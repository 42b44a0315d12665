"""Ragged batches: what the native lengths path costs against the two ways a user has without it.

usage: python tools/ragged_bench.py [--steps 20] [--out DIR]

Workloads (one JSON line each, after a line naming the card and its power limit):
  1. C2-shaped kNN: B = 8, padded 16384 x 16384, k = 16, form 0, lengths drawn (seeded) uniformly in [8192, 16384] on both
     sides.  (a) ops.knn_ragged; (b) the dense op on NaN-padded copies (a NaN ref is never selected, a NaN query row is
     empty) -- its valid rows are asserted equal to (a); (c) a loop of 8 dense calls on the exact slices.
  2. The same batch with every length full: (a) against the dense op, i.e. what the lengths path costs when unused.
  3. Chamfer, B = 8 at 16384 padded points (PointINet's frame size), ragged lengths: the ragged op against a per-item loop of
     the dense op, forward, and forward + backward.
Timing: CUDA events around each step, the 126 MB L2 overwritten before every step (a 256 MB memset outside the events),
mean over --steps after warm-up.  "pair_share" = sum_b len1[b] len2[b] / (B N S), the share of the dense pair work.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "point-cloud-interpolation-_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from b200pc import ops, synth  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return {"card": name, "power_limit": power or "unknown", "sms": torch.cuda.get_device_properties(0).multi_processor_count}


class Timer:
    def __init__(self, dev, steps, warmup=3):
        self.flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
        self.steps, self.warmup = steps, warmup

    def __call__(self, fn):
        for _ in range(self.warmup):
            fn()
        torch.cuda.synchronize()
        total = 0.0
        for _ in range(self.steps):
            self.flush.zero_()
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            total += e0.elapsed_time(e1)
        return round(total / self.steps, 4)


def nan_padded(a, lens):
    a = a.clone()
    for b, n in enumerate(lens.tolist()):
        a[b, n:] = float("nan")
    return a


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the lines to DIR/ragged_bench.jsonl")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ragged_bench: needs a CUDA device")
    dev = torch.device("cuda:0")
    tm = Timer(dev, args.steps)
    lines = [card()]
    B, N, S, k = 8, 16384, 16384, 16
    a, q = synth.batch_pairs(7, B, N)
    ref, qry = torch.from_numpy(a).to(dev), torch.from_numpy(q).to(dev)
    rng = np.random.default_rng(2024)
    rl = torch.from_numpy(rng.integers(8192, 16385, B)).to(dev)
    ql = torch.from_numpy(rng.integers(8192, 16385, B)).to(dev)
    share = float((rl.double() * ql.double()).sum() / (B * N * S))

    # 1. ragged kNN, three arms
    ia, da = ops.knn_ragged(ref, qry, k, 0, rl, ql, want_dist=True)
    rn, qn = nan_padded(ref, rl), nan_padded(qry, ql)
    ib, db = ops.knn_search(rn, qn, k, 0, want_dist=True)
    for b in range(B):
        s = int(ql[b])
        assert torch.equal(ia[b, :s], ib[b, :s]) and torch.equal(da[b, :s].view(torch.int32), db[b, :s].view(torch.int32)), b
    slices = [(ref[b:b + 1, :int(rl[b])].contiguous(), qry[b:b + 1, :int(ql[b])].contiguous()) for b in range(B)]
    lines.append({"workload": "knn_ragged B8 16384x16384 k16 form0", "pair_share": round(share, 4),
                  "a_ragged_ms": tm(lambda: ops.knn_ragged(ref, qry, k, 0, rl, ql)),
                  "b_dense_nan_padded_ms": tm(lambda: ops.knn_search(rn, qn, k, 0)),
                  "c_loop_of_8_dense_ms": tm(lambda: [ops.knn_search(r_, q_, k, 0) for r_, q_ in slices])})

    # 2. lengths all full
    full = torch.full((B,), N, dtype=torch.int64, device=dev)
    assert torch.equal(ops.knn_ragged(ref, qry, k, 0, full, full), ops.knn_search(ref, qry, k, 0))
    lines.append({"workload": "knn lengths all full B8 16384x16384 k16 form0",
                  "a_ragged_ms": tm(lambda: ops.knn_ragged(ref, qry, k, 0, full, full)),
                  "dense_ms": tm(lambda: ops.knn_search(ref, qry, k, 0))})

    # 3. Chamfer, ragged lengths
    x = ref.clone().requires_grad_(); y = qry.clone().requires_grad_()
    xs = [(x[b:b + 1, :int(rl[b])], y[b:b + 1, :int(ql[b])]) for b in range(B)]

    def ragged_fwd():
        with torch.no_grad():
            return ops.chamfer_reduce(ops.chamfer_ragged(x, y, rl, ql)[0], rl, ql, N, N, "mean", None)

    def loop_fwd():
        with torch.no_grad():
            return torch.stack([ops.chamfer(a_, b_)[0] for a_, b_ in xs])

    def ragged_fb():
        ops.chamfer_reduce(ops.chamfer_ragged(x, y, rl, ql)[0], rl, ql, N, N, "mean", "sum").backward()

    def loop_fb():
        torch.stack([ops.chamfer(a_, b_)[0] for a_, b_ in xs]).sum().backward()

    got, want = ragged_fwd(), loop_fwd()
    assert torch.allclose(got, want, rtol=1e-5), (got, want)
    lines.append({"workload": "chamfer ragged B8 16384 padded", "pair_share": round(share, 4),
                  "ragged_fwd_ms": tm(ragged_fwd), "loop_fwd_ms": tm(loop_fwd),
                  "ragged_fwd_bwd_ms": tm(ragged_fb), "loop_fwd_bwd_ms": tm(loop_fb)})
    for line in lines:
        print(json.dumps(line))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "ragged_bench.jsonl"), "w") as f:
            f.writelines(json.dumps(line) + "\n" for line in lines)


if __name__ == "__main__":
    main()
