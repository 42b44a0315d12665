#!/usr/bin/env python
"""bench.py -- headline measurement of the geometric hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--extras 0|1] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], "C2"): knn_point k=16, 16384 queries vs 16384 refs, batch 8,
on synthetic HDL-64-shaped frame pairs (b200pc.synth, seeds fixed by pair index).  One "step" is one
pass of knn_point over that batch.  Metric: kNN Gqueries/s, whole job over all ranks (weak scaling:
every rank owns its own 8 frame pairs, no data-path collective).

Printed JSON line (rank 0): value = device-resident throughput; e2e = the same call with HOST
(pinned) buffers, H2D + D2H inside the timed region; roofline = FP32 CUDA-core roofline of the
search kernel (8 FLOP per (query, ref) pair, SURVEY section 8d); cpu_baseline = the reference's torch
CPU algorithm (oracle/ref_torch.py) timed on this box's host cores on a bounded sample.
`--impl reference` times only that CPU path, on the same config, and prints the same line shape.
"""
import argparse
import contextlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "point-cloud-interpolation-_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

NPTS = 16384
BATCH = 8
K_NN = 16
FLOP_PER_PAIR = 8.0                       # SURVEY 8(d): the reference's own un-fused count
FP32_NOMINAL_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # 74.4: SMs x lanes x 2 x max SM clock
METRIC = "knn_point_gqueries_per_s"
UNIT = "Gqueries/s"
WORKLOAD = "C2: knn_point k=16, 16384 queries x 16384 refs, batch 8 per GPU, synthetic HDL-64 pairs"


def bench_config(world):
    """the `config` object, identical in the product arm and in the reference arm (the reference arm's bounded sample is
    described in its cpu_baseline.sample / note)"""
    return {"workload": WORKLOAD, "l2": "256 MB buffer rewritten before every timed step (L2 flush)",
            "parallelism": "batch-sharded, %d x 8 frame pairs, no data-path collective" % world}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--extras", type=int, default=1, help="also time the other kernels of the path (rank 0)")
    ap.add_argument("--ref-queries", type=int, default=0, help="(--impl reference) queries per step; 0 = automatic")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy, so that two builds can be "
                         "compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the timed CUDA path (--impl b200)")
    return args


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def reference_knn_fn():
    """-> (fn(ref [B,N,3], qry [B,S,3]) -> idx [B,S,k], kind).  kind "reference": the reference's OWN square_distance
    (Utils/Pointnet2Utils.py:20-41, imported unmodified from the staged checkout oracle/_ref or /root/reference) followed
    by the topk/permute expression of Group.forward (Utils/Layers.py:51-52); kind "port": oracle/ref_torch.py where no
    checkout is available."""
    from oracle import ref_loader, ref_torch
    if ref_loader.available():
        try:
            sqd = ref_loader.pointnet2_utils().square_distance

            def fn(ref, qry):
                dist = sqd(ref, qry)                                                                  # Utils/Layers.py:51
                return dist.topk(K_NN, dim=1, largest=False)[1].permute(0, 2, 1).contiguous()         # Utils/Layers.py:52
            return fn, "reference"
        except Exception as e:  # pragma: no cover
            print("real reference not importable (%r): timing the port" % (e,), file=sys.stderr)
    return (lambda ref, qry: ref_torch.knn_topk(K_NN, ref, qry)), "port"


def cpu_reference_knn(a, b, reps, queries=NPTS):
    """the reference's CPU path for the step on ONE frame pair (1/8 of the batch).
    returns (Gq/s, seconds per call, threads, kind)."""
    fn, kind = reference_knn_fn()
    torch.set_num_threads(os.cpu_count() or 1)
    ref = torch.from_numpy(a[:1]); qry = torch.from_numpy(b[:1, :queries])
    fn(ref[:, :2048], qry[:, :512])           # warm the thread pool
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn(ref, qry)
        ts.append(time.perf_counter() - t0)
    t = statistics.median(ts)
    return queries / t / 1e9, t, torch.get_num_threads(), kind


def run_reference(args, rank, world):
    """--impl reference: the reference's torch-CPU path on the host cores, rank 0 only."""
    if rank != 0:
        return
    from b200pc import synth
    a, b = synth.batch_pairs(0, 1, NPTS)
    # bounded sample per step: one pair of the batch of 8; shrink the query set for long runs
    queries = NPTS if args.steps + args.warmup <= 40 else 4096
    if args.ref_queries:
        queries = args.ref_queries
    fn, kind = reference_knn_fn()
    torch.set_num_threads(os.cpu_count() or 1)
    ref = torch.from_numpy(a); qry = torch.from_numpy(b[:, :queries])
    for _ in range(args.warmup):
        fn(ref, qry)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn(ref, qry)
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    val = queries / dt / 1e9
    sample = "1 of the 8 frame pairs per step: %d queries x %d refs, k=%d (%s: dense [N,S] matrix + topk(dim=1))" % (
        queries, NPTS, K_NN, "the reference's own torch-CPU code" if kind == "reference" else "torch-CPU port of the reference")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(max(1, int(os.environ.get("WORLD_SIZE", "1")))),
            "note": "reference arm: " + sample,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
                             "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def timed_steps(fn, steps, warmup, flush, stream_sync, barrier):
    """W warm-ups, then K steps each bracketed by CUDA events on the current stream, an L2 flush
    (outside the events) before every step; returns total seconds over the K steps."""
    for _ in range(warmup):
        flush(); fn()
    stream_sync(); barrier()
    evs = []
    for _ in range(steps):
        flush()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        evs.append((e0, e1))
    stream_sync(); barrier()
    return sum(e0.elapsed_time(e1) for e0, e1 in evs) / 1e3


def bind_to_gpu_numa(dev):
    """pin this process (and therefore its pinned host buffers, first-touched by it) to the CPUs local to the GPU's PCIe
    root: eight ranks reading back indices at once otherwise share whatever node the launcher started them on.
    Returns the cpulist string, or None where sysfs does not say."""
    try:
        pr = torch.cuda.get_device_properties(dev)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        path = "/sys/bus/pci/devices/%s/local_cpulist" % bdf
        txt = open(path).read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                lo, hi = part.split("-"); cpus.update(range(int(lo), int(hi) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return txt
    except Exception:
        pass
    return None


def e2e_bench(dev, a, b, steps, flush, barrier, dist):
    """the C2 step through the host-buffer API (pinned host tensors in, pinned host indices out), three ways:
      serial   - hostio.knn_point_host per step, int64 indices, every step ends before the next starts (round 1's number)
      pipelined- hostio.KnnHostPipeline, int64: step i's read-back overlaps step i+1's upload + search (two streams);
                 every step still uploads its inputs and reads its result back; timed over the whole loop
      int32    - the same pipeline with the 32-bit index variant of the C ABI (half the read-back bytes)
    -> seconds per step (max over ranks) for each"""
    from b200pc import hostio
    h_ref = torch.from_numpy(a).pin_memory(); h_qry = torch.from_numpy(b).pin_memory()
    outs64 = [torch.empty(BATCH, NPTS, K_NN, dtype=torch.int64).pin_memory() for _ in range(2)]
    outs32 = [torch.empty(BATCH, NPTS, K_NN, dtype=torch.int32).pin_memory() for _ in range(2)]
    res = {}

    def reduce_max(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    secs = timed_steps(lambda: hostio.knn_point_host(K_NN, h_ref, h_qry, out=outs64[0], device=dev), steps, 3, flush,
                       torch.cuda.synchronize, barrier)
    res["serial"] = reduce_max(secs / steps)
    for name, outs, dt in (("pipelined", outs64, torch.int64), ("int32", outs32, torch.int32)):
        pipe = hostio.KnnHostPipeline(K_NN, device=dev, index_dtype=dt)
        for i in range(3):
            pipe.submit(h_ref, h_qry, outs[i % 2])
        pipe.finish(); torch.cuda.synchronize(); barrier()
        flush()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            pipe.submit(h_ref, h_qry, outs[i % 2])
        pipe.finish()
        e1.record(); torch.cuda.synchronize(); barrier()
        res[name] = reduce_max(e0.elapsed_time(e1) / 1e3 / steps)
    return res, int(h_ref.numel() * 4 + h_qry.numel() * 4), int(outs64[0].numel() * 8)


def multi_gpu_lines(dev, rank, world, dist, flush, barrier):
    """The two configurations of BASELINE.json that have an exchange step, timed on `world` ranks (max over ranks):
      C5  PolyPCI.rebuild (PolyPCI/Models/Models_V1.py:102-114): 4 frames x (65536 queries x 65536 refs, K=1, return_nn),
          queries sharded over the ranks, refs replicated, (index, neighbour) records all-gathered -- strong scaling.
          Reported: search ms (no exchange), NCCL all_gather ms, and the peer-store variant where the producing kernel
          writes its slab into every rank's symmetric buffer (no collective kernel).
      C4  FlowNet3D training step (PointINet20230424/train_sceneflow.py:132-185): global batch 32 x 8192 points split over
          the ranks, BatchNorm in train mode, Chamfer loss, backward, DDP gradient all-reduce, Adam -- strong scaling.
    Also re-runs the query-sharded kNN / ball query of tests/test_gpu_dist.py and compares with the unsharded result."""
    from b200pc import dist as bdist, ops, pointnet2_utils as P, synth
    out = {"world": world}

    def tmax(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, n=10, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize(); barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize(); barrier()
        return tmax(e0.elapsed_time(e1) / 1e3 / n)

    # ---- C5 ----
    F, NP = 4, 65536
    fr = [synth.frame_pair(200 + i, NP) for i in range(F)]
    refs = torch.from_numpy(np.stack([p[0] for p in fr])).to(dev)         # [4,65536,3] replicated on every rank
    qry = torch.from_numpy(np.stack([p[1] for p in fr])).to(dev)
    per = NP // world
    mine = qry[:, rank * per:(rank + 1) * per].contiguous()
    c5 = {"workload": "C5: PolyPCI.rebuild, 4 frames x 65536 queries x 65536 refs, K=1 + neighbour coordinates, query-sharded",
          "scaling": "strong", "queries_per_rank": F * per, "record_bytes": 16,
          "allgather_bytes_per_rank": F * per * 16, "allgather_bytes_total": F * NP * 16}
    c5["search_ms"] = timed(lambda: ops.rebuild_pack(refs, mine, 0, ())) * 1e3
    if world > 1:
        c5["nccl_ms"] = timed(lambda: bdist.rebuild_sharded(refs, qry, mode="nccl")) * 1e3
        c5["nccl_allgather_share_ms"] = c5["nccl_ms"] - c5["search_ms"]
        full = ops.rebuild_pack(refs, qry, 0, ()) if rank == 0 else None
        got = bdist.rebuild_sharded(refs, qry, mode="nccl")
        ok = torch.equal(got.view(torch.int32), full.view(torch.int32)) if rank == 0 else True
        try:
            slab = bdist.PeerSlab(NP, F, dev)
            c5["peer_ms"] = timed(lambda: bdist.rebuild_sharded(refs, qry, mode="peer", slab=slab)) * 1e3
            c5["peer_exchange_share_ms"] = c5["peer_ms"] - c5["search_ms"]
            gotp = bdist.rebuild_sharded(refs, qry, mode="peer", slab=slab)
            okp = torch.equal(gotp.view(torch.int32), full.view(torch.int32)) if rank == 0 else True
            c5["peer_identical_to_unsharded"] = bool(okp)
        except Exception as e:
            c5["peer_unavailable"] = repr(e)[:300]
        c5["nccl_identical_to_unsharded"] = bool(ok)
        c5["value_queries_per_s"] = F * NP / (min(c5["nccl_ms"], c5.get("peer_ms", 1e9)) / 1e3)
    else:
        c5["value_queries_per_s"] = F * NP / (c5["search_ms"] / 1e3)
    out["c5_query_sharded"] = c5
    del refs, qry, mine

    # ---- tests/test_gpu_dist.py inside the bench: sharded == unsharded, bit for bit ----
    if world > 1:
        a, b = synth.batch_pairs(4, 1, 8192)
        r = torch.from_numpy(a).to(dev); q = torch.from_numpy(b[:, :5001].copy()).to(dev)      # ragged shards
        idx = bdist.query_sharded(lambda s: P.knn_point(16, r, s), q)
        ball = bdist.query_sharded(lambda s: P.query_ball_point(1.0, 32, r, s), q)
        ok = torch.equal(idx, P.knn_point(16, r, q)) and torch.equal(ball, P.query_ball_point(1.0, 32, r, q))
        flag = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        out["query_sharded_check"] = "ok: sharded kNN / ball query identical to the unsharded call on every rank" if int(flag.item()) == 1 else "MISMATCH"

    # ---- C4 ----
    try:
        from b200pc import pointinet, pytorch3d_shim as S3
        GB, NP4 = 32, 8192
        lb = GB // world
        pa, pb = synth.batch_pairs(300 + rank * lb, lb, NP4)
        p1 = torch.from_numpy(pa).to(dev).transpose(1, 2).contiguous(); p2 = torch.from_numpy(pb).to(dev).transpose(1, 2).contiguous()
        f0 = torch.zeros(lb, 3, NP4, device=dev)
        torch.manual_seed(0)
        net = pointinet.FlowNet3D().train().to(dev)
        model = net
        if world > 1:
            model = torch.nn.parallel.DistributedDataParallel(net, device_ids=[dev.index])
        opt = torch.optim.Adam(net.parameters(), lr=1e-3)

        def step(sync=True):
            opt.zero_grad(set_to_none=True)
            ctx = model.no_sync() if (world > 1 and not sync) else contextlib.nullcontext()
            with ctx:
                flow = model(p1, p2, f0, f0)
                loss, _ = S3.chamfer_distance((p1 + flow).permute(0, 2, 1), p2.permute(0, 2, 1))
                loss.backward()
            opt.step()

        c4 = {"workload": "C4: FlowNet3D train step, global batch 32 x 8192 points, BatchNorm train mode, Chamfer loss, Adam",
              "scaling": "strong", "global_batch": GB, "batch_per_rank": lb}
        c4["step_ms"] = timed(lambda: step(True), n=5, warm=2) * 1e3
        if world > 1:
            c4["step_ms_without_allreduce"] = timed(lambda: step(False), n=5, warm=1) * 1e3
            c4["allreduce_share_ms"] = c4["step_ms"] - c4["step_ms_without_allreduce"]
            c4["gradient_bytes"] = int(sum(p.numel() for p in net.parameters() if p.requires_grad) * 4)
        c4["value_pairs_per_s"] = GB / (c4["step_ms"] / 1e3)
        out["c4_ddp"] = c4
    except Exception as e:  # pragma: no cover
        out["c4_ddp"] = {"error": repr(e)[:300]}
    return out


def extras(dev, a, b, flush):
    """other kernels of the path at their BASELINE configs (C2 ball query, C3 FPS / gather /
    three_interpolate, Chamfer), device-resident, 10 timed calls each."""
    from b200pc import ops, pointnet2_utils as P
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    out = {"hbm_peak_gbs": hbm, "hbm_peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}

    def t(fn, n=10):
        s = timed_steps(fn, n, 3, flush, torch.cuda.synchronize, lambda: None)
        return s / n

    def t_train(fn, n=10):
        """kernel time of a 10-100 us op without the per-launch event / launch latency (~5 us, a third of an 18 us
        kernel): a CUDA graph of n x [L2 flush, op] is replayed between two events, the same graph WITHOUT the op is
        timed the same way, and the difference is divided by n.  Every op still starts with a flushed L2."""
        def build(with_op):
            g = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                flush(); fn()
                with torch.cuda.graph(g, stream=side):
                    for _ in range(n):
                        flush()
                        if with_op:
                            keep = fn()      # noqa: F841  (outputs live in the graph's pool)
            torch.cuda.current_stream().wait_stream(side)
            return g

        def run(g):
            for _ in range(2):
                g.replay()
            torch.cuda.synchronize()
            best = None
            for _ in range(3):
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                best = ms if best is None or ms < best else best
            return best / 1e3
        return max(run(build(True)) - run(build(False)), 1e-9) / n

    ref = torch.from_numpy(a).to(dev); qry = torch.from_numpy(b).to(dev)
    pairs = BATCH * NPTS * NPTS
    s = t(lambda: P.query_ball_point(1.0, 32, ref, qry))
    out["ball_query_c2"] = {"ms": s * 1e3, "gqueries_per_s": BATCH * NPTS / s / 1e9,
                            "effective_tflops": pairs * FLOP_PER_PAIR / s / 1e12}
    s = t(lambda: ops.knn_search(ref, qry, 16, ops.FORM_DIRECT, want_dist=True))
    out["knn_points_direct_k16_c1x8"] = {"ms": s * 1e3, "tflops": pairs * FLOP_PER_PAIR / s / 1e12}

    # C3: FPS 16384 -> 4096, gather C=128, three_interpolate C=128, batch 16
    B3 = 16
    a3 = np.concatenate([a, b], 0)[:B3]
    xyz = torch.from_numpy(a3).to(dev)
    start = torch.arange(B3, device=dev, dtype=torch.long) * 7
    s = t(lambda: ops.fps(xyz, 4096, start), n=3)
    out["fps_c3"] = {"ms": s * 1e3, "us_per_round": s * 1e6 / 4096, "clouds": B3}
    s1 = t(lambda: ops.fps(xyz[:1], 1024, start[:1]), n=3)
    out["fps_16384_to_1024_b1"] = {"ms": s1 * 1e3, "us_per_round": s1 * 1e6 / 1024}
    fidx = ops.fps(xyz, 4096, start)
    feats = torch.randn(B3, NPTS, 128, device=dev)
    s = t(lambda: P.index_points(feats, fidx))
    sk = t_train(lambda: P.index_points(feats, fidx))
    gbytes = B3 * 4096 * (128 * 4 * 2 + 8)
    how = ("hbm_frac: kernel time from a CUDA graph of 10 x [L2 flush, op] minus the same graph without the op (ncu gpu__time_duration "
           "of the same launch agrees, profiles/r02_ncu_rowmovers_shipped.txt); hbm_frac_single_launch: one op between two CUDA events, "
           "which adds ~5 us of launch / event latency")
    out["index_points_c3"] = {"ms": sk * 1e3, "gb_per_s": gbytes / sk / 1e9, "hbm_frac": gbytes / sk / 1e9 / hbm,
                              "ms_single_launch": s * 1e3, "hbm_frac_single_launch": gbytes / s / 1e9 / hbm,
                              "algorithmic_bytes": gbytes, "timing": how}
    known = P.index_points(xyz, fidx)
    sfeat = P.index_points(feats, fidx)
    s = t(lambda: P.three_nn_weights(xyz, known))
    out["three_nn_c3"] = {"ms": s * 1e3, "tflops": B3 * NPTS * 4096 * FLOP_PER_PAIR / s / 1e12}
    _, i3, w3 = P.three_nn_weights(xyz, known)
    s = t(lambda: P.three_interpolate(sfeat, i3, w3))
    sk = t_train(lambda: P.three_interpolate(sfeat, i3, w3))
    ibytes = B3 * NPTS * 128 * 4 + B3 * 4096 * 128 * 4 + B3 * NPTS * (24 + 12)
    out["three_interpolate_c3"] = {"ms": sk * 1e3, "gb_per_s": ibytes / sk / 1e9, "hbm_frac": ibytes / sk / 1e9 / hbm,
                                   "ms_single_launch": s * 1e3, "hbm_frac_single_launch": ibytes / s / 1e9 / hbm,
                                   "algorithmic_bytes": ibytes}
    sf = t_train(lambda: P.feature_propagation(xyz, known, sfeat))
    out["feature_propagation_c3"] = {"ms": sf * 1e3, "note": "three-NN search -> weights -> mix behind ONE C call (b200pc_feature_propagation)"}
    # fused grouping (SURVEY 8f rank 1) on the C3 clouds: 4096 centres x 16 neighbours, D=64 feature channels
    gfeat = feats[:, :, :64].contiguous()
    gidx = P.knn_point(16, xyz, known)
    s = t(lambda: P.group_points(xyz, known, gfeat, gidx))
    sk = t_train(lambda: P.group_points(xyz, known, gfeat, gidx))

    def unfused():          # the reference's five ops (Utils/Layers.py:57-66) on this repo's own gather kernels
        rel = P.index_points(xyz, gidx) - known.view(B3, 4096, 1, 3)
        return torch.cat([rel, P.index_points(gfeat, gidx)], dim=-1).permute(0, 3, 2, 1).contiguous()
    su = t(unfused)
    gb = B3 * 4096 * 16 * (8 + 4 * 67) + B3 * NPTS * 4 * 67 + B3 * 4096 * 12     # idx + output + each table row once + centres
    out["group_points_c3"] = {"ms": sk * 1e3, "gb_per_s": gb / sk / 1e9, "hbm_frac": gb / sk / 1e9 / hbm, "algorithmic_bytes": gb,
                              "ms_single_launch": s * 1e3, "hbm_frac_single_launch": gb / s / 1e9 / hbm,
                              "unfused_ms": su * 1e3, "shape": "B=16 N=16384 S=4096 K=16 D=64 -> [16,67,16,4096]"}
    # PolyPCI polynomial fit (SURVEY 8f rank 4) at the C5 size: 65536 points, field 2 (5 frames), T=[0,-1,1,-2,2], t=0.5, degree 2
    try:
        from b200pc import polypci
        fr = [torch.randn(1, 3, 65536, device=dev) * 30 for _ in range(5)]
        Tl = [[0.0, -1.0, 1.0, -2.0, 2.0]]
        tq = torch.tensor([0.5])
        s = t(lambda: polypci.fit_and_predict(fr, Tl, tq, 2))
        pb = 6 * 4 * 3 * 65536
        out["poly_fit_predict_c5"] = {"ms": s * 1e3, "gb_per_s": pb / s / 1e9, "algorithmic_bytes": pb,
                                      "note": "includes the host-side float64 weight solve (np.polyfit on a 5x5 identity)"}
        from oracle import ref_polyfit                                    # CPU baseline leg: the reference's host path
        host = [f.cpu().numpy() for f in fr]
        t0 = time.perf_counter()
        back = torch.from_numpy(ref_polyfit.forward_tail([f.cpu().numpy() for f in fr], Tl, tq.numpy(), 2)).to(dev)
        torch.cuda.synchronize()
        out["poly_fit_predict_c5"]["reference_host_path_ms"] = (time.perf_counter() - t0) * 1e3   # D2H + np.polyfit + H2D
        del host, back
    except Exception as e:      # never let a side measurement break the headline line
        out["poly_fit_predict_c5"] = {"error": repr(e)}
    # Chamfer, C4 per-GPU share: 4 pairs x 8192 points
    x = ref[:4, :8192].contiguous(); y = qry[:4, :8192].contiguous()
    s = t(lambda: ops.chamfer(x, y))
    out["chamfer_c4_share"] = {"ms": s * 1e3, "tflops": 2 * 4 * 8192 * 8192 * FLOP_PER_PAIR / s / 1e12}
    # C4 per-GPU share: FlowNet3D training step (train_sceneflow.py:132-185 in the reference), 4 pairs x 8192 points,
    # BatchNorm in train mode, loss = chamfer(p1 + flow, p2), backward, Adam step
    try:
        from b200pc import pointinet, pytorch3d_shim as S3
        torch.manual_seed(0)
        net = pointinet.FlowNet3D().train().to(dev)
        opt = torch.optim.Adam(net.parameters(), lr=1e-3)
        p1 = ref[:4, :8192].transpose(1, 2).contiguous(); p2 = qry[:4, :8192].transpose(1, 2).contiguous()
        f0 = torch.zeros(4, 3, 8192, device=dev)

        def train_step():
            opt.zero_grad(set_to_none=True)
            flow = net(p1, p2, f0, f0)
            loss, _ = S3.chamfer_distance((p1 + flow).permute(0, 2, 1), p2.permute(0, 2, 1))
            loss.backward()
            opt.step()

        s = t(train_step, n=5)
        out["flownet3d_train_step_c4_share"] = {"ms": s * 1e3, "pairs_per_s": 4 / s, "batch": 4, "points": 8192}
    except Exception as e:  # pragma: no cover
        out["flownet3d_train_step_c4_share"] = {"error": repr(e)}
    return out


def pointinet_inputs(pair, n, dev=None, pinned=False):
    """one synthetic frame pair as PointINet inputs: points [1,4,n] (xyz + intensity), zero features, t=0.5"""
    from b200pc import synth
    a, b = synth.frame_pair(pair, n)
    g = torch.Generator().manual_seed(pair)
    mk = lambda f: torch.cat([torch.from_numpy(f).t(), torch.rand(1, n, generator=g)], 0).unsqueeze(0).contiguous()
    ts = [mk(a), mk(b), torch.zeros(1, 3, n), torch.zeros(1, 3, n), torch.tensor([0.5])]
    if pinned:
        ts = [x.pin_memory() for x in ts]
    if dev is not None:
        ts = [x.to(dev) for x in ts]
    return ts


def pointinet_bench(dev, rank, steps, flush, barrier, dist):
    """BASELINE metric (i): PointINet interpolated frames/s at 16384 points, batch 1, t=0.5, random
    weights (the reference ships none).  Every rank interpolates its own frame pairs.  Three variants,
    seconds per frame as the max over ranks:
      eager   - the module called like the reference calls it (one Python dispatch per op), inputs resident
      graph   - the same forward captured once as a CUDA graph (b200pc.pointinet.GraphedPointINet: RNG tape
                refilled on the CPU generator each frame, BatchNorm folded), inputs resident
      graph_e2e - graph variant fed from pinned HOST buffers, fused frame copied back to the host"""
    from b200pc import pointinet
    torch.manual_seed(0)
    net = pointinet.PointINet().eval().to(dev)
    dev_in = pointinet_inputs(100 + rank, NPTS, dev=dev)
    host_in = pointinet_inputs(100 + rank, NPTS, pinned=True)
    host_out = torch.empty(1, 4, NPTS).pin_memory()
    graphed = pointinet.GraphedPointINet(state_dict=net.state_dict(), batch=1, npoints=NPTS, extra=1, t=0.5, device=dev)
    graphed.capture(*dev_in[:4])

    def eager():
        with torch.no_grad():
            net(*dev_in)

    def graph():
        graphed(*dev_in[:4])

    def graph_e2e():
        host_out.copy_(graphed(*host_in[:4]), non_blocking=True)

    out = {}
    for name, fn in (("eager", eager), ("graph", graph), ("graph_e2e", graph_e2e)):
        torch.manual_seed(3000 + rank)
        secs = timed_steps(fn, steps, 3, flush, torch.cuda.synchronize, barrier)
        tm = torch.tensor([secs / steps], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        out[name] = float(tm.item())
    # the UNMODIFIED upstream PointINet (PointINet20230424/models/models.py:79-125, staged under oracle/_ref by
    # oracle/make_ref.py) on the CUDA ops through b200pc.dropin: eager, like the reference's own test.py calls it
    ref_dir = os.path.join(ROOT, "oracle", "_ref", "PointINet20230424")
    if not os.path.isdir(ref_dir):
        ref_dir = "/root/reference/PointINet20230424"
    if os.path.isdir(os.path.join(ref_dir, "models")):
        from b200pc import dropin
        try:
            up = dropin.import_reference(ref_dir, "models.models")
            torch.manual_seed(0)
            rnet = up.PointINet(freeze=1).eval().to(dev)

            def real_eager():
                with torch.no_grad():
                    rnet(*dev_in)

            torch.manual_seed(3000 + rank)
            secs = timed_steps(real_eager, steps, 3, flush, torch.cuda.synchronize, barrier)
            tm = torch.tensor([secs / steps], device=dev, dtype=torch.float64)
            if dist is not None:
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            out["real_dropin_eager"] = float(tm.item())
            del rnet
        except Exception as e:  # pragma: no cover
            print("real-reference drop-in measurement failed: %r" % (e,), file=sys.stderr)
        finally:
            dropin.uninstall()
    if dist is None:
        # throughput mode, one GPU only: 8 frame pairs per replay (FPS runs 8 clusters side by side, PointsFusion's
        # per-item loop collapses into batched searches, SURVEY 8f rank 2).  Not the C1 configuration (batch 1).
        try:
            del graphed
            B8 = 8
            ins8 = [torch.cat(x, 0) for x in zip(*[pointinet_inputs(100 + i, NPTS, dev=dev)[:4] for i in range(B8)])]
            g8 = pointinet.GraphedPointINet(state_dict=net.state_dict(), batch=B8, npoints=NPTS, extra=1, t=0.5, device=dev)
            g8.capture(*ins8)
            torch.manual_seed(3000)
            secs = timed_steps(lambda: g8(*ins8), 5, 3, flush, torch.cuda.synchronize, barrier)
            out["graph_batch8_per_frame"] = secs / 5 / B8
        except Exception as e:  # pragma: no cover
            print("pointinet batch-8 measurement failed: %r" % (e,), file=sys.stderr)
    return out


def pointinet_cpu_baseline():
    """one PointINet forward with the reference's torch-CPU primitives (oracle.cpu_backend), all host threads"""
    from b200pc import pointinet
    from oracle import cpu_backend
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    net = pointinet.PointINet(backend=cpu_backend.make()).eval()
    ins = pointinet_inputs(100, NPTS)
    torch.manual_seed(3000)
    t0 = time.perf_counter()
    with torch.no_grad():
        net(*ins)
    return time.perf_counter() - t0, torch.get_num_threads()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    from b200pc import ops, pointnet2_utils as P, synth, _lib
    _lib.load()                                     # fail loudly if the native library is missing
    assert torch.cuda.is_available(), "bench.py needs a CUDA device: the hot path has no CPU fallback"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()

    numa = bind_to_gpu_numa(dev) if world > 1 else None       # before any pinned buffer is allocated
    # every rank owns its own 8 frame pairs (weak scaling, batch sharding: no exchange in the path)
    a, b = synth.batch_pairs(rank * BATCH, BATCH, NPTS)
    ref = torch.from_numpy(a).to(dev); qry = torch.from_numpy(b).to(dev)
    flush_buf = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MB > 126 MB L2

    def flush():
        flush_buf.zero_()

    # ---- device-resident value --------------------------------------------------------------
    try:
        gpu_id = "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        gpu_id = str(local)
    sampler = ClockSampler(gpu_id)
    if rank == 0:
        sampler.start()
    ops.launch_count = 0
    last = []

    def step():
        last[:] = [P.knn_point(K_NN, ref, qry)]
    secs = timed_steps(step, args.steps, args.warmup, flush, torch.cuda.synchronize, barrier)
    abi_calls = ops.launch_count
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # [BATCH, NPTS, K_NN] neighbour indices of rank 0's frame pairs: 8 MB in float32, exact since they are < 2^24
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "knn_point_idx.npy"), last[0].cpu().numpy().astype(np.float32))
    del last
    # sustained rate: the same call back to back for >= 2 s (no flush in between: the kernel reads 3 MB, it is not
    # memory bound), clocks sampled over that window
    sustained = None
    if args.extras:
        n_sus = int(max(200, min(6000, 2.0 / max(secs / args.steps, 1e-4))))
        sampler2 = ClockSampler(gpu_id)
        if rank == 0:
            sampler2.start()
        torch.cuda.synchronize(); barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_sus):
            P.knn_point(K_NN, ref, qry)
        e1.record(); torch.cuda.synchronize(); barrier()
        sus = torch.tensor([e0.elapsed_time(e1) / 1e3 / n_sus], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(sus, op=dist.ReduceOp.MAX)
        sustained = {"ms_per_step": float(sus.item()) * 1e3, "steps": n_sus, "value": BATCH * NPTS * world / float(sus.item()) / 1e9,
                     "clocks": sampler2.stop() if rank == 0 else None}
    tmax = torch.tensor([secs], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    secs_max = float(tmax.item())
    queries_per_step = BATCH * NPTS * world
    value = queries_per_step * args.steps / secs_max / 1e9

    # ---- end to end: pinned host inputs -> H2D -> knn_point -> D2H of the indices, every step ---
    e2e_steps = max(3, min(args.steps, 50))
    e2e_res, h2d_bytes, d2h_bytes = e2e_bench(dev, a, b, e2e_steps, flush, barrier, dist)
    e2e_value = queries_per_step / e2e_res["int32"] / 1e9

    # ---- the configurations with an exchange step (C5 all-gather, C4 DDP) on these `world` ranks ----
    multi = None
    if args.extras:
        try:
            multi = multi_gpu_lines(dev, rank, world, dist, flush, barrier)
        except Exception as e:  # pragma: no cover
            multi = {"error": repr(e)[:300]}

    # ---- metric (i): PointINet frames/s, every rank on its own frame pairs ----------------------
    pn = None
    if args.extras:
        try:
            pn = pointinet_bench(dev, rank, max(3, min(args.steps, 20)), flush, barrier, dist)
        except Exception as e:  # pragma: no cover
            if rank == 0:
                print("pointinet bench failed: %r" % (e,), file=sys.stderr)

    if rank != 0:
        if dist is not None:
            dist.barrier(); dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (search_kernel): FP32 CUDA-core pipe -----------------
    per_launch_s = secs / args.steps                       # the whole knn_point call: grid / sort kernels (~50 us) + search kernel, this rank
    pairs = BATCH * NPTS * NPTS
    achieved = pairs * FLOP_PER_PAIR / per_launch_s / 1e12
    try:
        fma_tf, fma_ms = ops.fma_peak(1 << 15)
    except Exception as e:  # pragma: no cover
        fma_tf, fma_ms = None, None
    peak = fma_tf if fma_tf else FP32_NOMINAL_TFLOPS
    roofline = {"bound": "fp32_cuda_core", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                # dram__bytes_read.sum + dram__bytes_write.sum of search_kernel from one `ncu --set full` capture of this very
                # call (profiles/r02_ncu_knn.txt: 5.28 MB read = the packed refs, sorted queries and thresholds once, 14 KB written:
                # the 16.8 MB of indices stay in L2 until evicted); a counter, so a constant from the committed capture, not measured live
                "traffic": 5290496, "traffic_source": "profiles/r02_ncu_knn.txt (ncu --set full, same shape)",
                "peak_source": "b200pc_fma_peak FFMA2 micro-kernel measured in this run (MEASURED_PEAKS.json has no FP32 entry)"
                if fma_tf else "nominal",
                "peak_nominal": FP32_NOMINAL_TFLOPS, "frac_nominal": achieved / FP32_NOMINAL_TFLOPS,
                "algorithmic": "8 FLOP per (query, ref) pair x %d pairs per launch" % pairs,
                "note": "K=3 contraction on FP32 CUDA cores (tensor cores would break the rounding parity); the "
                        "contract's enum is hbm|tensor, this kernel is neither: ncu shows it bound by instruction issue (lane "
                        "filter 49 %, lock-step heap drain 29 % of 359 M warp instructions, profiles/r02_notes.md), DRAM "
                        "traffic is 5.3 MB against 17.2 GFLOP.  `achieved` divides by the whole call (5 grid / sort kernels "
                        "+ the search kernel), not by the search kernel alone"}

    # ---- CPU baseline beside it (bounded sample: one of the 8 pairs) --------------------------
    cval, csec, cthreads, ckind = cpu_reference_knn(a, b, reps=3)
    cpu_baseline = {"value": cval, "unit": UNIT, "cores": cthreads, "kind": ckind,
                    "sample": "1 of the 8 frame pairs (16384 q x 16384 refs, k=16), median of 3; %.2f s per call" % csec}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": secs_max / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": bench_config(world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes // 2,
                    "steps": e2e_steps,
                    "api": "b200pc.hostio.KnnHostPipeline(index_dtype=torch.int32): pinned host clouds in, pinned host indices out, every "
                           "step uploads its inputs and reads its result back; step i's read-back overlaps step i+1's upload and search; "
                           "32-bit indices (N < 2^31: same values as the reference's int64, half the PCIe bytes)",
                    "int64_value": queries_per_step / e2e_res["pipelined"] / 1e9, "int64_d2h_bytes_per_step": d2h_bytes,
                    "serial_int64_value": queries_per_step / e2e_res["serial"] / 1e9,
                    "numa_cpulist": numa},
            # per knn_point call at C2 (no ref split): grid_bbox, grid_count, grid_pyramid, grid_scan, grid_scatter (which also writes the
            # starting thresholds) and search_kernel (+ one memset node for the grid counters); timed steps only
            "gpu_launches": int(args.steps * 6), "abi_calls_incl_warmup": int(abi_calls),
            "roofline": roofline, "cpu_baseline": cpu_baseline}
    if pn:
        line["pointinet"] = {"metric": "pointinet_interp_frames_per_s", "workload": "C1: PointINet forward, 16384 points, batch 1 per GPU, t=0.5, random weights",
                             "value": world / pn["graph"], "e2e_value": world / pn["graph_e2e"], "eager_value": world / pn["eager"], "unit": "frames/s",
                             "ms_per_frame": pn["graph"] * 1e3, "ms_per_frame_e2e": pn["graph_e2e"] * 1e3, "ms_per_frame_eager": pn["eager"] * 1e3,
                             "note": "value/e2e_value: forward captured as one CUDA graph (RNG tape, folded BatchNorm); eager_value: per-op dispatch like the reference",
                             "paper_rtx2060_frames_per_s": 4.9}
        if "real_dropin_eager" in pn:
            line["pointinet"]["real_dropin_eager_value"] = world / pn["real_dropin_eager"]
            line["pointinet"]["ms_per_frame_real_dropin_eager"] = pn["real_dropin_eager"] * 1e3
            line["pointinet"]["real_dropin_note"] = ("the reference's own PointINet20230424/models/models.py, unmodified, on the CUDA ops via "
                                                     "b200pc.dropin.install() (eager, per-op dispatch through torch.ops.b200pc.*)")
        if "graph_batch8_per_frame" in pn:
            line["pointinet"]["batch8_frames_per_s"] = 1.0 / pn["graph_batch8_per_frame"]
            line["pointinet"]["batch8_note"] = "throughput mode, NOT the C1 configuration: 8 frame pairs per graph replay on one GPU"
        if world == 1:
            try:
                csec, cthr = pointinet_cpu_baseline()
                line["pointinet"]["cpu_baseline"] = {"value": 1.0 / csec, "unit": "frames/s", "cores": cthr, "kind": "port",
                                                     "sample": "one forward, %.1f s" % csec}
            except Exception as e:  # pragma: no cover
                line["pointinet"]["cpu_baseline"] = {"error": repr(e)}
    if sustained:
        line["sustained"] = sustained
    if multi:
        line["extra_multi"] = multi
    if args.extras and world == 1:
        try:
            line["extra"] = extras(dev, a, b, flush)
        except Exception as e:  # pragma: no cover
            line["extra"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    main()
