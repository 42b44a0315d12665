"""Time farthest point sampling of full-resolution sweeps: the wide tier (131 073 .. 262 144 points per cloud, csrc/fps.cu
fps_wide_kernel) against the register tier at 131 072 points, with CUDA events after a warm-up.

    python tools/fps_large_time.py [--reps 5]

Prints one line per (N, B, npoint): ms per call and us per round, the plan that ran, and for the wide tier how many of
its clusters the device can hold at once (cudaOccupancyMaxActiveClusters, read back from the B200PC_DEBUG_PLAN lines).
Then the comparator a user has without this library: the reference's own farthest_point_sample (oracle/ref_torch.fps),
which keeps its state on the host and so runs on the CPU, per round at 133 312 points.  The clouds are the synthetic
HDL-64 sweeps of b200pc/synth.py (133 312 returns each), laid end to end and cropped."""
import argparse
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "point-cloud-interpolation-_b200"))
import numpy as np
import torch

from b200pc import ops, synth
from oracle import ref_torch


def sweeps(i):
    rng = np.random.default_rng(1000 + i)
    walls, boxes = synth._scene(rng)
    return (synth._scan(walls, boxes, (0.0, 0.0, 0.0), rng), synth._scan(walls, boxes, (1.2, 0.0, np.deg2rad(1.0)), rng))


def plan_lines(fn):
    """run fn once with B200PC_DEBUG_PLAN=1 and return what the library printed to stderr"""
    os.environ["B200PC_DEBUG_PLAN"] = "1"; ops.reload_tuning()
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            fn(); torch.cuda.synchronize()
        finally:
            os.dup2(saved, 2); os.close(saved)
        f.seek(0)
        text = f.read()
    del os.environ["B200PC_DEBUG_PLAN"]; ops.reload_tuning()
    return text


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    try:
        smi = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                      text=True).strip()
    except (OSError, subprocess.CalledProcessError) as e:
        smi = "nvidia-smi unavailable (%s)" % e
    print("device: %s | nvidia-smi: %s" % (torch.cuda.get_device_name(dev), smi), flush=True)

    clouds = [np.concatenate(sweeps(i)) for i in range(8)]          # 266 624 points each
    assert sweeps(0)[0].shape[0] == 133312
    host = np.ascontiguousarray(np.stack(clouds))
    for N in (131072, 133312, 196608, 262144):
        for B in (1, 8):
            x = torch.from_numpy(np.ascontiguousarray(host[:B, :N])).to(dev)
            st = torch.zeros(B, dtype=torch.long, device=dev)
            for npoint in (4096, 16384):
                plan = plan_lines(lambda: ops.fps(x, npoint, st))
                for _ in range(2):
                    ops.fps(x, npoint, st)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.reps):
                    ops.fps(x, npoint, st)
                e1.record(); torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / args.reps
                m = re.search(r"-> (cluster \d+, \d+ points/thread, exchange [\w-]+(?:, shared \d+ points/thread)?)", plan)
                occ = re.search(r"at most (\d+) clusters", plan)
                print("N=%6d B=%d npoint=%5d: %8.3f ms  %.3f us/round | %s | co-resident clusters: %s"
                      % (N, B, npoint, ms, ms * 1e3 / npoint, m.group(1) if m else "?", occ.group(1) if occ else "n/a (register tier)"),
                      flush=True)

    # the reference algorithm on the CPU (its state is allocated on the host), per round, a few rounds
    cpu = torch.from_numpy(host[:1, :133312].copy())
    npoint = 8
    ref_torch.fps(cpu, 2, torch.zeros(1, dtype=torch.long))
    t0 = time.perf_counter()
    ref_torch.fps(cpu, npoint, torch.zeros(1, dtype=torch.long))
    dt = time.perf_counter() - t0
    print("reference farthest_point_sample on the CPU, N=133312 B=1: %.3f ms/round (%d rounds timed, %d torch threads)"
          % (dt * 1e3 / npoint, npoint, torch.get_num_threads()), flush=True)


if __name__ == "__main__":
    main()
