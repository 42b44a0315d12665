"""randomised parity fuzz of the neighbour searches against the strict oracle (test infrastructure; GPU needed).
usage: python tools/fuzz_search.py [cases] [seed]"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "point-cloud-interpolation-_b200")); sys.path.insert(0, os.path.join(ROOT, "tests"))
import collections
import numpy as np
import torch
from b200pc import ops, pointnet2_utils as P
import b200pc.ops as _b200pc_ops; _b200pc_ops.TUNING_AUTORELOAD = True   # this probe flips B200PC_* knobs between calls (the library caches them)
from oracle import strict
import prune_geometry as PG


def run(cases, seed, dev="cuda:0"):
  rng = np.random.default_rng(seed)
  dev = torch.device(dev)
  bad = 0
  modes = collections.Counter()
  old = os.environ.get("B200PC_SMALL_PATH")
  for c in range(cases):
      B = int(rng.integers(1, 4)); N = int(rng.integers(1, int(os.environ.get("FUZZ_NMAX", "3000")))); S = int(rng.integers(1, int(os.environ.get("FUZZ_SMAX", "1500"))))
      scale = float(10.0 ** rng.uniform(-2, 2.5)); off = rng.normal(size=3) * scale * float(rng.choice([0, 0, 1, 20]))
      ref = (rng.normal(size=(B, N, 3)) * scale + off).astype(np.float32)
      qry = (rng.normal(size=(B, S, 3)) * scale + off).astype(np.float32)
      if rng.random() < 0.3:                                       # duplicates and exact ties
          ref = np.round(ref / (scale / 4)).astype(np.float32) * np.float32(scale / 4)
          qry = np.round(qry / (scale / 4)).astype(np.float32) * np.float32(scale / 4)
      if rng.random() < 0.3 and S <= N:
          qry = ref[:, :S].copy()                                  # queries are refs
      if rng.random() < 0.3:                                       # clustered cloud with a few far outliers: empty cells, wide boxes
          centres = rng.normal(size=(B, 6, 3)) * scale * 5
          ref = (centres[:, rng.integers(0, 6, N)][np.arange(B), :, :] if False else np.stack([centres[b][rng.integers(0, 6, N)] for b in range(B)]))
          ref = (ref + rng.normal(size=(B, N, 3)) * scale * 0.05).astype(np.float32)
          ref[:, :: max(1, N // 7)] *= np.float32(30.0)
          qry = (np.stack([centres[b][rng.integers(0, 6, S)] for b in range(B)]) + rng.normal(size=(B, S, 3)) * scale * 0.2).astype(np.float32)
      if rng.random() < 0.3:                                       # the pruned search's adversarial families, one per item
          ref, qry = PG.batch([str(f) for f in rng.choice(PG.FAMILIES, B)], int(rng.integers(0, 1 << 30)), N, S)
          sc = np.float32(2.0 ** int(rng.integers(-8, 9))); ref *= sc; qry *= sc               # a power of two keeps the ties
      os.environ["B200PC_SMALL_PATH"] = str(int(rng.integers(0, 2)))
      # the occupancy-grid variants of the top-k search (search.cu section 1b), forced on shapes the default would run blind
      # and the pruned search (section 3b, GRID=4), sometimes at a forced warp count
      grid = str(rng.choice(["", "0", "2", "3", "3", "4", "4", "4"]))
      for kk in ("B200PC_GRID", "B200PC_SEED", "B200PC_INTERLEAVE", "B200PC_FORCE_WARPS"): os.environ.pop(kk, None)
      if grid:
          os.environ["B200PC_GRID"] = grid
          if grid in ("2", "3", "4"): os.environ["B200PC_SMALL_PATH"] = "0"
          if grid == "3":
              os.environ["B200PC_SEED"] = str(rng.choice([0, 0, 2, 5])); os.environ["B200PC_INTERLEAVE"] = str(int(rng.integers(0, 2)))
          if grid == "4" and rng.random() < 0.3:
              os.environ["B200PC_FORCE_WARPS"] = str(int(rng.integers(1, 17)))
      form = int(rng.integers(0, 3)); k = int(rng.integers(1, min(N, 48) + 1))
      if grid == "4" and rng.random() < 0.1:                       # long lists: fewer warps per CTA, up to the largest that fits
          k = int(rng.integers(1, min(N, 876) + 1))
      modes[grid or "default"] += 1
      idx, dist = ops.knn_search(torch.from_numpy(ref).to(dev), torch.from_numpy(qry).to(dev), k, form, want_dist=True)
      oi, od = strict.knn(ref, qry, k, form)
      ok = np.array_equal(idx.cpu().numpy(), oi) and np.array_equal(dist.cpu().numpy().view(np.int32), od.view(np.int32))
      r = float(scale * rng.uniform(0.05, 1.5)); ns = int(rng.integers(1, 40))
      if grid == "4":                                              # the ball query has no pruned path: one of the other modes
          os.environ["B200PC_GRID"] = str(rng.choice(["0", "2", "3"])); os.environ.pop("B200PC_FORCE_WARPS", None)
      ball = P.query_ball_point(r, ns, torch.from_numpy(ref).to(dev), torch.from_numpy(qry).to(dev))
      okb = np.array_equal(ball.cpu().numpy(), strict.query_ball_point(r, ns, ref, qry))
      if not (ok and okb):
          bad += 1
          print("MISMATCH case %d: B=%d N=%d S=%d k=%d form=%d scale=%g off=%s small=%s grid=%s seed=%s drain=%s warps=%s knn_ok=%s ball_ok=%s (r=%g ns=%d)" % (
              c, B, N, S, k, form, scale, off, os.environ["B200PC_SMALL_PATH"], grid, os.environ.get("B200PC_SEED"),
              os.environ.get("B200PC_INTERLEAVE"), os.environ.get("B200PC_FORCE_WARPS"), ok, okb, r, ns), flush=True)
  for kk in ("B200PC_GRID", "B200PC_SEED", "B200PC_INTERLEAVE", "B200PC_FORCE_WARPS"): os.environ.pop(kk, None)
  print("fuzz grid modes: %s" % dict(sorted(modes.items())), flush=True)
  if old is None: os.environ.pop("B200PC_SMALL_PATH", None)
  else: os.environ["B200PC_SMALL_PATH"] = old
  return bad


if __name__ == "__main__":
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 150
    nbad = run(n, int(sys.argv[2]) if len(sys.argv) > 2 else 0)
    print("fuzz: %d cases, %d mismatches" % (n, nbad))
    sys.exit(1 if nbad else 0)
