"""Host simulation of the pruned search's block visits (csrc/search.cu section 3b) on the C2 clouds.

Refs and queries are sorted by level-0 cell (the grid of grid_bbox_kernel: <= 128 cells along the longest axis, <= 131072
cells) in raster or brick order; the sorted refs are cut into blocks, the sorted queries into groups, and a group visits a
block when some query of the group has boxdist^2(q, block box) <= tau_q.  tau_q is the exact k-th distance (float64, a
k-d tree): the limit the kernel's tightening thresholds approach, so the counts are a lower bound of what it visits.
usage: python tools/prune_sim.py [pairs=3] [k=16]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "point-cloud-interpolation-_b200"))
import numpy as np
from scipy.spatial import cKDTree

from b200pc import synth


def grid(ref):
    lo, hi = ref.min(0), ref.max(0)
    ext = hi - lo
    h = ext.max() / 128.0
    while True:
        dim = np.clip(np.ceil(ext / h).astype(int), 1, 128)
        if dim.prod() <= 131072:
            return lo, h, dim
        h *= 2.0


def brick_rank(dim):
    """raster cell -> rank of the brick order (the inverse of search.cu's brick_cell)"""
    gx, gy, gz = (int(v) for v in dim)
    c = np.arange(gx * gy * gz)
    x, y, z = c % gx, (c // gx) % gy, c // (gx * gy)
    bx, by, bz, lx, ly, lz = x // 4, y // 4, z // 4, x % 4, y % 4, z % 4
    d = np.minimum(4, gz - 4 * bz)
    h = np.minimum(4, gy - 4 * by)
    w = np.minimum(4, gx - 4 * bx)
    return bz * 4 * gx * gy + by * 4 * gx * d + bx * 4 * h * d + (lz * h + ly) * w + lx


def visits(ref, qry, k, order, block, group):
    lo, h, dim = grid(ref)
    def cell(p):                                   # raster index (cz * gy + cy) * gx + cx, clamped into the grid
        c = np.clip(((p - lo) / h).astype(int), 0, dim - 1)
        return (c[:, 2] * dim[1] + c[:, 1]) * dim[0] + c[:, 0]
    key = brick_rank(dim) if order == "brick" else np.arange(dim.prod())
    r = ref[np.argsort(key[cell(ref)], kind="stable")]
    q = qry[np.argsort(key[cell(qry)], kind="stable")]
    tau = cKDTree(r).query(q, k)[0][:, -1] ** 2
    nb = -(-len(r) // block)
    rb = np.pad(r, ((0, nb * block - len(r)), (0, 0)), mode="edge").reshape(nb, block, 3)
    blo, bhi = rb.min(1), rb.max(1)
    counts = []
    for g0 in range(0, len(q), group):
        qs, ts = q[g0:g0 + group, None], tau[g0:g0 + group, None]
        gap = np.maximum(np.maximum(blo[None] - qs, qs - bhi[None]), 0.0)
        counts.append(int(((gap ** 2).sum(-1) <= ts).any(0).sum()))
    counts = np.array(counts)
    return counts.sum() * block * group / (len(r) * len(q)), counts.mean(), counts.max()


def main():
    pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 3
    k = int(sys.argv[2]) if len(sys.argv) > 2 else 16
    print("order   group  block   visited pairs   blocks per group (mean, max)")
    for order, group, block in (("raster", 32, 64), ("brick", 32, 64), ("brick", 32, 512), ("brick", 448, 64)):
        res = [visits(*(p.astype(np.float64) for p in synth.frame_pair(i, 16384)), k, order, block, group) for i in range(pairs)]
        print("%-7s %5d %6d   %5.3f .. %5.3f   %6.1f  %4d" % (order, group, block, min(r[0] for r in res), max(r[0] for r in res),
                                                            np.mean([r[1] for r in res]), max(r[2] for r in res)))


if __name__ == "__main__":
    main()
