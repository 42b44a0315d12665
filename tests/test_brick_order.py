"""The brick order of the level-0 cells (csrc/search.cu brick_cell), restated on the host.

The pruned search sorts refs and queries in this order, and grid_pyramid_kernel / grid_scan_kernel walk its ranks while the
counters stay indexed by raster cell.  A rank that mapped to no cell, or two ranks to one cell, would drop or double a
cell's points.  The partial bricks (min(BRICK, g - BRICK * b)) only occur when a grid dimension is not a multiple of 4, and
which dimensions occur depends on the shape of the cloud, so the map is checked exhaustively on small grids, on random
grids up to GRID_MAX_CELLS, and on the grids that the adversarial clouds of the pruned-search tests produce.
tools/prune_sim.py's brick_rank (the host model of the block visits) must be its inverse."""
import importlib.util
import os

import numpy as np
import pytest

import prune_geometry as PG

BRICK, GRID_AXIS, GRID_MAX_CELLS = 4, 128, 131072          # search.cu
_spec = importlib.util.spec_from_file_location("prune_sim", os.path.join(os.path.dirname(os.path.dirname(__file__)), "tools", "prune_sim.py"))
prune_sim = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(prune_sim)


def brick_cell(dim, r):
    """search.cu brick_cell: rank r of the brick order -> raster cell (cz * gy + cy) * gx + cx, in int64 numpy"""
    gx, gy, gz = (int(v) for v in dim)
    r = np.asarray(r, np.int64).copy()
    bz = r // (BRICK * gx * gy)
    r -= bz * BRICK * gx * gy
    d = np.minimum(BRICK, gz - BRICK * bz)
    by = r // (BRICK * gx * d)
    r -= by * BRICK * gx * d
    h = np.minimum(BRICK, gy - BRICK * by)
    bx = r // (BRICK * h * d)
    r -= bx * BRICK * h * d
    w = np.minimum(BRICK, gx - BRICK * bx)
    lz = r // (h * w)
    r -= lz * h * w
    ly = r // w
    lx = r - ly * w
    return ((BRICK * bz + lz) * gy + BRICK * by + ly) * gx + BRICK * bx + lx


def _check(dim):
    n = int(np.prod(dim))
    c = brick_cell(dim, np.arange(n))
    assert c.min() >= 0 and c.max() < n, dim
    assert np.array_equal(np.sort(c), np.arange(n)), dim              # a bijection of [0, cells)
    rank = prune_sim.brick_rank(dim)
    assert np.array_equal(rank[c], np.arange(n)), dim                 # brick_rank is its inverse
    gx, gy, gz = (int(v) for v in dim)
    x, y, z = c % gx, (c // gx) % gy, c // (gx * gy)
    # every full 4 x 4 x 4 brick occupies 64 consecutive ranks; every brick (full or not) one contiguous run of ranks
    key = ((z // BRICK) * -(-gy // BRICK) + y // BRICK) * -(-gx // BRICK) + x // BRICK
    assert np.all(np.diff(key) >= 0), dim                              # bricks in raster order, each one run
    runs = np.bincount(key)
    full = (np.minimum(BRICK, gx - BRICK * np.arange(-(-gx // BRICK)))[None, None, :] *
            np.minimum(BRICK, gy - BRICK * np.arange(-(-gy // BRICK)))[None, :, None] *
            np.minimum(BRICK, gz - BRICK * np.arange(-(-gz // BRICK)))[:, None, None]).ravel()
    assert np.array_equal(runs, full), dim
    assert np.all(runs[full == 64] == 64)
    # inside a brick the cells are in raster order
    inner = (z % BRICK) * 16 + (y % BRICK) * 4 + x % BRICK
    same = np.diff(key) == 0
    assert np.all(np.diff(inner)[same] > 0), dim


@pytest.mark.parametrize("gz", range(1, 13))
def test_brick_order_is_a_bijection_on_every_small_grid(gz):
    # every residue mod 4 on every axis, and dimensions below one brick
    for gx in range(1, 13):
        for gy in range(1, 13):
            _check((gx, gy, gz))


def test_brick_order_on_random_grids_up_to_the_cell_limit():
    rng = np.random.default_rng(2024)
    seen = 0
    while seen < 300:
        dim = rng.integers(1, GRID_AXIS + 1, 3)
        if dim.prod() > GRID_MAX_CELLS:
            continue
        _check(dim)
        seen += 1
    for dim in ((128, 32, 32), (128, 128, 8), (127, 33, 31), (1, 1, 128), (128, 1, 1), (1, 128, 1), (65, 65, 31)):
        assert np.prod(dim) <= GRID_MAX_CELLS
        _check(dim)


def test_grid_sizing_of_the_adversarial_clouds():
    """the dimensions grid_bbox_kernel gives the clouds of tests/test_gpu_pruned_stress.py (restated as prune_sim.grid
    does), bijective too -- and among them flat and linear grids (an axis of one cell) and dimensions that are not
    multiples of 4"""
    dims = set()
    for name in PG.FAMILIES:
        for seed in range(3):
            ref, _ = PG.family(name, seed)
            finite = ref[np.isfinite(ref).all(1)].astype(np.float64)
            if np.ptp(finite, 0).max() == 0:
                continue                                              # all refs coincide: one cell
            _, _, dim = prune_sim.grid(finite)
            assert np.prod(dim) <= GRID_MAX_CELLS and dim.max() <= GRID_AXIS
            dims.add(tuple(int(v) for v in dim))
    for dim in sorted(dims):
        _check(dim)
    assert any(1 in d for d in dims) and any(d.count(1) >= 2 for d in dims), dims
    assert any(any(v % 4 for v in d) for d in dims), dims
