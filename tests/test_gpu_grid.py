"""The occupancy-grid variants of the top-k search (csrc/search.cu section 1b) against the strict oracle.

The variants only change the ORDER in which refs and queries are visited and the threshold a query starts from; results
must stay bit-identical to the oracle on every row.  The default only switches them on for large searches, so the knobs
force them here on small and awkward shapes: B200PC_GRID=2 (starting thresholds only), 3 (refs and queries in cell order),
B200PC_SEED=n (k-th distance inside the cell box up to level n-1 instead of the box's corner), B200PC_INTERLEAVE=1 (cell-ordered
queries dealt out warp by warp)."""
import numpy as np
import pytest
import torch

from b200pc import ops, synth
from oracle import strict
from test_gpu_plans import Knobs     # reads back the plan that ran (B200PC_DEBUG_PLAN)

pytestmark = pytest.mark.gpu

VARIANTS = [
    {"B200PC_GRID": "2"},
    {"B200PC_GRID": "3"},
    {"B200PC_GRID": "3", "B200PC_INTERLEAVE": "1"},
    {"B200PC_GRID": "3", "B200PC_SEED": "5"},
    {"B200PC_GRID": "3", "B200PC_SEED": "2", "B200PC_INTERLEAVE": "1"},
]
IDS = ["thresholds", "sorted", "sorted-interleaved", "sorted-seed5", "sorted-seed2-interleaved"]


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


def _force(monkeypatch, env):
    monkeypatch.setenv("B200PC_SMALL_PATH", "0")          # always the streaming kernel: that is where the grid lives
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    ops.reload_tuning()


def _check(dev, ref, qry, k, form):
    idx, dist = ops.knn_search(_t(ref, dev), _t(qry, dev), k, form, want_dist=True)
    oi, od = strict.knn(ref, qry, k, form)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))


SHAPES = [
    # (B, N, S, k)
    (2, 4096, 2048, 16),
    (3, 513, 31, 3),        # one ref past a tile boundary, fewer queries than a warp
    (1, 1000, 777, 1),
    (1, 5, 9, 5),           # k == N: every box is the whole cloud
    (1, 3000, 1500, 64),
    (2, 2500, 4100, 8),     # ragged on both sides, several query blocks
]


@pytest.mark.parametrize("env", VARIANTS, ids=IDS)
@pytest.mark.parametrize("B,N,S,k", SHAPES)
@pytest.mark.parametrize("form", [0, 1, 2])
def test_grid_variants_match_oracle(cuda_dev, monkeypatch, env, B, N, S, k, form):
    _force(monkeypatch, env)
    a, b = synth.batch_pairs(20, B, max(N, S))
    _check(cuda_dev, a[:, :N].copy(), b[:, :S].copy(), k, form)


@pytest.mark.parametrize("env", VARIANTS, ids=IDS)
def test_grid_variants_ties_and_duplicates(cuda_dev, monkeypatch, env):
    _force(monkeypatch, env)
    ref = synth.grid_snapped(7, 2, 3000, span=6)       # exact arithmetic, many equal distances and duplicate points
    qry = synth.grid_snapped(8, 2, 500, span=6)
    for form in (0, 1, 2):
        _check(cuda_dev, ref, qry, 16, form)
    same = np.repeat(np.array([[[1.5, -2.0, 0.25]]], np.float32), 700, axis=1)     # all refs coincide: cell size 0
    _check(cuda_dev, same, qry[:1, :64].copy(), 5, 0)


@pytest.mark.parametrize("env", VARIANTS, ids=IDS)
def test_grid_variants_split_and_far_queries(cuda_dev, monkeypatch, capfd, env):
    _force(monkeypatch, env)
    knobs = Knobs(monkeypatch, capfd)
    knobs.set()
    a, b = synth.batch_pairs(3, 1, 16384)
    _, plans, _ = knobs.run(lambda: _check(cuda_dev, a, b[:, :1024].copy(), 16, 2))   # few queries: the ref range is split and merged
    assert len(plans) == 1 and int(plans[0]["split"]) > 1, plans
    assert plans[0]["grid"] == ("thresholds" if env["B200PC_GRID"] == "2" else "sorted"), plans
    _check(cuda_dev, a[:, :6000].copy(), (b[:, :300] + 500.0).astype(np.float32), 8, 0)     # queries outside the ref box
    sparse = a[:, :4000].copy()
    sparse[:, ::7] *= 40.0                              # a few refs far away: most cells empty, wide boxes
    _check(cuda_dev, sparse, b[:, :900].copy(), 16, 1)


@pytest.mark.parametrize("env", VARIANTS, ids=IDS)
def test_grid_variants_non_finite_points(cuda_dev, monkeypatch, env):
    _force(monkeypatch, env)
    a, b = synth.batch_pairs(5, 2, 3000)
    ref, qry = a.copy(), b[:, :700].copy()
    ref[0, 5] = np.nan; ref[0, 77, 1] = np.inf; ref[1, 100:110] = -np.inf
    qry[0, 3] = np.nan; qry[1, 9, 2] = np.inf
    # non-finite refs never enter the grid and go behind the finite ones in the cell order; a non-finite query starts from
    # +inf.  The blind search is the yardstick here (it is pinned to the oracle on finite inputs by test_gpu_search.py).
    idx, dist = ops.knn_search(_t(ref, cuda_dev), _t(qry, cuda_dev), 16, 0, want_dist=True)
    monkeypatch.setenv("B200PC_GRID", "0"); ops.reload_tuning()
    idx0, dist0 = ops.knn_search(_t(ref, cuda_dev), _t(qry, cuda_dev), 16, 0, want_dist=True)
    assert torch.equal(idx, idx0) and torch.equal(dist.view(torch.int32), dist0.view(torch.int32))


def test_int32_output_and_three_nn_through_the_sorted_grid(cuda_dev, monkeypatch):
    _force(monkeypatch, {"B200PC_GRID": "3"})
    a, b = synth.batch_pairs(9, 2, 5000)
    i32 = ops.knn_search_i32(_t(a, cuda_dev), _t(b[:, :3000].copy(), cuda_dev), 16, 0)
    oi, _ = strict.knn(a, b[:, :3000].copy(), 16, 0)
    np.testing.assert_array_equal(i32.cpu().numpy(), oi.astype(np.int32))
    from b200pc import pointnet2_utils as P
    d3, i3 = P.three_nn(_t(b, cuda_dev), _t(a[:, :2500].copy(), cuda_dev))
    o3i, o3d = strict.knn(a[:, :2500].copy(), b, 3, 1)
    np.testing.assert_array_equal(i3.cpu().numpy(), o3i)
