"""The pruned top-k search (csrc/search.cu section 3b, B200PC_GRID=4) against the strict oracle.

Refs and queries are sorted in brick order, and each warp of 32 sorted queries visits only the 64-ref blocks whose box
bound does not exceed some lane's threshold.  Pruning changes which refs are looked at, never the keys, so every row must
be bit-identical to oracle/strict in all three distance forms and both index widths.  The plan that ran is read back from
B200PC_DEBUG_PLAN (grid "pruned", order "cell"), so that a knob that did not take effect fails instead of comparing the
brute-force search with itself."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

import guarded as G
import ragged_oracle as RO
from b200pc import _lib, ops, synth
from oracle import strict
from test_gpu_plans import Knobs, expect

pytestmark = pytest.mark.gpu

PRUNED = dict(SMALL_PATH=0, GRID=4)


@pytest.fixture
def knobs(cuda_dev, monkeypatch, capfd):
    k = Knobs(monkeypatch, capfd)
    k.set(**PRUNED)
    return k


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


def _expect_pruned(plans, n):
    expect(plans, n, grid="pruned", order="cell", mode=0)
    assert all(p["split"] == "1" for p in plans), plans


def _check(knobs, dev, ref, qry, k, forms=(0, 1, 2)):
    r, q = _t(ref, dev), _t(qry, dev)
    for form in forms:
        (idx, dist), plans, _ = knobs.run(lambda: ops.knn_search(r, q, k, form, want_dist=True))
        i32, plans32, _ = knobs.run(lambda: ops.knn_search_i32(r, q, k, form))
        _expect_pruned(plans + plans32, 2)
        oi, od = strict.knn(ref, qry, k, form)
        np.testing.assert_array_equal(idx.cpu().numpy(), oi)
        np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))
        np.testing.assert_array_equal(i32.cpu().numpy(), oi.astype(np.int32))


@functools.lru_cache(maxsize=None)
def _c2(first, B, n=16384):
    return synth.batch_pairs(first, B, n)


def test_c2_clouds(knobs, cuda_dev):
    a, b = _c2(0, 2)
    _check(knobs, cuda_dev, a, b, 16)


def test_c2_batch_matches_brute_force_bit_for_bit(knobs, cuda_dev):
    # the benchmark's shape (8 x 16384 x 16384, k = 16): the pruned search against the brute-force cell-order search
    a, b = _c2(0, 8)
    r, q = _t(a, cuda_dev), _t(b, cuda_dev)
    (pi, pd), plans, _ = knobs.run(lambda: ops.knn_search(r, q, 16, 0, want_dist=True))
    _expect_pruned(plans, 1)
    knobs.set(SMALL_PATH=0, GRID=3)
    (si, sd), plans, _ = knobs.run(lambda: ops.knn_search(r, q, 16, 0, want_dist=True))
    expect(plans, 1, grid="sorted")
    assert torch.equal(pi, si) and torch.equal(pd.view(torch.int32), sd.view(torch.int32))


def test_default_plan_of_the_long_searches_is_pruned(knobs, cuda_dev):
    # wherever the planner would sort refs and queries by cell (k >= 8, >= 2^29 pairs) it runs the pruned search
    knobs.set(GRID=None)                                   # no grid knob: the planner's own choice
    a, b = _c2(0, 8)
    r, q = _t(a, cuda_dev), _t(b, cuda_dev)
    for B, k in ((8, 16), (8, 64), (2, 16)):
        _, plans, _ = knobs.run(lambda: ops.knn_search_i32(r[:B], q[:B], k, 0))
        _expect_pruned(plans, 1)
    _, plans, _ = knobs.run(lambda: ops.knn_search_i32(r[:1], q[:1], 16, 0))     # 2^28 pairs: thresholds only
    expect(plans, 1, grid="thresholds")


def test_k64_and_small_shapes(knobs, cuda_dev):
    a, b = _c2(3, 1)
    _check(knobs, cuda_dev, a[:, :8000].copy(), b[:, :5000].copy(), 64)
    for B, N, S, k in ((3, 513, 31, 3), (1, 5, 9, 5), (2, 2500, 4100, 8), (1, 65, 40, 64)):
        x, y = synth.batch_pairs(20, B, max(N, S))
        _check(knobs, cuda_dev, x[:, :N].copy(), y[:, :S].copy(), k)


def test_grid_snapped_ties(knobs, cuda_dev):
    ref = synth.grid_snapped(7, 2, 3000, span=6)           # exact arithmetic, many equal distances and duplicate points
    qry = synth.grid_snapped(8, 2, 500, span=6)
    _check(knobs, cuda_dev, ref, qry, 16)
    wide = synth.grid_snapped(9, 1, 20000)                 # ties spread over many blocks
    _check(knobs, cuda_dev, wide, synth.grid_snapped(10, 1, 3000), 16)
    same = np.repeat(np.array([[[1.5, -2.0, 0.25]]], np.float32), 700, axis=1)     # all refs coincide: cell size 0
    _check(knobs, cuda_dev, same, qry[:1, :64].copy(), 5, forms=(0,))


def test_far_queries_and_sparse_outliers(knobs, cuda_dev):
    a, b = _c2(5, 1)
    _check(knobs, cuda_dev, a[:, :6000].copy(), (b[:, :700] + 500.0).astype(np.float32), 8)     # 500 m outside the refs
    sparse = a[:, :9000].copy()
    sparse[:, ::7] *= 40.0                                 # a few refs far away: wide boxes, most cells empty
    _check(knobs, cuda_dev, sparse, b[:, :2000].copy(), 16)


def test_non_finite_points_and_huge_coordinates(knobs, cuda_dev):
    a, b = synth.batch_pairs(5, 2, 5000)
    ref, qry = a.copy(), b[:, :1500].copy()
    ref[0, 5] = np.nan; ref[0, 77, 1] = np.inf; ref[1, 100:110] = -np.inf; ref[1, 4000:4064, 2] = np.nan
    qry[0, 3] = np.nan; qry[1, 9, 2] = np.inf; qry[1, 10, 0] = -np.inf
    _check(knobs, cuda_dev, ref, qry, 16)
    few = a[:1, :3000].copy()
    few[0, 10:] = np.nan                                   # 10 finite refs < k: every block is visited
    _check(knobs, cuda_dev, few, b[:1, :300].copy(), 16)
    for s in (2.0 ** 61, -(2.0 ** 61)):                    # |r|^2 near the top of the fp32 range
        big = (a[:1, :3000] * np.float32(2.0 ** 50) + np.float32(s)).astype(np.float32)
        bq = (b[:1, :500] * np.float32(2.0 ** 50) + np.float32(s)).astype(np.float32)
        _check(knobs, cuda_dev, big, bq, 16)


def test_ragged_lengths(knobs, cuda_dev):
    B, N, S, k = 8, 5000, 1500, 16
    a, b = synth.batch_pairs(80, B, N)
    ref, qry = a, b[:, :S].copy()
    rl = [0, 1, k - 1, k, 511, 512, 513, 5000]
    ql = [1500, 777, 33, 1, 1499, 0, 1000, 130]
    r, q = _t(ref, cuda_dev), _t(qry, cuda_dev)
    for form in (0, 2):
        (idx, dist), plans, _ = knobs.run(lambda: ops.knn_ragged(r, q, k, form, torch.tensor(rl, device=cuda_dev),
                                                                 torch.tensor(ql, device=cuda_dev), want_dist=True))
        _expect_pruned(plans, 1)
        oi, od = RO.knn(ref, qry, rl, ql, k, form)
        np.testing.assert_array_equal(idx.cpu().numpy(), oi)
        np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))


@pytest.mark.parametrize("knob", [dict(FORCE_SPLIT=3), dict(FORCE_Q=2), dict(SEED=5), dict(FILTER=0)])
def test_knobs_it_cannot_honour_are_refused(knobs, cuda_dev, knob):
    a, b = _c2(0, 1)
    knobs.set(**PRUNED, **knob)
    name = list(knob)[0]
    with pytest.raises(RuntimeError, match=name):
        ops.knn_search_i32(_t(a, cuda_dev), _t(b[:, :2000].copy(), cuda_dev), 16, 0)


def test_forced_split_without_forced_grid_keeps_the_sorted_search(knobs, cuda_dev):
    # a forced split without a forced grid is honoured by the brute-force cell order, and agrees with the pruned search
    a, b = _c2(0, 2)
    knobs.set(GRID=None, FORCE_SPLIT=3)
    r, q = _t(a, cuda_dev), _t(b, cuda_dev)
    idx, plans, _ = knobs.run(lambda: ops.knn_search(r, q, 16, 0))
    expect(plans, 1, grid="sorted", order="cell")
    assert int(plans[0]["split"]) == 3
    knobs.set(**PRUNED, FORCE_SPLIT=None)
    want, plans, _ = knobs.run(lambda: ops.knn_search(r, q, 16, 0))
    _expect_pruned(plans, 1)
    assert torch.equal(idx, want)


def test_forced_warps(knobs, cuda_dev):
    a, b = _c2(1, 1)
    for w in (1, 5):
        knobs.set(**PRUNED, FORCE_WARPS=w)
        _, plans, _ = knobs.run(lambda: ops.knn_search_i32(_t(a[:, :4000], cuda_dev), _t(b[:, :3000], cuda_dev), 16, 0))
        expect(plans, 1, warps=w, grid="pruned")
    _check(knobs, cuda_dev, a[:, :4000].copy(), b[:, :3000].copy(), 16, forms=(1,))


def test_run_to_run_determinism(knobs, cuda_dev):
    a, b = _c2(2, 4)
    r, q = _t(a, cuda_dev), _t(b, cuda_dev)
    first = ops.knn_search(r, q, 16, 2, want_dist=True)
    for _ in range(3):
        again = ops.knn_search(r, q, 16, 2, want_dist=True)
        assert torch.equal(first[0], again[0]) and torch.equal(first[1].view(torch.int32), again[1].view(torch.int32))


def test_buffer_hygiene(knobs, cuda_dev):
    """guarded, poisoned buffers (tests/guarded.py): nothing written outside the outputs, nothing read that the call did not
    write; item 0 holds non-finite refs and a NaN query, the last item two finite refs (rows that end in -1 / +inf)"""
    B, N, S, k = 2, 3000, 333, 16
    a, b = synth.batch_pairs(90, B, N)
    ref, qry = a.copy(), b[:, :S].copy()
    ref[0, 5] = np.nan; ref[0, N // 2, 1] = np.inf; ref[0, N - 1, 2] = -np.inf; qry[0, 3] = np.nan; ref[B - 1, 2:] = np.nan
    L = _lib.load()
    ops.reload_tuning()
    nws = L.b200pc_search_workspace_bytes(B, N, S, k)
    for i32 in (False, True):
        bufs = [G.inp("ref", ref), G.inp("qry", qry), G.out("idx", (B, S, k), torch.int32 if i32 else torch.int64),
                G.out("dist", (B, S, k), torch.float32), G.ws("ws", nws)]
        fn = L.b200pc_knn_i32 if i32 else L.b200pc_knn

        def call(lay):
            rc = fn(lay.ptr("ref"), lay.ptr("qry"), B, N, S, k, 1, lay.ptr("idx"), lay.ptr("dist"), lay.ptr("ws"), nws,
                    C.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert rc == 0, _lib.last_error()

        (res, _), plans, _ = knobs.run(lambda: G.check_call(bufs, call, cuda_dev))
        _expect_pruned(plans, len(G.POISONS) * len(G.ALIGNMENTS))
        oi, od = strict.knn(ref, qry, k, 1)
        np.testing.assert_array_equal(res["idx"], oi.astype(res["idx"].dtype))
        np.testing.assert_array_equal(_bits(res["dist"]), _bits(od))
