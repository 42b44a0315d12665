"""The pruned top-k search (csrc/search.cu section 3b, B200PC_GRID=4) on the geometry, list lengths, block and window edges
and entry points that stress it, against the strict oracle.

A skipped block that held a neighbour returns a plausible list that is a little wrong, so every comparison is exact:
indices and distance bits equal oracle/strict (or, for the shapes too large for the host oracle, the brute-force cell-order
search B200PC_GRID=3, which tests/test_gpu_plans.py checks against it).  Every forced call reads back, from
B200PC_DEBUG_PLAN, that the pruned plan ran, with the warp count expected for its k.

Per-warp shared memory grows with k (pruned_warp_bytes), so the warps per CTA run from 16 down to 1; k = 876 is the
largest list that fits.  A block is 64 sorted refs, the walk tests blocks 32 at a time (one window) and stages them
PRUNE_BATCH = 4 at a time, so the finite-ref counts around 64, 2048 and 4096 put the last block, the window edge and the
batch tail on both sides of their edges.  The geometry families are tests/prune_geometry.py's; the host model of their
block visits (tools/prune_sim.py, exact tau from a k-d tree) shows that each of them does prune."""
import ctypes as C
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import prune_geometry as PG
import ragged_oracle as RO
from b200pc import _lib, ops, pytorch3d_shim as S3, synth
from oracle import strict
from test_gpu_plans import Knobs, _fused, expect

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "point-cloud-interpolation-_b200")
_spec = importlib.util.spec_from_file_location("prune_sim", os.path.join(ROOT, "tools", "prune_sim.py"))
prune_sim = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(prune_sim)

gpu = pytest.mark.gpu
PRUNED = dict(SMALL_PATH=0, GRID=4)
BLOCK, MAX_SMEM, MAX_WARPS = 64, 227 * 1024, 16              # search.cu PRUNE_BLOCK, kMaxSmem, PRUNED_MAX_WARPS
REC, CHUNK, CAND_CAP, PRUNE_BATCH = 8, 8, 8, 4


def pruned_warp_bytes(k):
    """search.cu pruned_warp_bytes: query records, staged chunks, their indices, query positions, thresholds, heap [k+1],
    candidate buffer, block list; rounded up to 128 bytes"""
    b = 32 * 16 + 32 * REC * 16 + 32 * CHUNK * 4 + 32 * 16 + 32 * 4 + (k + 1) * 32 * 8 + CAND_CAP * 32 * 2 + PRUNE_BATCH * 4
    return -(-b // 128) * 128


def pruned_warps(k):
    """warps per CTA of the pruned plan (0: the list does not fit)"""
    return min(MAX_WARPS, (MAX_SMEM - 1024) // pruned_warp_bytes(k))


K_MAX = max(k for k in range(1, 2000) if pruned_warps(k) >= 1)
K_FOR_WARPS = {w: max(k for k in range(1, K_MAX + 1) if pruned_warps(k) == w) for w in range(1, MAX_WARPS + 1)}


@pytest.fixture
def knobs(cuda_dev, monkeypatch, capfd):
    k = Knobs(monkeypatch, capfd)
    k.set(**PRUNED)
    return k


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


def _expect_pruned(plans, n, k=None):
    expect(plans, n, grid="pruned", order="cell", mode=0, warps=None if k is None else pruned_warps(k))
    assert all(p["split"] == "1" for p in plans), plans


def _check(knobs, dev, ref, qry, k, forms=(0, 1, 2)):
    """forced pruned search, int64 and int32 entries, against oracle/strict bit for bit"""
    r, q = _t(ref, dev), _t(qry, dev)
    for form in forms:
        (idx, dist), plans, _ = knobs.run(lambda: ops.knn_search(r, q, k, form, want_dist=True))
        i32, plans32, _ = knobs.run(lambda: ops.knn_search_i32(r, q, k, form))
        _expect_pruned(plans + plans32, 2, k)
        oi, od = strict.knn(ref, qry, k, form)
        np.testing.assert_array_equal(idx.cpu().numpy(), oi)
        np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))
        np.testing.assert_array_equal(i32.cpu().numpy(), oi.astype(np.int32))


def _same(a, b):
    return torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a, b.view(torch.int32) if b.dtype == torch.float32 else b)


def _vs_sorted(knobs, call, n_plans, k=None, exact=None):
    """call under GRID=4 (pruned) and under GRID=3 (brute-force cell order): bit for bit the same outputs (the first `exact`
    of them; the rest are returned for the caller to compare)"""
    knobs.set(**PRUNED)
    got, plans, _ = knobs.run(call)
    _expect_pruned(plans, n_plans, k)
    knobs.set(SMALL_PATH=0, GRID=3)
    want, plans, _ = knobs.run(call)
    expect(plans, n_plans, grid="sorted")
    knobs.set(**PRUNED)
    got = got if isinstance(got, tuple) else (got,)
    want = want if isinstance(want, tuple) else (want,)
    for g, w in list(zip(got, want))[:exact]:
        assert _same(g, w)
    return got if exact is None else (got, want)


# ---- 2. adversarial geometry -------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", PG.FAMILIES)
def test_family_matches_oracle(knobs, cuda_dev, name):
    ref, qry = PG.batch((name, name), 0, 3000, 600)          # two items: per-item descriptors and block tables
    _check(knobs, cuda_dev, ref, qry, 16)


@gpu
@pytest.mark.parametrize("extent,offset", PG.PRECISION)
def test_precision_tight_every_form(knobs, cuda_dev, extent, offset):
    i = PG.PRECISION.index((extent, offset))
    ref, qry = PG.family("precision", i, 4000, 700)
    _check(knobs, cuda_dev, ref[None], qry[None], 16)
    _check(knobs, cuda_dev, ref[None], qry[None], 3, forms=(1,))


@gpu
def test_mixed_batch(knobs, cuda_dev):
    ref, qry = PG.mixed(0, k=16)
    assert np.isfinite(ref[4]).all(1).sum() < 16 and not np.isfinite(ref[1]).all()
    _check(knobs, cuda_dev, ref, qry, 16)


def _visited_fraction(name, seed=0, k=16):
    ref, qry = PG.family(name, seed)
    _, mean, _ = prune_sim.visits(ref.astype(np.float64), qry.astype(np.float64), k, "brick", BLOCK, 32)
    return mean / -(-len(ref) // BLOCK)


def test_each_family_prunes_in_the_host_model():
    """visited (group, block) pairs over all of them, in the host model of the walk (a lower bound of what the kernel visits:
    its thresholds only approach the exact tau): every family prunes, except the shell around its centre, which is meant to
    visit nearly everything and is the highest"""
    frac = {name: _visited_fraction(name) for name in PG.FAMILIES}
    near_all = ("shell", "shell_snapped")
    for name, f in frac.items():
        if name not in near_all:
            assert f < 0.9, (name, frac)
    assert frac["shell"] > 0.95 and frac["shell"] == max(frac.values()), frac


# ---- 3. k, warp counts and edges -------------------------------------------------------------------------------------
def test_warp_count_model():
    """the restated sizes: 16 warps up to k = 28, one warp from k = 425, and 876 the largest list that fits"""
    assert K_MAX == 876 and pruned_warps(877) == 0
    assert sorted(set(pruned_warps(k) for k in range(1, K_MAX + 1))) == list(range(1, 17))
    assert K_FOR_WARPS[16] == 28 and min(k for k in range(1, K_MAX + 1) if pruned_warps(k) == 1) == 425


@gpu
@pytest.mark.parametrize("warps", range(1, MAX_WARPS + 1))
def test_every_warp_count(knobs, cuda_dev, warps):
    k = K_FOR_WARPS[warps]
    name = PG.FAMILIES[warps % len(PG.FAMILIES)]
    ref, qry = PG.family(name, warps, max(2000, k + 300), 300)
    _check(knobs, cuda_dev, ref[None], qry[None], k)


@gpu
@pytest.mark.parametrize("k", [1, 2, 3, 4, 7, 9, 17, 31, 33, 65, 127, 255, 256, 876])
def test_other_list_lengths(knobs, cuda_dev, k):
    a, b = synth.batch_pairs(k, 1, 2500)
    _check(knobs, cuda_dev, a, b[:, :400].copy(), k, forms=(0, 2) if k > 64 else (0, 1, 2))


@gpu
def test_k877_does_not_fit(knobs, cuda_dev):
    a, b = synth.batch_pairs(3, 1, 2000)
    with pytest.raises(RuntimeError, match="does not fit"):
        ops.knn_search(_t(a, cuda_dev), _t(b[:, :64].copy(), cuda_dev), 877, 0)


@gpu
def test_longest_lists_of_the_default_plan(knobs, cuda_dev):
    """2^29 pairs, k >= 8: the planner's pruned range.  k = 876 runs there, although search_kernel's own lists end at
    k = 774 (the planner used to refuse every k > 774 before it looked at the pruned plan); k = 877 fits neither and fails
    cleanly"""
    knobs.set(GRID=None)
    ref = PG.family("ground_objects", 5, 1 << 21, 300)[0][None]
    qry = PG.family("ground_objects", 6, 300, 256)[1][None]
    r, q = _t(ref, cuda_dev), _t(qry, cuda_dev)
    (idx, dist), plans, _ = knobs.run(lambda: ops.knn_search(r, q, 876, 2, want_dist=True))
    _expect_pruned(plans, 1, 876)
    oi, od = strict.knn(ref, qry, 876, 2)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))
    with pytest.raises(RuntimeError, match="does not fit"):
        ops.knn_search(r, q, 877, 2)
    with pytest.raises(RuntimeError, match="does not fit"):                # below 2^29 pairs: search_kernel's limit
        ops.knn_search(r[:, : 1 << 20], q, 775, 2)


EDGE_COUNTS = [1, 63, 64, 65, 2047, 2048, 2049, 4095, 4096, 4097]


@gpu
@pytest.mark.parametrize("S", [1, 31, 32, 33])
@pytest.mark.parametrize("nf", EDGE_COUNTS)
def test_block_and_window_edges(knobs, cuda_dev, nf, S):
    """nf finite refs: the last block partly filled or not, the block count on both sides of a 32-block window, the tail
    batch of fewer than PRUNE_BATCH blocks; S queries: a partly dead last warp.  Once with N = nf, once with NaN refs
    spread through a larger N (they sort behind the finite ones)"""
    name = PG.FAMILIES[(nf + S) % len(PG.FAMILIES)]
    ref, qry = PG.family(name, nf, nf + 200, S)
    k = min(16, nf)
    _check(knobs, cuda_dev, ref[None, :nf].copy(), qry[None], k, forms=(0, 2))
    holes = ref.copy()
    holes[np.random.default_rng(nf).choice(nf + 200, 200, replace=False)] = np.nan
    _check(knobs, cuda_dev, holes[None], qry[None], 16, forms=(1,))


@gpu
def test_ragged_items_at_the_edges(knobs, cuda_dev):
    B, N, S, k = len(EDGE_COUNTS), 4097, 300, 16
    ref, qry = PG.batch([PG.FAMILIES[i % len(PG.FAMILIES)] for i in range(B)], 7, N, S)
    rl = EDGE_COUNTS
    ql = [1, 31, 32, 33, 300, 299, 64, 0, 257, 100]
    r, q = _t(ref, cuda_dev), _t(qry, cuda_dev)
    for form in (0, 1, 2):
        (idx, dist), plans, _ = knobs.run(lambda: ops.knn_ragged(r, q, k, form, torch.tensor(rl, device=cuda_dev),
                                                                 torch.tensor(ql, device=cuda_dev), want_dist=True))
        _expect_pruned(plans, 1, k)
        oi, od = RO.knn(ref, qry, rl, ql, k, form)
        np.testing.assert_array_equal(idx.cpu().numpy(), oi)
        np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))


@gpu
def test_persistent_warps_loop_over_many_groups(knobs, cuda_dev):
    # k = 512: one warp per CTA and one CTA per SM; 2 x 16384 queries are 1024 groups, several per resident warp
    ref, qry = PG.batch(("two_clusters", "lattice"), 3, 4096, 16384)
    _check(knobs, cuda_dev, ref, qry, 512, forms=(0,))


# ---- 4. every entry point that reaches the search ----------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["fusion_group", "feature_propagation", "chamfer", "rebuild_pack", "knn_point"])
def test_fused_entries_forced_pruned(knobs, cuda_dev, name):
    """the entries of test_gpu_plans.py (fusion_group with features, feature_propagation form 1 k = 3, Chamfer k = 1 direct
    form in both directions, rebuild_pack with int32 indices, knn_point) under GRID=4: the oracle, and bit for bit GRID=3"""
    call, check, n_plans = _fused(cuda_dev, name)
    got = _vs_sorted(knobs, call, n_plans)
    check(got)


@gpu
def test_fusion_group_without_features(knobs, cuda_dev):
    ref, qry = PG.batch(("ground_objects", "two_clusters"), 11, 5000, 700)
    r, q = _t(ref, cuda_dev), _t(qry, cuda_dev)
    resi, nn, gf, idx = _vs_sorted(knobs, lambda: ops.fusion_group(q, r, 16), 1, 16)
    od, oi = strict.knn_points(qry, ref, 16)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    assert gf.shape[1] == 0
    np.testing.assert_array_equal(_bits(nn.cpu().numpy()), _bits(strict.index_points(ref, oi).transpose(0, 3, 1, 2)))


@gpu
def test_three_nn_forced_pruned(knobs, cuda_dev):
    dense, _ = PG.batch(("plane", "density"), 12, 6000, 10)
    sparse, _ = PG.batch(("plane", "density"), 13, 2500, 10)
    u, kn = _t(dense, cuda_dev), _t(sparse, cuda_dev)
    dist, idx, w = _vs_sorted(knobs, lambda: ops.three_nn(u, kn), 1, 3)
    od, oi = strict.three_nn(dense, sparse)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))
    np.testing.assert_array_equal(_bits(w.cpu().numpy()), _bits(strict.three_weights(od, 0)))


@gpu
def test_chamfer_backward_and_ragged_forced_pruned(knobs, cuda_dev):
    x, _ = PG.batch(("two_clusters", "outside"), 14, 4000, 10)
    y, _ = PG.batch(("two_clusters", "outside"), 15, 3500, 10)

    def fwd_bwd():
        xt, yt = _t(x, cuda_dev).requires_grad_(), _t(y, cuda_dev).requires_grad_()
        loss, dx, ix, dy, iy = ops.chamfer(xt, yt)
        loss.backward()
        return loss.detach(), dx.detach(), ix, dy.detach(), iy, xt.grad, yt.grad
    got, want = _vs_sorted(knobs, fwd_bwd, 2, 1, exact=5)
    loss, dx, ix, dy, iy, gx, gy = got
    for g, w in zip(got[5:], want[5:]):          # same indices; the backward scatters with atomics, in no fixed order
        torch.testing.assert_close(g, w, rtol=1e-5, atol=1e-6 * w.abs().max().item())
    ol, odx, oix, ody, oiy = strict.chamfer(x, y)
    np.testing.assert_array_equal(ix.cpu().numpy(), oix)
    np.testing.assert_array_equal(iy.cpu().numpy(), oiy)
    np.testing.assert_array_equal(_bits(dx.cpu().numpy()), _bits(odx))
    np.testing.assert_array_equal(_bits(dy.cpu().numpy()), _bits(ody))
    assert abs(loss.item() - ol) <= 1e-5 * abs(ol)
    assert torch.isfinite(gx).all() and torch.isfinite(gy).all()

    xl, yl = [4000, 1777], [65, 3500]
    xt, yt = _t(x, cuda_dev), _t(y, cuda_dev)
    lx, ly = torch.tensor(xl, device=cuda_dev), torch.tensor(yl, device=cuda_dev)
    sums, dx, ix, dy, iy = _vs_sorted(knobs, lambda: ops.chamfer_ragged(xt, yt, lx, ly), 2, 1)
    osums, odx, oix, ody, oiy = RO.chamfer_terms(x, y, xl, yl)
    np.testing.assert_array_equal(ix.cpu().numpy(), oix)
    np.testing.assert_array_equal(iy.cpu().numpy(), oiy)
    np.testing.assert_array_equal(_bits(dx.cpu().numpy()), _bits(odx))
    np.testing.assert_array_equal(_bits(dy.cpu().numpy()), _bits(ody))
    np.testing.assert_allclose(sums.detach().cpu().numpy(), osums, rtol=1e-6)


@gpu
def test_knn_points_shim_with_lengths_forced_pruned(knobs, cuda_dev):
    p2, p1 = PG.batch(("lattice", "shell_snapped", "ground_objects"), 16, 3000, 500)
    l1, l2 = [500, 33, 1], [3000, 2049, 64]
    a, b = _t(p1, cuda_dev), _t(p2, cuda_dev)
    t1, t2 = torch.tensor(l1, device=cuda_dev), torch.tensor(l2, device=cuda_dev)
    dists, idx = _vs_sorted(knobs, lambda: tuple(S3.knn_points(a, b, t1, t2, K=16)[:2]), 1, 16)
    oi, od = RO.knn(p2, p1, l2, l1, 16, strict.FORM_DIRECT)
    pad = (np.arange(500)[None, :, None] >= np.array(l1)[:, None, None]) | (np.arange(16)[None, None, :] >= np.array(l2)[:, None, None])
    np.testing.assert_array_equal(idx.cpu().numpy(), np.where(pad, 0, oi))
    np.testing.assert_array_equal(_bits(dists.cpu().numpy()), _bits(np.where(pad, np.float32(0), od)))


@gpu
def test_knn_async_host_forced_pruned(knobs, cuda_dev):
    L = _lib.load()
    ref, qry = PG.batch(("density", "line_diag"), 17, 5000, 900)
    B, N, S, k = 2, 5000, 900, 16
    h_ref, h_qry = torch.from_numpy(ref).pin_memory(), torch.from_numpy(qry).pin_memory()

    def call():
        need = L.b200pc_knn_async_host_workspace_bytes(B, N, S, k)          # the plan, and its workspace, follow the knobs
        arena = torch.empty(need, dtype=torch.uint8, device=cuda_dev)
        out = torch.empty(B, S, k, dtype=torch.int32).pin_memory()
        dist = torch.empty(B, S, k, dtype=torch.float32).pin_memory()
        rc = L.b200pc_knn_async_host(C.c_void_p(h_ref.data_ptr()), C.c_void_p(h_qry.data_ptr()), B, N, S, k, 0,
                                     C.c_void_p(out.data_ptr()), C.c_void_p(dist.data_ptr()), C.c_void_p(arena.data_ptr()), need,
                                     C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, _lib.last_error()
        torch.cuda.current_stream().synchronize()
        return out, dist
    out, dist = _vs_sorted(knobs, call, 1, k)
    oi, od = strict.knn(ref, qry, k, 0)
    np.testing.assert_array_equal(out.numpy(), oi.astype(np.int32))
    np.testing.assert_array_equal(_bits(dist.numpy()), _bits(od))


@gpu
def test_default_plans_of_the_entries_at_the_benchmark_shapes(knobs, cuda_dev):
    """which entries the default planner sends to the pruned search at the shapes bench.py runs them: the k >= 8 searches
    of >= 2^29 pairs (C2's knn_points / knn_point / async host, the fused grouping of batch-8 PointINet), not three-NN (k = 3)
    and not the k = 1 searches of Chamfer and PolyPCI.rebuild"""
    knobs.set(SMALL_PATH=None, GRID=None)
    a, b = synth.batch_pairs(0, 8, 16384)
    r, q = _t(a, cuda_dev), _t(b, cuda_dev)
    _, plans, _ = knobs.run(lambda: S3.knn_points(q, r, K=16))
    _expect_pruned(plans, 1, 16)
    _, plans, _ = knobs.run(lambda: S3.knn_points(q, r, torch.full((8,), 16000, device=cuda_dev), None, K=16))
    _expect_pruned(plans, 1, 16)
    _, plans, _ = knobs.run(lambda: ops.fusion_group(q, r, 16, r))
    _expect_pruned(plans, 1, 16)
    L = _lib.load()
    need = L.b200pc_knn_async_host_workspace_bytes(8, 16384, 16384, 16)
    arena = torch.empty(need, dtype=torch.uint8, device=cuda_dev)
    h_ref, h_qry = torch.from_numpy(a).pin_memory(), torch.from_numpy(b).pin_memory()
    out = torch.empty(8, 16384, 16, dtype=torch.int32).pin_memory()

    def host():
        assert L.b200pc_knn_async_host(C.c_void_p(h_ref.data_ptr()), C.c_void_p(h_qry.data_ptr()), 8, 16384, 16384, 16, 0,
                                       C.c_void_p(out.data_ptr()), None, C.c_void_p(arena.data_ptr()), need,
                                       C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0, _lib.last_error()
    _, plans, _ = knobs.run(host)
    _expect_pruned(plans, 1, 16)
    known = r[:, :4096].contiguous()
    _, plans, _ = knobs.run(lambda: ops.three_nn(q, known))           # C3 shape, batch 8: k = 3
    assert all(p["grid"] != "pruned" for p in plans) and len(plans) == 1, plans
    _, plans, _ = knobs.run(lambda: ops.chamfer(q, r))
    assert all(p["grid"] != "pruned" for p in plans), plans
    _, plans, _ = knobs.run(lambda: ops.rebuild_pack(r[:4], q[:4]))
    assert all(p["grid"] != "pruned" for p in plans), plans


# ---- 5. large shapes ---------------------------------------------------------------------------------------------------
LARGE_FAMILIES = [n for n in PG.FAMILIES if n != "precision"]


@gpu
@pytest.mark.parametrize("seed", range(10))
def test_large_batches_match_the_brute_force_search(knobs, cuda_dev, seed):
    """8 x 16384^2, k = 16, eight families per batch, all three forms: too large for the host oracle, so bit for bit the
    brute-force cell-order search"""
    names = [LARGE_FAMILIES[(seed + i) % len(LARGE_FAMILIES)] for i in range(8)]
    ref, qry = PG.batch(names, 100 + seed, 16384, 16384)
    r, q = _t(ref, cuda_dev), _t(qry, cuda_dev)
    for form in (0, 1, 2):
        _vs_sorted(knobs, lambda: ops.knn_search(r, q, 16, form, want_dist=True), 1, 16)


@gpu
def test_one_large_cloud_matches_the_brute_force_search(knobs, cuda_dev):
    ref, qry = PG.family("ground_objects", 200, 65536, 65536)
    r, q = _t(ref[None], cuda_dev), _t(qry[None], cuda_dev)
    _vs_sorted(knobs, lambda: ops.knn_search(r, q, 16, 0, want_dist=True), 1, 16)


# ---- 6. bounds-checked build -------------------------------------------------------------------------------------------
BOUNDS_SCRIPT = r"""
import os, sys
sys.path[:0] = [%(root)r, %(pkg)r, %(tests)r]
import numpy as np, torch
from b200pc import _lib, ops
import prune_geometry as PG
assert _lib.LIB_PATH.endswith("libb200pc_bounds.so"), _lib.LIB_PATH
os.environ.update(B200PC_SMALL_PATH="0", B200PC_GRID="4")
ops.reload_tuning()
dev = torch.device("cuda:0")
t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
for name in PG.FAMILIES:
    ref, qry = PG.batch((name, name), 0, 3000, 600)
    for form in (0, 1, 2):
        ops.knn_search(t(ref), t(qry), 16, form, want_dist=True); ops.knn_search_i32(t(ref), t(qry), 16, form)
ref, qry = PG.mixed(0)
ops.knn_search(t(ref), t(qry), 16, 0, want_dist=True)
for k in %(ks)r:
    ref, qry = PG.family("ground_objects", k, max(2000, k + 300), 300)
    ops.knn_search(t(ref[None]), t(qry[None]), k, 0, want_dist=True)
for nf in %(edges)r:
    ref, qry = PG.family("lattice", nf, nf, 33)
    ops.knn_search(t(ref[None]), t(qry[None]), min(16, nf), 2, want_dist=True)
ref, qry = PG.batch([PG.FAMILIES[i] for i in range(10)], 7, 4097, 300)
ops.knn_ragged(t(ref), t(qry), 16, 0, t(np.array(%(edges)r)), t(np.array([1, 31, 32, 33, 300, 299, 64, 0, 257, 100])), want_dist=True)
torch.cuda.synchronize()
print("pruned bounds ok")
"""


@gpu
def test_stress_cases_under_the_bounds_checked_build():
    lib = os.path.join(PKG, "b200pc", "libb200pc_bounds.so")
    assert os.path.exists(lib), "libb200pc_bounds.so is not built (make -C point-cloud-interpolation-_b200 bounds)"
    ks = sorted(set(K_FOR_WARPS.values()) | {1, 2, 3, 4, 7, 9, 17, 31, 33, 65, 127, 255, 256, 876})
    code = BOUNDS_SCRIPT % {"root": ROOT, "pkg": PKG, "tests": os.path.dirname(os.path.abspath(__file__)), "ks": ks,
                            "edges": EDGE_COUNTS}
    p = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, B200PC_LIBRARY="bounds"), capture_output=True, text=True,
                       timeout=900)
    out = p.stdout + p.stderr
    assert "device assert failed" not in out, out[-4000:]
    assert p.returncode == 0 and "pruned bounds ok" in out, out[-4000:]
