"""NaN and +-inf coordinates through every search path and every entry that consumes a search, against the strict oracle.

The rule (include/b200pc.h, "Non-finite coordinates"): a (query, ref) pair is a top-k candidate only if its distance is
finite.  A row holds its candidates in ascending (distance, index) order, then -1 with distance +inf.  It must hold on
the warp-per-query kernel (int64 entries, N <= 1024), on the streaming kernel in every grid mode and forced plan, and for
both index widths.  Each test forces its path through the B200PC_* knobs and reads back the plan that ran (Knobs, from
test_gpu_plans.py), so a knob that did not take effect fails the test.

Bar: indices and distance bits equal to oracle/strict on every row.  Where a NaN is computed (weights of a row without
neighbours, features of a -1 slot, square_distance) the NaN positions must be equal: the payload of a generated NaN
differs between the host and the device.  FPS picks are also checked against oracle/ref_torch's loop, which is the
reference's own algorithm."""
import functools

import numpy as np
import pytest
import torch

from b200pc import ops, pointnet2_utils as P, pytorch3d_shim as S3, synth
from oracle import ref_torch, strict
from test_gpu_backward import _assert_within, _scatter64
from test_gpu_plans import GRID_NAME, Knobs, expect, topk_order

pytestmark = pytest.mark.gpu

NAN, INF = np.float32(np.nan), np.float32(np.inf)


@pytest.fixture
def knobs(cuda_dev, monkeypatch, capfd):
    return Knobs(monkeypatch, capfd)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def _same(got, want, what=""):
    """NaN exactly where want has NaN, every other element bit for bit"""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    np.testing.assert_array_equal(np.isnan(got), np.isnan(want), err_msg=what)
    keep = ~np.isnan(want)
    np.testing.assert_array_equal(_bits(got)[keep], _bits(want)[keep], err_msg=what)


def _spoil(ref, b, rows):
    """make the given refs non-finite, cycling through NaN in all or one coordinate, +inf, -inf and mixed infinities"""
    for j, n in enumerate(rows):
        c = j % 5
        if c == 0:
            ref[b, n] = NAN
        elif c == 1:
            ref[b, n, 1] = NAN
        elif c == 2:
            ref[b, n, 0] = INF
        elif c == 3:
            ref[b, n, 2] = -INF
        else:
            ref[b, n] = [INF, -INF, 1.0]


BAD_QUERIES = [[INF, 0, 0], [-INF, 0, 0], [0, INF, 0], [0, 0, -INF], [NAN, 0, 0], [NAN, NAN, NAN], [INF, INF, INF],
               [-INF, -INF, -INF], [INF, -INF, NAN], [1.0, 2.0, INF]]


def _mixed(rng, B, n):
    """mixed-sign coordinates, a few refs with x = 0 (the (+inf, 0, 0) query gives them a NaN distance)"""
    p = (rng.normal(size=(B, n, 3)) * 4).astype(np.float32)
    p[:, 1:4, 0] = 0.0
    return p


@functools.lru_cache(maxsize=None)
def _case(name, N):
    """(ref [B,N,3], qry [B,S,3], k) of one non-finite case at N refs"""
    rng = np.random.default_rng(N + len(name))
    ref, qry, k = _mixed(rng, 1, N), _mixed(rng, 1, 40), 16
    tiles = -(-N // 512)
    if name == "few":                  # a few NaN and +-inf refs, k below the finite count
        _spoil(ref, 0, [3, 10, 20, 21, 22, 23, 24, 25, N // 2, N - 1])
    elif name == "k_above":            # 8 finite refs, k = 16: every row ends in -1 slots
        _spoil(ref, 0, rng.permutation(N)[8:])
    elif name == "bad_queries":        # one or three coordinates NaN / +inf / -inf, including (+inf, 0, 0) (x > 0, < 0 and = 0 refs)
        qry[0, :len(BAD_QUERIES)] = BAD_QUERIES
        _spoil(ref, 0, [7, N - 2])
    elif name == "dead_item":          # batch item 0: every ref non-finite (and the grid's bounding box empty); item 1: normal
        ref, qry = _mixed(rng, 2, N), _mixed(rng, 2, 40)
        _spoil(ref, 0, range(N))
        k = 8
    elif name == "range":              # every non-finite ref in one tile of the strided order: a whole split range
        _spoil(ref, 0, range(1, N, tiles))
    elif name == "last_tile":          # every ref of the last tile of the natural order, ending at ref N-1
        _spoil(ref, 0, range(512 * (tiles - 1), N))
    elif name == "ties":               # grid-snapped coordinates (exact arithmetic, many equal distances) plus NaN refs
        ref = synth.grid_snapped(N, 1, N, span=4).copy()
        qry = synth.grid_snapped(N + 1, 1, 40, span=4)
        ref[0, 5::11] = NAN
    else:                              # finite clouds at +-2^61: every pair is still a candidate
        assert name == "huge"
        ref = (rng.uniform(-1, 1, size=(1, N, 3)) * 2.0 ** 61).astype(np.float32)
        qry = (rng.uniform(-1, 1, size=(1, 40, 3)) * 2.0 ** 61).astype(np.float32)
    return np.ascontiguousarray(ref), np.ascontiguousarray(qry), k


CASES = ["few", "k_above", "bad_queries", "dead_item", "range", "last_tile", "ties", "huge"]


@functools.lru_cache(maxsize=None)
def _oracle(name, N, form):
    ref, qry, k = _case(name, N)
    return strict.knn(ref, qry, k, form)


# ---- the path matrix ---------------------------------------------------------------------------------------------------
PATHS = {
    "small": dict(SMALL_PATH=1, GRID=0),
    "stream": dict(SMALL_PATH=0, GRID=0),
    "grid2": dict(SMALL_PATH=0, GRID=2),
    "grid3": dict(SMALL_PATH=0, GRID=3),
    "split2": dict(SMALL_PATH=0, GRID=0, FORCE_SPLIT=2),
    "split4": dict(SMALL_PATH=0, GRID=0, FORCE_SPLIT=4),
    "filter0": dict(SMALL_PATH=0, GRID=0, FILTER=0),
    "q2": dict(SMALL_PATH=0, GRID=0, FORCE_Q=2),
    "natural0": dict(SMALL_PATH=0, GRID=0, NATURAL_ORDER=0),
    "natural1": dict(SMALL_PATH=0, GRID=0, NATURAL_ORDER=1),
}


def _path_n(path):
    return 2000 if path == "split4" else 1000       # 4 tiles for four ranges; otherwise N <= 1024 (the small path's limit)


def _want(path, form):
    """plan fields of the streaming call of this path (the int32 entry of the small path included)"""
    env = dict(PATHS[path])
    if path == "small":
        env = dict(GRID=0)
    nat = env.get("NATURAL_ORDER")
    want = dict(grid=GRID_NAME[env["GRID"]], filter="broadcast" if env.get("FILTER") == 0 else "lane",
                order=topk_order(form, env["GRID"], None if nat is None else bool(nat)), mode=0)
    if "FORCE_SPLIT" in env:
        want["split"] = env["FORCE_SPLIT"]
    if "FORCE_Q" in env:
        want["q"] = env["FORCE_Q"]
    return want


def knn_i32_with_dist(ref, qry, k, form):
    """b200pc_knn_i32 with its distance output (the facade returns the indices only)"""
    from b200pc import _lib
    B, N, _ = ref.shape; S = qry.shape[1]
    dev = ref.device
    idx = torch.empty(B, S, k, dtype=torch.int32, device=dev)
    dist = torch.empty(B, S, k, dtype=torch.float32, device=dev)
    lib = _lib.load()
    nws = ops._search_ws(lib, B, N, S, k)
    ws = ops._workspace(nws, dev)
    ops._call(dev, lib.b200pc_knn_i32, ops._ptr(ref), ops._ptr(qry), B, N, S, k, int(form), ops._ptr(idx), ops._ptr(dist),
              ops._ptr(ws), nws, ops._stream(dev))
    return idx, dist


@pytest.mark.parametrize("form", [0, 1, 2])
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("path", list(PATHS))
def test_topk_every_path_matches_oracle(knobs, cuda_dev, path, case, form):
    N = _path_n(path)
    ref, qry, k = _case(case, N)
    oi, od = _oracle(case, N, form)
    if case == "huge":
        assert (oi >= 0).all() and np.isfinite(od).all()
    if case == "k_above":
        assert (oi[..., 8:] == -1).all() and (od[..., 8:] == np.inf).all()
    knobs.set(**PATHS[path])
    r, q = _t(ref, cuda_dev), _t(qry, cuda_dev)
    (idx, dist), plans, _ = knobs.run(lambda: ops.knn_search(r, q, k, form, want_dist=True))
    want = _want(path, form)
    if path == "small":
        assert plans == [], plans                     # the warp-per-query kernel prints no streaming plan
    else:
        expect(plans, 1, **want)
    (i32, d32), plans, _ = knobs.run(lambda: knn_i32_with_dist(r, q, k, form))
    expect(plans, 1, **want)                          # the int32 entry always streams
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))
    np.testing.assert_array_equal(i32.cpu().numpy(), oi.astype(np.int32))
    np.testing.assert_array_equal(_bits(d32.cpu().numpy()), _bits(od))


# ---- entries through their facades, on the small and the streaming path ---------------------------------------------
@functools.lru_cache(maxsize=None)
def _cloud(seed, B, N, S):
    """refs and queries with a fifth of the points non-finite, the bad queries above, and (B > 1) a last batch item whose
    refs keep only two finite points (fewer than three-NN needs)"""
    rng = np.random.default_rng(seed)
    ref, qry = _mixed(rng, B, N), _mixed(rng, B, S)
    for b in range(B):
        _spoil(ref, b, rng.choice(N, size=N // 5, replace=False))
        _spoil(qry, b, rng.choice(np.arange(len(BAD_QUERIES), S), size=S // 10, replace=False))
    qry[:, :len(BAD_QUERIES)] = BAD_QUERIES
    if B > 1:
        _spoil(ref, B - 1, range(2, N))
    return ref, qry


SMALL = pytest.mark.parametrize("small", [1, 0], ids=["small", "stream"])


def _plans_per_search(small):
    return 0 if small else 1


@SMALL
def test_knn_point_and_knn_points(knobs, cuda_dev, small):
    ref, qry = _cloud(1, 2, 900, 300)
    knobs.set(SMALL_PATH=small, GRID=0)
    r, q = _t(ref, cuda_dev), _t(qry, cuda_dev)
    idx, plans, _ = knobs.run(lambda: P.knn_point(16, r, q))
    assert len(plans) == _plans_per_search(small)
    np.testing.assert_array_equal(idx.cpu().numpy(), strict.knn_point(16, ref, qry))
    knn, plans, _ = knobs.run(lambda: S3.knn_points(q, r, K=12))
    assert len(plans) == _plans_per_search(small)
    od, oi = strict.knn_points(qry, ref, 12)
    np.testing.assert_array_equal(knn.idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(knn.dists.cpu().numpy()), _bits(od))


@SMALL
@pytest.mark.parametrize("variant", [0, 1])
def test_three_nn_weights_and_feature_propagation(knobs, cuda_dev, small, variant):
    known, dense = _cloud(2, 2, 700, 500)
    feat = np.random.default_rng(3).normal(size=(2, 700, 12)).astype(np.float32)
    knobs.set(SMALL_PATH=small, GRID=0)
    u, kn, f = _t(dense, cuda_dev), _t(known, cuda_dev), _t(feat, cuda_dev)
    (d, i, w), plans, _ = knobs.run(lambda: ops.three_nn(u, kn, variant=variant))
    assert len(plans) == _plans_per_search(small)
    od, oi = strict.three_nn(dense, known)
    ow = strict.three_weights(od, variant)
    assert (oi[1] == -1).any() and (oi == -1).all(-1).any()         # rows with one and with no neighbour
    np.testing.assert_array_equal(i.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(d.cpu().numpy()), _bits(od))
    _same(w.cpu().numpy(), ow, "weights")
    # feature propagation = three-NN, then interpolate, where -1 wraps once to the last known point
    (out, fi, fw), plans, _ = knobs.run(lambda: torch.ops.b200pc.feature_propagation(u, kn, f, variant))
    assert len(plans) == _plans_per_search(small)
    assert torch.equal(fi, i)
    _same(fw.cpu().numpy(), w.cpu().numpy(), "feature_propagation weights")
    _same(out.cpu().numpy(), ops.three_interpolate(f, i, w).cpu().numpy(), "feature_propagation vs composition")
    _same(out.cpu().numpy(), strict.three_interpolate(feat, oi, ow), "feature_propagation vs oracle")


@SMALL
def test_fusion_group(knobs, cuda_dev, small):
    ref, qry = _cloud(4, 2, 800, 200)
    feat = np.random.default_rng(5).normal(size=(2, 800, 5)).astype(np.float32)
    knobs.set(SMALL_PATH=small, GRID=0)
    r, q, f = _t(ref, cuda_dev), _t(qry, cuda_dev), _t(feat, cuda_dev)
    (resi, nn, gf, idx), plans, _ = knobs.run(lambda: ops.fusion_group(q, r, 8, f))
    assert len(plans) == _plans_per_search(small)
    _, oi = strict.knn_points(qry, ref, 8)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    assert (oi[:, :len(BAD_QUERIES)] == -1).all()
    # the unfused composition on the slots that have a neighbour; a -1 slot (every slot of a non-finite query) is NaN
    ok = oi >= 0
    safe = np.where(ok, oi, 0)
    want_nn = np.where(ok[..., None], strict.index_points(ref, safe), NAN)
    with np.errstate(invalid="ignore"):
        d = (want_nn - qry[:, :, None, :]).astype(np.float32)
        n2 = ((d[..., 0] * d[..., 0]).astype(np.float32) + (d[..., 1] * d[..., 1]).astype(np.float32)).astype(np.float32)
        n2 = (n2 + (d[..., 2] * d[..., 2]).astype(np.float32)).astype(np.float32)
    want_resi = np.concatenate([d, np.sqrt(n2)[..., None]], -1)
    want_gf = np.where(ok[..., None], strict.index_points(feat, safe), NAN)
    _same(nn.cpu().numpy(), want_nn.transpose(0, 3, 1, 2), "nn")
    _same(resi.cpu().numpy(), want_resi.transpose(0, 3, 1, 2), "resi")
    _same(gf.cpu().numpy(), want_gf.transpose(0, 3, 1, 2), "grouped features")
    assert np.isnan(nn.cpu().numpy()[:, :, :len(BAD_QUERIES)]).all()


def _chamfer_grad_ref(x, y, ix, iy, scale):
    """float64 gradient of scale * loss with the kernel's nearest-neighbour choice; a point with index -1 gives and takes
    no term"""
    B, N, _ = x.shape; M = y.shape[1]
    x64, y64 = x.astype(np.float64), y.astype(np.float64)
    bn = np.arange(B)[:, None]
    with np.errstate(invalid="ignore"):
        tx = 2.0 * scale / (B * N) * (x64 - y64[bn, np.maximum(ix, 0)])
        ty = 2.0 * scale / (B * M) * (y64 - x64[bn, np.maximum(iy, 0)])
    fx = (bn * N + np.arange(N)[None]).reshape(-1)
    fy = (bn * M + np.arange(M)[None]).reshape(-1)
    ixf = np.where(ix >= 0, ix + bn * M, -1).reshape(-1)
    iyf = np.where(iy >= 0, iy + bn * N, -1).reshape(-1)
    own_x, own_y = np.where(ix >= 0, fx.reshape(B, N), -1).reshape(-1), np.where(iy >= 0, fy.reshape(B, M), -1).reshape(-1)
    tx, ty = np.nan_to_num(tx.reshape(-1, 3)), np.nan_to_num(ty.reshape(-1, 3))      # rows of -1 points are dropped anyway
    sx = _scatter64(B * N, np.concatenate([own_x, iyf]), np.concatenate([tx, -ty]))
    sy = _scatter64(B * M, np.concatenate([own_y, ixf]), np.concatenate([ty, -tx]))
    return sx, sy


@SMALL
def test_chamfer_forward_and_backward(knobs, cuda_dev, small):
    x_np, y_np = _cloud(6, 2, 600, 500)                  # M <= 1024 and B * N <= 4096: the small path serves it by default
    knobs.set(SMALL_PATH=small, GRID=0)
    x = _t(x_np, cuda_dev).requires_grad_(True); y = _t(y_np, cuda_dev).requires_grad_(True)
    (loss, dx, ix, dy, iy), plans, _ = knobs.run(lambda: ops.chamfer(x, y))
    assert len(plans) == 2 * _plans_per_search(small)
    ol, odx, oix, ody, oiy = strict.chamfer(x_np, y_np)
    np.testing.assert_array_equal(ix.cpu().numpy(), oix)
    np.testing.assert_array_equal(iy.cpu().numpy(), oiy)
    np.testing.assert_array_equal(_bits(dx.detach().cpu().numpy()), _bits(odx))
    np.testing.assert_array_equal(_bits(dy.detach().cpu().numpy()), _bits(ody))
    assert ol == np.inf and loss.item() == np.inf           # a point without a candidate adds +inf
    (loss * 3.5).backward()
    (sx, ax, mx), (sy, ay, my) = _chamfer_grad_ref(x_np, y_np, oix, oiy, 3.5)
    gx, gy = x.grad.cpu().numpy().reshape(-1, 3), y.grad.cpu().numpy().reshape(-1, 3)
    fin_x, fin_y = np.isfinite(x_np).all(-1).reshape(-1), np.isfinite(y_np).all(-1).reshape(-1)
    assert np.isfinite(gx[fin_x]).all() and np.isfinite(gy[fin_y]).all()
    assert (gx[~fin_x] == 0).all() and (gy[~fin_y] == 0).all()       # no gradient into a point without a candidate
    _assert_within(gx[fin_x], sx[fin_x], ax[fin_x], mx[fin_x], k=4, what="gx")
    _assert_within(gy[fin_y], sy[fin_y], ay[fin_y], my[fin_y], k=4, what="gy")


@SMALL
def test_chamfer_of_finite_clouds_at_large_scale(knobs, cuda_dev, small):
    x_np, y_np, _ = _case("huge", 1000)
    knobs.set(SMALL_PATH=small, GRID=0)
    loss, dx, ix, dy, iy = ops.chamfer(_t(x_np, cuda_dev), _t(y_np, cuda_dev))
    ol, odx, oix, ody, oiy = strict.chamfer(x_np, y_np)
    assert np.isfinite(ol) and abs(loss.item() - ol) <= 1e-5 * ol
    np.testing.assert_array_equal(ix.cpu().numpy(), oix)
    np.testing.assert_array_equal(iy.cpu().numpy(), oiy)


@pytest.mark.parametrize("split", [None, 2])
def test_rebuild_pack_minus_one_record_holds_nan(knobs, cuda_dev, split):
    ref, qry = _cloud(7, 2, 1000, 300)
    knobs.set(FORCE_SPLIT=split, GRID=0)
    rec, plans, _ = knobs.run(lambda: ops.rebuild_pack(_t(ref, cuda_dev), _t(qry, cuda_dev)))
    expect(plans, 1, split=split)
    idx, nn = ops.unpack_rebuild(rec)
    _, oi = strict.knn_points(qry, ref, 1)
    oi = oi[..., 0]
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    want = np.where((oi >= 0)[..., None], strict.index_points(ref, np.maximum(oi, 0)), NAN)
    assert (oi == -1).any()
    _same(nn.cpu().numpy(), want, "rebuild records")


@pytest.mark.parametrize("split", [None, 3])
@pytest.mark.parametrize("small", [1, 0], ids=["small", "stream"])
def test_ball_query(knobs, cuda_dev, small, split):
    N = 6000 if split else 900                          # 12 tiles for a forced split; N <= 1024 for the small path
    ref, qry = _cloud(8, 2, N, 300)
    knobs.set(SMALL_PATH=small, FORCE_SPLIT=split)
    out, plans, _ = knobs.run(lambda: P.query_ball_point(1.5, 16, _t(ref, cuda_dev), _t(qry, cuda_dev)))
    if small and not split:
        assert plans == []
    else:
        expect(plans, 1, split=split, mode=1)
    want = strict.query_ball_point(1.5, 16, ref, qry)
    np.testing.assert_array_equal(out.cpu().numpy(), want)
    assert (want[:, :len(BAD_QUERIES)] == N).all()


# ---- FPS ---------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _fps_cloud(N, start_kind):
    """item 0: +-1e30 points among finite ones (their squared distances overflow to +inf, so only their own pick lowers
    their minimum); item 1: NaN and +-inf points spread over the cloud (their minimum stays 1e10 for good, so the lowest
    index of them is picked again and again).  start: finite, or a 1e30 / NaN point."""
    a, _ = synth.batch_pairs(81, 2, N)
    a = a.copy()
    a[0, 50] = 1e30; a[0, N // 3, 1] = -1e30; a[0, N - 7, 2] = 1e30; a[0, N - 2] = -1e30
    _spoil(a, 1, range(17, N, N // 12))
    start = np.array([5, 9]) if start_kind == "finite" else np.array([N // 3, 17])
    want = strict.farthest_point_sample(a, 200, start)
    np.testing.assert_array_equal(want, ref_torch.fps(torch.from_numpy(a), 200, torch.from_numpy(start)).numpy())
    return a, start, want


FPS_CASES = [(N, C) for N in (3000, 20000) for C in (1, 2, 4, 8, 16) if C * 8192 >= N]


@pytest.mark.parametrize("start_kind", ["finite", "non_finite"])
@pytest.mark.parametrize("flat", [0, 1])
@pytest.mark.parametrize("N,C", FPS_CASES)
def test_fps_clusters(knobs, cuda_dev, N, C, flat, start_kind):
    cloud, start, want = _fps_cloud(N, start_kind)
    knobs.set(FPS_CLUSTER=C, FPS_FLAT=flat)
    out, _, fplans = knobs.run(lambda: ops.fps(_t(cloud, cuda_dev), 200, _t(start, cuda_dev)))
    assert len(fplans) == 1 and (int(fplans[0]["C"]), fplans[0]["exchange"]) == (C, "flat" if flat else "two-level"), fplans
    np.testing.assert_array_equal(out.cpu().numpy(), want)


# ---- square_distance, channel_max --------------------------------------------------------------------------------------
def test_square_distance(cuda_dev):
    ref, qry = _cloud(9, 2, 500, 300)
    got = P.square_distance(_t(qry, cuda_dev), _t(ref, cuda_dev)).cpu().numpy()
    want = strict.square_distance(qry, ref)
    assert np.isnan(want).any() and np.isinf(want).any()
    _same(got, want, "square_distance")


@pytest.mark.parametrize("C", [4, 132])
def test_channel_max(cuda_dev, C):
    from b200pc import _lib
    rows = 16 * _lib.load().b200pc_device_sm_count() * 8 * 2 + 37        # more rows than one pass of the grid-stride loop
    x = np.random.default_rng(C).uniform(0.5, 2.0, size=(rows, C)).astype(np.float32) * np.where(np.arange(C) % 2, 1, -1).astype(np.float32)
    x[0] = -INF                                          # only -inf
    x[1, ::2] = INF; x[1, 1::2] = -INF                   # +-inf mixed
    x[2, -1] = NAN                                       # NaN only in the last float4
    x[3, 124 if C > 4 else 0] = NAN                      # NaN only in lane 31's slice (C = 132: float4 #31)
    x[4, :] = -INF; x[4, C // 2] = INF
    x[5, :] = NAN
    x[rows - 1, -2] = NAN; x[rows - 2] = -INF            # in the last pass of the grid-stride loop
    got = ops.channel_max(_t(x, cuda_dev)).cpu().numpy()
    want = torch.from_numpy(x).max(dim=1)[0].numpy()
    _same(got, want, "channel_max")
