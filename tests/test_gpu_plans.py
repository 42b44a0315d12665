"""Every launch plan of the streaming search and of FPS, forced through the B200PC_* knobs, against the strict oracle.

The planner picks, per call, a ref split (the reference range divided over gridDim.z, partial lists combined by
merge_topk_kernel / merge_ball_kernel), the warps per CTA, the queries per thread, the filter and the ref order; FPS picks
a cluster size and an exchange.  Which plan the default picks depends on the shape and on the SM count, so these tests
force each plan and read back, from the B200PC_DEBUG_PLAN=1 line on stderr, the plan that actually ran: a knob that did
not take effect fails the test instead of quietly comparing the default plan with itself.

Bar: top-k indices and distances (as int32 bits) and ball indices bit-exact against oracle/strict on every row; both the
int64 and the int32 search entries, because the merge writes idx, idx32 and dist.
"""
import functools
import re

import numpy as np
import pytest
import torch

from b200pc import ops, pointnet2_utils as P, synth
from oracle import strict

pytestmark = pytest.mark.gpu

TILE, MAX_SPLIT, FPS_CTA_POINTS = 512, 32, 8192      # search.cu TILE / MAX_SPLIT; fps.cu FPS_T * 16 points per CTA

PLAN = re.compile(r"b200pc plan: B=(?P<B>\d+) N=(?P<N>\d+) S=(?P<S>\d+) k=(?P<k>\d+) mode=(?P<mode>\d+) -> (?P<warps>\d+) warps/CTA, "
                  r"(?P<qpc>\d+) queries/CTA, ref split (?P<split>\d+) \((?P<tps>\d+) tiles each\), grid (?P<grid>\w+), "
                  r"filter (?P<filter>\w+), order (?P<order>\w+), ")
FPS_PLAN = re.compile(r"b200pc fps plan: B=(?P<B>\d+) N=(?P<N>\d+) npoint=(?P<npoint>\d+) -> cluster (?P<C>\d+), "
                      r"(?P<P>\d+) points/thread, exchange (?P<exchange>[\w-]+)")
GRID_NAME = {0: "off", 2: "thresholds", 3: "sorted"}


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


def forced_split(N, f):
    """(ranges, tiles per range) the planner must use for B200PC_FORCE_SPLIT=f: f clamped to the tile count and to the
    32 lists of one merge warp, then ceil(tiles / ceil(tiles / f)) ranges"""
    tiles = -(-N // TILE)
    f = min(f, tiles, MAX_SPLIT)
    tps = -(-tiles // f)
    return -(-tiles // tps), tps


def topk_order(form, grid=0, natural=None):
    if grid == 3:
        return "cell"
    if natural is not None:
        return "natural" if natural else "strided"
    return "natural" if form == 1 else "strided"


class Knobs:
    """sets B200PC_* knobs (plus B200PC_DEBUG_PLAN=1), makes the library re-read them, runs a call and parses its plans"""

    def __init__(self, monkeypatch, capfd):
        self.mp, self.capfd = monkeypatch, capfd

    def set(self, **env):
        self.mp.setenv("B200PC_DEBUG_PLAN", "1")
        for name, v in env.items():
            if v is None:
                self.mp.delenv("B200PC_" + name, raising=False)
            else:
                self.mp.setenv("B200PC_" + name, str(v))
        ops.reload_tuning()

    def run(self, fn):
        torch.cuda.synchronize()
        self.capfd.readouterr()
        out = fn()
        torch.cuda.synchronize()
        err = self.capfd.readouterr().err
        return out, [m.groupdict() for m in PLAN.finditer(err)], [m.groupdict() for m in FPS_PLAN.finditer(err)]


@pytest.fixture
def knobs(cuda_dev, monkeypatch, capfd):
    return Knobs(monkeypatch, capfd)


def expect(plans, n=1, split=None, warps=None, q=None, **want):
    """every plan line matches; split = forced split value (checked against the ceil formula for that line's N)"""
    assert len(plans) == n, "expected %d search plan line(s), got %r" % (n, plans)
    for p in plans:
        if split is not None:
            ns, tps = forced_split(int(p["N"]), split)
            assert (int(p["split"]), int(p["tps"])) == (ns, tps), p
        if warps is not None:
            assert int(p["warps"]) == warps, p
        if q is not None:
            assert int(p["qpc"]) == 32 * q * int(p["warps"]), p
        for key, v in want.items():
            assert p[key] == str(v), (key, p)


@functools.lru_cache(maxsize=None)
def _pairs(seed, B, N, S):
    a, b = synth.batch_pairs(seed, B, max(N, S))
    return a[:, :N].copy(), b[:, :S].copy()


@functools.lru_cache(maxsize=None)
def _knn_oracle(seed, B, N, S, k, form):
    ref, qry = _pairs(seed, B, N, S)
    return strict.knn(ref, qry, k, form)


def _check_topk(knobs, dev, ref, qry, k, form, oi, od, n_plans=1, **want):
    r, q = _t(ref, dev), _t(qry, dev)
    (idx, dist), plans, _ = knobs.run(lambda: ops.knn_search(r, q, k, form, want_dist=True))
    expect(plans, n_plans, **want)
    i32, plans, _ = knobs.run(lambda: ops.knn_search_i32(r, q, k, form))
    expect(plans, n_plans, **want)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))
    assert i32.dtype == torch.int32
    np.testing.assert_array_equal(i32.cpu().numpy(), oi.astype(np.int32))


# ---- C.1: split matrix, top-k ----------------------------------------------------------------------------------------
SPLIT_CASES = [
    # ((B, N, S, k), forced split)
    ((1, 513, 77, 300), 2),        # 2 tiles: every range holds fewer than k refs (partial lists end in sentinels)
    ((2, 2048, 333, 600), 2),      # 4 tiles, k > 512 refs per range
    ((2, 2048, 333, 600), 3),      # -> 2 ranges of 2 tiles
    ((2, 2048, 333, 600), 4),
    ((1, 5000, 700, 16), 3),       # 10 tiles: 4+4+2
    ((1, 5000, 700, 16), 4),       # 3+3+3+1
    ((1, 5000, 700, 16), 5),       # 5 ranges of 2 (not in the planner's own 1, 2, 3, 4, 8, ... sequence)
    ((1, 5000, 700, 16), 7),       # 5 ranges of 2
    ((1, 5000, 700, 16), 8),       # 5 ranges of 2
    ((2, 16384, 1024, 16), 32),    # 32 tiles: one tile per range
    ((1, 20000, 300, 64), 32),     # 40 tiles -> 20 ranges of 2
    ((1, 20000, 300, 64), 40),     # clamped to the 32 lists of a merge warp -> 20 ranges of 2
]


@pytest.mark.parametrize("grid", [0, 2, 3])
@pytest.mark.parametrize("form", [0, 1, 2])
@pytest.mark.parametrize("shape,split", SPLIT_CASES, ids=["%dx%dx%dx%d-split%d" % (s + (f,)) for s, f in SPLIT_CASES])
def test_forced_split_topk_matches_oracle(knobs, cuda_dev, shape, split, form, grid):
    B, N, S, k = shape
    knobs.set(SMALL_PATH=0, GRID=grid, FORCE_SPLIT=split)
    assert forced_split(N, split)[0] > 1
    ref, qry = _pairs(40, B, N, S)
    oi, od = _knn_oracle(40, B, N, S, k, form)
    _check_topk(knobs, cuda_dev, ref, qry, k, form, oi, od, split=split, grid=GRID_NAME[grid], filter="lane",
                order=topk_order(form, grid), mode=0)


@pytest.mark.parametrize("grid", [0, 3])
@pytest.mark.parametrize("form", [0, 1, 2])
@pytest.mark.parametrize("split", [2, 3, 5])
def test_forced_split_ties_merge_by_index(knobs, cuda_dev, split, form, grid):
    # grid-snapped coordinates: exact arithmetic, many equal distances, so equal keys from different ranges must merge by index
    ref = synth.grid_snapped(7, 2, 3000, span=6)
    qry = synth.grid_snapped(8, 2, 500, span=6)
    knobs.set(SMALL_PATH=0, GRID=grid, FORCE_SPLIT=split)
    oi, od = strict.knn(ref, qry, 16, form)
    assert (od[:, :, 1:] == od[:, :, :-1]).any(-1).mean() > 0.5
    _check_topk(knobs, cuda_dev, ref, qry, 16, form, oi, od, split=split, grid=GRID_NAME[grid], order=topk_order(form, grid))


# ---- C.2: split matrix, ball query -----------------------------------------------------------------------------------
BALL_N = 6000          # 12 tiles: splits 2, 3, 8 give ranges of 6, 4 and 2 tiles


@functools.lru_cache(maxsize=None)
def _x_sorted_cloud(kind):
    """a cloud sorted along x, so that index ranges are slabs of space"""
    rng = np.random.default_rng(61)
    if kind == "line":            # a thin rod along x: one ref per 0.01 on average
        x = np.sort(rng.uniform(0.0, 60.0, BALL_N))
        c = np.stack([x, rng.uniform(0, 0.01, BALL_N), rng.uniform(0, 0.01, BALL_N)], -1)
    else:                          # a synthetic scan, sorted along x
        a, _ = synth.batch_pairs(62, 1, BALL_N)
        c = a[0][np.argsort(a[0][:, 0], kind="stable")]
    return c[None].astype(np.float32)


def _ball_queries(cloud, radius):
    """queries placed so that, for every tile boundary t*512, the ball's left edge sits m refs before it (m = 0, 1, 16, 64):
    a ball that fills nsample partway through the range after a boundary; plus balls at the far end (hits only in the last
    range), random refs, and one far outside the cloud (empty ball)"""
    x = cloud[0, :, 0]
    yz = cloud[0, :, 1:].mean(0)
    q = []
    for t in range(1, BALL_N // TILE + 1):
        for m in (0, 1, 16, 64):
            q.append([x[t * TILE - m] + radius, yz[0], yz[1]])
    q += [cloud[0, -1], cloud[0, -3], cloud[0, BALL_N // 2], [x[-1] + 1e4, 0, 0]]
    q += list(cloud[0, np.random.default_rng(63).integers(0, BALL_N, 40)])
    return np.asarray(q, np.float32)[None]


@pytest.mark.parametrize("split", [2, 3, 8])
@pytest.mark.parametrize("nsample", [1, 32, 128])
@pytest.mark.parametrize("radius", [1e-4, 0.05, 1.0, 1e3])        # (mostly) empty balls ... every ref in the ball
@pytest.mark.parametrize("kind", ["line", "scan"])
def test_forced_split_ball_query_matches_oracle(knobs, cuda_dev, kind, radius, nsample, split):
    cloud = _x_sorted_cloud(kind)
    qry = _ball_queries(cloud, radius)
    knobs.set(FORCE_SPLIT=split)
    out, plans, _ = knobs.run(lambda: ops.ball_query(radius, nsample, _t(cloud, cuda_dev), _t(qry, cuda_dev)))
    expect(plans, split=split, grid="off", order="natural", mode=1)
    exp = strict.query_ball_point(radius, nsample, cloud, qry)
    np.testing.assert_array_equal(out.cpu().numpy(), exp)
    if radius == 1e-4:
        assert (exp == BALL_N).any()                      # the sentinel N of an empty ball went through the merge
    if radius == 1e3:                                     # every query inside the cloud: range 0 filled its ball alone
        assert (exp[0, :, -1] == nsample - 1).sum() >= 40


# ---- C.3 / C.4: warps per CTA and queries per thread ------------------------------------------------------------------
WARP_OPS = [("topk", 0, {}), ("topk", 2, {}), ("ball", None, {}),
            ("topk", 0, {"GRID": 3, "INTERLEAVE": 1}), ("topk", 2, {"GRID": 3, "INTERLEAVE": 1})]
WARP_IDS = ["topk-form0", "topk-form2", "ball", "topk-form0-cell-interleaved", "topk-form2-cell-interleaved"]


def _run_op(knobs, dev, op, form, ref, qry, k, radius=1.0):
    """one forced call (both index widths for top-k) against the oracle; returns the plans of the calls"""
    r, q = _t(ref, dev), _t(qry, dev)
    if op == "ball":
        out, plans, _ = knobs.run(lambda: ops.ball_query(radius, k, r, q))
        np.testing.assert_array_equal(out.cpu().numpy(), strict.query_ball_point(radius, k, ref, qry))
        return plans
    (idx, dist), plans, _ = knobs.run(lambda: ops.knn_search(r, q, k, form, want_dist=True))
    i32, plans32, _ = knobs.run(lambda: ops.knn_search_i32(r, q, k, form))
    oi, od = strict.knn(ref, qry, k, form)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    np.testing.assert_array_equal(_bits(dist.cpu().numpy()), _bits(od))
    np.testing.assert_array_equal(i32.cpu().numpy(), oi.astype(np.int32))
    return plans + plans32


@pytest.mark.parametrize("op,form,env", WARP_OPS, ids=WARP_IDS)
@pytest.mark.parametrize("S", [33, 777, 4100])                   # the last CTA has whole warps without a query
@pytest.mark.parametrize("warps", [1, 2, 5, 14])
@pytest.mark.parametrize("q", [1, 2])
def test_forced_warps_and_queries_per_thread(knobs, cuda_dev, q, warps, S, op, form, env):
    ref, qry = _pairs(41, 1, 3000, S)
    knobs.set(SMALL_PATH=0, FORCE_WARPS=warps, FORCE_Q=q, **env)
    plans = _run_op(knobs, cuda_dev, op, form, ref, qry, 16 if op == "topk" else 32)
    want = {"grid": "sorted", "order": "cell"} if env else {"order": "natural" if op == "ball" else "strided"}
    expect(plans, 2 if op == "topk" else 1, warps=warps, q=q, filter="lane", **want)


@pytest.mark.parametrize("op,form,split", [("topk", 0, 4), ("topk", 2, 4), ("ball", None, 3)])
def test_forced_two_queries_per_thread_with_split(knobs, cuda_dev, op, form, split):
    ref, qry = _pairs(42, 1, 5000, 700)
    knobs.set(SMALL_PATH=0, GRID=0, FORCE_Q=2, FORCE_SPLIT=split)
    plans = _run_op(knobs, cuda_dev, op, form, ref, qry, 16)
    expect(plans, 2 if op == "topk" else 1, q=2, split=split)


def test_forced_two_queries_per_thread_that_cannot_fit_is_an_error(knobs, cuda_dev):
    # k = 600: 64 query lists do not fit in shared memory; the call must fail, not run as one query per thread
    ref, qry = _pairs(43, 1, 2048, 100)
    knobs.set(FORCE_Q=2)
    with pytest.raises(RuntimeError, match="FORCE_Q"):
        ops.knn_search_i32(_t(ref, cuda_dev), _t(qry, cuda_dev), 600, 0)


# ---- C.5: filter and ref order ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("split", [None, 4])
@pytest.mark.parametrize("knob", ["filter", "order"])
@pytest.mark.parametrize("form", [0, 1, 2])
def test_filter_and_order_knobs(knobs, cuda_dev, form, knob, split):
    ref, qry = _pairs(23, 1, 5000, 1500)
    natural = form != 1                     # the order that is NOT the form's default
    env = {"FILTER": 0} if knob == "filter" else {"NATURAL_ORDER": int(natural)}
    knobs.set(SMALL_PATH=0, GRID=0, FORCE_SPLIT=split, **env)
    oi, od = _knn_oracle(23, 1, 5000, 1500, 16, form)
    want = {"filter": "broadcast", "order": topk_order(form)} if knob == "filter" else \
           {"filter": "lane", "order": topk_order(form, natural=natural)}
    if split:
        want["split"] = split
    _check_topk(knobs, cuda_dev, ref, qry, 16, form, oi, od, **want)


# ---- C.6: fused entries under a forced split -------------------------------------------------------------------------
def _fused(dev, name):
    """(call, oracle check); the call returns a tuple of tensors"""
    ref, qry = _pairs(44, 2, 5000, 700)
    r, q = _t(ref, dev), _t(qry, dev)
    if name == "fusion_group":
        feat = np.random.default_rng(5).normal(size=(2, 5000, 3)).astype(np.float32)
        f = _t(feat, dev)

        def check(out):
            resi, nn, gf, idx = out
            od, oi = strict.knn_points(qry, ref, 16)
            np.testing.assert_array_equal(idx.cpu().numpy(), oi)
            want_nn = strict.index_points(ref, oi)
            np.testing.assert_array_equal(_bits(nn.cpu().numpy()), _bits(want_nn.transpose(0, 3, 1, 2)))
            want_resi = (want_nn - qry[:, :, None, :]).astype(np.float32)
            np.testing.assert_array_equal(_bits(resi[:, :3].cpu().numpy()), _bits(want_resi.transpose(0, 3, 1, 2)))
            np.testing.assert_array_equal(_bits(gf.cpu().numpy()), _bits(strict.index_points(feat, oi).transpose(0, 3, 1, 2)))
        return (lambda: ops.fusion_group(q, r, 16, f)), check, 1
    if name == "feature_propagation":
        dense, sparse = qry.copy(), ref                         # refs of the three-NN search: the 5000 "known" points
        feat = np.random.default_rng(6).normal(size=(2, 5000, 12)).astype(np.float32)
        args = (_t(dense, dev), r, _t(feat, dev), 0)

        def check(out):
            o, idx, w = out
            od, oi = strict.three_nn(dense, sparse)
            ow = strict.three_weights(od, 0)
            np.testing.assert_array_equal(idx.cpu().numpy(), oi)
            np.testing.assert_array_equal(_bits(w.cpu().numpy()), _bits(ow))
            np.testing.assert_array_equal(_bits(o.cpu().numpy()), _bits(strict.three_interpolate(feat, oi, ow)))
        return (lambda: torch.ops.b200pc.feature_propagation(*args)), check, 1
    if name == "chamfer":
        x, y = ref, _pairs(45, 2, 4600, 10)[0]                  # 10 and 9 tiles: both searches split
        xt, yt = _t(x, dev), _t(y, dev)

        def check(out):
            loss, dx, ix, dy, iy = out
            ol, odx, oix, ody, oiy = strict.chamfer(x, y)
            np.testing.assert_array_equal(ix.cpu().numpy(), oix)
            np.testing.assert_array_equal(iy.cpu().numpy(), oiy)
            np.testing.assert_array_equal(_bits(dx.cpu().numpy()), _bits(odx))
            np.testing.assert_array_equal(_bits(dy.cpu().numpy()), _bits(ody))
            assert abs(loss.item() - ol) <= 1e-5 * abs(ol)
        return (lambda: ops.chamfer(xt, yt)), check, 2
    if name == "rebuild_pack":
        def check(out):
            idx, nn = ops.unpack_rebuild(out[0])
            od, oi = strict.knn_points(qry, ref, 1)
            np.testing.assert_array_equal(idx.cpu().numpy(), oi[..., 0])
            np.testing.assert_array_equal(_bits(nn.cpu().numpy()), _bits(strict.index_points(ref, oi)[:, :, 0]))
        return (lambda: (ops.rebuild_pack(r, q),)), check, 1
    assert name == "knn_point"

    def check(out):
        np.testing.assert_array_equal(out[0].cpu().numpy(), strict.knn_point(16, ref, qry))
    return (lambda: (P.knn_point(16, r, q),)), check, 1


@pytest.mark.parametrize("split", [3, 4])
@pytest.mark.parametrize("name", ["fusion_group", "feature_propagation", "chamfer", "rebuild_pack", "knn_point"])
def test_fused_entries_under_forced_split(knobs, cuda_dev, name, split):
    call, check, n_plans = _fused(cuda_dev, name)
    knobs.set(FORCE_SPLIT=None)
    want, _, _ = knobs.run(call)
    knobs.set(FORCE_SPLIT=split)
    got, plans, _ = knobs.run(call)
    expect(plans, n_plans, split=split)
    assert all(int(p["split"]) > 1 for p in plans)
    check(got)
    for w, g in zip(want, got):                   # bit for bit the unforced call's outputs
        assert torch.equal(w.view(torch.int32) if w.dtype == torch.float32 else w,
                           g.view(torch.int32) if g.dtype == torch.float32 else g)


# ---- C.7: FPS cluster matrix -----------------------------------------------------------------------------------------
FPS_CASES = [(N, C) for N in (40, 301, 3000, 8193, 16384, 40000, "dup") for C in (1, 2, 4, 8, 16)
             if C * FPS_CTA_POINTS >= (3072 if N == "dup" else N)]


@functools.lru_cache(maxsize=None)
def _fps_cloud(N):
    if N == "dup":                  # the padded-duplicate cloud of test_fps_duplicates_first_argmax
        a, _ = synth.batch_pairs(71, 1, 2048)
        a = np.concatenate([a, a[:, :1024]], 1)
        a = np.concatenate([a, a[:, ::-1]], 0).copy()
    else:
        a, _ = synth.batch_pairs(72, 2, N)
    start = np.random.default_rng(a.shape[1]).integers(0, a.shape[1], 2)
    return a, start, strict.farthest_point_sample(a, a.shape[1], start)     # npoint = N: the last picks tie at 0


@pytest.mark.parametrize("flat", [0, 1])
@pytest.mark.parametrize("N,C", FPS_CASES)
def test_fps_forced_cluster_matches_oracle(knobs, cuda_dev, N, C, flat):
    cloud, start, want = _fps_cloud(N)
    n = cloud.shape[1]
    knobs.set(FPS_CLUSTER=C, FPS_FLAT=flat)
    x, s = _t(cloud, cuda_dev), _t(start, cuda_dev)
    for npoint in (n, min(n, 37)):
        out, _, fplans = knobs.run(lambda: ops.fps(x, npoint, s))
        assert len(fplans) == 1, fplans
        P_ = 1
        while C * 512 * P_ < n:
            P_ *= 2
        assert (int(fplans[0]["C"]), int(fplans[0]["P"]), fplans[0]["exchange"]) == (C, P_, "flat" if flat else "two-level")
        np.testing.assert_array_equal(out.cpu().numpy(), want[:, :npoint])
