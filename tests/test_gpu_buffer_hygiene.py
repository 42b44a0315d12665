"""Every compute entry of include/b200pc.h through the C ABI, on guarded and poisoned buffers (tests/guarded.py).

Each case calls the entry directly (ctypes, torch's current stream) on buffers carved out of one allocation, with 16 KB
guards around every buffer and the outputs, the workspace and the guards filled with a poison (all 0x00, all 0xFF, seeded
random bytes), once with every buffer 256-byte aligned and once at the smallest offset the contract allows.  Every case
requires (a) the guards untouched, (b) the inputs unchanged, (c) every output bit-identical across the poisons and both
alignments, and (d) the outputs at the bar the suite holds for that entry against oracle/strict.  (c) is what tells a
result computed by the call from a value left in the buffer: a missed write, a read of workspace this call never wrote, a
read past the end of an input.  Outputs the kernels accumulate into start from a random non-zero base instead of a
poison: rows that receive nothing must keep the base bit for bit, the others must lie within the test_gpu_backward bound
with the base counted as one more term.  Forced plans are read back from B200PC_DEBUG_PLAN like in test_gpu_plans.
"""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

import guarded as G
from b200pc import _lib, ops, synth
from oracle import strict
from test_gpu_backward import _assert_within, _chamfer_ref, _gather_ref, _group_ref, _interp_ref, _wrap
from test_gpu_plans import BALL_N, Knobs, _ball_queries, _x_sorted_cloud, expect

pytestmark = pytest.mark.gpu

RUNS = len(G.POISONS) * len(G.ALIGNMENTS)         # C calls per case


@pytest.fixture
def knobs(cuda_dev, monkeypatch, capfd):
    return Knobs(monkeypatch, capfd)


def _L():
    return _lib.load()


def _ok(rc):
    assert rc == 0, "rc %d: %s" % (rc, _lib.last_error())


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


def _same(got, want, what=""):
    """bit-identical, except that any NaN matches any NaN (its payload differs between host and device)"""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    nan = np.isnan(got) & np.isnan(want)
    bad = (_bits(got) != _bits(want)) & ~nan
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError("%s: %d element(s) differ, first at %s: got %r, want %r" % (what, bad.sum(), i, got[i], want[i]))


def _ws_search(B, N, S, k):
    ops.reload_tuning()                        # the size under the tuning state the call will see
    return _L().b200pc_search_workspace_bytes(B, N, S, k)


def _run(bufs, call, dev):
    return G.check_call(bufs, call, dev)


# ==========================================================================================================================
# searches: knn (int64 with / without dist), knn_i32, ball_query, three_nn (with / without weight) on every path
# ==========================================================================================================================
@functools.lru_cache(maxsize=None)
def _search_clouds(B, N, S):
    """batch item 0: a few NaN / +-inf refs and a NaN query (a row of -1 / +inf); the last item: two finite refs, so every
    top-k row with k > 2 ends in -1 / +inf slots -- the slots where a missed write hides under the 0xFF poison"""
    a, b = synth.batch_pairs(90, B, max(N, S))
    ref, qry = a[:, :N].copy(), b[:, :S].copy()
    ref[0, 5] = np.nan
    ref[0, N // 2, 1] = np.inf
    ref[0, N - 1, 2] = -np.inf
    qry[0, 3] = np.nan
    ref[B - 1, 2:] = np.nan
    return ref, qry


# name: ((B, N, S, k), form, knobs, plan fields of every top-k line, plan fields of every line)
SEARCH_PATHS = {
    "small": ((2, 700, 333, 16), 0, dict(SMALL_PATH=1), {}, {}),
    "stream": ((2, 3000, 333, 16), 2, dict(SMALL_PATH=0, GRID=0), dict(grid="off"), dict(filter="lane")),
    "grid2": ((2, 3000, 333, 16), 0, dict(SMALL_PATH=0, GRID=2), dict(grid="thresholds"), {}),
    "grid3": ((2, 3000, 333, 16), 2, dict(SMALL_PATH=0, GRID=3), dict(grid="sorted", order="cell"), {}),
    "grid3-split3": ((2, 5000, 700, 16), 0, dict(SMALL_PATH=0, GRID=3, FORCE_SPLIT=3), dict(grid="sorted"), dict(split=3)),
    "split2-lt-k": ((2, 513, 77, 300), 0, dict(SMALL_PATH=0, GRID=0, FORCE_SPLIT=2), {}, dict(split=2)),
    "split32": ((2, 16384, 200, 16), 1, dict(SMALL_PATH=0, GRID=0, FORCE_SPLIT=32), {}, dict(split=32)),
    "q2": ((2, 3000, 333, 16), 0, dict(SMALL_PATH=0, GRID=0, FORCE_Q=2), {}, dict(q=2)),
    "filter0": ((2, 3000, 333, 16), 2, dict(SMALL_PATH=0, GRID=0, FILTER=0), {}, dict(filter="broadcast")),
    "natural": ((2, 3000, 333, 16), 0, dict(SMALL_PATH=0, GRID=0, NATURAL_ORDER=1), dict(order="natural"), {}),
}
SEARCH_ENTRIES = ["knn", "knn_nodist", "knn_i32", "ball", "three_nn", "three_nn_noweight"]
RADIUS = 1.0


def _search_case(entry, B, N, S, k, form):
    """(buffers, call, oracle check, mode of the plan line) of one search entry"""
    ref, qry = _search_clouds(B, N, S)
    L = _L()
    if entry.startswith("knn"):
        i32 = entry == "knn_i32"
        want_dist = entry != "knn_nodist"
        nws = _ws_search(B, N, S, k)
        bufs = [G.inp("ref", ref), G.inp("qry", qry), G.out("idx", (B, S, k), torch.int32 if i32 else torch.int64),
                G.ws("ws", nws)]
        if want_dist:
            bufs.append(G.out("dist", (B, S, k), torch.float32))
        fn = L.b200pc_knn_i32 if i32 else L.b200pc_knn

        def call(lay):
            _ok(fn(lay.ptr("ref"), lay.ptr("qry"), B, N, S, k, form, lay.ptr("idx"), lay.ptr("dist") if want_dist else None,
                   lay.ptr("ws"), nws, _st()))

        def check(res):
            oi, od = strict.knn(ref, qry, k, form)
            assert (oi == -1).any() and (oi[0] >= 0).any()
            np.testing.assert_array_equal(res["idx"], oi.astype(res["idx"].dtype))
            if want_dist:
                np.testing.assert_array_equal(_bits(res["dist"]), _bits(od))
        return bufs, call, check, 0
    if entry == "ball":
        ns = min(k, 64)
        nws = _ws_search(B, N, S, ns)
        bufs = [G.inp("xyz", ref), G.inp("new_xyz", qry), G.out("idx", (B, S, ns), torch.int64), G.ws("ws", nws)]

        def call(lay):
            _ok(L.b200pc_ball_query(lay.ptr("xyz"), lay.ptr("new_xyz"), B, N, S, C.c_float(float(strict.radius_sq(RADIUS))), ns,
                                    lay.ptr("idx"), lay.ptr("ws"), nws, _st()))

        def check(res):
            exp = strict.query_ball_point(RADIUS, ns, ref, qry)
            assert (exp == N).any()                     # empty balls: the sentinel N
            np.testing.assert_array_equal(res["idx"], exp)
        return bufs, call, check, 1
    # three_nn: the queries are the dense `unknown` cloud, the refs the sparse `known` one
    want_w = entry == "three_nn"
    nws = _ws_search(B, N, S, 3)
    bufs = [G.inp("unknown", qry), G.inp("known", ref), G.out("dist", (B, S, 3), torch.float32), G.out("idx", (B, S, 3), torch.int64),
            G.ws("ws", nws)]
    if want_w:
        bufs.append(G.out("weight", (B, S, 3), torch.float32))
    variant = form % 2

    def call(lay):
        _ok(L.b200pc_three_nn(lay.ptr("unknown"), lay.ptr("known"), B, S, N, variant, lay.ptr("dist"), lay.ptr("idx"),
                              lay.ptr("weight") if want_w else None, lay.ptr("ws"), nws, _st()))

    def check(res):
        od, oi = strict.three_nn(qry, ref)
        np.testing.assert_array_equal(res["idx"], oi)
        np.testing.assert_array_equal(_bits(res["dist"]), _bits(od))
        if want_w:
            _same(res["weight"], strict.three_weights(od, variant), "weight")
    return bufs, call, check, 0


@pytest.mark.parametrize("entry", SEARCH_ENTRIES)
@pytest.mark.parametrize("path", list(SEARCH_PATHS))
def test_search_entries(knobs, cuda_dev, path, entry):
    (B, N, S, k), form, env, want_topk, want_all = SEARCH_PATHS[path]
    knobs.set(**env)
    bufs, call, check, mode = _search_case(entry, B, N, S, k, form)
    (res, _), plans, _ = knobs.run(lambda: _run(bufs, call, cuda_dev))
    small = path == "small" and entry != "knn_i32"         # the int32 entry always streams
    want = dict(want_all, **(want_topk if mode == 0 else {}))
    if mode == 1 and "grid" in want_topk:
        want["grid"] = "off"                                # the ball query never builds the grid
    expect(plans, 0 if small else RUNS, **({} if small else dict(want, mode=mode)))
    check(res)


@pytest.mark.parametrize("radius", [1e-4, 0.05, 1.0])
def test_ball_query_merge_of_split_ranges(knobs, cuda_dev, radius):
    """a cloud sorted along x under a 3-range split: empty balls (the merge writes the sentinel N into every slot) and
    balls that fill nsample partway through a later range"""
    cloud = _x_sorted_cloud("line")
    qry = _ball_queries(cloud, radius)
    B, N, S, ns = 1, cloud.shape[1], qry.shape[1], 32
    knobs.set(FORCE_SPLIT=3)
    nws = _ws_search(B, N, S, ns)
    bufs = [G.inp("xyz", cloud), G.inp("new_xyz", qry), G.out("idx", (B, S, ns), torch.int64), G.ws("ws", nws)]

    def call(lay):
        _ok(_L().b200pc_ball_query(lay.ptr("xyz"), lay.ptr("new_xyz"), B, N, S, C.c_float(float(strict.radius_sq(radius))), ns,
                                   lay.ptr("idx"), lay.ptr("ws"), nws, _st()))

    (res, _), plans, _ = knobs.run(lambda: _run(bufs, call, cuda_dev))
    expect(plans, RUNS, split=3, mode=1)
    exp = strict.query_ball_point(radius, ns, cloud, qry)
    np.testing.assert_array_equal(res["idx"], exp)
    if radius == 1e-4:
        assert (exp == BALL_N).any()
    elif radius == 0.05:                                        # balls with fewer than nsample hits, padded with the first
        assert ((exp[0, :, -1] == exp[0, :, 0]) & (exp[0, :, 1] != exp[0, :, 0])).any()
    else:                                                       # full balls whose hits start in range 0 and go on in range 1
        last = exp[0].max(-1)
        assert ((exp[0, :, 0] < 4 * 512) & (last >= 4 * 512) & (last < BALL_N)).any()


# ==========================================================================================================================
# fps, fps_sample
# ==========================================================================================================================
@functools.lru_cache(maxsize=None)
def _fps_cloud():
    a, _ = synth.batch_pairs(72, 2, 3001)
    start = np.array([17, 2999], np.int64)
    return a, start, strict.farthest_point_sample(a, a.shape[1], start)          # npoint = N: the last picks tie at 0


@pytest.mark.parametrize("flat", [0, 1])
@pytest.mark.parametrize("cluster", [1, 2, 4, 8, 16])
@pytest.mark.parametrize("entry", ["fps", "fps_sample"])
def test_fps(knobs, cuda_dev, entry, cluster, flat):
    cloud, start, want = _fps_cloud()
    B, N = cloud.shape[:2]
    knobs.set(FPS_CLUSTER=cluster, FPS_FLAT=flat)
    L = _L()
    bufs = [G.inp("xyz", cloud), G.inp("start", start), G.out("idx", (B, N), torch.int64)]
    if entry == "fps":
        # documented as ignored: a non-null workspace full of random bytes must come back untouched
        nws = L.b200pc_fps_workspace_bytes(B, N)
        bufs.append(G.inp("ws", np.random.default_rng(3).integers(0, 256, nws, dtype=np.uint8), align=16))

        def call(lay):
            _ok(L.b200pc_fps(lay.ptr("xyz"), B, N, N, lay.ptr("start"), lay.ptr("idx"), lay.ptr("ws"), nws, _st()))
    else:
        bufs.append(G.out("new_xyz", (B, N, 3), torch.float32))

        def call(lay):
            _ok(L.b200pc_fps_sample(lay.ptr("xyz"), B, N, N, lay.ptr("start"), lay.ptr("idx"), lay.ptr("new_xyz"), _st()))

    (res, _), _, fplans = knobs.run(lambda: _run(bufs, call, cuda_dev))
    assert len(fplans) == RUNS and all((int(p["C"]), p["exchange"]) == (cluster, "flat" if flat else "two-level") for p in fplans), fplans
    np.testing.assert_array_equal(res["idx"], want)
    if entry == "fps_sample":
        np.testing.assert_array_equal(_bits(res["new_xyz"]), _bits(cloud[np.arange(B)[:, None], want]))


# ==========================================================================================================================
# row movers: gather, three_interpolate, group_points
# ==========================================================================================================================
def _gather_want(points, idx):
    N = points.shape[1]
    w = _wrap(idx, N)
    rows = points[np.arange(points.shape[0])[:, None], np.maximum(w, 0)]
    return np.where((w >= 0)[..., None], rows, np.float32(0)).astype(np.float32)


GATHER_CASES = [  # (C, knobs, out-of-range indices)
    (3, {}, True), (5, {}, False),
    (4, dict(GATHER_FLAT=1), True), (64, dict(GATHER_FLAT=1), False),
    (64, dict(GATHER_FLAT=0, GATHER_ROWS=8), True), (128, dict(GATHER_FLAT=0, GATHER_ROWS=2), True),
    (132, dict(GATHER_FLAT=0, GATHER_ROWS=4), False),
]


@pytest.mark.parametrize("C_,env,oob", GATHER_CASES, ids=["C%d-%s-%s" % (c, "-".join("%s%s" % kv for kv in e.items()) or "default",
                                                                          "oob" if o else "inrange") for c, e, o in GATHER_CASES])
def test_gather(knobs, cuda_dev, C_, env, oob):
    """the aligned runs take the vector kernel the knobs force (C % 4 == 0), the offset runs the scalar one; the flag is
    zero-initialised by the caller and must come back exactly 0 or 1"""
    B, N, R = 2, 300, 777
    rng = np.random.default_rng(C_)
    points = rng.normal(size=(B, N, C_)).astype(np.float32)
    idx = rng.integers(-N, N, size=(B, R))
    if oob:
        idx[:, ::37] = N
        idx[1, 5::41] = -N - 1
    knobs.set(**env)
    L = _L()
    bufs = [G.inp("points", points), G.inp("idx", idx), G.out("out", (B, R, C_), torch.float32),
            G.acc("flag", np.zeros(1, np.int32), exact=True)]

    def call(lay):
        _ok(L.b200pc_gather(lay.ptr("points"), lay.ptr("idx"), B, N, C_, R, lay.ptr("out"), lay.ptr("flag"), _st()))

    res, _ = _run(bufs, call, cuda_dev)
    np.testing.assert_array_equal(_bits(res["out"]), _bits(_gather_want(points, idx)))
    assert int(res["flag"][0]) == (1 if oob else 0)


INTERP_CASES = [(3, {}), (12, dict(INTERP_FLAT=1)), (128, dict(INTERP_FLAT=0, INTERP_ROWS=1)), (64, dict(INTERP_FLAT=0, INTERP_ROWS=2)),
                (132, dict(INTERP_FLAT=0, INTERP_ROWS=4)), (128, dict(INTERP_FLAT=0, INTERP_ROWS=8))]


@pytest.mark.parametrize("C_,env", INTERP_CASES, ids=["C%d-%s" % (c, "-".join("%s%s" % kv for kv in e.items()) or "default")
                                                      for c, e in INTERP_CASES])
def test_three_interpolate(knobs, cuda_dev, C_, env):
    B, S, N = 2, 300, 1001
    rng = np.random.default_rng(400 + C_)
    feat = rng.normal(size=(B, S, C_)).astype(np.float32)
    idx = rng.integers(0, S, size=(B, N, 3))
    idx[:, ::13, 2] = -1                                       # wraps once, to the last row
    w = rng.uniform(0.05, 1.0, size=(B, N, 3)).astype(np.float32)
    knobs.set(**env)
    L = _L()
    bufs = [G.inp("feat", feat), G.inp("idx", idx), G.inp("weight", w), G.out("out", (B, N, C_), torch.float32)]

    def call(lay):
        _ok(L.b200pc_three_interpolate(lay.ptr("feat"), lay.ptr("idx"), lay.ptr("weight"), B, S, N, C_, lay.ptr("out"), _st()))

    res, _ = _run(bufs, call, cuda_dev)
    np.testing.assert_array_equal(_bits(res["out"]), _bits(strict.three_interpolate(feat, idx, w)))


def _group_want(xyz, new, feat, idx, xyz_first):
    B, N, _ = xyz.shape
    w = _wrap(idx, N)
    ok = (w >= 0)[..., None]
    bi = np.arange(B)[:, None, None]
    rel = (np.where(ok, xyz[bi, np.maximum(w, 0)], np.float32(0)) - new[:, :, None, :]).astype(np.float32)
    parts = [rel]
    if feat is not None:
        g = np.where(ok, feat[bi, np.maximum(w, 0)], np.float32(0)).astype(np.float32)
        parts = [rel, g] if xyz_first else [g, rel]
    return np.ascontiguousarray(np.concatenate(parts, -1).transpose(0, 3, 2, 1))


@pytest.mark.parametrize("xyz_first", [1, 0])
@pytest.mark.parametrize("bulk", [0, 1])
@pytest.mark.parametrize("D", [0, 3, 64])
def test_group_points(knobs, cuda_dev, D, bulk, xyz_first):
    B, N, S, K = 2, 900, 123, 16
    a, b = synth.batch_pairs(36, B, N)
    xyz, new = a, b[:, :S].copy()
    rng = np.random.default_rng(D + 10 * bulk)
    feat = rng.normal(size=(B, N, D)).astype(np.float32) if D else None
    idx = rng.integers(-N, N, size=(B, S, K))
    idx[0, 5] = N                                              # an empty ball: the sentinel in every slot
    idx[1, 7, 3:] = N                                          # a ball that filled three slots, padded with the sentinel
    idx[1, 9, -1] = -1
    knobs.set(BULK=bulk)
    L = _L()
    bufs = [G.inp("xyz", xyz), G.inp("new_xyz", new), G.inp("idx", idx), G.out("out", (B, 3 + D, K, S), torch.float32)]
    if D:
        bufs.append(G.inp("feat", feat))

    def call(lay):
        _ok(L.b200pc_group_points(lay.ptr("xyz"), lay.ptr("new_xyz"), lay.ptr("feat") if D else None, lay.ptr("idx"), B, N, S, K, D,
                                  xyz_first, lay.ptr("out"), _st()))

    res, _ = _run(bufs, call, cuda_dev)
    np.testing.assert_array_equal(_bits(res["out"]), _bits(_group_want(xyz, new, feat, idx, xyz_first)))


# ==========================================================================================================================
# fused entries: feature_propagation, fusion_group, chamfer, rebuild_pack
# ==========================================================================================================================
@pytest.mark.parametrize("variant", [0, 1])
def test_feature_propagation(cuda_dev, variant):
    """the distances of the three-NN search live in the workspace, behind the search's own scratch"""
    B, N, S, Cc = 2, 1500, 400, 12
    a, b = synth.batch_pairs(46, B, N)
    dense, sparse = a, b[:, :S].copy()
    feat = np.random.default_rng(6).normal(size=(B, S, Cc)).astype(np.float32)
    L = _L()
    ops.reload_tuning()
    nws = L.b200pc_feature_propagation_workspace_bytes(B, N, S)
    bufs = [G.inp("unknown", dense), G.inp("known", sparse), G.inp("feat", feat), G.out("out", (B, N, Cc), torch.float32),
            G.out("idx", (B, N, 3), torch.int64), G.out("weight", (B, N, 3), torch.float32), G.ws("ws", nws)]

    def call(lay):
        _ok(L.b200pc_feature_propagation(lay.ptr("unknown"), lay.ptr("known"), lay.ptr("feat"), B, N, S, Cc, variant, lay.ptr("out"),
                                         lay.ptr("idx"), lay.ptr("weight"), lay.ptr("ws"), nws, _st()))

    res, _ = _run(bufs, call, cuda_dev)
    od, oi = strict.three_nn(dense, sparse)
    ow = strict.three_weights(od, variant)
    np.testing.assert_array_equal(res["idx"], oi)
    np.testing.assert_array_equal(_bits(res["weight"]), _bits(ow))
    np.testing.assert_array_equal(_bits(res["out"]), _bits(strict.three_interpolate(feat, oi, ow)))


@pytest.mark.parametrize("Cf", [0, 13])
def test_fusion_group(cuda_dev, Cf):
    B, N, S, k = 2, 1200, 333, 16
    a, b = synth.batch_pairs(31, B, N)
    ref, qry = a, b[:, :S].copy()
    feat = np.random.default_rng(Cf).normal(size=(B, N, Cf)).astype(np.float32)
    L = _L()
    nws = _ws_search(B, N, S, k)
    bufs = [G.inp("qry", qry), G.inp("ref", ref), G.out("resi", (B, 4, S, k), torch.float32), G.out("nn", (B, 3, S, k), torch.float32),
            G.out("idx", (B, S, k), torch.int64), G.ws("ws", nws)]
    if Cf:
        bufs += [G.inp("feat", feat), G.out("gfeat", (B, Cf, S, k), torch.float32)]

    def call(lay):
        _ok(L.b200pc_fusion_group(lay.ptr("qry"), lay.ptr("ref"), lay.ptr("feat") if Cf else None, B, N, S, k, Cf, lay.ptr("resi"),
                                  lay.ptr("nn"), lay.ptr("gfeat") if Cf else None, lay.ptr("idx"), lay.ptr("ws"), nws, _st()))

    res, _ = _run(bufs, call, cuda_dev)
    od, oi = strict.knn_points(qry, ref, k)
    np.testing.assert_array_equal(res["idx"], oi)
    want_nn = strict.index_points(ref, oi)
    want_resi = (want_nn - qry[:, :, None, :]).astype(np.float32)
    np.testing.assert_array_equal(_bits(res["nn"]), _bits(want_nn.transpose(0, 3, 1, 2)))
    np.testing.assert_array_equal(_bits(res["resi"][:, :3]), _bits(want_resi.transpose(0, 3, 1, 2)))
    np.testing.assert_allclose(res["resi"][:, 3], np.linalg.norm(want_resi, axis=-1), rtol=1e-6, atol=1e-30)
    if Cf:
        np.testing.assert_array_equal(_bits(res["gfeat"]), _bits(strict.index_points(feat, oi).transpose(0, 3, 1, 2)))


CHAMFER_SHAPES = [(2, 700, 333), (3, 1000, 1500)]


@pytest.mark.parametrize("B,N,M", CHAMFER_SHAPES)
def test_chamfer_fwd(cuda_dev, B, N, M):
    a, b = synth.batch_pairs(93, B, max(N, M))
    x, y = a[:, :N].copy(), b[:, :M].copy()
    L = _L()
    nws = max(_ws_search(B, M, N, 1), _ws_search(B, N, M, 1))
    bufs = [G.inp("x", x), G.inp("y", y), G.out("dx", (B, N), torch.float32), G.out("ix", (B, N), torch.int64),
            G.out("dy", (B, M), torch.float32), G.out("iy", (B, M), torch.int64), G.out("loss", (1,), torch.float32), G.ws("ws", nws)]

    def call(lay):
        _ok(L.b200pc_chamfer_fwd(lay.ptr("x"), lay.ptr("y"), B, N, M, lay.ptr("dx"), lay.ptr("ix"), lay.ptr("dy"), lay.ptr("iy"),
                                 lay.ptr("loss"), lay.ptr("ws"), nws, _st()))

    res, _ = _run(bufs, call, cuda_dev)
    ol, odx, oix, ody, oiy = strict.chamfer(x, y)
    np.testing.assert_array_equal(res["ix"], oix)
    np.testing.assert_array_equal(res["iy"], oiy)
    np.testing.assert_array_equal(_bits(res["dx"]), _bits(odx))
    np.testing.assert_array_equal(_bits(res["dy"]), _bits(ody))
    assert abs(float(res["loss"][0]) - ol) <= 1e-5 * abs(ol)


@pytest.mark.parametrize("B,N,M", CHAMFER_SHAPES)
def test_chamfer_bwd(cuda_dev, B, N, M):
    """gx / gy are zero-filled by the entry itself: poisoned like any output (atomic sums: compared with the bound, not
    across runs)"""
    a, b = synth.batch_pairs(94, B, max(N, M))
    x, y = a[:, :N].copy(), b[:, :M].copy()
    _, _, ix, _, iy = strict.chamfer(x, y)
    L = _L()
    bufs = [G.inp("x", x), G.inp("y", y), G.inp("ix", ix), G.inp("iy", iy), G.inp("gloss", np.array([3.5], np.float32)),
            G.out("gx", (B, N, 3), torch.float32, exact=False), G.out("gy", (B, M, 3), torch.float32, exact=False)]

    def call(lay):
        _ok(L.b200pc_chamfer_bwd(lay.ptr("x"), lay.ptr("y"), lay.ptr("ix"), lay.ptr("iy"), lay.ptr("gloss"), B, N, M, lay.ptr("gx"),
                                 lay.ptr("gy"), _st()))

    _, runs = _run(bufs, call, cuda_dev)
    (sx, ax, mx), (sy, ay, my) = _chamfer_ref(x, y, ix, iy, 3.5)
    for res in runs:
        _assert_within(res["gx"].reshape(-1, 3), sx, ax, mx, k=4, what="gx")
        _assert_within(res["gy"].reshape(-1, 3), sy, ay, my, k=4, what="gy")


def _records(ref, qry):
    _, oi = strict.knn_points(qry, ref, 1)
    i = oi[..., 0]                                                           # [B,S]
    nn = strict.index_points(ref, oi)[:, :, 0]                               # [B,S,3]
    rec = np.concatenate([i.astype(np.int32).view(np.float32)[..., None], nn], -1)
    return np.ascontiguousarray(rec.transpose(1, 0, 2))                     # [S,B,4]


@pytest.mark.parametrize("n_peers", [0, 1, 8])
def test_rebuild_pack(cuda_dev, n_peers):
    """local_out and 1 or 8 same-device "peer" buffers [S_total, B, 4]: only the slab [s_offset, s_offset + S_local) of a
    peer may change"""
    B, N, S_local, s_offset, S_total = 3, 2000, 500, 700, 1500
    a, b = synth.batch_pairs(35, B, N)
    ref, qry = a, b[:, :S_local].copy()
    L = _L()
    ops.reload_tuning()
    nws = L.b200pc_rebuild_pack_workspace_bytes(B, N, S_local)
    rng = np.random.default_rng(n_peers)
    bases = [rng.normal(size=(S_total, B, 4)).astype(np.float32) for _ in range(n_peers)]
    bufs = [G.inp("ref", ref), G.inp("qry", qry), G.out("local", (S_local, B, 4), torch.float32, align=16), G.ws("ws", nws)]
    bufs += [G.acc("peer%d" % p, bases[p], align=16, exact=True) for p in range(n_peers)]

    def call(lay):
        arr = (C.c_void_p * 8)(*[lay.ptr("peer%d" % p) for p in range(n_peers)])
        _ok(L.b200pc_rebuild_pack(lay.ptr("ref"), lay.ptr("qry"), B, N, S_local, s_offset, lay.ptr("local"), arr if n_peers else None,
                                  n_peers, lay.ptr("ws"), nws, _st()))

    res, _ = _run(bufs, call, cuda_dev)
    want = _records(ref, qry)
    _same(res["local"], want, "local_out")
    for p in range(n_peers):
        got = res["peer%d" % p]
        _same(got[s_offset:s_offset + S_local], want, "peer %d slab" % p)
        outside = np.ones(S_total, bool); outside[s_offset:s_offset + S_local] = False
        np.testing.assert_array_equal(_bits(got[outside]), _bits(bases[p][outside]))


def test_rebuild_pack_refuses_misaligned_records(cuda_dev):
    """the records are 16-byte stores: a destination 4 bytes past a 16-byte boundary is refused before anything launches"""
    B, N, S = 1, 600, 50
    a, b = synth.batch_pairs(35, B, N)
    ref, qry = torch.from_numpy(a).to(cuda_dev), torch.from_numpy(b[:, :S].copy()).to(cuda_dev)
    L = _L()
    nws = L.b200pc_rebuild_pack_workspace_bytes(B, N, S)
    ws = torch.empty(nws, dtype=torch.uint8, device=cuda_dev)
    buf = torch.zeros(S * B * 4 + 4, dtype=torch.float32, device=cuda_dev)
    good, bad = buf.data_ptr(), buf.data_ptr() + 4
    assert good % 16 == 0
    for local, peers in ((bad, []), (good, [good, bad])):
        arr = (C.c_void_p * 8)(*peers)
        rc = L.b200pc_rebuild_pack(ref.data_ptr(), qry.data_ptr(), B, N, S, 0, local, arr if peers else None, len(peers), ws.data_ptr(), nws,
                                   _st())
        assert rc == _lib.EINVAL and "16-byte aligned" in _lib.last_error()
    torch.cuda.synchronize()
    assert not buf.any()                                       # nothing ran
    _ok(L.b200pc_rebuild_pack(ref.data_ptr(), qry.data_ptr(), B, N, S, 0, good, None, 0, ws.data_ptr(), nws, _st()))


# ==========================================================================================================================
# channel_max, square_distance, poly_predict
# ==========================================================================================================================
@pytest.mark.parametrize("rows,C_", [(1001, 4), (77, 260)])
def test_channel_max(cuda_dev, rows, C_):
    x = np.random.default_rng(rows).normal(size=(rows, C_)).astype(np.float32)
    x[rows - 2, C_ // 2] = np.nan
    L = _L()
    bufs = [G.inp("x", x, align=16), G.out("out", (rows,), torch.float32)]

    def call(lay):
        _ok(L.b200pc_channel_max(lay.ptr("x"), rows, C_, lay.ptr("out"), _st()))

    res, _ = _run(bufs, call, cuda_dev)
    _same(res["out"], x.max(axis=1), "channel_max")
    assert np.isnan(res["out"][rows - 2])


@pytest.mark.parametrize("M", [1003, 1004])
def test_square_distance(cuda_dev, M):
    """M % 4 == 0 takes the 16-byte stores in the aligned runs and the scalar ones at the offset output"""
    B, N = 2, 77
    a, b = synth.batch_pairs(12, B, max(N, M))
    src, dst = a[:, :N].copy(), b[:, :M].copy()
    L = _L()
    bufs = [G.inp("src", src), G.inp("dst", dst), G.out("out", (B, N, M), torch.float32)]

    def call(lay):
        _ok(L.b200pc_square_distance(lay.ptr("src"), lay.ptr("dst"), B, N, M, lay.ptr("out"), _st()))

    res, _ = _run(bufs, call, cuda_dev)
    np.testing.assert_array_equal(_bits(res["out"]), _bits(strict.square_distance(src, dst)))


@pytest.mark.parametrize("F", [1, 16])
@pytest.mark.parametrize("per_batch", [999, 1200])
def test_poly_predict(cuda_dev, F, per_batch):
    """frames: a HOST array of F device pointers; weights [B, F] float64"""
    B = 3
    rng = np.random.default_rng(F * per_batch)
    frames = [(rng.normal(size=(B, per_batch)) * 30).astype(np.float32) for _ in range(F)]
    w = rng.normal(size=(B, F))
    L = _L()
    bufs = [G.inp("f%d" % f, frames[f]) for f in range(F)] + [G.inp("w", w), G.out("out", (B, per_batch), torch.float32)]

    def call(lay):
        ptrs = (C.c_void_p * F)(*[lay.ptr("f%d" % f) for f in range(F)])
        _ok(L.b200pc_poly_predict(ptrs, lay.ptr("w"), B, F, per_batch, lay.ptr("out"), _st()))

    res, _ = _run(bufs, call, cuda_dev)
    want = sum(w[:, f:f + 1] * frames[f].astype(np.float64) for f in range(F)).astype(np.float32)
    np.testing.assert_allclose(res["out"], want, rtol=1e-6, atol=1e-6)


# ==========================================================================================================================
# the kernels that accumulate into a caller-zeroed output: gather_bwd, three_interpolate_bwd, group_points_bwd
# ==========================================================================================================================
def _check_acc(got, base, s, a, m, k, what):
    """rows without a term keep the base bit for bit; the others lie within the bound with the base as one more term"""
    got = np.asarray(got); base = np.asarray(base)
    m = np.broadcast_to(m, got.shape)
    none = m == 0
    np.testing.assert_array_equal(_bits(got[none]), _bits(base[none]), err_msg=what + ": rows without a term")
    assert (~none).any()
    _assert_within(got, s + base, a + np.abs(base.astype(np.float64)), m + 1, k=k, what=what)


@pytest.mark.parametrize("C_", [3, 64])
def test_gather_bwd(cuda_dev, C_):
    B, N, R = 2, 500, 700
    rng = np.random.default_rng(200 + C_)
    idx = rng.integers(-N, N // 2, size=(B, R))                 # rows in [N/2, N) only through negative indices
    idx[:, ::29] = N                                            # out of range: no contribution
    gout = rng.normal(size=(B, R, C_)).astype(np.float32)
    base = rng.normal(size=(B, N, C_)).astype(np.float32)
    L = _L()
    bufs = [G.inp("gout", gout), G.inp("idx", idx), G.acc("gpoints", base)]

    def call(lay):
        _ok(L.b200pc_gather_bwd(lay.ptr("gout"), lay.ptr("idx"), B, N, C_, R, lay.ptr("gpoints"), _st()))

    _, runs = _run(bufs, call, cuda_dev)
    s, a, m = _gather_ref(gout, idx, N)
    assert (m == 0).any()
    for res in runs:
        _check_acc(res["gpoints"], base, s, a, m, 0, "gather_bwd C=%d" % C_)


@pytest.mark.parametrize("C_", [3, 64])
def test_three_interpolate_bwd(cuda_dev, C_):
    B, S, N = 2, 400, 900
    rng = np.random.default_rng(600 + C_)
    idx = rng.integers(0, S - 50, size=(B, N, 3))                # the last 50 rows of feat receive nothing
    idx[:, ::7, 0] = S                                          # dropped neighbour
    idx[:, 3::11, 1] = -1
    w = rng.uniform(0.05, 1.0, size=(B, N, 3)).astype(np.float32)
    feat = rng.normal(size=(B, S, C_)).astype(np.float32)
    gout = rng.normal(size=(B, N, C_)).astype(np.float32)
    base = rng.normal(size=(B, S, C_)).astype(np.float32)
    L = _L()
    bufs = [G.inp("gout", gout), G.inp("feat", feat), G.inp("idx", idx), G.inp("weight", w), G.acc("gfeat", base),
            G.out("gweight", (B, N, 3), torch.float32)]

    def call(lay):
        _ok(L.b200pc_three_interpolate_bwd(lay.ptr("gout"), lay.ptr("feat"), lay.ptr("idx"), lay.ptr("weight"), B, S, N, C_,
                                           lay.ptr("gfeat"), lay.ptr("gweight"), _st()))

    first, runs = _run(bufs, call, cuda_dev)
    (sf, af, mf), (sw, aw) = _interp_ref(gout, feat, idx, w)
    for res in runs:
        _check_acc(res["gfeat"], base, sf, af, mf, 1, "three_interpolate_bwd gfeat C=%d" % C_)
    _assert_within(first["gweight"], sw, aw, C_, k=1, what="gweight")
    assert (first["gweight"][_wrap(idx, S) < 0] == 0).all()


@pytest.mark.parametrize("xyz_first", [1, 0])
@pytest.mark.parametrize("D", [3, 64])
def test_group_points_bwd(cuda_dev, D, xyz_first):
    B, N, S, K = 2, 600, 77, 8
    rng = np.random.default_rng(D * 7 + xyz_first)
    idx = rng.integers(-N // 2, N // 2, size=(B, S, K))
    idx.reshape(-1)[::17] = N                                   # the ball query's empty-ball sentinel
    gout = rng.normal(size=(B, 3 + D, K, S)).astype(np.float32)
    base = rng.normal(size=(B, N, D)).astype(np.float32)
    L = _L()
    bufs = [G.inp("gout", gout), G.inp("idx", idx), G.acc("grad_feat", base)]

    def call(lay):
        _ok(L.b200pc_group_points_bwd(lay.ptr("gout"), lay.ptr("idx"), B, N, S, K, D, xyz_first, lay.ptr("grad_feat"), _st()))

    _, runs = _run(bufs, call, cuda_dev)
    (sf, af, mf), _, _ = _group_ref(idx, gout, N, D, xyz_first)
    assert (mf == 0).any()
    for res in runs:
        _check_acc(res["grad_feat"].reshape(B * N, D), base.reshape(B * N, D), sf, af, mf, 0, "group_points_bwd D=%d" % D)


# ==========================================================================================================================
# host-buffer entries
# ==========================================================================================================================
def test_host_entries(cuda_dev):
    """knn_host, ball_query_host and fps_host with guarded host arrays"""
    B, N, S, k = 2, 1500, 300, 8
    ref, qry = _search_clouds(B, N, S)
    L = _L()
    H = dict(space="host")
    bufs = [G.inp("ref", ref, **H), G.inp("qry", qry, **H), G.out("idx", (B, S, k), torch.int64, **H),
            G.out("dist", (B, S, k), torch.float32, **H)]

    def knn(lay):
        _ok(L.b200pc_knn_host(lay.ptr("ref"), lay.ptr("qry"), B, N, S, k, 0, lay.ptr("idx"), lay.ptr("dist")))

    res, _ = _run(bufs, knn, cuda_dev)
    oi, od = strict.knn(ref, qry, k, 0)
    np.testing.assert_array_equal(res["idx"], oi)
    np.testing.assert_array_equal(_bits(res["dist"]), _bits(od))

    bufs = [G.inp("xyz", ref, **H), G.inp("new_xyz", qry, **H), G.out("idx", (B, S, 16), torch.int64, **H)]

    def ball(lay):
        _ok(L.b200pc_ball_query_host(lay.ptr("xyz"), lay.ptr("new_xyz"), B, N, S, C.c_float(float(strict.radius_sq(0.7))), 16, lay.ptr("idx")))

    res, _ = _run(bufs, ball, cuda_dev)
    np.testing.assert_array_equal(res["idx"], strict.query_ball_point(0.7, 16, ref, qry))

    cloud = synth.batch_pairs(5, B, N)[0]
    start = np.array([3, 1400], np.int64)
    bufs = [G.inp("xyz", cloud, **H), G.inp("start", start, **H), G.out("idx", (B, 100), torch.int64, **H)]

    def fps(lay):
        _ok(L.b200pc_fps_host(lay.ptr("xyz"), B, N, 100, lay.ptr("start"), lay.ptr("idx")))

    res, _ = _run(bufs, fps, cuda_dev)
    np.testing.assert_array_equal(res["idx"], strict.farthest_point_sample(cloud, 100, start))


@pytest.mark.parametrize("want_dist", [True, False])
def test_knn_async_host(cuda_dev, want_dist):
    """pinned host clouds in, pinned int32 indices (and distances) out, a poisoned 256-byte aligned device arena"""
    B, N, S, k = 2, 3000, 700, 16
    ref, qry = _search_clouds(B, N, S)
    L = _L()
    ops.reload_tuning()
    need = L.b200pc_knn_async_host_workspace_bytes(B, N, S, k)
    P_ = dict(space="pinned")
    bufs = [G.inp("ref", ref, **P_), G.inp("qry", qry, **P_), G.out("idx", (B, S, k), torch.int32, **P_), G.ws("arena", need, align=256)]
    if want_dist:
        bufs.append(G.out("dist", (B, S, k), torch.float32, **P_))

    def call(lay):
        _ok(L.b200pc_knn_async_host(lay.ptr("ref"), lay.ptr("qry"), B, N, S, k, 0, lay.ptr("idx"), lay.ptr("dist") if want_dist else None,
                                    lay.ptr("arena"), need, _st()))

    res, _ = _run(bufs, call, cuda_dev)
    oi, od = strict.knn(ref, qry, k, 0)
    np.testing.assert_array_equal(res["idx"], oi.astype(np.int32))
    if want_dist:
        np.testing.assert_array_equal(_bits(res["dist"]), _bits(od))
