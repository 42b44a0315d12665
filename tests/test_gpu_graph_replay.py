"""Every op under CUDA-graph replay on new clouds, and off the current device, against the oracle.

A graph runs the host once, at capture; every replay reuses what the host decided then.  A graph stays correct only if every
data-dependent step runs on the device inside it: the grid's bounding box, the zeroed grid and work counters, the ragged
lengths, the FPS start indices, the zero-fill of every gradient.  So each case here captures one public call (forward, or
forward and backward together) on static inputs, then copies input sets of the same shapes into those inputs, replays and
compares the static outputs with the oracle of that set:

  1. the capture set;  2. another scene;  3. the capture scene scaled by 1e3 and shifted by ~3e5 (new bounding box and cell
  sizes);  4. a tie-heavy grid-snapped cloud;  5. non-finite refs, one batch item with fewer finite refs than k;  6. the
  capture set again, so that nothing carries over between replays.

The oracle's answer for every new set must differ from its answer for the capture set: a graph that returns stale outputs
cannot pass.  The forced plan of a path is read from the B200PC_DEBUG_PLAN=1 lines printed at capture.

Bar (DESIGN section 2): indices, search distances, square_distance, gather / grouping / three_interpolate, FPS and rebuild_pack
records bit-exact (NaN where the oracle has NaN); weights and the Chamfer scalar within 1e-5; gradients within the float64
summation bound of test_gpu_backward.py.
"""
import numpy as np
import pytest
import torch

import prune_geometry
import ragged_oracle as RO
from b200pc import ops, pointinet, pointnet2_utils as P, pytorch3d_shim as S3, synth
from oracle import strict
from test_gpu_backward import U, _assert_within, _chamfer_ref, _group_ref, _interp_ref, _scatter64, _wrap
from test_gpu_fps_large import WIDE_PLAN
from test_gpu_non_finite import _same, _spoil
from test_gpu_plans import GRID_NAME, PLAN, Knobs, expect, topk_order

pytestmark = pytest.mark.gpu

F32 = np.float32
SETS = ["capture", "other scene", "scaled 1e3 + 3e5", "grid-snapped ties", "non-finite", "capture again"]
SHIFT = np.array([3.0e5, -2.7e5, 3.2e5], F32)
GRID_NAME = {**GRID_NAME, 4: "pruned"}


def _c(a):
    """a C-contiguous copy that keeps a 0-d array 0-d (np.ascontiguousarray makes it [1])"""
    return np.array(a, order="C")


def _dev(a, dev):
    return torch.from_numpy(_c(a)).to(dev)


def _host(t):
    return t.detach().cpu().numpy()


# ---- harness -----------------------------------------------------------------------------------------------------------
class GraphKnobs(Knobs):
    """Knobs that also keep the stderr of the last run (the wide FPS tier's plan line carries one more field)"""

    def run(self, fn):
        torch.cuda.synchronize()
        self.capfd.readouterr()
        out = fn()
        torch.cuda.synchronize()
        self.last_err = self.capfd.readouterr().err
        return out, [m.groupdict() for m in PLAN.finditer(self.last_err)], [m.groupdict() for m in WIDE_PLAN.finditer(self.last_err)]


@pytest.fixture
def knobs(cuda_dev, monkeypatch, capfd):
    return GraphKnobs(monkeypatch, capfd)


class Replay:
    """fn(statics) captured into a CUDA graph after one warm-up on a side stream; run(set) copies the set into the static
    inputs, replays, synchronises and returns the static outputs on the host.  `plans` / `fps_plans`: the plan lines that
    the capture printed (knobs given)."""

    def __init__(self, knobs, statics, fn, dev):
        self.statics, self.dev = statics, dev
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            fn(statics)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()

        def capture():
            with torch.cuda.graph(self.graph):
                return fn(statics)
        if knobs is None:
            self.out, self.plans, self.fps_plans = capture(), [], []
        else:
            self.out, self.plans, self.fps_plans = knobs.run(capture)

    def run(self, inputs):
        with torch.no_grad():
            for name, a in inputs.items():
                self.statics[name].copy_(torch.from_numpy(_c(a)))
        self.graph.replay()
        torch.cuda.synchronize(self.dev)
        return [_host(o) for o in self.out]


def _key(x):
    """bytes of an oracle answer, for the stale-output check"""
    return b"".join(np.ascontiguousarray(np.asarray(a)).tobytes() for a in (x if isinstance(x, (list, tuple)) else [x]))


def _exact(got, want, what):
    for i, (g, w) in enumerate(zip(got, want)):
        g, w = np.asarray(g), np.asarray(w)
        assert g.shape == w.shape, (what, i, g.shape, w.shape)
        if w.dtype.kind == "f":
            _same(g, w, "%s, output %d" % (what, i))
        else:
            np.testing.assert_array_equal(g, w.astype(g.dtype), err_msg="%s, output %d" % (what, i))


def drive(knobs, dev, sets, fn, oracle, check=_exact):
    """capture fn on sets[0], then replay every set in order against oracle(set); returns the Replay"""
    statics = {name: _dev(a, dev) for name, a in sets[0].items()}
    rep = Replay(knobs, statics, fn, dev)
    wants = [oracle(s) for s in sets]
    for i, (s, want) in enumerate(zip(sets, wants)):
        if 0 < i < len(sets) - 1:
            assert _key(want) != _key(wants[0]), "set %d (%s): the oracle gives the capture set's answer" % (i, SETS[i])
        check(rep.run(s), want, "set %d (%s)" % (i, SETS[i]))
    return rep


# ---- input sets --------------------------------------------------------------------------------------------------------
def cloud_sets(seed, B, N, S, k):
    """six (ref [B,N,3], qry [B,S,3]) pairs in the order of SETS; set 5: NaN / +-inf refs in item 0, and item B-1 keeps
    only k-1 finite refs"""
    a, b = synth.batch_pairs(seed, B, max(N, S))
    ref, qry = a[:, :N].copy(), b[:, :S].copy()
    other = prune_geometry.batch(("ground_objects", "shell", "two_clusters", "plane")[:B], seed, N, S)
    scaled = ((ref * F32(1e3)) + SHIFT).astype(F32), ((qry * F32(1e3)) + SHIFT).astype(F32)
    snapped = synth.grid_snapped(seed, B, N, span=12), synth.grid_snapped(seed + 1, B, S, span=12)
    bad = ref.copy()
    rng = np.random.default_rng(seed)
    _spoil(bad, 0, rng.choice(N, N // 10, replace=False))
    _spoil(bad, B - 1, rng.permutation(N)[max(k - 1, 0):])
    return [(ref, qry), other, scaled, snapped, (bad, qry), (ref, qry)]


def _sets(pairs, names=("ref", "qry")):
    return [dict(zip(names, p)) for p in pairs]


# ---- forward: top-k search ---------------------------------------------------------------------------------------------
SMALL_SHAPE, STREAM_SHAPE = (2, 1000, 300), (2, 5000, 700)
TOPK_PATHS = {
    "small": (dict(SMALL_PATH=1, GRID=0), SMALL_SHAPE, 16),
    "grid0": (dict(SMALL_PATH=0, GRID=0), STREAM_SHAPE, 16),
    "grid2": (dict(SMALL_PATH=0, GRID=2), STREAM_SHAPE, 16),
    "grid3": (dict(SMALL_PATH=0, GRID=3), STREAM_SHAPE, 16),
    "pruned-k1": (dict(SMALL_PATH=0, GRID=4), STREAM_SHAPE, 1),
    "pruned-k16": (dict(SMALL_PATH=0, GRID=4), STREAM_SHAPE, 16),
    "pruned-k128": (dict(SMALL_PATH=0, GRID=4), STREAM_SHAPE, 128),
    "split3": (dict(SMALL_PATH=0, GRID=0, FORCE_SPLIT=3), STREAM_SHAPE, 16),
}
# entry -> (form, call on the static refs / queries, oracle of one (ref, qry) set)
TOPK_ENTRIES = {
    "knn_point": (0, lambda s, k: (P.knn_point(k, s["ref"], s["qry"]),),
                  lambda ref, qry, k: (strict.knn(ref, qry, k, 0)[0],)),
    "knn_points": (2, lambda s, k: tuple(S3.knn_points(s["qry"], s["ref"], K=k)[:2]),
                   lambda ref, qry, k: strict.knn(ref, qry, k, 2)[::-1]),
    "three_nn": (1, lambda s, k: tuple(P.three_nn(s["qry"], s["ref"])),
                 lambda ref, qry, k: strict.knn(ref, qry, 3, 1)[::-1]),
    "knn_search_i32": (0, lambda s, k: (ops.knn_search_i32(s["ref"], s["qry"], k, 0),),
                       lambda ref, qry, k: (strict.knn(ref, qry, k, 0)[0].astype(np.int32),)),
}


TOPK_CASES = [(p, e) for p in TOPK_PATHS for e in TOPK_ENTRIES if not (e == "three_nn" and p in ("pruned-k1", "pruned-k128"))]


@pytest.mark.parametrize("path,entry", TOPK_CASES, ids=["%s-%s" % c for c in TOPK_CASES])
def test_topk_search_replays_new_clouds(knobs, cuda_dev, path, entry):
    env, (B, N, S), k = TOPK_PATHS[path]
    form, call, oracle = TOPK_ENTRIES[entry]
    kk = 3 if entry == "three_nn" else k
    knobs.set(**env)
    rep = drive(knobs, cuda_dev, _sets(cloud_sets(11 + kk, B, N, S, kk)), lambda s: call(s, k),
                lambda s: oracle(s["ref"], s["qry"], k))
    if path == "small" and entry != "knn_search_i32":
        assert rep.plans == [], rep.plans                  # the warp-per-query kernel prints no streaming plan
        return
    grid = env["GRID"]
    want = dict(grid=GRID_NAME[grid], mode=0, k=kk, order="cell" if grid >= 3 else topk_order(form, grid))
    if "FORCE_SPLIT" in env:
        want["split"] = env["FORCE_SPLIT"]
    expect(rep.plans, 1, **want)


# ---- forward: ragged kNN and Chamfer -----------------------------------------------------------------------------------
RAGGED_B, RAGGED_N, RAGGED_S, RAGGED_K = 4, 3000, 500, 16
# per set: (lengths of the refs, lengths of the queries); 0, 1, fewer than k and full, in a new order every replay
REF_LENS = [[3000, 15, 1, 0], [0, 3000, 15, 1], [1, 0, 3000, 15], [15, 1, 0, 3000], [3000, 2999, 7, 16], [3000, 15, 1, 0]]
QRY_LENS = [[500, 0, 1, 250], [1, 500, 0, 499], [250, 1, 500, 0], [0, 250, 1, 500], [500, 1, 300, 500], [500, 0, 1, 250]]


def _ragged_sets(seed, k):
    pairs = cloud_sets(seed, RAGGED_B, RAGGED_N, RAGGED_S, k)
    return [dict(p2=ref, p1=qry, l2=np.array(rl, np.int64), l1=np.array(ql, np.int64))
            for (ref, qry), rl, ql in zip(pairs, REF_LENS, QRY_LENS)]


def _knn_points_ragged_oracle(s, k):
    """pytorch3d padding: rows beyond lengths1 and slots beyond lengths2 hold idx 0 and dist 0"""
    oi, od = RO.knn(s["p2"], s["p1"], s["l2"], s["l1"], k, strict.FORM_DIRECT)
    n1, n2 = RO.clamp_lengths(s["l1"], RAGGED_S, RAGGED_B), RO.clamp_lengths(s["l2"], RAGGED_N, RAGGED_B)
    pad = (np.arange(RAGGED_S)[None, :, None] >= n1[:, None, None]) | (np.arange(k)[None, None, :] >= n2[:, None, None])
    return np.where(pad, F32(0), od), np.where(pad, 0, oi)


def test_knn_points_with_lengths_replays_new_lengths(cuda_dev):
    k = RAGGED_K
    drive(None, cuda_dev, _ragged_sets(21, k),
          lambda s: tuple(S3.knn_points(s["p1"], s["p2"], s["l1"], s["l2"], K=k)[:2]),
          lambda s: _knn_points_ragged_oracle(s, k))


def _chamfer_sets(seed):
    """x [B,3000,3], y [B,500,3] with lengths; set 5: another scene with NaN / inf in the padding beyond the lengths, which
    must not matter"""
    pairs = cloud_sets(seed, RAGGED_B, RAGGED_N, RAGGED_S, 1)
    pairs[4] = (pairs[1][0].copy(), pairs[1][1].copy())
    sets = []
    for i, (x, y) in enumerate(pairs):
        s = dict(x=x, y=y, xl=np.array(REF_LENS[i], np.int64), yl=np.array(QRY_LENS[i], np.int64))
        if i == 4:
            for b in range(RAGGED_B):
                _spoil(x, b, range(REF_LENS[i][b], RAGGED_N))
                _spoil(y, b, range(QRY_LENS[i][b], RAGGED_S))
        sets.append(s)
    return sets


def _loss_close(got, want, what):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    inf = np.isinf(want)
    assert (got[inf] == want[inf]).all(), (what, got, want)
    assert (np.abs(got[~inf] - want[~inf]) <= 1e-5 * np.abs(want[~inf]) + 1e-30).all(), (what, got, want)


@pytest.mark.parametrize("batch_reduction", [None, "mean"])
def test_chamfer_distance_with_lengths_replays_new_lengths(cuda_dev, batch_reduction):
    def call(s):
        return (S3.chamfer_distance(s["x"], s["y"], x_lengths=s["xl"], y_lengths=s["yl"], batch_reduction=batch_reduction)[0],)

    def oracle(s):
        x64, y64 = torch.from_numpy(s["x"]).double(), torch.from_numpy(s["y"]).double()
        return (RO.chamfer_distance64(x64, y64, s["xl"], s["yl"], "mean", batch_reduction).numpy(),)

    drive(None, cuda_dev, _chamfer_sets(23), call, oracle, lambda g, w, what: _loss_close(g[0], w[0], what))


def test_dense_chamfer_replays_new_clouds(cuda_dev):
    def check(got, want, what):
        _loss_close(got[0], want[0], what + " loss")
        _exact(got[1:], want[1:], what)

    drive(None, cuda_dev, _sets(cloud_sets(25, 2, 3000, 2600, 1), ("x", "y")), lambda s: tuple(ops.chamfer(s["x"], s["y"])),
          lambda s: strict.chamfer(s["x"], s["y"]), check)


# ---- forward: ball query -----------------------------------------------------------------------------------------------
BALL_PATHS = {"small": (dict(SMALL_PATH=1), (2, 900, 300)), "stream": (dict(SMALL_PATH=0), (2, 5000, 700)),
              "split3": (dict(SMALL_PATH=0, FORCE_SPLIT=3), (2, 6000, 700))}
RADIUS, NSAMPLE = 0.8, 16


@pytest.mark.parametrize("path", list(BALL_PATHS))
def test_ball_query_replays_new_clouds(knobs, cuda_dev, path):
    env, (B, N, S) = BALL_PATHS[path]
    sets = _sets(cloud_sets(31, B, N, S, NSAMPLE))
    for s in sets:                                        # the last queries lie far outside every cloud: empty balls
        s["qry"] = s["qry"].copy()
        s["qry"][:, -5:] = s["ref"][:, :5] + F32(1e7)
    knobs.set(**env)
    # the radius is a capture-time constant: ball_query squares it on the host and passes r2 as a scalar argument
    rep = drive(knobs, cuda_dev, sets, lambda s: (P.query_ball_point(RADIUS, NSAMPLE, s["ref"], s["qry"]),),
                lambda s: (strict.query_ball_point(RADIUS, NSAMPLE, s["ref"], s["qry"]),))
    if path == "small":
        assert rep.plans == []
    else:
        expect(rep.plans, 1, mode=1, split=env.get("FORCE_SPLIT"))
    assert (strict.query_ball_point(RADIUS, NSAMPLE, sets[0]["ref"], sets[0]["qry"])[:, -5:] == N).all()


# ---- forward: FPS and sample_points ------------------------------------------------------------------------------------
FPS_CASES = {"C1": (1, 2, 3000, 300), "C8": (8, 2, 20000, 300), "C16": (16, 2, 20000, 300), "wide": (None, 2, 140000, 200)}


def _fps_sets(seed, B, N):
    rng = np.random.default_rng(seed)
    starts = [rng.integers(0, N, B) for _ in range(5)]
    return [dict(xyz=ref, start=st) for (ref, _), st in zip(cloud_sets(seed, B, N, 8, 1), starts + [starts[0]])]


@pytest.mark.parametrize("want_xyz", [False, True], ids=["farthest_point_sample", "sample_points"])
@pytest.mark.parametrize("case", list(FPS_CASES))
def test_fps_replays_new_clouds_and_starts(knobs, cuda_dev, case, want_xyz):
    C, B, N, npoint = FPS_CASES[case]
    knobs.set(FPS_CLUSTER=C)
    if want_xyz:
        call = lambda s: tuple(P.sample_points(s["xyz"], npoint, s["start"]))

        def oracle(s):
            idx = strict.farthest_point_sample(s["xyz"], npoint, s["start"])
            return idx, strict.index_points(s["xyz"], idx)
    else:
        call = lambda s: (P.farthest_point_sample_from(s["xyz"], npoint, s["start"]),)
        oracle = lambda s: (strict.farthest_point_sample(s["xyz"], npoint, s["start"]),)
    sets = _fps_sets(41, B, N)
    rep = drive(knobs, cuda_dev, sets, call, oracle)
    assert len(rep.fps_plans) == 1, rep.fps_plans
    line = rep.fps_plans[0]
    if C is None:
        assert line["Q"] is not None, line                # the shared-memory (wide) tier, fps_wide_kernel
    else:
        assert int(line["C"]) == C and line["Q"] is None, line


# ---- forward: everything else ------------------------------------------------------------------------------------------
def _value_sets(seed, shape, spread=1.0):
    """six fp32 arrays of one shape in the order of SETS (set 5 holds NaN and +-inf)"""
    rng = np.random.default_rng(seed)
    a = (rng.normal(size=shape) * spread).astype(F32)
    b = (rng.normal(size=shape) * spread * 3).astype(F32)
    c = (a * F32(1e3) + F32(3e5)).astype(F32)
    d = (rng.integers(-4, 5, size=shape) * F32(0.25)).astype(F32)
    e = a.copy().reshape(-1)
    e[::7], e[3::11], e[5::13] = np.nan, np.inf, -np.inf
    return [a, b, c, d, e.reshape(shape), a]


def _index_sets(seed, shape, N):
    """six index arrays in [-N, N) (torch indexing: a negative index wraps once); set 3 all the same row, set 4 the edges"""
    rng = np.random.default_rng(seed)
    a = rng.integers(-N, N, size=shape)
    e = a.copy().reshape(-1)
    e[::3], e[1::3] = N - 1, -N
    return [a, rng.integers(-N, N, size=shape), rng.integers(0, N, size=shape), np.full(shape, 7), e.reshape(shape), a]


@pytest.mark.parametrize("C", [64, 3], ids=["vec4", "scalar"])
def test_index_points_replays(cuda_dev, C):
    B, N = 2, 3000
    pts, idx = _value_sets(51, (B, N, C)), _index_sets(52, (B, 400, 16), N)
    drive(None, cuda_dev, [dict(p=p, i=i) for p, i in zip(pts, idx)], lambda s: (P.index_points(s["p"], s["i"]),),
          lambda s: (strict.index_points(s["p"], s["i"]),))


@pytest.mark.parametrize("bulk", [None, 1], ids=["registers", "bulk"])
@pytest.mark.parametrize("xyz_first", [True, False])
def test_group_points_replays(knobs, cuda_dev, xyz_first, bulk):
    B, N, S, K, D = 2, 3000, 500, 16, 32
    knobs.set(BULK=bulk)
    clouds = cloud_sets(53, B, N, S, K)
    feats, idx = _value_sets(54, (B, N, D)), _index_sets(55, (B, S, K), N)
    sets = [dict(xyz=r, new=q, f=f, i=i) for (r, q), f, i in zip(clouds, feats, idx)]
    drive(knobs, cuda_dev, sets, lambda s: (P.group_points(s["xyz"], s["new"], s["f"], s["i"], xyz_first),),
          lambda s: (strict.group_points(s["xyz"], s["new"], s["f"], s["i"], xyz_first),))


def _interp_idx_sets(seed, B, N, S):
    rng = np.random.default_rng(seed)
    sets = [rng.integers(0, S, size=(B, N, 3)) for _ in range(5)]
    sets[3][:] = 2                                        # every row reads the same known point
    sets[4][:, ::5] = [S - 1, 0, S - 1]
    return sets + [sets[0]]


def test_three_interpolate_replays(cuda_dev):
    B, S, N, C = 2, 700, 4000, 24
    feats = _value_sets(56, (B, S, C))
    ws = [np.abs(w[..., :3]).astype(F32) for w in _value_sets(57, (B, N, 3))]
    ws[4] = np.random.default_rng(58).uniform(0, 1, size=(B, N, 3)).astype(F32)      # finite weights, non-finite features
    sets = [dict(f=f, i=i, w=w) for f, i, w in zip(feats, _interp_idx_sets(59, B, N, S), ws)]
    drive(None, cuda_dev, sets, lambda s: (P.three_interpolate(s["f"], s["i"], s["w"]),),
          lambda s: (strict.three_interpolate(s["f"], s["i"], s["w"]),))


def _three_nn_weights_oracle(dense, sparse, variant=0):
    od, oi = strict.three_nn(dense, sparse)
    return od, oi, strict.three_weights(od, variant)


def test_feature_propagation_replays(cuda_dev):
    B, N, S, C = 2, 4000, 1000, 16
    clouds = cloud_sets(61, B, S, N, 3)
    feats = _value_sets(62, (B, S, C))
    sets = [dict(known=r, dense=q, f=f) for (r, q), f in zip(clouds, feats)]

    def call(s):
        out, idx, w = torch.ops.b200pc.feature_propagation(s["dense"], s["known"], s["f"], 0)
        return P.feature_propagation(s["dense"], s["known"], s["f"]), idx, w

    def oracle(s):
        od, oi, ow = _three_nn_weights_oracle(s["dense"], s["known"])
        return strict.three_interpolate(s["f"], oi, ow), oi, ow

    def check(got, want, what):
        _exact(got[:2], want[:2], what)
        g, w = got[2], want[2]
        np.testing.assert_array_equal(np.isnan(g), np.isnan(w), err_msg=what + " weights")
        ok = ~np.isnan(w)
        assert (np.abs(g[ok] - w[ok]) <= 1e-5 * np.abs(w[ok]) + 1e-30).all(), what + " weights"

    drive(None, cuda_dev, sets, call, oracle, check)


def _fusion_oracle(qry, ref, feat, k):
    _, oi = strict.knn_points(qry, ref, k)
    ok = oi >= 0
    safe = np.where(ok, oi, 0)
    nn = np.where(ok[..., None], strict.index_points(ref, safe), F32(np.nan))
    with np.errstate(invalid="ignore", over="ignore"):
        d = (nn - qry[:, :, None, :]).astype(F32)
        n2 = ((d[..., 0] * d[..., 0]).astype(F32) + (d[..., 1] * d[..., 1]).astype(F32)).astype(F32)
        n2 = (n2 + (d[..., 2] * d[..., 2]).astype(F32)).astype(F32)
    resi = np.concatenate([d, np.sqrt(n2)[..., None]], -1)
    out = [resi.transpose(0, 3, 1, 2), nn.transpose(0, 3, 1, 2)]
    if feat is not None:
        out.append(np.where(ok[..., None], strict.index_points(feat, safe), F32(np.nan)).transpose(0, 3, 1, 2))
    return out + [oi]


@pytest.mark.parametrize("Cf", [0, 5])
def test_fusion_group_replays(cuda_dev, Cf):
    B, N, S, k = 2, 3000, 800, 16
    clouds = cloud_sets(63, B, N, S, k)
    feats = _value_sets(64, (B, N, max(Cf, 1)))
    sets = [dict(ref=r, qry=q, **({"f": f} if Cf else {})) for (r, q), f in zip(clouds, feats)]

    def call(s):
        resi, nn, gf, idx = P.fusion_group(s["qry"], s["ref"], k, s.get("f"))
        return (resi, nn) + ((gf,) if Cf else ()) + (idx,)

    drive(None, cuda_dev, sets, call, lambda s: _fusion_oracle(s["qry"], s["ref"], s.get("f"), k))


@pytest.mark.parametrize("C", [4, 132])
def test_channel_max_replays(cuda_dev, C):
    rows = 16 * 148 * 8 * 2 + 37
    sets = [dict(x=x) for x in _value_sets(65 + C, (rows, C))]

    def oracle(s):
        x = s["x"]
        return (np.where(np.isnan(x).any(1), F32(np.nan), np.nanmax(np.where(np.isnan(x), -np.inf, x), 1)).astype(F32),)

    drive(None, cuda_dev, sets, lambda s: (ops.channel_max(s["x"]),), oracle)


def test_square_distance_replays(cuda_dev):
    sets = _sets(cloud_sets(67, 2, 700, 300, 1), ("dst", "src"))
    drive(None, cuda_dev, sets, lambda s: (P.square_distance(s["src"], s["dst"]),),
          lambda s: (strict.square_distance(s["src"], s["dst"]),))


@pytest.mark.parametrize("split", [None, 3])
def test_rebuild_pack_with_a_peer_buffer_replays(knobs, cuda_dev, split):
    B, N, S, off = 2, 6000, 500, 120
    knobs.set(FORCE_SPLIT=split, GRID=0)
    peer = torch.full((S + 2 * off, B, 4), -7.0, device=cuda_dev)       # a same-device peer of [S_total, B, 4] rows

    def call(s):
        return ops.rebuild_pack(s["ref"], s["qry"], off, [peer.data_ptr()]), peer

    def oracle(s):
        _, oi = strict.knn_points(s["qry"], s["ref"], 1)
        oi = oi[..., 0]
        nn = np.where((oi >= 0)[..., None], strict.index_points(s["ref"], np.maximum(oi, 0)), F32(np.nan))
        rec = np.concatenate([oi.astype(np.int32).view(F32)[..., None], nn], -1).transpose(1, 0, 2)     # [S,B,4]
        full = np.full((S + 2 * off, B, 4), -7.0, F32)
        full[off:off + S] = rec
        return rec, full

    rep = drive(knobs, cuda_dev, _sets(cloud_sets(69, B, N, S, 1)), call, oracle)
    expect(rep.plans, 1, split=split)


def test_poly_predict_replays_new_weights(cuda_dev):
    B, Fr, shape = 3, 4, (3, 3, 1000)
    frames = [_value_sets(70 + f, shape) for f in range(Fr)]
    rng = np.random.default_rng(75)
    ws = [rng.normal(size=(B, Fr)) for _ in range(5)]
    ws = ws + [ws[0]]
    sets = [dict(w=w, **{"f%d" % f: frames[f][i] for f in range(Fr)}) for i, w in enumerate(ws)]

    def oracle(s):
        with np.errstate(invalid="ignore"):               # inf - inf in the non-finite set
            acc = sum(s["w"][:, f].reshape(B, 1, 1) * s["f%d" % f].astype(np.float64) for f in range(Fr))
        mag = sum(np.abs(s["w"][:, f].reshape(B, 1, 1) * s["f%d" % f].astype(np.float64)) for f in range(Fr))
        return acc, mag

    def check(got, want, what):
        acc, mag = want
        g = got[0].astype(np.float64)
        fin = np.isfinite(acc)
        np.testing.assert_array_equal(np.isfinite(g), fin, err_msg=what)
        # one fp32 rounding of a float64 sum of F fma terms
        assert (np.abs(g - acc)[fin] <= U * np.abs(acc)[fin] + 2 * Fr * 2.0 ** -53 * mag[fin] + 1e-38).all(), what

    drive(None, cuda_dev, sets, lambda s: (ops.poly_predict([s["f%d" % f] for f in range(Fr)], s["w"]),), oracle, check)


# ---- backward under capture --------------------------------------------------------------------------------------------
def drive_backward(dev, sets, grads, fn, check):
    """capture fn's forward and torch.autograd.grad of its outputs with respect to `grads` (static upstream gradients)
    together; replay every set against check(), then the last set once more: the gradients must still pass (a doubled
    gradient does not), so their zero-fill is inside the graph.  Atomic scatters sum in any order, so two replays of one set
    may differ in the last bits."""
    statics = {name: _dev(a, dev) for name, a in sets[0].items()}
    for name in grads:
        statics[name].requires_grad_(True)
    rep = Replay(None, statics, lambda st: _fwd_bwd(st, grads, fn), dev)
    results = []
    for i, s in enumerate(sets):
        results.append(rep.run(s))
        check(results[-1], s, "set %d (%s)" % (i, SETS[i]))
        if 0 < i < len(sets) - 1:
            assert _key(results[-1]) != _key(results[0]), "set %d (%s): the capture set's outputs" % (i, SETS[i])
    check(rep.run(sets[-1]), sets[-1], "set %d (%s) replayed twice" % (len(sets) - 1, SETS[-1]))


def _fwd_bwd(s, grads, fn):
    """fn(s) -> (differentiated outputs, their upstream gradients[, outputs that ride along])"""
    res = fn(s)
    outs, gouts, extra = res[0], res[1], (res[2] if len(res) > 2 else ())
    return (*outs, *extra, *torch.autograd.grad(outs, [s[g] for g in grads], gouts))


def _gout_sets(seed, shape):
    rng = np.random.default_rng(seed)
    g = [rng.normal(size=shape).astype(F32) for _ in range(5)]
    return g + [g[0]]


def test_index_points_backward_replays(cuda_dev):
    B, N, C = 2, 1500, 8
    pts = _value_sets(81, (B, N, C))[:4]
    pts = pts + [pts[1], pts[0]]
    idx = _index_sets(82, (B, 300, 16), N)
    idx[4] = idx[4].copy(); idx[4].reshape(-1)[::2] = 3       # one row gets half of all the terms
    sets = [dict(p=p, i=i, g=g) for p, i, g in zip(pts, idx, _gout_sets(83, (B, 300, 16, C)))]

    def check(got, s, what):
        out, gp = got
        np.testing.assert_array_equal(out, strict.index_points(s["p"], s["i"]))
        flat = np.where(_wrap(s["i"], N) >= 0, _wrap(s["i"], N) + np.arange(B)[:, None, None] * N, -1).reshape(-1)
        sg, ag, mg = _scatter64(B * N, flat, s["g"].reshape(-1, C))
        _assert_within(gp.reshape(B * N, C), sg, ag, mg, what=what + " gpoints")

    drive_backward(cuda_dev, sets, ["p"], lambda s: ((P.index_points(s["p"], s["i"]),), (s["g"],)), check)


def _group_forward(xyz, new, feat, idx, xyz_first):
    """strict.group_points where a slot still out of range after one wrap (the ball query's sentinel N) reads a zero row:
    the kernel fills it with 0 - centre and zero features"""
    N = xyz.shape[1]
    wr = _wrap(idx, N)
    pad = lambda a: np.concatenate([a, np.zeros_like(a[:, :1])], 1)
    return strict.group_points(pad(xyz), new, pad(feat), np.where(wr >= 0, wr, N), xyz_first)


@pytest.mark.parametrize("xyz_first", [True, False])
def test_group_points_backward_replays(cuda_dev, xyz_first):
    B, N, S, K, D = 2, 1200, 300, 16, 12
    clouds = cloud_sets(84, B, N, S, K)[:4]
    feats = _value_sets(85, (B, N, D))[:4]
    idx = _index_sets(86, (B, S, K), N)
    idx[4] = idx[4].copy(); idx[4].reshape(-1)[::5] = N          # the ball query's empty-ball sentinel
    sets = [dict(xyz=c[0], new=c[1], f=f, i=i, g=g) for c, f, i, g in
            zip(clouds + [clouds[1], clouds[0]], feats + [feats[1], feats[0]], idx, _gout_sets(87, (B, 3 + D, K, S)))]

    def check(got, s, what):
        out, gx, gn, gf = got
        _same(out, _group_forward(s["xyz"], s["new"], s["f"], s["i"], xyz_first), what + " forward")
        (sf, af, mf), (sx, ax, mx), (sn, an) = _group_ref(s["i"], s["g"], N, D, xyz_first)
        _assert_within(gf.reshape(B * N, D), sf, af, mf, what=what + " feat")
        _assert_within(gx.reshape(B * N, 3), sx, ax, mx, what=what + " xyz")
        _assert_within(gn, sn, an, K, what=what + " new_xyz")

    drive_backward(cuda_dev, sets, ["xyz", "new", "f"],
                   lambda s: ((P.group_points(s["xyz"], s["new"], s["f"], s["i"], xyz_first),), (s["g"],)), check)


def test_three_interpolate_backward_replays(cuda_dev):
    B, S, N, C = 2, 400, 3000, 16
    feats = _value_sets(88, (B, S, C))[:4]
    ws = [np.random.default_rng(89 + i).uniform(0.05, 1, size=(B, N, 3)).astype(F32) for i in range(5)]
    sets = [dict(f=f, i=i, w=w, g=g) for f, i, w, g in
            zip(feats + [feats[1], feats[0]], _interp_idx_sets(90, B, N, S), ws + [ws[0]], _gout_sets(91, (B, N, C)))]

    def check(got, s, what):
        out, gf, gw = got
        np.testing.assert_array_equal(out, strict.three_interpolate(s["f"], s["i"], s["w"]))
        (sf, af, mf), (sw, aw) = _interp_ref(s["g"], s["f"], s["i"], s["w"])
        _assert_within(gf, sf, af, mf, k=1, what=what + " gfeat")
        _assert_within(gw, sw, aw, C, k=1, what=what + " gweight")

    drive_backward(cuda_dev, sets, ["f", "w"], lambda s: ((P.three_interpolate(s["f"], s["i"], s["w"]),), (s["g"],)), check)


def _fp_grads64(dense, known, feat, gout, od, oi):
    """float64 gradient of feature propagation with differentiable coordinates: the distances' VALUES are the search's
    (od), their gradients those of |u - k|^2 (ops.three_nn_autograd)"""
    u = torch.from_numpy(dense).double().requires_grad_(True)
    kn = torch.from_numpy(known).double().requires_grad_(True)
    f = torch.from_numpy(feat).double().requires_grad_(True)
    idx = torch.from_numpy(oi)
    bi = torch.arange(u.shape[0])[:, None, None]
    diff = u.unsqueeze(2) - kn[bi, idx]
    dt = (diff * diff).sum(-1)
    d = torch.from_numpy(od).double() + (dt - dt.detach())
    inv = 1.0 / torch.where(d < 1e-10, torch.full_like(d, 1e-10), d)
    w = inv / inv.sum(2, keepdim=True)
    out = (f[bi, idx] * w.unsqueeze(-1)).sum(2)
    out.backward(torch.from_numpy(gout).double())
    return u.grad.numpy(), kn.grad.numpy(), f.grad.numpy()


def test_feature_propagation_coordinate_backward_replays(cuda_dev):
    B, N, S, C = 2, 2000, 400, 8
    clouds = cloud_sets(92, B, S, N, 3)[:4]
    known_dup = clouds[1][0].copy()
    known_dup[:, 1::2] = known_dup[:, ::2]                       # every known point twice: tied neighbours
    clouds = clouds + [(known_dup, clouds[1][1]), clouds[0]]
    feats = _value_sets(93, (B, S, C))[:4]
    sets = [dict(known=c[0], dense=c[1], f=f, g=g) for c, f, g in zip(clouds, feats + [feats[1], feats[0]], _gout_sets(94, (B, N, C)))]
    fn = lambda s: ((P.feature_propagation(s["dense"], s["known"], s["f"]),), (s["g"],))

    def check(got, s, what):
        # the replay against the eager call on the same set: the same kernels and torch ops, so only the order of the
        # atomic scatters differs
        st = {name: _dev(a, cuda_dev).requires_grad_(name != "g") for name, a in s.items()}
        eager = [_host(t) for t in _fwd_bwd(st, ["dense", "known", "f"], fn)]
        for name, g, w in zip(("out", "dense", "known", "feat"), got, eager):
            np.testing.assert_allclose(g, w, rtol=1e-5, atol=1e-6 * np.abs(w).max(), err_msg=what + " " + name)
        # and against float64 (test_gpu_round2's bar) where the weights' expanded-form distance values are well conditioned:
        # far from the origin (set 3) they carry the rounding of |q|^2 + |r|^2, which the fp32 chain through 1 / d amplifies
        # past any fixed tolerance
        if SETS[2] not in what:
            od, oi = strict.three_nn(s["dense"], s["known"])
            want = _fp_grads64(s["dense"], s["known"], s["f"], s["g"], od, oi)
            for name, g, w in zip(("dense", "known", "feat"), got[1:], want):
                np.testing.assert_allclose(g, w, rtol=2e-3, atol=1e-5 * np.abs(w).max(), err_msg=what + " " + name)

    drive_backward(cuda_dev, sets, ["dense", "known", "f"], fn, check)


def test_dense_chamfer_backward_replays(cuda_dev):
    B, N, M = 2, 2000, 1500
    clouds = cloud_sets(95, B, max(N, M), max(N, M), 1)[:4]
    clouds = clouds + [clouds[1], clouds[0]]
    scales = [1.0, -2.5, 0.75, 3.0, 0.5, 1.0]
    sets = [dict(x=c[0][:, :N].copy(), y=c[1][:, :M].copy(), g=np.array(sc, F32)) for c, sc in zip(clouds, scales)]

    def check(got, s, what):
        loss, ix, iy, gx, gy = got
        ol, _, oix, _, oiy = strict.chamfer(s["x"], s["y"])
        _loss_close(loss, ol, what + " loss")
        np.testing.assert_array_equal(ix, oix); np.testing.assert_array_equal(iy, oiy)
        (sx, ax, mx), (sy, ay, my) = _chamfer_ref(s["x"], s["y"], oix, oiy, float(s["g"]))
        _assert_within(gx.reshape(-1, 3), sx, ax, mx, k=4, what=what + " gx")
        _assert_within(gy.reshape(-1, 3), sy, ay, my, k=4, what=what + " gy")

    def fn(s):
        loss, _, ix, _, iy = ops.chamfer(s["x"], s["y"])
        return (loss,), (s["g"],), (ix, iy)

    drive_backward(cuda_dev, sets, ["x", "y"], fn, check)


def _ragged_chamfer_grad64(x, y, xl, yl, g):
    """float64 gradient of sum_b g[b] * loss[b] (point_reduction "mean", batch_reduction None) with the oracle's nearest
    neighbours (test_gpu_backward's _chamfer_ref for a ragged batch): x_i (i < nx) gets 2 g / nx (x_i - y_ix[i]) and y_ix[i]
    the negative; the y direction mirrors it.  Padded points and points without a candidate give and take nothing."""
    _, _, ix, _, iy = RO.chamfer_terms(x, y, xl, yl)
    B, N, M = x.shape[0], x.shape[1], y.shape[1]
    nx, ny = RO.clamp_lengths(xl, N, B), RO.clamp_lengths(yl, M, B)
    x64, y64, g = x.astype(np.float64), y.astype(np.float64), np.asarray(g, np.float64)
    bn = np.arange(B)[:, None]
    okx = (np.arange(N)[None] < nx[:, None]) & (ix >= 0)
    oky = (np.arange(M)[None] < ny[:, None]) & (iy >= 0)
    with np.errstate(invalid="ignore"):
        tx = (2.0 * g / np.maximum(nx, 1))[:, None, None] * (x64 - y64[bn, np.maximum(ix, 0)])
        ty = (2.0 * g / np.maximum(ny, 1))[:, None, None] * (y64 - x64[bn, np.maximum(iy, 0)])
    tx = np.where(okx[..., None], tx, 0.0).reshape(-1, 3)
    ty = np.where(oky[..., None], ty, 0.0).reshape(-1, 3)
    own_x = np.where(okx, bn * N + np.arange(N)[None], -1).reshape(-1)
    own_y = np.where(oky, bn * M + np.arange(M)[None], -1).reshape(-1)
    to_y = np.where(okx, ix + bn * M, -1).reshape(-1)
    to_x = np.where(oky, iy + bn * N, -1).reshape(-1)
    return (_scatter64(B * N, np.concatenate([own_x, to_x]), np.concatenate([tx, -ty])),
            _scatter64(B * M, np.concatenate([own_y, to_y]), np.concatenate([ty, -tx])))


def test_ragged_chamfer_backward_replays(cuda_dev):
    sets = _chamfer_sets(96)
    for i, s in enumerate(sets):
        s["g"] = np.linspace(0.5, 1.5, RAGGED_B).astype(F32) * F32([1, -2, 0.5, 3, 1.5, 1][i])

    def check(got, s, what):
        loss, gx, gy = got
        x64, y64 = torch.from_numpy(s["x"]).double(), torch.from_numpy(s["y"]).double()
        _loss_close(loss, RO.chamfer_distance64(x64, y64, s["xl"], s["yl"], "mean", None).numpy(), what + " loss")
        (sx, ax, mx), (sy, ay, my) = _ragged_chamfer_grad64(s["x"], s["y"], s["xl"], s["yl"], s["g"])
        _assert_within(gx.reshape(-1, 3), sx, ax, mx, k=4, what=what + " gx")
        _assert_within(gy.reshape(-1, 3), sy, ay, my, k=4, what=what + " gy")

    drive_backward(cuda_dev, sets, ["x", "y"],
                   lambda s: ((S3.chamfer_distance(s["x"], s["y"], x_lengths=s["xl"], y_lengths=s["yl"], batch_reduction=None)[0],),
                              (s["g"],)), check)


# ---- GraphedPointINet on new clouds ------------------------------------------------------------------------------------
def _frames(first, B, n, transform=None):
    a, b = synth.batch_pairs(first, B, n)
    if transform is not None:
        a, b = transform(a), transform(b)
    g = torch.Generator().manual_seed(first)
    p1 = torch.cat([torch.from_numpy(a).transpose(1, 2), torch.rand(B, 1, n, generator=g)], 1).contiguous()
    p2 = torch.cat([torch.from_numpy(b).transpose(1, 2), torch.rand(B, 1, n, generator=g)], 1).contiguous()
    z = torch.zeros(B, 3, n)
    return [p1, p2, z, z.clone()]


def _rotate_and_move(a):
    c, s = np.cos(0.6), np.sin(0.6)
    rot = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1]], np.float64)
    return (a.astype(np.float64) @ rot.T + [100.0, -60.0, 2.0]).astype(F32)


@pytest.mark.parametrize("B,n", [(2, 4096), (8, 16384)])
def test_graphed_pointinet_on_new_clouds(knobs, cuda_dev, B, n):
    """captured on pair 0; replayed on other scenes, on pair 0 rotated and moved by ~100 m, and on pinned host inputs.  Each
    result equals the eager forward under the same seed (no BN folding), at test_gpu_pointinet's bar.  Batch 2 x 4096 takes
    the side-stream fork of _concurrently; 8 x 16384 sends the fusion's k = 16 searches to the pruned search."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(0)
    eager = pointinet.PointINet().eval().to(cuda_dev)
    graphed = pointinet.GraphedPointINet(state_dict=eager.state_dict(), batch=B, npoints=n, extra=1, t=0.5, device=cuda_dev,
                                         fold_bn=False)
    inputs = {"pair 0": _frames(0, B, n), "other scene 1": _frames(B, B, n), "other scene 2": _frames(2 * B, B, n),
              "pair 0 rotated and moved": _frames(0, B, n, _rotate_and_move)}
    inputs["pinned host"] = [x.pin_memory() for x in _frames(3 * B, B, n)]
    knobs.set()
    _, plans, _ = knobs.run(lambda: graphed.capture(*[x.to(cuda_dev) for x in inputs["pair 0"]]))
    if B == 8:
        assert any(p["grid"] == "pruned" and (p["B"], p["N"], p["S"], p["k"]) == ("8", str(n), str(n), "16") for p in plans), plans
    t = torch.full((B,), 0.5, device=cuda_dev)
    first = None
    for i, (name, ins) in enumerate(list(inputs.items()) + [("pair 0 again", inputs["pair 0"])]):
        torch.manual_seed(100 + i)
        with torch.no_grad():
            want = eager(*[x.to(cuda_dev) for x in ins], t)
        if first is None:
            first = want
        elif name != "pair 0 again":
            assert not torch.equal(want, first), name
        torch.manual_seed(100 + i)
        got = graphed(*(ins if name == "pinned host" else [x.to(cuda_dev) for x in ins])).clone()
        err = (got - want).abs().amax(dim=1).reshape(-1)
        assert (err < 5e-5).float().mean() > 0.995, (name, float(err.max()), float((err < 5e-5).float().mean()))


# ---- off the current device --------------------------------------------------------------------------------------------
def _two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs (tensors on cuda:1 while cuda:0 is current)")
    return torch.device("cuda:0"), torch.device("cuda:1")


def _default_plan_calls(seed):
    """(name, call on device tensors, oracle) of the forward matrix's default-plan cases"""
    (ref, qry) = cloud_sets(seed, 2, 5000, 700, 16)[0]
    small = cloud_sets(seed + 1, 2, 900, 300, 16)[0]
    feat = np.random.default_rng(seed).normal(size=(2, 5000, 8)).astype(F32)
    idx = np.random.default_rng(seed + 2).integers(-5000, 5000, size=(2, 700, 16))
    start = np.array([3, 4000])
    x, y = ref[:, :3000].copy(), qry
    return [
        ("knn_point", lambda d: P.knn_point(16, d(ref), d(qry)), lambda: strict.knn_point(16, ref, qry)),
        ("knn_points", lambda d: S3.knn_points(d(qry), d(ref), K=16).dists, lambda: strict.knn(ref, qry, 16, 2)[1]),
        ("knn small", lambda d: P.knn_point(16, d(small[0]), d(small[1])), lambda: strict.knn_point(16, *small)),
        ("three_nn", lambda d: P.three_nn(d(qry), d(ref))[1], lambda: strict.three_nn(qry, ref)[1]),
        ("knn_search_i32", lambda d: ops.knn_search_i32(d(ref), d(qry), 16, 0), lambda: strict.knn_point(16, ref, qry).astype(np.int32)),
        ("ball_query", lambda d: P.query_ball_point(RADIUS, NSAMPLE, d(ref), d(qry)),
         lambda: strict.query_ball_point(RADIUS, NSAMPLE, ref, qry)),
        ("fps", lambda d: P.farthest_point_sample_from(d(ref), 300, d(start)), lambda: strict.farthest_point_sample(ref, 300, start)),
        ("index_points", lambda d: P.index_points(d(feat), d(idx)), lambda: strict.index_points(feat, idx)),
        ("group_points", lambda d: P.group_points(d(ref), d(qry), d(feat), d(idx)), lambda: strict.group_points(ref, qry, feat, idx)),
        ("feature_propagation", lambda d: P.feature_propagation(d(qry), d(ref), d(feat)),
         lambda: strict.three_interpolate(feat, *(lambda od, oi: (oi, strict.three_weights(od, 0)))(*strict.three_nn(qry, ref)))),
        ("fusion_group", lambda d: P.fusion_group(d(qry), d(ref), 16, d(feat))[3], lambda: strict.knn_points(qry, ref, 16)[1]),
        ("square_distance", lambda d: P.square_distance(d(qry), d(small[0])), lambda: strict.square_distance(qry, small[0])),
        ("chamfer", lambda d: ops.chamfer(d(x), d(y))[2], lambda: strict.chamfer(x, y)[2]),
    ]


def test_default_plans_off_the_current_device_interleaved(cuda_dev):
    dev0, dev1 = _two_gpus()
    torch.cuda.set_device(dev0)
    for name, call, oracle in _default_plan_calls(101):
        want = oracle()
        for dev in (dev1, dev0, dev1):                    # the per-thread SM-count cache flips on every call
            got = _host(call(lambda a: _dev(a, dev)))
            assert torch.cuda.current_device() == 0
            _exact([got], [want], "%s on %s" % (name, dev))


def test_search_and_fps_graphs_on_the_second_device(cuda_dev):
    dev0, dev1 = _two_gpus()
    torch.cuda.set_device(dev0)
    with torch.cuda.device(dev1):
        drive(None, dev1, _sets(cloud_sets(103, 2, 5000, 700, 16)), lambda s: (P.knn_point(16, s["ref"], s["qry"]),),
              lambda s: (strict.knn_point(16, s["ref"], s["qry"]),))
        drive(None, dev1, _fps_sets(104, 2, 20000), lambda s: (P.farthest_point_sample_from(s["xyz"], 300, s["start"]),),
              lambda s: (strict.farthest_point_sample(s["xyz"], 300, s["start"]),))
    assert torch.cuda.current_device() == 0
