"""The PyTorch face of every op: torch.library.opcheck, torch.compile, autocast and the tensors real callers pass, against
eager and the oracle.

The kernels sit behind two Python layers: the `torch.library` registration in b200pc/ops.py (schemas, fake kernels,
autograd formulas) and the public functions that normalise a caller's tensors before the C ABI sees them.  A wrong fake
shape, stride or dtype, a backward formula that drops a term, or a view the facade hands on unaligned passes every test
that calls the ops eagerly on fresh contiguous tensors.  Here:

  * opcheck with every test util (test_aot_dispatch_dynamic included) on all 23 ops, on a small and an edge input each;
  * torch.compile(fullgraph=True), dynamic shapes on and off, of every public function: equal to eager bit for bit on two
    input sets of one shape and on a new shape, and equal to oracle/strict on the first; forward and backward compiled
    together for the differentiable ops; the CPU-RNG draw of farthest_point_sample under inductor; the PointINet mirror;
  * autocast (fp16, bf16) and fp16 / bf16 / fp64 inputs: the fp32 call's outputs and dtypes, bit for bit;
  * channel-first views, storage offsets of 4, 8 and 12 bytes, batch slices, stride-0 batches and int32 / uint8 /
    strided int64 indices, against the oracle.

Bar (DESIGN section 2): indices, distances, gathers, groupings and interpolations bit-exact; weights and Chamfer values within
1e-5; gradients within the float64 summation bound of test_gpu_backward.py.
"""
import types

import numpy as np
import pytest
import torch

import ragged_oracle as RO
from b200pc import ops, pointnet2_utils as P, pytorch3d_shim as S3
from oracle import strict
from test_gpu_backward import U, _assert_within, _chamfer_ref, _gather_ref, _group_ref, _interp_ref
from test_gpu_graph_replay import _exact, _fp_grads64, _fusion_oracle, _loss_close, _ragged_chamfer_grad64

pytestmark = pytest.mark.gpu

F32 = np.float32
SHAPES = [dict(B=2, N=201, S=71), dict(B=2, N=201, S=71), dict(B=3, N=255, S=101)]    # two sets of one shape, then a new one
K = 8                                                                                 # neighbours; N stays < 256 for uint8 indices


# ---- the public functions, their inputs and their oracles --------------------------------------------------------------
def _cloud(rng, B, n):
    return rng.normal(size=(B, n, 3)).astype(F32)


def _pair(seed, sh):
    rng = np.random.default_rng(seed)
    return rng, _cloud(rng, sh["B"], sh["N"]), _cloud(rng, sh["B"], sh["S"])


def _lens(values, B):
    return np.array(values[:B], np.int64)


def _weights_close(got, want, what):
    assert got.shape == want.shape, what
    assert (np.abs(got - want) <= 1e-5 * np.abs(want) + 1e-30).all(), what


class Case:
    """make(seed, shape) -> dict of numpy inputs (fp32 values, int64 indices, lists of arrays); call(tensors) -> outputs;
    oracle(numpy inputs) -> expected outputs; check(got, want, what) compares them (default: bit-exact)"""

    def __init__(self, make, call, oracle, check=_exact):
        self.make, self.call, self.oracle, self.check = make, call, oracle, check


def _ref_qry(seed, sh):
    _, ref, qry = _pair(seed, sh)
    return dict(ref=ref, qry=qry)


def _ragged(seed, sh):
    d = _ref_qry(seed, sh)
    d["rl"] = _lens([9, sh["N"], 0], sh["B"])                 # fewer than k refs / full / none
    d["ql"] = _lens([sh["S"], sh["S"] - 3, 4], sh["B"])
    return d


def _ball(seed, sh):
    d = _ref_qry(seed, sh)
    d["qry"][:, -1] = 100.0                                   # an empty ball: N in every slot
    return d


def _fps_in(seed, sh):
    rng, ref, _ = _pair(seed, sh)
    return dict(xyz=ref, start=rng.integers(0, sh["N"], sh["B"]))


def _gather_in(seed, sh):
    rng, _, _ = _pair(seed, sh)
    return dict(p=rng.normal(size=(sh["B"], sh["N"], 8)).astype(F32), i=rng.integers(0, sh["N"], (sh["B"], sh["S"], 4)))


def _group_in(seed, sh):
    rng, ref, qry = _pair(seed, sh)
    return dict(xyz=ref, new=qry, f=rng.normal(size=(sh["B"], sh["N"], 8)).astype(F32),
                i=rng.integers(0, sh["N"], (sh["B"], sh["S"], 6)))


def _interp_in(seed, sh):
    rng, _, _ = _pair(seed, sh)
    B, N, S = sh["B"], sh["N"], sh["S"]
    return dict(f=rng.normal(size=(B, S, 8)).astype(F32), i=rng.integers(0, S, (B, N, 3)),
                w=rng.uniform(0.05, 1.0, (B, N, 3)).astype(F32))


def _fp_in(seed, sh):
    rng, dense, known = _pair(seed, sh)
    return dict(dense=dense, known=known, f=rng.normal(size=(sh["B"], sh["S"], 8)).astype(F32))


def _fusion_in(cf):
    def make(seed, sh):
        rng, ref, qry = _pair(seed, sh)
        d = dict(ref=ref, qry=qry)
        if cf:
            d["f"] = rng.normal(size=(sh["B"], sh["N"], cf)).astype(F32)
        return d
    return make


def _rows_in(seed, sh):
    rng = np.random.default_rng(seed)
    return dict(x=rng.normal(size=(sh["B"] * sh["S"], 12)).astype(F32))


def _chamfer_in(seed, sh):
    _, x, y = _pair(seed, sh)
    return dict(x=x, y=y)


def _chamfer_ragged_in(seed, sh):
    d = _chamfer_in(seed, sh)
    d["xl"] = _lens([sh["N"], 5, 0], sh["B"])
    d["yl"] = _lens([sh["S"] - 2, sh["S"], 0], sh["B"])       # item 2: both clouds empty
    return d


def _chamfer_shim_in(seed, sh):
    d = _chamfer_in(seed, sh)
    d["xl"] = _lens([sh["N"], 5, 0], sh["B"])
    d["yl"] = _lens([sh["S"] - 2, 0, 3], sh["B"])             # an empty y cloud, an empty x cloud
    return d


def _poly_in(seed, sh):
    rng = np.random.default_rng(seed)
    B = sh["B"]
    return dict(frames=[rng.normal(size=(B, 3, sh["S"])).astype(F32) for _ in range(3)], w=rng.normal(size=(B, 3)))


def _knn_points_in(seed, sh):
    d = _ref_qry(seed, sh)
    d["l1"] = _lens([sh["S"], 0, 4], sh["B"])
    d["l2"] = _lens([5, sh["N"], sh["N"]], sh["B"])
    return d


def _knn_gather_in(seed, sh):
    d = _gather_in(seed, sh)
    d["len"] = _lens([2, sh["N"], 0], sh["B"])
    return d


def _fp_oracle(d):
    od, oi = strict.three_nn(d["dense"], d["known"])
    return (strict.three_interpolate(d["f"], oi, strict.three_weights(od, 0)),)


def _three_nn_check(got, want, what):
    _exact(got[:2], want[:2], what)
    _weights_close(got[2], want[2], what + " weights")


def _chamfer_check(got, want, what):
    _loss_close(got[0], want[0], what + " loss")
    _exact(got[1:], want[1:], what)


def _chamfer_ragged_oracle(d):
    sums, dx, ix, dy, iy = RO.chamfer_terms(d["x"], d["y"], d["xl"], d["yl"])
    x64, y64 = torch.from_numpy(d["x"]).double(), torch.from_numpy(d["y"]).double()
    return RO.chamfer_distance64(x64, y64, d["xl"], d["yl"]).numpy(), sums, dx, ix, dy, iy


def _chamfer_ragged_check(got, want, what):
    _loss_close(got[0], want[0], what + " loss")
    _loss_close(got[1], want[1], what + " sums")
    _exact(got[2:], want[2:], what)


def _poly_oracle(d):
    B, Fr = d["w"].shape
    acc = sum(d["w"][:, f].reshape(B, 1, 1) * d["frames"][f].astype(np.float64) for f in range(Fr))
    mag = sum(np.abs(d["w"][:, f].reshape(B, 1, 1) * d["frames"][f].astype(np.float64)) for f in range(Fr))
    return acc, mag


def _poly_check(got, want, what):
    acc, mag = want
    g = got[0].astype(np.float64)
    assert g.shape == acc.shape, what
    assert (np.abs(g - acc) <= U * np.abs(acc) + 2 * 3 * 2.0 ** -53 * mag + 1e-38).all(), what    # one fp32 rounding


def _knn_points_oracle(d, lengths):
    B, S, N = d["qry"].shape[0], d["qry"].shape[1], d["ref"].shape[1]
    l1, l2 = (d["l1"], d["l2"]) if lengths else (None, None)
    oi, od = RO.knn(d["ref"], d["qry"], l2, l1, K, strict.FORM_DIRECT)
    n1, n2 = RO.clamp_lengths(l1, S, B), RO.clamp_lengths(l2, N, B)
    pad = (np.arange(S)[None, :, None] >= n1[:, None, None]) | (np.arange(K)[None, None, :] >= n2[:, None, None])
    oi = np.where(pad, 0, oi)
    return np.where(pad, F32(0), od), oi, np.where(pad[..., None], F32(0), strict.index_points(d["ref"], oi))


def _knn_gather_oracle(d, lengths):
    out = strict.index_points(d["p"], d["i"])
    if lengths:
        out = np.where((np.arange(d["i"].shape[-1])[None, :] >= d["len"][:, None])[:, None, :, None], F32(0), out)
    return (out,)


def _rebuild_oracle(d):
    _, oi = strict.knn_points(d["qry"], d["ref"], 1)
    oi = oi[..., 0]
    rec = np.concatenate([oi.astype(np.int32).view(F32)[..., None], strict.index_points(d["ref"], oi)], -1).transpose(1, 0, 2)
    return rec, oi, strict.index_points(d["ref"], oi)


CASES = {
    "square_distance": Case(_ref_qry, lambda t: P.square_distance(t["qry"], t["ref"]),
                            lambda d: (strict.square_distance(d["qry"], d["ref"]),)),
    "knn_search_form0": Case(_ref_qry, lambda t: ops.knn_search(t["ref"], t["qry"], K, ops.FORM_REF_NORM_FIRST),
                             lambda d: (strict.knn(d["ref"], d["qry"], K, 0)[0],)),
    "knn_search_form2": Case(_ref_qry, lambda t: ops.knn_search(t["ref"], t["qry"], K, ops.FORM_DIRECT, want_dist=True),
                             lambda d: strict.knn(d["ref"], d["qry"], K, 2)),
    "knn_ragged": Case(_ragged, lambda t: ops.knn_ragged(t["ref"], t["qry"], K, ops.FORM_DIRECT, t["rl"], t["ql"], want_dist=True),
                       lambda d: RO.knn(d["ref"], d["qry"], d["rl"], d["ql"], K, 2)),
    "knn_search_i32": Case(_ref_qry, lambda t: ops.knn_search_i32(t["ref"], t["qry"], K, ops.FORM_REF_NORM_FIRST),
                           lambda d: (strict.knn(d["ref"], d["qry"], K, 0)[0],)),
    "ball_query": Case(_ball, lambda t: P.query_ball_point(0.6, K, t["ref"], t["qry"]),
                       lambda d: (strict.query_ball_point(0.6, K, d["ref"], d["qry"]),)),
    "fps": Case(_fps_in, lambda t: P.farthest_point_sample_from(t["xyz"], 32, t["start"]),
                lambda d: (strict.farthest_point_sample(d["xyz"], 32, d["start"]),)),
    "sample_points": Case(_fps_in, lambda t: P.sample_points(t["xyz"], 32, t["start"]),
                          lambda d: (strict.farthest_point_sample(d["xyz"], 32, d["start"]),
                                     strict.index_points(d["xyz"], strict.farthest_point_sample(d["xyz"], 32, d["start"])))),
    "gather": Case(_gather_in, lambda t: P.index_points(t["p"], t["i"]), lambda d: (strict.index_points(d["p"], d["i"]),)),
    "group_points_xyz_first": Case(_group_in, lambda t: P.group_points(t["xyz"], t["new"], t["f"], t["i"], True),
                                   lambda d: (strict.group_points(d["xyz"], d["new"], d["f"], d["i"], True),)),
    "group_points_feat_first": Case(_group_in, lambda t: P.group_points(t["xyz"], t["new"], t["f"], t["i"], False),
                                    lambda d: (strict.group_points(d["xyz"], d["new"], d["f"], d["i"], False),)),
    "three_nn": Case(_fp_in, lambda t: ops.three_nn(t["dense"], t["known"]),
                     lambda d: (*strict.three_nn(d["dense"], d["known"]),
                                strict.three_weights(strict.three_nn(d["dense"], d["known"])[0], 0)), _three_nn_check),
    "three_interpolate": Case(_interp_in, lambda t: P.three_interpolate(t["f"], t["i"], t["w"]),
                              lambda d: (strict.three_interpolate(d["f"], d["i"], d["w"]),)),
    "feature_propagation": Case(_fp_in, lambda t: P.feature_propagation(t["dense"], t["known"], t["f"]), _fp_oracle),
    "fusion_group": Case(_fusion_in(0), lambda t: [o for j, o in enumerate(P.fusion_group(t["qry"], t["ref"], K)) if j != 2],
                         lambda d: _fusion_oracle(d["qry"], d["ref"], None, K)),
    "fusion_group_feat": Case(_fusion_in(5), lambda t: P.fusion_group(t["qry"], t["ref"], K, t["f"]),
                              lambda d: _fusion_oracle(d["qry"], d["ref"], d["f"], K)),
    "channel_max": Case(_rows_in, lambda t: ops.channel_max(t["x"]), lambda d: (d["x"].max(1),)),
    "rebuild_pack": Case(_ref_qry, lambda t: (lambda r: (r, *ops.unpack_rebuild(r)))(ops.rebuild_pack(t["ref"], t["qry"])),
                         _rebuild_oracle),
    "chamfer": Case(_chamfer_in, lambda t: ops.chamfer(t["x"], t["y"]), lambda d: strict.chamfer(d["x"], d["y"]), _chamfer_check),
    "chamfer_ragged": Case(_chamfer_ragged_in,
                           lambda t: (lambda r: (ops.chamfer_reduce(r[0], t["xl"], t["yl"], t["x"].shape[1], t["y"].shape[1]), *r))(
                               ops.chamfer_ragged(t["x"], t["y"], t["xl"], t["yl"])),
                           _chamfer_ragged_oracle, _chamfer_ragged_check),
    "poly_predict": Case(_poly_in, lambda t: ops.poly_predict(t["frames"], t["w"]), _poly_oracle, _poly_check),
    "knn_points": Case(_knn_points_in, lambda t: S3.knn_points(t["qry"], t["ref"], K=K, return_nn=True),
                       lambda d: _knn_points_oracle(d, False)),
    "knn_points_lengths": Case(_knn_points_in, lambda t: S3.knn_points(t["qry"], t["ref"], t["l1"], t["l2"], K=K, return_nn=True),
                               lambda d: _knn_points_oracle(d, True)),
    "knn_gather": Case(_knn_gather_in, lambda t: S3.knn_gather(t["p"], t["i"]), lambda d: _knn_gather_oracle(d, False)),
    "knn_gather_lengths": Case(_knn_gather_in, lambda t: S3.knn_gather(t["p"], t["i"], t["len"]), lambda d: _knn_gather_oracle(d, True)),
    "chamfer_distance": Case(_chamfer_in, lambda t: S3.chamfer_distance(t["x"], t["y"])[0],
                             lambda d: (strict.chamfer(d["x"], d["y"])[0],), lambda g, w, what: _loss_close(g[0], w[0], what)),
    "chamfer_distance_lengths": Case(
        _chamfer_shim_in, lambda t: S3.chamfer_distance(t["x"], t["y"], t["xl"], t["yl"])[0],
        lambda d: (RO.chamfer_distance64(torch.from_numpy(d["x"]).double(), torch.from_numpy(d["y"]).double(), d["xl"], d["yl"]).numpy(),),
        lambda g, w, what: _loss_close(g[0], w[0], what)),
}


# ---- plumbing -----------------------------------------------------------------------------------------------------------
def _flat(out):
    """outputs as a flat list of tensors (tuples, lists and namedtuples flattened, None dropped)"""
    if out is None:
        return []
    if isinstance(out, torch.Tensor):
        return [out]
    return [t for o in out for t in _flat(o)]


def _host(outs):
    return [o.detach().cpu().numpy() for o in outs]


def _dev(d, dev, fn=None):
    """numpy inputs -> device tensors; fn(array) -> tensor replaces the plain contiguous upload"""
    up = fn or (lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev))
    return {k: ([up(x) for x in v] if isinstance(v, list) else up(v)) for k, v in d.items()}


def _bits_equal(got, want, what):
    got, want = _flat(got), _flat(want)
    assert len(got) == len(want), (what, len(got), len(want))
    for i, (g, w) in enumerate(zip(got, want)):
        assert g.dtype == w.dtype and g.shape == w.shape, (what, i, g.dtype, w.dtype, g.shape, w.shape)
        g8 = g.detach().reshape(-1).contiguous().view(torch.uint8)
        w8 = w.detach().reshape(-1).contiguous().view(torch.uint8)
        assert torch.equal(g8, w8), "%s: output %d differs from eager" % (what, i)


def _check_oracle(case, d, outs, what):
    case.check(_host(_flat(outs)), case.oracle(d), what)


@pytest.fixture
def fresh_dynamo(monkeypatch):
    """every compile test starts from an empty dynamo cache (the case lambdas share code objects), with inductor's fp32
    division correctly rounded like eager's (Triton's default x / y is approximate, which moves the last bit of the torch
    arithmetic the facade does after the ops: chamfer_reduce, the differentiable three-NN weights), and with CPU tensors
    left to ATen (the host RNG draw and t's host copy need no C++ toolchain)"""
    import torch._inductor.config as ic
    monkeypatch.setattr(ic.eager_numerics, "division_rounding", True)
    monkeypatch.setattr(ic, "disable_cpp_codegen", True)
    torch._dynamo.reset()
    yield
    torch._dynamo.reset()


# ---- 1. opcheck ---------------------------------------------------------------------------------------------------------
def _opcheck_samples(dev):
    """-> (op name -> list of (label, args): a small input and the edge inputs of each op; buffers the caller keeps alive).
    rebuild_pack's peer buffer is passed as a raw address: the tensor behind it must outlive every call, or the kernel
    writes into whatever the allocator has put there since (opcheck's clones of the inputs, for one)."""
    g = torch.Generator().manual_seed(11)
    r = lambda *s: torch.randn(*s, generator=g).to(dev)
    i64 = lambda hi, *s: torch.randint(0, hi, s, generator=g).to(dev)
    lens = lambda *v: torch.tensor(v, dtype=torch.int64, device=dev)
    grad = lambda t: t.clone().requires_grad_(True)
    ref, qry, feat = r(2, 40, 3), r(2, 17, 3), r(2, 40, 16)
    idx = torch.ops.b200pc.knn(ref, qry, 4, 0, False)[0]
    idx3 = i64(40, 2, 17, 3)
    w3 = torch.rand(2, 17, 3, generator=g).to(dev)
    x1, y1 = r(3, 1, 3), r(3, 9, 3)                               # a one-point cloud
    cx, cy = r(3, 30, 3), r(3, 20, 3)
    ix, iy = torch.ops.b200pc.chamfer_fwd(cx, cy)[2], torch.ops.b200pc.chamfer_fwd(cx, cy)[4]
    rl, rix, riy = (lens(0, 7, 30), lens(20, 0, 3)), *torch.ops.b200pc.chamfer_ragged_fwd(cx, cy, lens(0, 7, 30), lens(20, 0, 3))[2::2]
    peer = torch.zeros(17, 2, 4, device=dev)
    return {
        "square_distance": [("small", (qry, ref)), ("S=0", (qry[:, :0], ref))],
        "knn": [("small", (ref, qry, 4, 0, True)), ("k=N", (ref, qry, 40, 2, True)), ("S=0", (ref, qry[:, :0], 4, 1, False))],
        "knn_ragged": [("lengths 0 / <k / full", (r(3, 40, 3), r(3, 17, 3), lens(0, 3, 40), lens(17, 5, 0), 4, 2, True)),
                       ("no lengths, k=N", (ref, qry, None, None, 40, 0, False))],
        "knn_i32": [("small", (ref, qry, 4, 0)), ("k=N", (ref, qry, 40, 2)), ("B=0", (ref[:0], qry[:0], 4, 0))],
        "ball_query": [("small", (ref, qry, 0.5, 8)), ("S=0", (ref, qry[:, :0], 0.5, 8))],
        "fps": [("small", (ref, 10, i64(40, 2))), ("npoint=N", (ref, 40, i64(40, 2))), ("B=0", (ref[:0], 5, i64(40, 0)))],
        "fps_sample": [("small", (ref, 10, i64(40, 2))), ("npoint=N", (ref, 40, i64(40, 2)))],
        "gather": [("small", (grad(feat), idx.reshape(2, -1), False)), ("checked, R=0", (grad(feat), idx[:, :0, 0], True))],
        "gather_bwd": [("small", (r(2, 68, 16), idx.reshape(2, -1), 40)), ("C=1", (r(2, 68, 1), idx.reshape(2, -1), 40))],
        "group_points": [("small", (grad(ref), grad(qry), grad(feat), idx, True)),
                         ("feat=None", (grad(ref), grad(qry), None, idx, False)),
                         ("S=0", (ref, qry[:, :0], feat, idx[:, :0], True))],
        "group_points_bwd": [("small", (r(2, 19, 4, 17), idx, 40, 16, True)), ("features first", (r(2, 19, 4, 17), idx, 40, 16, False))],
        "three_nn": [("small", (qry, ref, 0, True)), ("3 known, no weights", (qry, ref[:, :3].contiguous(), 1, False))],
        "three_interpolate": [("small", (grad(r(2, 40, 8)), idx3, grad(w3))),
                              ("N=0", (grad(r(2, 40, 8)), idx3[:, :0], grad(w3[:, :0])))],
        "three_interpolate_bwd": [("small", (r(2, 17, 8), r(2, 40, 8), idx3, w3, True)), ("no gweight", (r(2, 17, 8), r(2, 40, 8), idx3, w3, False))],
        "feature_propagation": [("small", (qry, ref, grad(r(2, 40, 8)), 0)), ("3 known", (qry, ref[:, :3].contiguous(), grad(r(2, 3, 1)), 1)),
                                ("N=0", (qry[:, :0], ref, grad(r(2, 40, 8)), 0))],
        "fusion_group": [("small", (qry, ref, feat, 4)), ("feat=None, k=N", (qry, ref, None, 40)), ("S=0", (qry[:, :0], ref, feat, 4))],
        "channel_max": [("small", (r(37, 12),)), ("C=4", (r(5, 4),)), ("rows=0", (r(0, 8),))],
        "rebuild_pack": [("no peers", (ref, qry, 0, [])), ("one peer", (ref, qry, 0, [peer.data_ptr()])), ("S=0", (ref, qry[:, :0], 0, []))],
        "chamfer_fwd": [("small", (grad(cx), grad(cy))), ("N=1", (grad(x1), grad(y1)))],
        "chamfer_bwd": [("small", (cx, cy, ix, iy, r(1))), ("N=1", (x1, y1, *torch.ops.b200pc.chamfer_fwd(x1, y1)[2::2], r(1)))],
        "chamfer_ragged_fwd": [("lengths 0 / part / full", (grad(cx), grad(cy), *rl)), ("no lengths", (grad(cx), grad(cy), None, None))],
        "chamfer_ragged_bwd": [("small", (cx, cy, rix, riy, *rl, r(3, 2))), ("no lengths", (cx, cy, ix, iy, None, None, r(3, 2)))],
        "poly_predict": [("F=1", ([r(2, 3, 50)], r(2, 1).double())), ("F=16", ([r(2, 3, 50) for _ in range(16)], r(2, 16).double()))],
    }, [peer]


def test_torch_ops_pass_opcheck(cuda_dev):
    """every op of OP_SCHEMAS on its small and edge inputs: schema, fake kernel (shapes, strides, dtypes, symbolic shapes),
    autograd registration and AOT dispatch with dynamic shapes agree with what the CUDA implementation returns.  Every op and
    input runs; the failures are reported together."""
    samples, peers = _opcheck_samples(cuda_dev)
    assert set(samples) == set(ops.OP_SCHEMAS), set(ops.OP_SCHEMAS) ^ set(samples)
    failures = []
    for name in sorted(samples):
        assert len(samples[name]) >= 2, name
        for label, args in samples[name]:
            try:
                torch.library.opcheck(getattr(torch.ops.b200pc, name), args)
            except Exception as e:                              # noqa: BLE001  (collected, reported below)
                failures.append("%s (%s): %s" % (name, label, str(e).split("\n")[0]))
    assert not failures, "opcheck failed on %d input(s):\n%s" % (len(failures), "\n".join(failures))
    # the peer buffer (still alive) holds the records of the last call
    ref, qry = samples["rebuild_pack"][1][1][:2]
    assert torch.equal(peers[0].view(torch.int32), ops.rebuild_pack(ref, qry).view(torch.int32))


# ---- 2. torch.compile ---------------------------------------------------------------------------------------------------
# chamfer_reduce's batch mean divides by the Python int B.  Eager CUDA multiplies by its fp32 reciprocal (a CPU scalar
# divisor); with dynamic shapes inductor divides by the symbolic size instead, one rounding apart.  Every op output stays
# bit-exact; the reduced loss is held to one rounding there.
_DYNAMIC_GLUE = {"chamfer_ragged"}


@pytest.mark.parametrize("dynamic", [False, True], ids=["static", "dynamic"])
@pytest.mark.parametrize("name", list(CASES))
def test_compiled_equals_eager(cuda_dev, fresh_dynamo, name, dynamic):
    case = CASES[name]
    fn = torch.compile(case.call, fullgraph=True, dynamic=dynamic)
    for i, sh in enumerate(SHAPES):
        d = case.make(100 + i, sh)
        t = _dev(d, cuda_dev)
        want = case.call(t)
        got = fn(t)
        if dynamic and name in _DYNAMIC_GLUE:
            g0, w0 = _host(_flat(got)[:1])[0], _host(_flat(want)[:1])[0]
            assert (np.abs(g0 - w0) <= 2 * U * np.abs(w0)).all(), "%s, set %d: loss beyond one rounding" % (name, i)
            _bits_equal(_flat(got)[1:], _flat(want)[1:], "%s, set %d" % (name, i))
        else:
            _bits_equal(got, want, "%s, set %d" % (name, i))
        if i == 0:
            _check_oracle(case, d, got, name + " compiled")


def _leaves(d, dev, grads):
    t = _dev(d, dev)
    for k in grads:
        t[k].requires_grad_(True)
    return t


AUTOGRAD = {
    # name: (make, forward(t), names that require grad)
    "index_points": (_gather_in, lambda t: P.index_points(t["p"], t["i"]), ["p"]),
    "group_points_xyz_first": (_group_in, lambda t: P.group_points(t["xyz"], t["new"], t["f"], t["i"], True), ["xyz", "new", "f"]),
    "group_points_feat_first": (_group_in, lambda t: P.group_points(t["xyz"], t["new"], t["f"], t["i"], False), ["xyz", "new", "f"]),
    "three_interpolate": (_interp_in, lambda t: P.three_interpolate(t["f"], t["i"], t["w"]), ["f", "w"]),
    "feature_propagation": (_fp_in, lambda t: P.feature_propagation(t["dense"], t["known"], t["f"]), ["f"]),
    "feature_propagation_coordinates": (_fp_in, lambda t: P.feature_propagation(t["dense"], t["known"], t["f"]), ["dense", "known", "f"]),
    "chamfer": (_chamfer_in, lambda t: ops.chamfer(t["x"], t["y"])[0], ["x", "y"]),
    "chamfer_distance_lengths": (_chamfer_ragged_in, lambda t: S3.chamfer_distance(t["x"], t["y"], t["xl"], t["yl"], batch_reduction=None)[0],
                                 ["x", "y"]),
}


def _permuted(name, d, sh):
    """the same inputs with every index a permutation: each gradient row receives one term, so every kernel-made gradient
    is deterministic and compiled must equal eager bit for bit"""
    rng = np.random.default_rng(7)
    B, N = sh["B"], sh["N"]
    d = dict(d)
    if name == "index_points":
        d["i"] = np.stack([rng.permutation(N) for _ in range(B)])
    elif name.startswith("group_points"):
        S = N // 3                                               # S * K == N with K = 3
        d["new"], d["i"] = d["new"][:, :S].copy(), np.stack([rng.permutation(N) for _ in range(B)]).reshape(B, S, 3)
    elif name == "three_interpolate":                            # 3N known rows, each read once
        d["f"] = rng.normal(size=(B, N * 3, d["f"].shape[2])).astype(F32)
        d["i"] = np.stack([rng.permutation(N * 3) for _ in range(B)]).reshape(B, N, 3)
    return d


def _grad_bound(name, d, t, grads, gout):
    """the float64 bound of test_gpu_backward.py (what every gradient must meet, eager or compiled); t: the device inputs"""
    B = next(iter(d.values())).shape[0]
    if name == "index_points":
        N, C = d["p"].shape[1], d["p"].shape[2]
        s, a, m = _gather_ref(gout.reshape(B, -1, C), d["i"].reshape(B, -1), N)
        _assert_within(grads[0], s, a, m, what=name)
    elif name.startswith("group_points"):
        N, D = d["xyz"].shape[1], d["f"].shape[2]
        (sf, af, mf), (sx, ax, mx), (sn, an) = _group_ref(d["i"], gout, N, D, name.endswith("xyz_first"))
        gx, gn, gf = grads
        _assert_within(gf.reshape(B * N, D), sf, af, mf, what=name + " feat")
        _assert_within(gx.reshape(B * N, 3), sx, ax, mx, what=name + " xyz")
        _assert_within(gn, sn, an, d["i"].shape[2], what=name + " new_xyz")
    elif name == "three_interpolate":
        (sf, af, mf), (sw, aw) = _interp_ref(gout, d["f"], d["i"], d["w"])
        _assert_within(grads[0], sf, af, mf, k=1, what=name + " gfeat")
        _assert_within(grads[1], sw, aw, d["f"].shape[2], k=1, what=name + " gweight")
    elif name == "feature_propagation":                           # the terms of the op's own indices and weights
        _, oi, ow = torch.ops.b200pc.feature_propagation(t["dense"], t["known"], t["f"].detach(), 0)
        (sf, af, mf), _ = _interp_ref(gout, d["f"], oi.cpu().numpy(), ow.cpu().numpy())
        _assert_within(grads[0], sf, af, mf, k=1, what=name + " gfeat")
    elif name == "feature_propagation_coordinates":
        od, oi = strict.three_nn(d["dense"], d["known"])
        want = _fp_grads64(d["dense"], d["known"], d["f"], gout, od, oi)
        for what, g, w in zip(("dense", "known", "feat"), grads, want):
            np.testing.assert_allclose(g, w, rtol=2e-3, atol=1e-5 * np.abs(w).max(), err_msg=name + " " + what)
    elif name == "chamfer":
        _, _, oix, _, oiy = strict.chamfer(d["x"], d["y"])
        (sx, ax, mx), (sy, ay, my) = _chamfer_ref(d["x"], d["y"], oix, oiy, float(gout))
        _assert_within(grads[0].reshape(-1, 3), sx, ax, mx, k=4, what=name + " gx")
        _assert_within(grads[1].reshape(-1, 3), sy, ay, my, k=4, what=name + " gy")
    else:
        (sx, ax, mx), (sy, ay, my) = _ragged_chamfer_grad64(d["x"], d["y"], d["xl"], d["yl"], gout)
        _assert_within(grads[0].reshape(-1, 3), sx, ax, mx, k=4, what=name + " gx")
        _assert_within(grads[1].reshape(-1, 3), sy, ay, my, k=4, what=name + " gy")


# gradients that eager computes deterministically whatever the indices (no atomic scatter, no torch reduction that inductor
# may regenerate in another order): three_interpolate's gweight (a per-row dot product in the kernel)
_ALWAYS_EXACT = {"three_interpolate": [1]}
# ... and with permutation indices, the kernels' scatters too (one term per element)
_EXACT_ON_PERMUTATION = {"index_points": [0], "group_points_xyz_first": [0, 2], "group_points_feat_first": [0, 2],
                         "three_interpolate": [0, 1]}


# the differentiable three-NN weights are torch arithmetic on the kernel's distances (ops.three_nn_autograd); inductor
# regenerates it, and its fused kernels round the weights differently in the last bit: the compiled output is held to the
# bar of that path in test_gpu_graph_replay.py instead of bit equality
_GLUE_FORWARD = {"feature_propagation_coordinates"}


@pytest.mark.parametrize("dynamic", [False, True], ids=["static", "dynamic"])
@pytest.mark.parametrize("name", list(AUTOGRAD))
def test_compiled_backward_equals_eager(cuda_dev, fresh_dynamo, name, dynamic):
    """forward and backward compiled together (AOTAutograd's joint graph): outputs bit-exact with eager; gradients bit-exact
    where eager is deterministic, and within the float64 bound everywhere"""
    make, fwd, grads = AUTOGRAD[name]
    fn = torch.compile(fwd, fullgraph=True, dynamic=dynamic)
    for i, sh in enumerate(SHAPES):
        d = make(200 + i, sh)
        sets = [("random", d)] + ([("permutation", _permuted(name, d, sh))] if name in _EXACT_ON_PERMUTATION else [])
        for label, dd in sets:
            te = _leaves(dd, cuda_dev, grads)
            tc = _leaves(dd, cuda_dev, grads)
            oe = fwd(te)
            gout_np = np.random.default_rng(300 + i).normal(size=tuple(oe.shape)).astype(F32)
            gout = torch.from_numpy(gout_np).to(cuda_dev)
            oe.backward(gout)
            oc = fn(tc)
            oc.backward(gout)
            what = "%s, set %d (%s)" % (name, i, label)
            if name in _GLUE_FORWARD:
                np.testing.assert_allclose(_host([oc])[0], _host([oe])[0], rtol=1e-5, atol=1e-6 * oe.abs().max().item(), err_msg=what)
            else:
                _bits_equal(oc, oe, what + " forward")
            ge = [_host([te[k].grad])[0] for k in grads]
            gc = [_host([tc[k].grad])[0] for k in grads]
            exact = _ALWAYS_EXACT.get(name, []) + (_EXACT_ON_PERMUTATION.get(name, []) if label == "permutation" else [])
            for j in exact:
                np.testing.assert_array_equal(gc[j].view(np.int32), ge[j].view(np.int32), err_msg="%s grad %s" % (what, grads[j]))
            for g in (ge, gc):
                _grad_bound(name, dd, te, g, gout_np)


def test_compiled_fps_draws_the_eager_start_with_fallback_random(cuda_dev, fresh_dynamo, monkeypatch):
    """farthest_point_sample / sample_points draw the first centroid with torch.randint on the CPU generator.  Inductor
    replaces that draw with its own generator unless torch._inductor.config.fallback_random is set; with it, the compiled
    call reproduces the eager picks under the same manual_seed, and both are the oracle's FPS from that start."""
    import torch._inductor.config as ic
    monkeypatch.setattr(ic, "fallback_random", True)
    fps = torch.compile(lambda x: P.farthest_point_sample(x, 32), fullgraph=True)
    sample = torch.compile(lambda x: P.sample_points(x, 32), fullgraph=True)
    for i, sh in enumerate(SHAPES):
        d = _fps_in(400 + i, sh)
        xyz = torch.from_numpy(d["xyz"]).to(cuda_dev)
        for name, eager, comp in (("farthest_point_sample", lambda x: P.farthest_point_sample(x, 32), fps),
                                  ("sample_points", lambda x: P.sample_points(x, 32), sample)):
            torch.manual_seed(1000 + i)
            want = eager(xyz)
            torch.manual_seed(1000 + i)
            start = torch.randint(0, sh["N"], (sh["B"],), dtype=torch.long).numpy()
            torch.manual_seed(1000 + i)
            got = comp(xyz)
            _bits_equal(got, want, "%s, set %d" % (name, i))
            np.testing.assert_array_equal(_flat(got)[0].cpu().numpy(), strict.farthest_point_sample(d["xyz"], 32, start))


def test_compiled_fps_without_fallback_random_is_still_an_exact_sample(cuda_dev, fresh_dynamo, monkeypatch):
    """without fallback_random inductor may replace the draw with its own generator, so the start need not be the eager
    one; it is still reproducible under manual_seed, and the picks are the oracle's FPS from the start that was drawn"""
    import torch._inductor.config as ic
    monkeypatch.setattr(ic, "fallback_random", False)
    fps = torch.compile(lambda x: P.farthest_point_sample(x, 32), fullgraph=True)
    d = _fps_in(410, SHAPES[2])
    xyz = torch.from_numpy(d["xyz"]).to(cuda_dev)
    torch.manual_seed(5)
    got = fps(xyz).cpu().numpy()
    torch.manual_seed(5)
    assert np.array_equal(fps(xyz).cpu().numpy(), got)
    np.testing.assert_array_equal(got, strict.farthest_point_sample(d["xyz"], 32, got[:, 0]))


def test_compiled_pointinet_mirror_forward(cuda_dev, fresh_dynamo, monkeypatch):
    """b200pc.pointinet's eager forward at 2 x 4 096 points under torch.compile (graph breaks allowed: the host read of t,
    the CPU-RNG draws) against the eager forward with the same weights and seed.  The geometric ops run the same kernels; the
    1x1 convolutions + BatchNorm + ReLU are regenerated by inductor and round differently, which can flip a near-tie in the
    fusion kNN for a few points, hence the existing end-to-end bar (test_gpu_pointinet.py)."""
    from b200pc import pointinet, synth
    import torch._inductor.config as ic
    monkeypatch.setattr(ic, "fallback_random", True)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    n = 4096
    a, b = synth.frame_pair(5, n)
    g = torch.Generator().manual_seed(1)
    mk = lambda f: torch.cat([torch.from_numpy(f).t(), torch.rand(1, n, generator=g)], 0)
    p1 = torch.stack([mk(a), mk(b)]).to(cuda_dev)
    p2 = torch.stack([mk(b), mk(a)]).to(cuda_dev)
    z = torch.zeros(2, 3, n, device=cuda_dev)
    t = torch.tensor([0.5, 0.5], device=cuda_dev)
    torch.manual_seed(0)
    net = pointinet.PointINet().eval().to(cuda_dev)
    comp = torch.compile(net)
    for seed in (3000, 3001):
        torch.manual_seed(seed)
        with torch.no_grad():
            want = net(p1, p2, z, z, t)
        torch.manual_seed(seed)
        with torch.no_grad():
            got = comp(p1, p2, z, z, t)
        assert got.shape == want.shape == (2, 4, n) and torch.isfinite(got).all()
        err = (got - want).abs().amax(dim=1).reshape(-1)
        assert (err < 1e-3).float().mean() > 0.995, "only %.4f of the points agree" % (err < 1e-3).float().mean()


def test_compiled_dropin_group_and_fusion(cuda_dev, fresh_dynamo):
    """the drop-in's Group.forward (kNN and ball branches) under fullgraph compile on channel-first inputs, and, where the
    reference is staged, the real reference's PointsFusion.knn_group after dropin.install()"""
    from b200pc import dropin
    from oracle import ref_loader
    rng = np.random.default_rng(12)
    pts = torch.from_numpy(rng.normal(size=(2, 3, 300)).astype(F32)).to(cuda_dev)
    new = pts[:, :, ::3].contiguous()
    feat = torch.from_numpy(rng.normal(size=(2, 8, 300)).astype(F32)).to(cuda_dev)
    for knn in (True, False):
        layer = types.SimpleNamespace(knn=knn, num_samples=16, radius=0.7)
        fn = lambda p, q, f: dropin._group_forward(layer, p, q, f)
        want = fn(pts, new, feat)
        got = torch.compile(fn, fullgraph=True)(pts, new, feat)
        _bits_equal(got, want, "Group.forward knn=%s" % knn)
        idx = (strict.knn_point(16, _host([pts.transpose(1, 2)])[0], _host([new.transpose(1, 2)])[0]) if knn else
               strict.query_ball_point(0.7, 16, _host([pts.transpose(1, 2)])[0], _host([new.transpose(1, 2)])[0]))
        np.testing.assert_array_equal(_host([got])[0], strict.group_points(
            _host([pts.transpose(1, 2)])[0], _host([new.transpose(1, 2)])[0], _host([feat.transpose(1, 2)])[0], idx))
    if not ref_loader.available():
        pytest.skip("reference not staged (python oracle/make_ref.py): the real PointsFusion.knn_group case did not run")
    lay = ref_loader.layers(ref_loader.strict_provider())
    dropin.install(force_pytorch3d=True)
    try:
        fusion = lay.PointsFusion([64, 64, 128]).eval().to(cuda_dev)
        fn = lambda a, b: fusion.knn_group(a, b, 8)
        with torch.no_grad():
            want = fn(new, pts)
            got = torch.compile(fn, fullgraph=True)(new, pts)
        _bits_equal(got, want, "PointsFusion.knn_group")
    finally:
        dropin.uninstall()


# ---- 3. autocast and other input dtypes ---------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("name", list(CASES))
def test_autocast_returns_the_fp32_result(cuda_dev, name, dtype):
    """the ops compute in fp32 by contract: inside an autocast region every public function returns the fp32 call's outputs,
    dtypes included, bit for bit"""
    case = CASES[name]
    t = _dev(case.make(500, SHAPES[0]), cuda_dev)
    want = case.call(t)
    with torch.autocast("cuda", dtype=dtype):
        got = case.call(t)
    _bits_equal(got, want, "%s under autocast(%s)" % (name, dtype))


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float64], ids=["fp16", "bf16", "fp64"])
@pytest.mark.parametrize("name", list(CASES))
def test_other_float_inputs_are_cast_to_fp32(cuda_dev, name, dtype):
    """fp16 / bf16 / fp64 coordinates and features are cast to fp32 and the outputs are fp32: the same bits as the fp32 call
    on the cast values (poly_predict's weights are float64 by contract and stay so)"""
    case = CASES[name]
    d = case.make(600, SHAPES[0])
    cast = lambda a: (lambda t: t.to(dtype) if a.dtype == F32 else t)(torch.from_numpy(np.ascontiguousarray(a)).to(cuda_dev))
    low = _dev(d, cuda_dev, cast)
    was_f32 = lambda k: (d[k][0] if isinstance(d[k], list) else d[k]).dtype == F32
    fp32 = {k: (([x.float() for x in v] if isinstance(v, list) else v.float()) if was_f32(k) else v) for k, v in low.items()}
    got = case.call(low)
    want = case.call(fp32)
    _bits_equal(got, want, "%s on %s inputs" % (name, dtype))
    assert all(o.dtype != dtype for o in _flat(got) if o.dtype.is_floating_point), name


# ---- 4. inputs as callers pass them -------------------------------------------------------------------------------------
def _channel_first(a, dev):
    """the [.., C, N] storage of a channel-first tensor handed over as its [.., N, C] view (x.permute(0, 2, 1))"""
    t = torch.from_numpy(np.ascontiguousarray(a))
    if t.dim() < 2:
        return t.to(dev)
    return t.transpose(-1, -2).contiguous().to(dev).transpose(-1, -2)


def _offset(nbytes):
    """a contiguous view into a flat buffer, starting nbytes past a 512-byte aligned allocation"""
    def up(a, dev):
        t = torch.from_numpy(np.ascontiguousarray(a))
        o = max(1, nbytes // t.element_size())
        flat = torch.empty(t.numel() + o, dtype=t.dtype, device=dev)
        v = flat[o:].view(t.shape)
        v.copy_(t)
        assert v.is_contiguous() and v.storage_offset() == o
        return v
    return up


def _batch_slice(a, dev):
    """items 1..B of a batch of B + 2: a contiguous view whose storage offset is one item"""
    t = torch.from_numpy(np.ascontiguousarray(a))
    big = torch.zeros((t.shape[0] + 2,) + tuple(t.shape[1:]), dtype=t.dtype, device=dev)
    big[1:-1] = t
    return big[1:-1]


def _values(fn):
    """apply a layout to the value tensors only (indices and lengths keep their plain int64 upload)"""
    return lambda a, dev: fn(a, dev) if a.dtype.kind == "f" else torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _indices(kind):
    def up(a, dev):
        t = torch.from_numpy(np.ascontiguousarray(a))
        if a.dtype.kind == "f":
            return t.to(dev)
        if kind == "int32":
            return t.int().to(dev)
        if kind == "uint8":
            assert a.min() >= 0 and a.max() < 256
            return t.to(torch.uint8).to(dev)
        v = torch.stack([t, torch.full_like(t, -99)], -1).to(dev)[..., 0]           # strided int64
        assert not v.is_contiguous() or v.numel() <= 1
        return v
    return up


LAYOUTS = {
    "channel_first": _values(_channel_first),
    "offset4": _values(_offset(4)), "offset8": _values(_offset(8)), "offset12": _values(_offset(12)),
    "batch_slice": _values(_batch_slice),
    "expanded": None,                                  # below: item 0 broadcast over the batch with stride 0
    "int32": _indices("int32"), "uint8": _indices("uint8"), "int64_strided": _indices("int64_strided"),
}
_HAS_INDICES = [n for n, c in CASES.items() if any(np.asarray(v).dtype.kind == "i" for v in c.make(0, SHAPES[0]).values()
                                                   if not isinstance(v, list))]


def _layout_params():
    for layout in LAYOUTS:
        for name in CASES:
            if layout.startswith(("int", "uint")) and name not in _HAS_INDICES:
                continue
            yield pytest.param(name, layout, id="%s-%s" % (name, layout))


@pytest.mark.parametrize("name,layout", list(_layout_params()))
def test_caller_layouts_match_the_oracle(cuda_dev, name, layout):
    case = CASES[name]
    d = case.make(700, SHAPES[0])
    if layout == "expanded":
        one = lambda a: np.broadcast_to(a[:1], a.shape)
        d = {k: ([np.ascontiguousarray(one(x)) for x in v] if isinstance(v, list) else np.ascontiguousarray(one(v))) for k, v in d.items()}
        t = _dev(d, cuda_dev, lambda a: torch.from_numpy(np.ascontiguousarray(a[:1])).to(cuda_dev).expand(a.shape))
        assert all(x.stride(0) == 0 for v in t.values() for x in (v if isinstance(v, list) else [v]))
    else:
        t = _dev(d, cuda_dev, lambda a: LAYOUTS[layout](a, cuda_dev))
    _check_oracle(case, d, case.call(t), "%s, %s" % (name, layout))


def test_channel_max_on_an_unaligned_flat_buffer_view(cuda_dev):
    """a contiguous [rows, C] view that starts 4 bytes into a flat buffer: the kernel needs 16-byte aligned rows, so the op
    copies the view first; the answer is torch.max(x, 1) bit for bit"""
    rows, C = 33, 16
    flat = torch.randn(1 + rows * C + 3, generator=torch.Generator().manual_seed(4)).to(cuda_dev)
    for start in (1, 2, 3, 4):
        x = flat[start:start + rows * C].view(rows, C)
        assert x.is_contiguous() and (x.data_ptr() % 16 == 0) == (start == 4)
        _bits_equal(ops.channel_max(x), x.max(1)[0], "channel_max at element offset %d" % start)
        _bits_equal(torch.ops.b200pc.channel_max(x), x.max(1)[0], "the op at element offset %d" % start)
