"""Backward passes against float64 references: gather_bwd (vec4 / scalar scatter), three_interpolate_bwd (gfeat, gweight),
group_points_bwd + the xyz gradients of group_points, chamfer_bwd.

A gradient element that sums m fp32 terms in some order is off the exact sum by at most about (m-1) * 2^-24 * sum|terms|,
and each term computed on the device in fp32 adds its own roundings (k of them).  The bound used here is twice that,
2 * (m + k) * 2^-24 * sum|terms|, with m and sum|terms| counted per element by the same float64 scatter on absolute values.
Shapes keep m below ~2 000, so one dropped or doubled term is well outside it.  Elements that get exactly one term
(permutation indices) must be bit-exact."""
import numpy as np
import pytest
import torch

from b200pc import ops, pointnet2_utils as P, synth

U = 2.0 ** -24
TINY = 1e-30


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _misaligned(a, dev):
    """a copy of `a` on `dev` that is contiguous but starts 4 bytes past a 16-byte boundary: kernels take their scalar path"""
    a = np.ascontiguousarray(a, np.float32)
    t = torch.empty(a.size + 1, dtype=torch.float32, device=dev)[1:].view(a.shape)
    t.copy_(torch.from_numpy(a))
    assert t.data_ptr() % 16 == 4 and t.is_contiguous()
    return t


def _scatter64(n, index, vals):
    """float64 sums of vals [R, C] into n rows by index [R] (entries outside [0, n) dropped) -> (sum, sum of |vals|, count)"""
    index = torch.as_tensor(np.asarray(index, np.int64)).reshape(-1)
    vals = torch.as_tensor(np.asarray(vals, np.float64)).reshape(index.numel(), -1)
    keep = (index >= 0) & (index < n)
    index, vals = index[keep], vals[keep]
    s = torch.zeros(n, vals.shape[1], dtype=torch.float64).index_add_(0, index, vals)
    a = torch.zeros(n, vals.shape[1], dtype=torch.float64).index_add_(0, index, vals.abs())
    m = torch.zeros(n, dtype=torch.float64).index_add_(0, index, torch.ones(index.numel(), dtype=torch.float64))
    return s.numpy(), a.numpy(), m.numpy()[:, None]


def _assert_within(got, ref, abs_sum, m, k=0, what=""):
    """|got - ref| <= 2 (m + k) 2^-24 sum|terms| + tiny, element by element (a NaN fails)"""
    got = np.asarray(got, np.float64)
    ref, abs_sum, m = np.broadcast_arrays(np.asarray(ref, np.float64), np.asarray(abs_sum, np.float64), np.asarray(m, np.float64))
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    bound = 2.0 * (m + k) * U * abs_sum + TINY
    bad = ~(np.abs(got - ref) <= bound)
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError("%s: %d of %d elements outside the fp32 summation bound; first at %s: got %r, float64 %r, bound %r "
                             "(%d terms)" % (what, bad.sum(), bad.size, i, got[i], ref[i], bound[i], m[i]))


def _wrap(idx, n):
    """torch indexing: a negative index wraps once; -1 marks what is still out of range (no contribution)"""
    w = np.where(idx < 0, idx + n, idx)
    return np.where((w >= 0) & (w < n), w, -1)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


# ==========================================================================================
# group_points: xyz gradient on CPU (torch ops only; the feature gradient is D = 0 here)
# ==========================================================================================
class _Ctx:
    def __init__(self, idx, N, xyz_first):
        self.saved_tensors = (idx,)
        self.N, self.D, self.xyz_first = N, 0, xyz_first
        self.needs_input_grad = (True, True, False, False, False)


@pytest.mark.parametrize("xyz_first", [True, False])
def test_group_xyz_backward_masks_out_of_range_slots_cpu(xyz_first):
    """ball query's empty-ball sentinel N, -1, -N (wrap) and -N-1 (dropped): dropped slots read as zeros in the forward
    pass, so they give xyz nothing; new_xyz still gets -gout there (that output is 0 - centre)"""
    B, N, S, K = 2, 10, 7, 5
    rng = np.random.default_rng(0)
    idx = rng.integers(0, N, size=(B, S, K))
    idx[0, 0] = N                                  # a whole empty ball
    idx[0, 1, :4] = [-1, -N, -N - 1, N]
    idx[1, 3, 2] = 3 * N
    idx[1, 4, 1] = -N - 1
    gout = torch.from_numpy(rng.normal(size=(B, 3, K, S)).astype(np.float32))
    gxyz, gnew, gfeat, _, _ = ops._group_backward(_Ctx(torch.from_numpy(idx), N, xyz_first), gout)
    assert gfeat is None

    xyz = torch.zeros(B, N, 3, dtype=torch.float64, requires_grad=True)
    new = torch.zeros(B, S, 3, dtype=torch.float64, requires_grad=True)
    w = torch.from_numpy(_wrap(idx, N))
    ok = (w >= 0).unsqueeze(-1)
    rows = xyz[torch.arange(B).view(B, 1, 1), w.clamp(min=0)]            # unfused formula, dropped slots masked to 0
    rel = torch.where(ok, rows, torch.zeros((), dtype=torch.float64)) - new.unsqueeze(2)
    rel.permute(0, 3, 2, 1).backward(gout.double())
    _, a, m = _scatter64(B * N, (w + torch.arange(B).view(B, 1, 1) * N).where(w >= 0, -1).numpy(),
                         gout.permute(0, 3, 2, 1).reshape(-1, 3).numpy())
    _assert_within(gxyz.numpy().reshape(-1, 3), xyz.grad.numpy().reshape(-1, 3), a, m, what="xyz")
    _assert_within(gnew.numpy(), new.grad.numpy(), np.abs(gout.double().numpy()).sum(2).transpose(0, 2, 1), K, what="new_xyz")
    assert gxyz.shape == (B, N, 3) and gnew.shape == (B, S, 3)


# ==========================================================================================
# gather_bwd (index_points backward)
# ==========================================================================================
GATHER_C = [1, 3, 4, 5, 8, 64, 128, 130, 256]


def _gather_bwd(gout_np, idx_np, N, dev, misaligned):
    gout = _misaligned(gout_np, dev) if misaligned else _t(gout_np.astype(np.float32), dev)
    return torch.ops.b200pc.gather_bwd(gout, _t(idx_np, dev), N).cpu().numpy()


def _gather_ref(gout, idx, N):
    B, R, C = gout.shape
    w = _wrap(idx, N)
    flat = np.where(w >= 0, w + np.arange(B)[:, None] * N, -1)
    s, a, m = _scatter64(B * N, flat, gout.reshape(B * R, C))
    return s.reshape(B, N, C), a.reshape(B, N, C), m.reshape(B, N, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("misaligned", [False, True], ids=["vec4", "scalar"])
@pytest.mark.parametrize("C", GATHER_C)
def test_gather_bwd_random_and_bad_indices(cuda_dev, C, misaligned):
    B, N, R = 2, 300, 1500
    rng = np.random.default_rng(C)
    idx = rng.integers(-N, N, size=(B, R))
    idx[:, ::37] = N                                       # out of range: no contribution
    idx[:, 5::41] = -N - 1
    idx[1, 7] = 1 << 40
    gout = rng.normal(size=(B, R, C)).astype(np.float32)
    got = _gather_bwd(gout, idx, N, cuda_dev, misaligned)
    s, a, m = _gather_ref(gout, idx, N)
    _assert_within(got, s, a, m, what="gather_bwd C=%d" % C)


@pytest.mark.gpu
@pytest.mark.parametrize("misaligned", [False, True], ids=["vec4", "scalar"])
@pytest.mark.parametrize("C", GATHER_C)
def test_gather_bwd_permutation_is_bit_exact(cuda_dev, C, misaligned):
    B, N = 3, 777
    rng = np.random.default_rng(100 + C)
    idx = np.stack([rng.permutation(N) for _ in range(B)])
    idx[1] -= N                                            # the same rows, written as negative indices
    gout = rng.normal(size=(B, N, C)).astype(np.float32)
    got = _gather_bwd(gout, idx, N, cuda_dev, misaligned)
    want = np.zeros_like(gout)
    for b in range(B):
        want[b, idx[b] % N] = gout[b]
    np.testing.assert_array_equal(_bits(got), _bits(want))


@pytest.mark.gpu
@pytest.mark.parametrize("misaligned", [False, True], ids=["vec4", "scalar"])
@pytest.mark.parametrize("C", [3, 4, 64, 130])
def test_gather_bwd_duplicate_heavy(cuda_dev, C, misaligned):
    """every row lands on one of three targets: ~500 atomic adds per element"""
    B, N, R = 2, 50, 1600
    rng = np.random.default_rng(200 + C)
    targets = np.array([3, -7, N - 1])
    idx = targets[rng.integers(0, 3, size=(B, R))]
    idx[:, ::53] = N
    gout = rng.normal(size=(B, R, C)).astype(np.float32)
    got = _gather_bwd(gout, idx, N, cuda_dev, misaligned)
    s, a, m = _gather_ref(gout, idx, N)
    assert m.max() > 400
    _assert_within(got, s, a, m, what="gather_bwd duplicates C=%d" % C)
    untouched = np.ones(N, bool); untouched[targets % N] = False
    assert not got[:, untouched].any()


@pytest.mark.gpu
@pytest.mark.parametrize("ndim", [2, 3])
@pytest.mark.parametrize("C", [3, 64])
def test_index_points_autograd(cuda_dev, ndim, C):
    B, N = 2, 400
    rng = np.random.default_rng(300 + C + ndim)
    shape = (B, 700) if ndim == 2 else (B, 70, 10)
    idx = rng.integers(-N, N, size=shape)
    pts = _t(rng.normal(size=(B, N, C)).astype(np.float32), cuda_dev).requires_grad_(True)
    g = rng.normal(size=shape + (C,)).astype(np.float32)
    P.index_points(pts, _t(idx, cuda_dev)).backward(_t(g, cuda_dev))
    s, a, m = _gather_ref(g.reshape(B, -1, C), idx.reshape(B, -1), N)
    _assert_within(pts.grad.cpu().numpy(), s, a, m, what="index_points.backward")


# ==========================================================================================
# three_interpolate_bwd
# ==========================================================================================
def _interp_ref(gout, feat, idx, w):
    """gfeat[b, i_j] += gout * w_j (one fp32 product per term), gweight[b, n, j] = <gout, feat[i_j]> (C products);
    dropped neighbours give nothing"""
    B, N, C = gout.shape
    S = feat.shape[1]
    wr = _wrap(idx, S)                                                   # [B,N,3]
    flat = np.where(wr >= 0, wr + np.arange(B)[:, None, None] * S, -1).reshape(-1)
    terms = (gout.astype(np.float64)[:, :, None, :] * w.astype(np.float64)[..., None]).reshape(-1, C)
    sf, af, mf = _scatter64(B * S, flat, terms)
    rows = feat.reshape(B * S, C).astype(np.float64)[np.maximum(flat, 0)].reshape(B, N, 3, C)
    prod = gout.astype(np.float64)[:, :, None, :] * rows * (wr >= 0)[..., None]
    return (sf.reshape(B, S, C), af.reshape(B, S, C), mf.reshape(B, S, 1)), (prod.sum(-1), np.abs(prod).sum(-1))


def _check_interp_bwd(dev, gout, feat, idx, w, want_gweight=True, what=""):
    C = gout.shape[2]
    gfeat, gw = torch.ops.b200pc.three_interpolate_bwd(_t(gout, dev), _t(feat, dev), _t(idx, dev), _t(w, dev), want_gweight)
    (sf, af, mf), (sw, aw) = _interp_ref(gout, feat, idx, w)
    _assert_within(gfeat.cpu().numpy(), sf, af, mf, k=1, what=what + " gfeat")
    if want_gweight:
        _assert_within(gw.cpu().numpy(), sw, aw, C, k=1, what=what + " gweight")
    else:
        assert gw.numel() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 3, 4, 12, 64, 128, 256, 300])
def test_three_interpolate_bwd_matches_float64(cuda_dev, C):
    B, S, N = 2, 500, 3000
    rng = np.random.default_rng(400 + C)
    idx = rng.integers(0, S, size=(B, N, 3))
    w = rng.uniform(0.05, 1.0, size=(B, N, 3)).astype(np.float32)
    feat = rng.normal(size=(B, S, C)).astype(np.float32)
    gout = rng.normal(size=(B, N, C)).astype(np.float32)
    for want in (True, False):
        _check_interp_bwd(cuda_dev, gout, feat, idx, w, want, what="C=%d want_gweight=%s" % (C, want))


@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 64])
def test_three_interpolate_bwd_grid_strides(cuda_dev, C):
    """80 000 rows: more warps than the capped grid has, so every warp handles several rows"""
    B, S, N = 2, 1000, 40000
    rng = np.random.default_rng(500 + C)
    idx = rng.integers(0, S, size=(B, N, 3))
    w = rng.uniform(0.05, 1.0, size=(B, N, 3)).astype(np.float32)
    feat = rng.normal(size=(B, S, C)).astype(np.float32)
    gout = rng.normal(size=(B, N, C)).astype(np.float32)
    assert B * N > 148 * 16 * 8
    _check_interp_bwd(cuda_dev, gout, feat, idx, w, True, what="grid-stride C=%d" % C)
    _check_interp_bwd(cuda_dev, gout, feat, idx, w, False, what="grid-stride C=%d" % C)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [3, 64])
def test_three_interpolate_bwd_dropped_neighbours(cuda_dev, C):
    """negative indices wrap once; a neighbour still out of range was dropped by the forward pass (row 0, weight 0):
    it gets gweight 0 and adds nothing to gfeat, not even a NaN from a non-finite upstream gradient"""
    B, S, N = 2, 40, 600
    rng = np.random.default_rng(600 + C)
    idx = rng.integers(1, S, size=(B, N, 3))                             # row 0 only through the wrapped -S below
    idx[:, ::7, 0] = S
    idx[:, 3::11, 1] = -S - 1
    idx[:, 5::13, 2] = -S
    idx[1, 9] = [S, 1 << 40, -(1 << 40)]                                 # every neighbour dropped
    w = rng.uniform(0.05, 1.0, size=(B, N, 3)).astype(np.float32)
    feat = rng.normal(size=(B, S, C)).astype(np.float32)
    gout = rng.normal(size=(B, N, C)).astype(np.float32)
    _check_interp_bwd(cuda_dev, gout, feat, idx, w, True, what="dropped C=%d" % C)
    # a NaN upstream gradient on a row whose neighbours are all dropped must not reach gfeat or gweight
    gout[1, 9] = np.nan
    gfeat, gw = torch.ops.b200pc.three_interpolate_bwd(_t(gout, cuda_dev), _t(feat, cuda_dev), _t(idx, cuda_dev), _t(w, cuda_dev), True)
    gfeat, gw = gfeat.cpu().numpy(), gw.cpu().numpy()
    assert np.isfinite(gfeat).all() and (gw[1, 9] == 0).all()
    assert (gw[_wrap(idx, S) < 0] == 0).all()


@pytest.mark.gpu
def test_feature_propagation_backward_large(cuda_dev):
    """autograd through the one-call feature propagation at a C3-like size: the gradient reaches feat through
    three_interpolate_bwd with the op's own indices and weights"""
    B, N, S, C = 2, 16384, 4096, 128
    a, _ = synth.batch_pairs(81, B, N)
    unknown = _t(a, cuda_dev)
    known = _t(a[:, ::4], cuda_dev)
    rng = np.random.default_rng(7)
    feat_np = rng.normal(size=(B, S, C)).astype(np.float32)
    feat = _t(feat_np, cuda_dev).requires_grad_(True)
    out, idx, w = torch.ops.b200pc.feature_propagation(unknown, known, feat, 0)
    assert torch.equal(out, P.feature_propagation(unknown, known, feat.detach()))
    gout = rng.normal(size=(B, N, C)).astype(np.float32)
    (gfeat,) = torch.autograd.grad(out, feat, _t(gout, cuda_dev))
    (sf, af, mf), _ = _interp_ref(gout, feat_np, idx.detach().cpu().numpy(), w.detach().cpu().numpy())
    _assert_within(gfeat.cpu().numpy(), sf, af, mf, k=1, what="feature_propagation gfeat")


# ==========================================================================================
# group_points: features through group_points_bwd, xyz / new_xyz through _group_backward
# ==========================================================================================
GROUP_D = [1, 3, 5, 16, 64, 255, 256, 257, 300, 520]
GROUP_SHAPES = [(3, 50, 1, 1), (2, 200, 33, 16), (1, 1000, 777, 64)]      # B, N, S, K


def _group_grads(dev, xyz, new, feat, idx, gout, xyz_first):
    x = _t(xyz, dev).requires_grad_(True)
    n = _t(new, dev).requires_grad_(True)
    f = _t(feat, dev).requires_grad_(True)
    P.group_points(x, n, f, _t(idx, dev), xyz_first).backward(_t(gout, dev))
    return x.grad.cpu().numpy(), n.grad.cpu().numpy(), f.grad.cpu().numpy()


def _group_ref(idx, gout, N, D, xyz_first):
    """float64: feat[b, i] += gout[b, foff + d, k, s]; xyz[b, i] += gout[b, xoff + c, k, s]; new[b, s] -= sum_k gout[b, xoff + c, k, s]"""
    B, S, K = idx.shape
    xoff, foff = (0, 3) if xyz_first else (D, 0)
    wr = _wrap(idx, N)
    flat = np.where(wr >= 0, wr + np.arange(B)[:, None, None] * N, -1).reshape(-1)      # (b, s, k) order
    g = gout.transpose(0, 3, 2, 1)                                                      # [B,S,K,C]
    fe = _scatter64(B * N, flat, g[..., foff:foff + D].reshape(-1, D))
    xy = _scatter64(B * N, flat, g[..., xoff:xoff + 3].reshape(-1, 3))
    gx = g[..., xoff:xoff + 3].astype(np.float64)
    nw = (-gx.sum(2), np.abs(gx).sum(2))
    return fe, xy, nw


@pytest.mark.gpu
@pytest.mark.parametrize("xyz_first", [True, False])
@pytest.mark.parametrize("B,N,S,K", GROUP_SHAPES)
@pytest.mark.parametrize("D", GROUP_D)
def test_group_points_backward_matches_float64(cuda_dev, D, B, N, S, K, xyz_first):
    rng = np.random.default_rng(D * 7 + S)
    a, b = synth.batch_pairs(44, B, max(N, S))
    xyz, new = a[:, :N].copy(), b[:, :S].copy()
    feat = rng.normal(size=(B, N, D)).astype(np.float32)
    idx = rng.integers(-N, N, size=(B, S, K))
    flat_idx = idx.reshape(-1)
    flat_idx[::17] = N                                    # the ball query's empty-ball sentinel
    flat_idx[3::29] = -N - 1
    gout = rng.normal(size=(B, 3 + D, K, S)).astype(np.float32)
    gx, gn, gf = _group_grads(cuda_dev, xyz, new, feat, idx, gout, xyz_first)
    (sf, af, mf), (sx, ax, mx), (sn, an) = _group_ref(idx, gout, N, D, xyz_first)
    _assert_within(gf.reshape(B * N, D), sf, af, mf, what="feat")
    _assert_within(gx.reshape(B * N, 3), sx, ax, mx, what="xyz")
    _assert_within(gn, sn, an, K, what="new_xyz")


@pytest.mark.gpu
@pytest.mark.parametrize("xyz_first", [True, False])
@pytest.mark.parametrize("D", [3, 64, 257])
def test_group_points_backward_permutation_is_bit_exact(cuda_dev, D, xyz_first):
    """every feature row fills exactly one (centre, slot): its feature and xyz gradients are single terms"""
    B, S, K = 2, 45, 16
    N = S * K
    rng = np.random.default_rng(900 + D)
    idx = np.stack([rng.permutation(N) for _ in range(B)]).reshape(B, S, K)
    idx[0] -= N
    a, b = synth.batch_pairs(45, B, N)
    feat = rng.normal(size=(B, N, D)).astype(np.float32)
    gout = rng.normal(size=(B, 3 + D, K, S)).astype(np.float32)
    gx, _, gf = _group_grads(cuda_dev, a, b[:, :S].copy(), feat, idx, gout, xyz_first)
    xoff, foff = (0, 3) if xyz_first else (D, 0)
    g = gout.transpose(0, 3, 2, 1).reshape(B, N, 3 + D)                 # (s, k) order, the order of idx's rows
    want_f = np.zeros((B, N, D), np.float32); want_x = np.zeros((B, N, 3), np.float32)
    for bb in range(B):
        rows = idx[bb].reshape(-1) % N
        want_f[bb, rows] = g[bb, :, foff:foff + D]
        want_x[bb, rows] = g[bb, :, xoff:xoff + 3]
    np.testing.assert_array_equal(_bits(gf), _bits(want_f))
    np.testing.assert_array_equal(_bits(gx), _bits(want_x))


# ==========================================================================================
# chamfer_bwd
# ==========================================================================================
def _chamfer_ref(x, y, ix, iy, scale):
    """float64 gradient of scale * loss with the kernel's own nearest-neighbour choice:
    x_i gets 2 s/(B N) (x_i - y_ix[i]) and each y_j with iy[j] = i adds 2 s/(B M) (x_i - y_j); y mirrors it"""
    B, N, _ = x.shape; M = y.shape[1]
    x64, y64 = x.astype(np.float64), y.astype(np.float64)
    bn = np.arange(B)[:, None]
    tx = 2.0 * scale / (B * N) * (x64 - y64[bn, ix])                    # [B,N,3]: term of x_i, and -term of y_ix[i]
    ty = 2.0 * scale / (B * M) * (y64 - x64[bn, iy])                    # [B,M,3]
    fx = (np.arange(B)[:, None] * N + np.arange(N)[None]).reshape(-1)
    fy = (np.arange(B)[:, None] * M + np.arange(M)[None]).reshape(-1)
    ixf = (ix + bn * M).reshape(-1)
    iyf = (iy + bn * N).reshape(-1)
    sx, ax, mx = _scatter64(B * N, np.concatenate([fx, iyf]), np.concatenate([tx.reshape(-1, 3), -ty.reshape(-1, 3)]))
    sy, ay, my = _scatter64(B * M, np.concatenate([fy, ixf]), np.concatenate([ty.reshape(-1, 3), -tx.reshape(-1, 3)]))
    return (sx, ax, mx), (sy, ay, my)


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,M", [(1, 1, 700), (3, 1000, 1500), (2, 4096, 333), (2, 1500, 1)])
def test_chamfer_backward_matches_float64(cuda_dev, B, N, M):
    a, b = synth.batch_pairs(93, B, max(N, M))
    x_np, y_np = a[:, :N].copy(), b[:, :M].copy()
    x = _t(x_np, cuda_dev).requires_grad_(True); y = _t(y_np, cuda_dev).requires_grad_(True)
    loss, _, ix, _, iy = ops.chamfer(x, y)
    (loss * 3.5).backward()
    (sx, ax, mx), (sy, ay, my) = _chamfer_ref(x_np, y_np, ix.cpu().numpy(), iy.cpu().numpy(), 3.5)
    if M == 1:
        assert my.max() == N + 1                       # y_0 is every x's nearest point, and its own term
    _assert_within(x.grad.cpu().numpy().reshape(-1, 3), sx, ax, mx, k=4, what="gx")
    _assert_within(y.grad.cpu().numpy().reshape(-1, 3), sy, ay, my, k=4, what="gy")
