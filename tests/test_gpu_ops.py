"""GPU parity of FPS, index_points, three_interpolate, square_distance and Chamfer vs the oracle."""
import numpy as np
import pytest
import torch

from b200pc import ops, pointnet2_utils as P, pytorch3d_shim as S3, synth
from oracle import strict

pytestmark = pytest.mark.gpu


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


# ---------------------------------------------------------------- square_distance (a1)
@pytest.mark.parametrize("B,N,M", [(2, 1024, 256), (1, 300, 1001), (3, 17, 5), (1, 4096, 4096)])
def test_square_distance_bit_exact(cuda_dev, B, N, M):
    a, b = synth.batch_pairs(60, B, max(N, M))
    src, dst = a[:, :N].copy(), b[:, :M].copy()
    out = P.square_distance(_t(src, cuda_dev), _t(dst, cuda_dev))
    np.testing.assert_array_equal(_bits(out.cpu().numpy()), _bits(strict.square_distance(src, dst)))


def test_square_distance_non_contiguous_input(cuda_dev):
    a, b = synth.batch_pairs(61, 2, 512)
    src = _t(a, cuda_dev).permute(0, 2, 1).contiguous().permute(0, 2, 1)   # SA-MSG passes a permuted view
    out = P.square_distance(src, _t(b, cuda_dev))
    np.testing.assert_array_equal(_bits(out.cpu().numpy()), _bits(strict.square_distance(a, b)))


# ---------------------------------------------------------------- farthest_point_sample (a3)
FPS_CASES = [(1, 16384, 1024), (2, 1024, 256), (2, 256, 64), (3, 64, 16), (1, 8192, 2048),
             (2, 5000, 500), (1, 40000, 256), (1, 70000, 128), (16, 16384, 64), (1, 3, 3)]


@pytest.mark.parametrize("flat", ["auto", "0", "1"])      # two-level arg-max / flat exchange of warp keys / launcher's choice
@pytest.mark.parametrize("B,N,npoint", FPS_CASES)
def test_fps_bit_exact(cuda_dev, monkeypatch, B, N, npoint, flat):
    if flat != "auto":
        monkeypatch.setenv("B200PC_FPS_FLAT", flat); ops.reload_tuning()
    a, _ = synth.batch_pairs(70, B, N)
    start = np.random.default_rng(N).integers(0, N, size=B)
    out = P.farthest_point_sample_from(_t(a, cuda_dev), npoint, _t(start, cuda_dev))
    assert out.dtype == torch.int64 and out.shape == (B, npoint)
    np.testing.assert_array_equal(out.cpu().numpy(), strict.farthest_point_sample(a, npoint, start))


def test_fps_duplicates_first_argmax(cuda_dev):
    # padded-duplicate cloud (the reference's loaders pad short frames by re-drawing points)
    a, _ = synth.batch_pairs(71, 1, 2048)
    dup = np.concatenate([a, a[:, :1024]], 1)
    start = np.array([7])
    out = P.farthest_point_sample_from(_t(dup, cuda_dev), 2500, _t(start, cuda_dev))
    np.testing.assert_array_equal(out.cpu().numpy(), strict.farthest_point_sample(dup, 2500, start))


@pytest.mark.parametrize("flat", ["0", "1"])
@pytest.mark.parametrize("N", [301, 1025, 2049, 4097, 8193, 16385, 40001])     # P = 1, 2, 4, 8, 16 and clusters of 2..8 CTAs
def test_fps_near_ties_no_fused_multiply_add(cuda_dev, monkeypatch, N, flat):
    monkeypatch.setenv("B200PC_FPS_FLAT", flat); ops.reload_tuning()
    """clouds built so that fma(dz,dz,fma(dy,dy,dx*dx)) picks a different point than the reference's
    (dx*dx + dy*dy) + dz*dz already in the first round (tests/adversarial.py)"""
    from adversarial import fps_rot90_cloud, first_round_pick
    clouds = np.stack([fps_rot90_cloud(900 + i, N // 2) for i in range(4)])
    for c in clouds:
        assert first_round_pick(c, False) != first_round_pick(c, True)
    start = np.zeros(4, np.int64)
    npoint = min(64, N)
    out = P.farthest_point_sample_from(_t(clouds, cuda_dev), npoint, _t(start, cuda_dev))
    np.testing.assert_array_equal(out.cpu().numpy(), strict.farthest_point_sample(clouds, npoint, start))


def test_fps_consumes_cpu_rng_like_reference(cuda_dev):
    a, _ = synth.batch_pairs(72, 2, 1024)
    torch.manual_seed(123)
    expect_start = torch.randint(0, 1024, (2,), dtype=torch.long)
    torch.manual_seed(123)
    out = P.farthest_point_sample(_t(a, cuda_dev), 8)
    assert torch.equal(out[:, 0].cpu(), expect_start)


# ---------------------------------------------------------------- index_points (a6)
@pytest.mark.parametrize("C", [3, 1, 64, 128, 130, 256])
def test_index_points_2d_and_3d_idx(cuda_dev, C):
    rng = np.random.default_rng(C)
    pts = rng.normal(size=(2, 1000, C)).astype(np.float32)
    i2 = rng.integers(0, 1000, size=(2, 333))
    i3 = rng.integers(0, 1000, size=(2, 77, 16))
    for idx in (i2, i3):
        out = P.index_points(_t(pts, cuda_dev), _t(idx, cuda_dev))
        assert out.shape == idx.shape + (C,)
        np.testing.assert_array_equal(out.cpu().numpy(), strict.index_points(pts, idx))


def test_index_points_int32_and_negative_indices(cuda_dev):
    pts = np.arange(2 * 10 * 4, dtype=np.float32).reshape(2, 10, 4)
    idx = np.array([[0, -1, 9, -10], [3, 3, -2, 5]], np.int32)
    out = P.index_points(_t(pts, cuda_dev), torch.from_numpy(idx).to(cuda_dev))
    np.testing.assert_array_equal(out.cpu().numpy(), strict.index_points(pts, idx.astype(np.int64)))


def test_index_points_out_of_range_raises_indexerror(cuda_dev, monkeypatch):
    monkeypatch.setattr(ops, "CHECK_BOUNDS", True)
    pts = torch.zeros(1, 10, 4, device=cuda_dev)
    with pytest.raises(IndexError):
        P.index_points(pts, torch.tensor([[10]], device=cuda_dev))


def test_index_points_backward_scatter_add(cuda_dev):
    rng = np.random.default_rng(1)
    pts = torch.tensor(rng.normal(size=(2, 50, 8)).astype(np.float32), device=cuda_dev, requires_grad=True)
    idx = torch.tensor(rng.integers(0, 50, size=(2, 40, 4)), device=cuda_dev)
    g = torch.tensor(rng.normal(size=(2, 40, 4, 8)).astype(np.float32), device=cuda_dev)
    P.index_points(pts, idx).backward(g)
    ref = pts.detach().clone().requires_grad_(True)
    ref[torch.arange(2, device=cuda_dev).view(2, 1, 1), idx].backward(g)
    torch.testing.assert_close(pts.grad, ref.grad, rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------- three_interpolate (a5)
@pytest.mark.parametrize("C", [128, 256, 3, 30, 64, 12])
def test_three_interpolate_forward(cuda_dev, C):
    a, _ = synth.batch_pairs(80, 2, 4096)
    known = a[:, ::8].copy()
    feats = np.random.default_rng(C).normal(size=(2, known.shape[1], C)).astype(np.float32)
    od, oi = strict.three_nn(a, known)
    for variant in (0, 1):
        ow = strict.three_weights(od, variant)
        out = P.three_interpolate(_t(feats, cuda_dev), _t(oi, cuda_dev), _t(ow, cuda_dev))
        exp = strict.three_interpolate(feats, oi, ow)
        np.testing.assert_allclose(out.cpu().numpy(), exp, rtol=1e-5, atol=1e-6)   # north_star tolerance


def test_three_interpolate_backward(cuda_dev):
    rng = np.random.default_rng(2)
    feat = torch.tensor(rng.normal(size=(2, 30, 16)).astype(np.float32), device=cuda_dev, requires_grad=True)
    w = torch.tensor(rng.uniform(0.1, 1, size=(2, 100, 3)).astype(np.float32), device=cuda_dev, requires_grad=True)
    idx = torch.tensor(rng.integers(0, 30, size=(2, 100, 3)), device=cuda_dev)
    g = torch.tensor(rng.normal(size=(2, 100, 16)).astype(np.float32), device=cuda_dev)
    P.three_interpolate(feat, idx, w).backward(g)
    f2 = feat.detach().clone().requires_grad_(True); w2 = w.detach().clone().requires_grad_(True)
    gathered = f2[torch.arange(2, device=cuda_dev).view(2, 1, 1), idx]
    (gathered * w2.unsqueeze(-1)).sum(2).backward(g)
    torch.testing.assert_close(feat.grad, f2.grad, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(w.grad, w2.grad, rtol=1e-4, atol=1e-5)


# ---------------------------------------------------------------- chamfer (a9)
@pytest.mark.parametrize("B,N,M", [(2, 2048, 2048), (1, 1000, 1500), (4, 8192, 8192)])
def test_chamfer_forward(cuda_dev, B, N, M):
    a, b = synth.batch_pairs(90, B, max(N, M))
    x, y = a[:, :N].copy(), b[:, :M].copy()
    loss, dx, ix, dy, iy = ops.chamfer(_t(x, cuda_dev), _t(y, cuda_dev))
    ol, odx, oix, ody, oiy = strict.chamfer(x, y)
    np.testing.assert_array_equal(ix.cpu().numpy(), oix)
    np.testing.assert_array_equal(iy.cpu().numpy(), oiy)
    np.testing.assert_array_equal(_bits(dx.cpu().numpy()), _bits(odx))
    np.testing.assert_array_equal(_bits(dy.cpu().numpy()), _bits(ody))
    assert abs(loss.item() - ol) <= 1e-5 * abs(ol)      # north_star: 1e-5 relative
    l2, none = S3.chamfer_distance(_t(x, cuda_dev), _t(y, cuda_dev))
    assert none is None and l2.dim() == 0 and l2.item() == loss.item()


def test_chamfer_backward_matches_autograd_of_dense_formula(cuda_dev):
    a, b = synth.batch_pairs(91, 2, 512)
    x = _t(a, cuda_dev).requires_grad_(True); y = _t(b, cuda_dev).requires_grad_(True)
    S3.chamfer_distance(x, y)[0].backward()
    x2 = x.detach().clone().requires_grad_(True); y2 = y.detach().clone().requires_grad_(True)
    d = ((x2.unsqueeze(2) - y2.unsqueeze(1)) ** 2).sum(-1)
    (d.min(2)[0].mean(1) + d.min(1)[0].mean(1)).mean().backward()
    torch.testing.assert_close(x.grad, x2.grad, rtol=1e-4, atol=1e-7)
    torch.testing.assert_close(y.grad, y2.grad, rtol=1e-4, atol=1e-7)


def test_chamfer_loss_reference_layout(cuda_dev):
    # Utils/Utils.py:39-48 passes [B,3,N] tensors permuted to [B,N,3] (non-contiguous views)
    a, b = synth.batch_pairs(92, 2, 1024)
    pc1 = _t(a, cuda_dev).permute(0, 2, 1).contiguous(); pc2 = _t(b, cuda_dev).permute(0, 2, 1).contiguous()
    loss, _ = S3.chamfer_distance(pc1.permute(0, 2, 1), pc2.permute(0, 2, 1))
    ol = strict.chamfer(a, b)[0]
    assert abs(loss.item() - ol) <= 1e-5 * abs(ol)


# ---------------------------------------------------------------- fused grouping (SURVEY 8f rank 1)
@pytest.mark.parametrize("xyz_first", [True, False])
@pytest.mark.parametrize("B,N,S,K,D", [(2, 4096, 512, 16, 5),     # the golden fixture's shape
                                       (1, 1024, 256, 16, 3),     # SetConv 1 of FlowNet3D
                                       (2, 256, 256, 64, 128),    # FlowEmbedding
                                       (1, 300, 77, 3, 0),        # ragged S, no feature channels
                                       (1, 64, 33, 8, 300),       # wide rows (16-byte row reads)
                                       (2, 128, 70, 5, 37),       # D not a multiple of 4: scalar row reads
                                       (3, 50, 1, 1, 2)])
def test_group_points_bit_exact(cuda_dev, B, N, S, K, D, xyz_first):
    a, b = synth.batch_pairs(40, B, max(N, S))
    xyz, new = a[:, :N].copy(), b[:, :S].copy()
    rng = np.random.default_rng(41)
    feat = rng.normal(size=(B, N, D)).astype(np.float32) if D else None
    idx = rng.integers(0, N, size=(B, S, K))
    out = P.group_points(_t(xyz, cuda_dev), _t(new, cuda_dev), None if feat is None else _t(feat, cuda_dev), _t(idx, cuda_dev), xyz_first)
    want = strict.group_points(xyz, new, feat, idx, xyz_first)
    assert out.shape == want.shape == (B, 3 + D, K, S) and out.is_contiguous()
    np.testing.assert_array_equal(_bits(out.cpu().numpy()), _bits(want))


def test_group_points_equals_the_unfused_reference_ops(cuda_dev):
    # the five ops of Group.forward (Utils/Layers.py:57-66) on the same kernels' outputs, including negative indices
    a, b = synth.batch_pairs(42, 2, 2048)
    xyz, new = _t(a, cuda_dev), _t(b[:, :300], cuda_dev)
    feat = torch.randn(2, 2048, 20, device=cuda_dev)
    idx = P.query_ball_point(2.0, 24, xyz, new)
    idx[0, :5] -= 2048                                                                  # python-style negative indices wrap
    rel = P.index_points(xyz, idx) - new.view(2, 300, 1, 3)
    want = torch.cat([rel, P.index_points(feat, idx)], dim=-1).permute(0, 3, 2, 1).contiguous()
    assert torch.equal(P.group_points(xyz, new, feat, idx), want)


def test_group_points_backward_matches_unfused_autograd(cuda_dev):
    a, b = synth.batch_pairs(43, 2, 1024)
    idx = torch.randint(0, 1024, (2, 200, 12), device=cuda_dev)
    gout = torch.randn(2, 3 + 16, 12, 200, device=cuda_dev)
    grads = []
    for fused in (True, False):
        xyz = _t(a, cuda_dev).requires_grad_(True); new = _t(b[:, :200], cuda_dev).requires_grad_(True)
        feat = torch.randn(2, 1024, 16, device=cuda_dev, generator=torch.Generator(cuda_dev).manual_seed(5)).requires_grad_(True)
        if fused:
            out = P.group_points(xyz, new, feat, idx)
        else:
            rel = xyz[torch.arange(2, device=cuda_dev).view(2, 1, 1), idx] - new.view(2, 200, 1, 3)
            out = torch.cat([rel, feat[torch.arange(2, device=cuda_dev).view(2, 1, 1), idx]], dim=-1).permute(0, 3, 2, 1)
        out.backward(gout)
        grads.append((xyz.grad, new.grad, feat.grad))
    for g_fused, g_ref in zip(*grads):
        torch.testing.assert_close(g_fused, g_ref, rtol=1e-5, atol=1e-5)                # fp32 sums in a different order


def test_group_points_rejects_bad_shapes(cuda_dev):
    xyz = torch.zeros(1, 10, 3, device=cuda_dev); new = torch.zeros(1, 4, 3, device=cuda_dev)
    with pytest.raises(ValueError):
        P.group_points(xyz, new, None, torch.zeros(1, 5, 2, dtype=torch.long, device=cuda_dev))
    with pytest.raises(RuntimeError):
        P.group_points(xyz.cpu(), new, None, torch.zeros(1, 4, 2, dtype=torch.long))


# ---------------------------------------------------------------- PolyPCI polynomial fit (SURVEY 8f rank 4)
@pytest.mark.parametrize("B,N,field,degree", [(2, 4096, 2, 3), (1, 16384, 3, 2), (3, 1001, 1, 1)])
def test_poly_fit_and_predict_matches_host_restatement(cuda_dev, B, N, field, degree):
    from b200pc import polypci
    from oracle import ref_polyfit
    F = 2 * field + 1
    rng = np.random.default_rng(50 + N)
    base = (rng.normal(size=(B, 3, N)) * 30).astype(np.float32)
    frames = [(base + rng.normal(size=(B, 3, N)).astype(np.float32) * (0.3 * f)).astype(np.float32) for f in range(F)]
    T_list = [[0.0] + [s * (i + 1) for i in range(field) for s in (-1.0, 1.0)] for _ in range(B)]   # key, fwd0, bwd0, fwd1, ...
    t = np.linspace(-0.5, 0.7, B)
    out = polypci.fit_and_predict([_t(f, cuda_dev) for f in frames], T_list, torch.from_numpy(t), degree)
    want = ref_polyfit.forward_tail(frames, T_list, t, degree)
    assert out.shape == (B, 3, N) and out.dtype == torch.float32
    # float64 accumulation on both sides, in a different association: fp32 results agree to the last bit or one ulp
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=1e-6, atol=1e-6)


def test_poly_fit_rejects_cpu_and_bad_counts(cuda_dev):
    from b200pc import polypci
    f = [torch.zeros(1, 3, 8) for _ in range(3)]
    with pytest.raises(RuntimeError):
        polypci.fit_and_predict(f, [[0.0, -1.0, 1.0]], [0.5], 1)
    g = [x.to(cuda_dev) for x in f]
    with pytest.raises(ValueError):
        polypci.fit_and_predict(g, [[0.0, -1.0]], [0.5], 1)


def test_poly_predict_rejects_weights_and_frames_it_cannot_read(cuda_dev):
    """the kernel reads B*F doubles from `weights` and F frames of one shape: anything else is refused before the call"""
    from b200pc import ops
    f = [torch.zeros(2, 3, 8, device=cuda_dev) for _ in range(3)]
    w = torch.zeros(2, 3, dtype=torch.float64, device=cuda_dev)
    assert ops.poly_predict(f, w).shape == (2, 3, 8)
    bad = {"float32 weights": (f, w.float()), "[B, F-1] weights": (f, w[:, :2].contiguous()),
           "[F, B] weights": (f, torch.zeros(3, 2, dtype=torch.float64, device=cuda_dev)), "[B*F] weights": (f, w.reshape(-1)),
           "weights on the host": (f, w.cpu()), "frames of two shapes": (f[:2] + [torch.zeros(2, 3, 9, device=cuda_dev)], w),
           "no frames": ([], w[:, :0])}
    for what, (frames, weights) in bad.items():
        with pytest.raises(ValueError):
            ops.poly_predict(frames, weights)
        torch.cuda.synchronize()


def test_sample_points_is_fps_plus_gather(cuda_dev):
    # Sample.forward (Utils/Layers.py:23-27): the FPS kernel also writes the picks' coordinates
    a, _ = synth.batch_pairs(60, 3, 16384)
    for N, npoint in ((16384, 1024), (5000, 300), (700, 700)):
        xyz = _t(a[:, :N], cuda_dev)
        start = torch.tensor([5, 0, N - 1], dtype=torch.long)
        idx, new_xyz = P.sample_points(xyz, npoint, start.to(cuda_dev))
        np.testing.assert_array_equal(idx.cpu().numpy(), strict.farthest_point_sample(a[:, :N], npoint, start.numpy()))
        assert torch.equal(new_xyz, P.index_points(xyz, idx))
    torch.manual_seed(77)
    i1, _ = P.sample_points(xyz, 64)
    torch.manual_seed(77)
    assert torch.equal(i1, P.farthest_point_sample(xyz, 64))           # same CPU-RNG draw as farthest_point_sample


def test_empty_work_is_accepted_everywhere(cuda_dev):
    # zero queries / clouds / samples / neighbours: empty tensors (null data pointers) in, empty tensors out, like torch
    from b200pc import pytorch3d_shim as S3
    x = torch.randn(2, 100, 3, device=cuda_dev)
    z = lambda *s: torch.zeros(*s, dtype=torch.long, device=cuda_dev)
    assert P.knn_point(4, x, x[:, :0]).shape == (2, 0, 4)
    assert P.knn_point(4, x[:0], x[:0, :10]).shape == (0, 10, 4)
    assert P.query_ball_point(1.0, 4, x, x[:, :0]).shape == (2, 0, 4)
    assert ops.fps(x, 0, z(2)).shape == (2, 0)
    assert P.index_points(x, z(2, 0)).shape == (2, 0, 3)
    assert P.group_points(x, x[:, :5].contiguous(), None, z(2, 5, 0)).shape == (2, 3, 0, 5)
    assert P.group_points(x, x[:, :0].contiguous(), None, z(2, 0, 3)).shape == (2, 3, 3, 0)
    assert S3.knn_points(x, x, K=0).idx.shape == (2, 100, 0)
    assert P.three_interpolate(torch.randn(2, 10, 8, device=cuda_dev), z(2, 0, 3), torch.zeros(2, 0, 3, device=cuda_dev)).shape == (2, 0, 8)
    assert P.knn_point(1, x[:, :1].contiguous(), x).eq(0).all()                      # a single reference point
    torch.cuda.synchronize()


def test_three_interpolate_index_hygiene(cuda_dev):
    # negative indices wrap once like torch indexing; an index that is still out of range contributes nothing
    feat = torch.randn(1, 10, 8, device=cuda_dev)
    idx = torch.tensor([[[0, 1, 2], [-1, -10, 9], [3, 10, 4], [5, -11, 6]]], device=cuda_dev)
    w = torch.tensor([[[0.2, 0.3, 0.5]] * 4], device=cuda_dev)
    out = P.three_interpolate(feat, idx, w)
    f = feat[0]
    want = torch.stack([0.2 * f[0] + 0.3 * f[1] + 0.5 * f[2], 0.2 * f[9] + 0.3 * f[0] + 0.5 * f[9],
                        0.2 * f[3] + 0.5 * f[4], 0.2 * f[5] + 0.5 * f[6]])[None]
    torch.testing.assert_close(out, want, rtol=1e-6, atol=1e-6)
