"""GPU parity of the entries added in round 2 (through torch.ops.b200pc.* -> C ABI): fusion_group, feature_propagation,
the int32-index search, rebuild_pack, the asynchronous-copy row movers and the host pipeline -- all against oracle/strict.c
or against the entry they fuse."""
import numpy as np
import pytest
import torch

from b200pc import hostio, ops, pointnet2_utils as P, synth
from oracle import strict

pytestmark = pytest.mark.gpu


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


@pytest.mark.parametrize("B,N,S,k,Cf", [(1, 4096, 4096, 16, 0), (2, 3000, 1777, 8, 1), (1, 700, 900, 32, 5), (2, 2048, 64, 1, 3)])
def test_fusion_group_matches_the_unfused_sequence(cuda_dev, B, N, S, k, Cf):
    """PointsFusion.knn_group / knn_group_withI (Utils/Layers.py:207-226, :384-402): indices bit-exact vs the strict
    knn_points oracle; nn and resi bit-exact (a gather and one fp32 subtraction); |resi| within 1e-6 relative of
    numpy's float32 norm (north_star: fp32 values within 1e-5)."""
    a, b = synth.batch_pairs(31, B, max(N, S))
    ref, qry = a[:, :N].copy(), b[:, :S].copy()
    feat = np.random.default_rng(k).normal(size=(B, N, Cf)).astype(np.float32) if Cf else None
    resi, nn, gf, idx = P.fusion_group(_t(qry, cuda_dev), _t(ref, cuda_dev), k, _t(feat, cuda_dev) if Cf else None)
    od, oi = strict.knn_points(qry, ref, k)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi)
    want_nn = strict.index_points(ref, oi)                                  # [B,S,k,3]
    want_resi = (want_nn - qry[:, :, None, :]).astype(np.float32)
    np.testing.assert_array_equal(_bits(nn.cpu().numpy()), _bits(want_nn.transpose(0, 3, 1, 2)))
    np.testing.assert_array_equal(_bits(resi[:, :3].cpu().numpy()), _bits(want_resi.transpose(0, 3, 1, 2)))
    np.testing.assert_allclose(resi[:, 3].cpu().numpy(), np.linalg.norm(want_resi, axis=-1), rtol=1e-6, atol=1e-30)
    assert resi.shape == (B, 4, S, k) and nn.shape == (B, 3, S, k) and gf.shape == (B, Cf, S, k)
    if Cf:
        np.testing.assert_array_equal(_bits(gf.cpu().numpy()), _bits(strict.index_points(feat, oi).transpose(0, 3, 1, 2)))


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("C", [128, 12])
def test_feature_propagation_is_three_nn_plus_interpolate(cuda_dev, variant, C):
    a, _ = synth.batch_pairs(32, 2, 4096)
    dense = _t(a, cuda_dev)
    sparse = dense[:, ::8].contiguous()
    feat = torch.randn(2, 512, C, device=cuda_dev)
    out = P.feature_propagation(dense, sparse, feat, variant=variant)
    _, i3, w3 = P.three_nn_weights(dense, sparse, variant=variant)
    assert torch.equal(out, P.three_interpolate(feat, i3, w3))
    od, oi = strict.three_nn(a, a[:, ::8])
    want = strict.three_interpolate(feat.cpu().numpy(), oi, strict.three_weights(od, variant))
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=1e-5, atol=1e-6)


def test_feature_propagation_backward_matches_the_two_step_path(cuda_dev):
    a, _ = synth.batch_pairs(33, 1, 1024)
    dense = _t(a, cuda_dev); sparse = dense[:, ::4].contiguous()
    f1 = torch.randn(1, 256, 32, device=cuda_dev, requires_grad=True)
    f2 = f1.detach().clone().requires_grad_(True)
    P.feature_propagation(dense, sparse, f1).square().sum().backward()
    _, i3, w3 = P.three_nn_weights(dense, sparse)
    P.three_interpolate(f2, i3, w3).square().sum().backward()
    torch.testing.assert_close(f1.grad, f2.grad, rtol=1e-5, atol=1e-6)


def test_three_nn_weights_carry_gradient_to_the_coordinates(cuda_dev):
    """values stay the kernel's, gradients are those of the dense torch formula (the reference's autograd)"""
    g = torch.Generator().manual_seed(3)
    dense = torch.randn(1, 300, 3, generator=g).to(cuda_dev).requires_grad_(True)
    sparse = torch.randn(1, 60, 3, generator=g).to(cuda_dev).requires_grad_(True)
    feat = torch.randn(1, 60, 8, generator=g).to(cuda_dev)
    for variant in (0, 1):
        dense.grad = sparse.grad = None
        P.feature_propagation(dense, sparse, feat, variant=variant).square().sum().backward()
        got = (dense.grad.clone(), sparse.grad.clone())
        d2 = dense.detach().clone().requires_grad_(True); s2 = sparse.detach().clone().requires_grad_(True)
        dist = ((d2.unsqueeze(2) - s2.unsqueeze(1)) ** 2).sum(-1)
        dd, ii = dist.sort(dim=-1)
        dd, ii = dd[:, :, :3], ii[:, :, :3]
        inv = 1.0 / torch.where(dd < 1e-10, torch.full_like(dd, 1e-10), dd) if variant == 0 else 1.0 / (dd + 1e-8)
        w = inv / inv.sum(2, keepdim=True)
        out = (feat[0][ii[0]] * w[0].unsqueeze(-1)).sum(1)
        out.square().sum().backward()
        torch.testing.assert_close(got[0], d2.grad, rtol=2e-3, atol=1e-5)
        torch.testing.assert_close(got[1], s2.grad, rtol=2e-3, atol=1e-5)


@pytest.mark.parametrize("B,N,S,k", [(2, 4096, 3000, 16), (1, 20000, 100, 4), (1, 600, 800, 8)])
def test_int32_index_variant_equals_int64(cuda_dev, B, N, S, k):
    a, b = synth.batch_pairs(34, B, max(N, S))
    ref, qry = _t(a[:, :N].copy(), cuda_dev), _t(b[:, :S].copy(), cuda_dev)
    for form in (0, 2):
        i64 = ops.knn_search(ref, qry, k, form)
        i32 = ops.knn_search_i32(ref, qry, k, form)
        assert i32.dtype == torch.int32 and torch.equal(i32.long(), i64)


def test_rebuild_pack_records(cuda_dev):
    """PolyPCI.rebuild (PolyPCI/Models/Models_V1.py:102-114): K=1 index bit-exact vs the oracle, neighbour = ref[index]"""
    a, b = synth.batch_pairs(35, 3, 5000)
    rec = ops.rebuild_pack(_t(a, cuda_dev), _t(b[:, 1000:3000].copy(), cuda_dev), s_offset=0)
    assert rec.shape == (2000, 3, 4)
    idx, nn = ops.unpack_rebuild(rec)
    od, oi = strict.knn_points(b[:, 1000:3000], a, 1)
    np.testing.assert_array_equal(idx.cpu().numpy(), oi[..., 0])
    np.testing.assert_array_equal(_bits(nn.cpu().numpy()), _bits(strict.index_points(a, oi)[:, :, 0]))
    # a "peer" buffer on the same device: the slab lands at its row offset
    full = torch.zeros(5000, 3, 4, device=cuda_dev)
    ops.rebuild_pack(_t(a, cuda_dev), _t(b[:, 1000:3000].copy(), cuda_dev), s_offset=1000, peer_ptrs=[full.data_ptr()])
    assert torch.equal(full[1000:3000].view(torch.int32), rec.view(torch.int32)) and not full[:1000].any() and not full[3000:].any()


def test_async_group_points_equals_the_register_path(cuda_dev, monkeypatch):
    """rowmove.cu (forced with B200PC_BULK=1, default for D <= 64) against group.cu (B200PC_BULK=0): identical bits,
    ragged sizes, both layouts, the ball query's empty-ball sentinel"""
    g = torch.Generator().manual_seed(7)
    a, b = synth.batch_pairs(36, 2, 3000)
    xyz = _t(a, cuda_dev); new = _t(b[:, :777].copy(), cuda_dev)
    for D, K in [(64, 16), (128, 5), (32, 9), (16, 3), (256, 2)]:
        feat = torch.randn(2, 3000, D, generator=g).to(cuda_dev)
        idx = P.knn_point(K, xyz, new)
        idx[0, 5, 0] = 3000                                            # the ball query's empty-ball sentinel
        idx[1, 7, K - 1] = -1                                          # wraps to the last point
        for first in (True, False):
            monkeypatch.setenv("B200PC_BULK", "0"); ops.reload_tuning()
            want = P.group_points(xyz, new, feat, idx, xyz_first=first)
            monkeypatch.setenv("B200PC_BULK", "1"); ops.reload_tuning()
            got = P.group_points(xyz, new, feat, idx, xyz_first=first)
            monkeypatch.delenv("B200PC_BULK"); ops.reload_tuning()
            assert torch.equal(got, want), (D, K, first)
            assert torch.equal(P.group_points(xyz, new, feat, idx, xyz_first=first), want)      # whichever the default picks


def test_host_pipeline_overlapped_calls(cuda_dev):
    a, b = synth.batch_pairs(37, 4, 4096)
    h_ref = torch.from_numpy(a).pin_memory(); h_qry = torch.from_numpy(b).pin_memory()
    want = strict.knn_point(8, a, b)
    for dt in (torch.int64, torch.int32):
        pipe = hostio.KnnHostPipeline(8, device=cuda_dev, index_dtype=dt)
        outs = [torch.empty(4, 4096, 8, dtype=dt).pin_memory() for _ in range(3)]
        for o in outs:
            pipe.submit(h_ref, h_qry, o)
        pipe.finish(); torch.cuda.synchronize()
        for o in outs:
            np.testing.assert_array_equal(o.numpy().astype(np.int64), want)


def test_loader_fps_on_device(cuda_dev, tmp_path):
    """b200pc.io (SURVEY 8f rank 3): .bin sweeps -> FPS on the device.  Real nuScenes / KITTI sweeps when the reference is
    staged (oracle/_ref), synthetic files otherwise; picks bit-exact against the oracle from start index 0."""
    from b200pc import io as bio
    from oracle import ref_loader
    files = []
    if ref_loader.available():
        kitti, nusc = ref_loader.demo_bins()
        files += [(p, 5) for p in nusc[:2]] + [(p, 4) for p in kitti[:1]]
    if not files:
        a, _ = synth.frame_pair(50, 30000)
        arr = np.concatenate([a, np.zeros((30000, 2), np.float32)], 1)
        p = tmp_path / "sweep.bin"; arr.tofile(p); files.append((str(p), 5))
    for path, cols in files:
        scan = bio.read_bin(path, cols)
        assert scan.shape[1] == cols and scan.shape[0] > 16000
        pts, idx = bio.load_and_sample(path, 2048, columns=cols, device=cuda_dev, return_index=True)
        want = strict.farthest_point_sample(scan[None, :, :3], 2048, np.array([0]))[0]
        np.testing.assert_array_equal(idx.cpu().numpy(), want)
        np.testing.assert_array_equal(pts.cpu().numpy(), scan[want, :3])
    if len(files) >= 2 and files[0][1] == files[1][1]:                  # ragged batch: one launch, padded with start-point copies
        pts, idx = bio.load_and_sample_many([f[0] for f in files[:2]], 1024, columns=files[0][1], device=cuda_dev, return_index=True)
        for i in range(2):
            scan = bio.read_bin(files[i][0], files[i][1])
            want = strict.farthest_point_sample(scan[None, :, :3], 1024, np.array([0]))[0]
            np.testing.assert_array_equal(idx[i].cpu().numpy(), want)


def test_error_behaviour_of_the_new_entries(cuda_dev):
    ref = torch.randn(1, 10, 3, device=cuda_dev); qry = torch.randn(1, 4, 3, device=cuda_dev)
    # fusion_group clamps k to the number of refs like pytorch3d.knn_points (K = min(K, P2))
    resi, nn, gf, idx = P.fusion_group(qry, ref, 64)
    assert idx.shape == (1, 4, 10) and resi.shape == (1, 4, 4, 10)
    with pytest.raises(RuntimeError):                       # three-NN needs three known points (the reference's slice [:3] of a shorter sort)
        P.feature_propagation(ref, qry[:, :2].contiguous(), torch.randn(1, 2, 8, device=cuda_dev))
    with pytest.raises(RuntimeError):                       # topk: k out of range
        ops.knn_search_i32(ref, qry, 11, 0)
    assert ops.rebuild_pack(ref, qry[:, :0].contiguous()).shape == (0, 1, 4)
    from b200pc import io as bio
    with pytest.raises(ValueError):
        bio.sample_clouds([np.zeros((100, 3), np.float32)], 101, device=cuda_dev)
    with pytest.raises(RuntimeError):
        bio.sample_clouds([np.zeros((100, 3), np.float32)], 10, device="cpu")
    with pytest.raises(RuntimeError):                       # CPU tensors never reach a kernel
        P.fusion_group(qry.cpu(), ref.cpu(), 2)


def test_channel_max(cuda_dev):
    g = torch.Generator().manual_seed(3)
    for rows, C in [(1000, 128), (7, 4), (4097, 64), (33, 260)]:
        x = torch.randn(rows, C, generator=g).to(cuda_dev)
        assert torch.equal(ops.channel_max(x), x.max(dim=1)[0])
    x = torch.randn(10, 128, generator=g).to(cuda_dev); x[3, 77] = float("nan")
    got = ops.channel_max(x)
    assert torch.isnan(got[3]) and torch.equal(got[[0, 1, 2, 4]], x.max(dim=1)[0][[0, 1, 2, 4]])
    y = torch.randn(5, 6, generator=g).to(cuda_dev)                     # C not a multiple of 4: served by torch
    assert torch.equal(ops.channel_max(y), y.max(dim=1)[0])


def test_c_level_async_host_knn_pipelined_over_two_streams(cuda_dev):
    """b200pc_knn_async_host (include/b200pc.h): a plain C caller's pipeline -- pinned host clouds in, pinned int32 indices
    out, two streams and two device arenas, nothing synchronised inside; every step must equal the oracle."""
    import ctypes as C
    from b200pc import _lib
    lib = _lib.load()
    B, N, S, k = 2, 6000, 3000, 16
    need = lib.b200pc_knn_async_host_workspace_bytes(B, N, S, k)
    assert need > B * (N + S) * 12
    streams = [torch.cuda.Stream(device=cuda_dev) for _ in range(2)]
    arenas = [torch.empty(need, dtype=torch.uint8, device=cuda_dev) for _ in range(2)]
    steps = []
    for i in range(5):
        a, b = synth.batch_pairs(60 + i, B, N)
        ref = torch.from_numpy(a).pin_memory(); qry = torch.from_numpy(b[:, :S].copy()).pin_memory()
        out = torch.empty(B, S, k, dtype=torch.int32).pin_memory(); dist = torch.empty(B, S, k, dtype=torch.float32).pin_memory()
        steps.append((ref, qry, out, dist))
    with torch.cuda.device(cuda_dev):
        for i, (ref, qry, out, dist) in enumerate(steps):
            st = streams[i % 2]                       # a call reuses its arena only after the previous call on ITS stream
            rc = lib.b200pc_knn_async_host(C.c_void_p(ref.data_ptr()), C.c_void_p(qry.data_ptr()), B, N, S, k, 0,
                                           C.c_void_p(out.data_ptr()), C.c_void_p(dist.data_ptr()), C.c_void_p(arenas[i % 2].data_ptr()),
                                           need, C.c_void_p(st.cuda_stream))
            assert rc == 0, lib.b200pc_last_error()
        for st in streams:
            st.synchronize()
    for ref, qry, out, dist in steps:
        oi, od = strict.knn(ref.numpy(), qry.numpy(), k, 0)
        np.testing.assert_array_equal(out.numpy(), oi.astype(np.int32))
        np.testing.assert_array_equal(dist.numpy().view(np.int32), od.view(np.int32))
    small = torch.empty(1024, dtype=torch.uint8, device=cuda_dev)
    ref, qry, out, dist = steps[0]
    rc = lib.b200pc_knn_async_host(C.c_void_p(ref.data_ptr()), C.c_void_p(qry.data_ptr()), B, N, S, k, 0, C.c_void_p(out.data_ptr()), None,
                                   C.c_void_p(small.data_ptr()), 1024, None)
    assert rc == _lib.EWORKSPACE and b"arena too small" in lib.b200pc_last_error()
