"""CPU side of the ragged-batch entries: the oracles against the dense oracle, the Chamfer reductions, argument handling of
the ops and the shim, and the fake kernels of the new ops."""
import numpy as np
import pytest
import torch

import ragged_oracle as RO
from b200pc import ops, pytorch3d_shim as shim, synth
from oracle import strict


@pytest.fixture
def knobs():
    """nothing to set on the CPU: the knobs only steer the device's launch plans (test_gpu_ragged.py)"""
    return None


def _cloud(seed, B, N, S):
    a, b = synth.batch_pairs(seed, B, max(N, S))
    return a[:, :N].copy(), b[:, :S].copy()


@pytest.mark.parametrize("form", [0, 1, 2])
def test_ragged_oracle_with_full_lengths_is_the_dense_oracle(knobs, form):
    ref, qry = _cloud(91, 3, 700, 200)
    want = strict.knn(ref, qry, 16, form)
    for rl, ql in ((None, None), ([700] * 3, [200] * 3), ([10 ** 6] * 3, [10 ** 6] * 3)):
        got = RO.knn(ref, qry, rl, ql, 16, form)
        np.testing.assert_array_equal(got[0], want[0])
        np.testing.assert_array_equal(got[1].view(np.int32), want[1].view(np.int32))


def test_ragged_oracle_pads_and_slices(knobs):
    ref, qry = _cloud(92, 3, 300, 50)
    idx, dist = RO.knn(ref, qry, [0, 5, 300], [50, 50, 7], 16, 2)
    assert (idx[0] == -1).all() and np.isinf(dist[0]).all()
    assert (idx[1, :, 5:] == -1).all() and (idx[1, :, :5] < 5).all() and (idx[1, :, :5] >= 0).all()
    assert (idx[2, 7:] == -1).all()
    want = strict.knn(ref[2:3], qry[2:3, :7].copy(), 16, 2)
    np.testing.assert_array_equal(idx[2:3, :7], want[0])


def test_chamfer_oracles_with_full_lengths_are_the_dense_oracle(knobs):
    x, y = _cloud(93, 2, 400, 300)
    ol, odx, oix, ody, oiy = strict.chamfer(x, y)
    sums, dx, ix, dy, iy = RO.chamfer_terms(x, y, None, None)
    np.testing.assert_array_equal(ix, oix); np.testing.assert_array_equal(iy, oiy)
    np.testing.assert_array_equal(dx, odx); np.testing.assert_array_equal(dy, ody)
    l64 = RO.chamfer_distance64(torch.from_numpy(x).double(), torch.from_numpy(y).double())
    assert abs(l64.item() - ol) <= 1e-5 * abs(ol)
    assert abs((sums[:, 0] / 400 + sums[:, 1] / 300).mean() - ol) <= 1e-5 * abs(ol)


@pytest.mark.parametrize("batch_reduction", ["mean", "sum", None])
@pytest.mark.parametrize("point_reduction", ["mean", "sum"])
def test_chamfer_reduce_follows_pytorch3d(knobs, point_reduction, batch_reduction):
    """ops.chamfer_reduce on the exact per-item sums equals the float64 restatement of pytorch3d's chamfer_distance"""
    x, y = _cloud(94, 4, 200, 150)
    xl, yl = [200, 17, 1, 0], [150, 150, 3, 9]
    sums, *_ = RO.chamfer_terms(x, y, xl, yl)
    sums[3, 1] = 0.0                       # x is empty: y's slots are padding (distance 0 in pytorch3d)
    got = ops.chamfer_reduce(torch.from_numpy(sums), torch.tensor(xl), torch.tensor(yl), 200, 150, point_reduction, batch_reduction)
    want = RO.chamfer_distance64(torch.from_numpy(x).double(), torch.from_numpy(y).double(), xl, yl, point_reduction, batch_reduction)
    assert tuple(got.shape) == tuple(want.shape)
    np.testing.assert_allclose(got.numpy(), want.numpy(), rtol=1e-6)
    full = ops.chamfer_reduce(torch.from_numpy(sums), None, None, 200, 150, point_reduction, batch_reduction)
    assert tuple(full.shape) == tuple(want.shape)


def test_chamfer_reduce_rejects_unknown_reductions(knobs):
    s = torch.zeros(2, 2)
    with pytest.raises(ValueError):
        ops.chamfer_reduce(s, None, None, 4, 4, "median", "mean")
    with pytest.raises(ValueError):
        ops.chamfer_reduce(s, None, None, 4, 4, "mean", "max")


def test_lengths_are_validated_without_reading_values(knobs):
    dev = torch.device("cpu")
    assert ops._lengths(None, 3, dev, "l") is None
    got = ops._lengths(torch.tensor([1, -2, 10 ** 12]), 3, dev, "l")
    assert got.dtype == torch.int64 and got.tolist() == [1, -2, 10 ** 12]       # clamping is the device's job
    assert ops._lengths(torch.tensor([1, 2, 3], dtype=torch.int32), 3, dev, "l").dtype == torch.int64
    with pytest.raises(ValueError):
        ops._lengths(torch.tensor([1, 2]), 3, dev, "l")
    with pytest.raises(TypeError):
        ops._lengths(torch.tensor([1.0, 2.0, 3.0]), 3, dev, "l")
    with pytest.raises(TypeError):
        ops._lengths([1, 2, 3], 3, dev, "l")


def test_shim_still_refuses_what_it_does_not_implement(knobs):
    x = torch.zeros(1, 4, 3)
    for kw in ({"weights": torch.ones(1)}, {"x_normals": x}, {"y_normals": x}, {"norm": 1}, {"point_reduction": "max"},
               {"point_reduction": None}):
        with pytest.raises(NotImplementedError):
            shim.chamfer_distance(x, x, **kw)
    with pytest.raises(NotImplementedError):
        shim.knn_points(x, x, torch.tensor([4]), None, norm=1)


def test_fake_kernels_of_the_ragged_ops(knobs):
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        ref = torch.empty(2, 100, 3, device="cuda"); qry = torch.empty(2, 50, 3, device="cuda")
        ln = torch.empty(2, dtype=torch.int64, device="cuda")
        idx, dist = torch.ops.b200pc.knn_ragged(ref, qry, ln, None, 4, 0, True)
        assert idx.shape == (2, 50, 4) and idx.dtype == torch.int64 and dist.shape == (2, 50, 4)
        sums, dx, ix, dy, iy = torch.ops.b200pc.chamfer_ragged_fwd(ref, qry, ln, ln)
        assert sums.shape == (2, 2) and dx.shape == (2, 100) and ix.dtype == torch.int64 and dy.shape == (2, 50)
        gx, gy = torch.ops.b200pc.chamfer_ragged_bwd(ref, qry, ix, iy, None, ln, sums)
        assert gx.shape == ref.shape and gy.shape == qry.shape


def test_ragged_ops_register_autograd_on_the_forward_only(knobs):
    op = torch.ops.b200pc.chamfer_ragged_fwd.default
    assert torch._C._dispatch_has_kernel_for_dispatch_key(op.name(), "Autograd")
    for name in ("knn_ragged", "chamfer_ragged_fwd", "chamfer_ragged_bwd"):
        o = getattr(torch.ops.b200pc, name).default
        assert torch._C._dispatch_has_kernel_for_dispatch_key(o.name(), "CUDA")
        assert not torch._C._dispatch_has_kernel_for_dispatch_key(o.name(), "CPU")
