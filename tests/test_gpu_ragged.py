"""Ragged batches on the GPU: b200pc_knn_ragged, b200pc_chamfer_ragged_fwd / _bwd, their ops and the pytorch3d shim with lengths.

Bar: valid rows bit-identical (indices and fp32 distance bits) to oracle/strict per item on the valid points, padded rows and
slots -1 / +inf, under every launch plan of the search (forced through the B200PC_* knobs and proven by the
B200PC_DEBUG_PLAN line); outputs that do not depend on what the padded rows hold nor on what the output buffers held; Chamfer
losses and gradients against a float64 restatement of pytorch3d's formulas.
"""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

import ragged_oracle as RO
from b200pc import _lib, ops, pytorch3d_shim as shim, synth
from oracle import strict

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "point-cloud-interpolation-_b200")
PLAN = re.compile(r"b200pc plan: B=(?P<B>\d+) N=(?P<N>\d+) S=(?P<S>\d+) k=(?P<k>\d+) mode=(?P<mode>\d+) -> (?P<warps>\d+) warps/CTA, "
                  r"(?P<qpc>\d+) queries/CTA, ref split (?P<split>\d+) \((?P<tps>\d+) tiles each\), grid (?P<grid>\w+), "
                  r"filter (?P<filter>\w+), order (?P<order>\w+), ")


class Knobs:
    """sets B200PC_* knobs (plus B200PC_DEBUG_PLAN=1), makes the library re-read them, runs a call and parses its plan lines"""

    def __init__(self, monkeypatch, capfd):
        self.mp, self.capfd = monkeypatch, capfd

    def set(self, **env):
        self.mp.setenv("B200PC_DEBUG_PLAN", "1")
        for name in ("SMALL_PATH", "GRID", "FORCE_SPLIT", "FORCE_Q", "INTERLEAVE"):
            self.mp.delenv("B200PC_" + name, raising=False)
        for name, v in env.items():
            self.mp.setenv("B200PC_" + name, str(v))
        ops.reload_tuning()

    def run(self, fn):
        torch.cuda.synchronize()
        self.capfd.readouterr()
        out = fn()
        torch.cuda.synchronize()
        err = self.capfd.readouterr().err
        return out, [m.groupdict() for m in PLAN.finditer(err)]


@pytest.fixture
def knobs(cuda_dev, monkeypatch, capfd):
    return Knobs(monkeypatch, capfd)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


def _cloud(seed, B, N, S):
    a, b = synth.batch_pairs(seed, B, max(N, S))
    return a[:, :N].copy(), b[:, :S].copy()


# ---- every launch plan -------------------------------------------------------------------------------------------------
K = 16
LARGE = (8, 5000, 1500)      # 10 tiles of refs
SMALL = (8, 1000, 700)       # the warp-per-query path serves N <= 1024
REF_LENS = {5000: [0, 1, K - 1, K, 511, 512, 513, 5000], 1000: [0, 1, K - 1, K, 511, 512, 513, 1000]}
QRY_LENS = {1500: [1500, 777, 33, 1, 1499, 0, 1000, 130], 700: [700, 333, 33, 1, 699, 0, 500, 130]}
# (knobs, expected plan fields, shape).  FORCE_SPLIT 8 on 10 tiles: 5 ranges of 2, so the items with 1 or 2 tiles have
# ranges that hold none of their tiles.
PLANS = [
    ({"SMALL_PATH": 1}, None, SMALL),
    ({"SMALL_PATH": 0, "GRID": 0}, {"grid": "off"}, SMALL),
    ({"SMALL_PATH": 0, "GRID": 0}, {"grid": "off"}, LARGE),
    ({"SMALL_PATH": 0, "GRID": 2}, {"grid": "thresholds"}, LARGE),
    ({"SMALL_PATH": 0, "GRID": 3}, {"grid": "sorted", "order": "cell"}, LARGE),
    ({"SMALL_PATH": 0, "GRID": 0, "FORCE_SPLIT": 2}, {"grid": "off", "split": "2"}, LARGE),
    ({"SMALL_PATH": 0, "GRID": 0, "FORCE_SPLIT": 3}, {"grid": "off", "split": "3"}, LARGE),
    ({"SMALL_PATH": 0, "GRID": 0, "FORCE_SPLIT": 8}, {"grid": "off", "split": "5"}, LARGE),
    ({"SMALL_PATH": 0, "GRID": 3, "FORCE_SPLIT": 3}, {"grid": "sorted", "split": "3"}, LARGE),
    ({"SMALL_PATH": 0, "GRID": 2, "FORCE_SPLIT": 8}, {"grid": "thresholds", "split": "5"}, LARGE),
    ({"SMALL_PATH": 0, "GRID": 0, "FORCE_Q": 2}, {"grid": "off", "q": 2}, LARGE),
    ({"SMALL_PATH": 0, "GRID": 3, "INTERLEAVE": 1}, {"grid": "sorted", "order": "cell"}, LARGE),
]
PLAN_IDS = ["-".join("%s%s" % (k_.lower(), v) for k_, v in env.items()) + "-N%d" % shape[1] for env, _, shape in PLANS]


def _expect(plans, want):
    if want is None:                  # the warp-per-query path prints no plan
        assert plans == [], plans
        return
    assert len(plans) == 1, plans
    p = plans[0]
    for key, v in want.items():
        if key == "q":
            assert int(p["qpc"]) == 32 * v * int(p["warps"]), p
        else:
            assert p[key] == v, (key, p)


def _run_ragged(knobs, dev, ref, qry, rl, ql, k, form):
    r, q = _t(ref, dev), _t(qry, dev)
    rlt = None if rl is None else torch.tensor(rl, dtype=torch.int64, device=dev)
    qlt = None if ql is None else torch.tensor(ql, dtype=torch.int64, device=dev)
    (idx, dist), plans = knobs.run(lambda: ops.knn_ragged(r, q, k, form, rlt, qlt, want_dist=True))
    return idx.cpu().numpy(), dist.cpu().numpy(), plans


def _assert_oracle(idx, dist, ref, qry, rl, ql, k, form):
    oi, od = RO.knn(ref, qry, rl, ql, k, form)
    np.testing.assert_array_equal(idx, oi)
    np.testing.assert_array_equal(_bits(dist), _bits(od))


@pytest.mark.parametrize("form", [0, 2])
@pytest.mark.parametrize("env,want,shape", PLANS, ids=PLAN_IDS)
def test_every_plan_matches_the_oracle(knobs, cuda_dev, env, want, shape, form):
    B, N, S = shape
    ref, qry = _cloud(80, B, N, S)
    knobs.set(**env)
    for rl, ql in ((REF_LENS[N], QRY_LENS[S]), (None, None), ([N] * B, [S] * B), ([0] * B, [S] * B), ([N] * B, [0] * B)):
        idx, dist, plans = _run_ragged(knobs, cuda_dev, ref, qry, rl, ql, K, form)
        _expect(plans, want)
        _assert_oracle(idx, dist, ref, qry, rl, ql, K, form)
    # NULL lengths and full lengths are the dense call, bit for bit
    r, q = _t(ref, cuda_dev), _t(qry, cuda_dev)
    di, dd = ops.knn_search(r, q, K, form, want_dist=True)
    idx, dist, _ = _run_ragged(knobs, cuda_dev, ref, qry, None, None, K, form)
    np.testing.assert_array_equal(idx, di.cpu().numpy())
    np.testing.assert_array_equal(_bits(dist), _bits(dd.cpu().numpy()))


@pytest.mark.parametrize("env", [{"SMALL_PATH": 1}, {"SMALL_PATH": 0, "GRID": 0, "FORCE_SPLIT": 3}, {"SMALL_PATH": 0, "GRID": 3}],
                         ids=["small", "split3", "sorted"])
def test_out_of_range_lengths_are_clamped_on_the_device(knobs, cuda_dev, env):
    B, N, S = 6, 1000, 300
    ref, qry = _cloud(81, B, N, S)
    rl = [-5, N + 100, 2 ** 40, -(2 ** 40), 7, N]
    ql = [S + 1, -1, 2 ** 40, 17, -(2 ** 62), 0]
    knobs.set(**env)
    idx, dist, _ = _run_ragged(knobs, cuda_dev, ref, qry, rl, ql, K, 0)
    _assert_oracle(idx, dist, ref, qry, rl, ql, K, 0)


def test_k_larger_than_some_lengths_and_k_equal_to_N(knobs, cuda_dev):
    B, N, S = 4, 600, 200
    ref, qry = _cloud(82, B, N, S)
    for env in ({"SMALL_PATH": 1}, {"SMALL_PATH": 0, "GRID": 0}, {"SMALL_PATH": 0, "GRID": 3}):
        knobs.set(**env)
        for k in (N, 100):
            rl, ql = [3, 99, 0, N], [S, 5, S, 1]
            idx, dist, _ = _run_ragged(knobs, cuda_dev, ref, qry, rl, ql, k, 2)
            _assert_oracle(idx, dist, ref, qry, rl, ql, k, 2)
    with pytest.raises(RuntimeError, match="out of range"):
        ops.knn_ragged(_t(ref, cuda_dev), _t(qry, cuda_dev), N + 1, 0)


# ---- no output depends on the padded rows or on the output buffers ------------------------------------------------------
def _fill_padding(a, lens, how, rng):
    a = a.copy()
    for b, n in enumerate(lens):
        n = int(np.clip(n, 0, a.shape[1]))
        tail = a.shape[1] - n
        if tail == 0:
            continue
        if how == "dup":
            src = a[b, :max(n, 1)] if n else a[(b + 1) % a.shape[0]]
            a[b, n:] = src[rng.integers(0, len(src), tail)]
        else:
            a[b, n:] = {"nan": np.nan, "inf": np.inf, "-inf": -np.inf, "big": 1e30}[how]
    return a


def _raw_ragged(dev, ref, qry, rl, ql, k, form, fill):
    """b200pc_knn_ragged through the C ABI into output buffers pre-filled with the byte `fill`"""
    B, N, _ = ref.shape; S = qry.shape[1]
    lib = _lib.load()
    idx = torch.full((B * S * k * 8,), fill, dtype=torch.uint8, device=dev)
    dist = torch.full((B * S * k * 4,), fill, dtype=torch.uint8, device=dev)
    nws = lib.b200pc_search_workspace_bytes(B, N, S, k)
    ws = torch.full((nws,), fill, dtype=torch.uint8, device=dev)
    rlt = torch.tensor(rl, dtype=torch.int64, device=dev); qlt = torch.tensor(ql, dtype=torch.int64, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(lib.b200pc_knn_ragged(C.c_void_p(ref.data_ptr()), C.c_void_p(qry.data_ptr()), C.c_void_p(rlt.data_ptr()),
                                     C.c_void_p(qlt.data_ptr()), B, N, S, k, form, C.c_void_p(idx.data_ptr()),
                                     C.c_void_p(dist.data_ptr()), C.c_void_p(ws.data_ptr()), nws, stream))
    torch.cuda.synchronize()
    return idx.cpu().numpy().tobytes(), dist.cpu().numpy().tobytes()


@pytest.mark.parametrize("env", [{"SMALL_PATH": 1}, {"SMALL_PATH": 0, "GRID": 0, "FORCE_SPLIT": 8}, {"SMALL_PATH": 0, "GRID": 2},
                                 {"SMALL_PATH": 0, "GRID": 3, "FORCE_SPLIT": 3}, {"SMALL_PATH": 0, "GRID": 3, "INTERLEAVE": 1}],
                         ids=["small", "split8", "thresholds", "sorted-split3", "sorted-interleave"])
def test_padding_contents_and_output_buffers_do_not_matter(knobs, cuda_dev, env):
    B, N, S = (8, 1000, 700) if env.get("SMALL_PATH") == 1 else LARGE
    ref, qry = _cloud(83, B, N, S)
    rl, ql = REF_LENS[N], QRY_LENS[S]
    knobs.set(**env)
    rng = np.random.default_rng(5)
    want = None
    for how in ("nan", "inf", "-inf", "big", "dup"):
        r = _t(_fill_padding(ref, rl, how, rng), cuda_dev)
        q = _t(_fill_padding(qry, ql, how, rng), cuda_dev)
        for fill in (0x00, 0xA5):
            got = _raw_ragged(cuda_dev, r, q, rl, ql, K, 0, fill)
            if want is None:
                want = got
                oi, od = RO.knn(ref, qry, rl, ql, K, 0)
                np.testing.assert_array_equal(np.frombuffer(got[0], np.int64).reshape(oi.shape), oi)
                np.testing.assert_array_equal(np.frombuffer(got[1], np.int32).reshape(od.shape), _bits(od))
            assert got == want, (how, fill)


def test_non_finite_points_inside_the_lengths(knobs, cuda_dev):
    B, N, S = 4, 3000, 800
    ref, qry = _cloud(84, B, N, S)
    ref[0, 5] = np.nan; ref[1, :2948] = np.inf; ref[2, 10:20, 1] = np.nan      # item 1: 2 finite refs of 2950 valid
    qry[0, 3] = np.nan; qry[3, 0] = [np.inf, 0, 0]
    rl, ql = [2000, 2950, 1500, 3000], [800, 700, 11, 1]
    for env in ({"SMALL_PATH": 0, "GRID": 0}, {"SMALL_PATH": 0, "GRID": 3}, {"SMALL_PATH": 0, "GRID": 0, "FORCE_SPLIT": 3}):
        knobs.set(**env)
        idx, dist, _ = _run_ragged(knobs, cuda_dev, ref, qry, rl, ql, K, 2)
        _assert_oracle(idx, dist, ref, qry, rl, ql, K, 2)
    assert (idx[1, :700, 2:] == -1).all() and (idx[0, 3] == -1).all()
    # the shim leaves the non-finite slots inside the lengths at -1 / +inf and zero-pads only the slots the lengths empty
    knn = shim.knn_points(_t(qry, cuda_dev), _t(ref, cuda_dev), torch.tensor(ql, device=cuda_dev), torch.tensor(rl, device=cuda_dev), K=K)
    si, sd = knn.idx.cpu().numpy(), knn.dists.cpu().numpy()
    assert (si[1, :700, 2:] == -1).all() and np.isinf(sd[1, :700, 2:]).all()
    assert (si[0, 3] == -1).all()
    assert (si[2, 11:] == 0).all() and (sd[2, 11:] == 0).all()


# ---- Chamfer -----------------------------------------------------------------------------------------------------------
def _chamfer_case(seed=85):
    B, N, M = 5, 3000, 2600
    x, y = _cloud(seed, B, N, M)
    xl, yl = [3000, 1700, 513, 1, 2000], [2600, 2500, 1, 700, 0]
    return x, y, xl, yl


@pytest.mark.parametrize("env", [{}, {"SMALL_PATH": 0, "GRID": 0, "FORCE_SPLIT": 3}], ids=["default", "split3"])
def test_chamfer_ragged_forward_matches_the_oracle(knobs, cuda_dev, env):
    x, y, xl, yl = _chamfer_case()
    knobs.set(**env)
    dev = cuda_dev
    out = ops.chamfer_ragged(_t(x, dev), _t(y, dev), torch.tensor(xl, device=dev), torch.tensor(yl, device=dev))
    sums, dx, ix, dy, iy = [t.cpu().numpy() for t in out]
    osums, odx, oix, ody, oiy = RO.chamfer_terms(x, y, xl, yl)
    np.testing.assert_array_equal(ix, oix); np.testing.assert_array_equal(iy, oiy)
    np.testing.assert_array_equal(_bits(dx), _bits(odx)); np.testing.assert_array_equal(_bits(dy), _bits(ody))
    fin = np.isfinite(osums)
    np.testing.assert_allclose(sums[fin], osums[fin], rtol=1e-6)
    assert (np.isinf(sums) == np.isinf(osums)).all()
    assert sums[4, 1] == 0.0 and np.isinf(sums[4, 0])           # item 4: y is empty
    # repeated calls: the same bits
    again = ops.chamfer_ragged(_t(x, dev), _t(y, dev), torch.tensor(xl, device=dev), torch.tensor(yl, device=dev))
    for a, b in zip(out, again):
        assert torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a, b.view(torch.int32) if b.dtype == torch.float32 else b)


@pytest.mark.parametrize("batch_reduction", ["mean", "sum", None])
@pytest.mark.parametrize("point_reduction", ["mean", "sum"])
def test_chamfer_distance_loss_and_gradients(cuda_dev, point_reduction, batch_reduction):
    x, y, xl, yl = _chamfer_case(86)
    dev = cuda_dev
    xt = _t(x, dev).requires_grad_(); yt = _t(y, dev).requires_grad_()
    loss, none = shim.chamfer_distance(xt, yt, x_lengths=torch.tensor(xl, device=dev), y_lengths=torch.tensor(yl, device=dev),
                                       batch_reduction=batch_reduction, point_reduction=point_reduction)
    assert none is None
    x64 = torch.from_numpy(x).double().requires_grad_(); y64 = torch.from_numpy(y).double().requires_grad_()
    ol = RO.chamfer_distance64(x64, y64, xl, yl, point_reduction, batch_reduction)
    assert tuple(loss.shape) == tuple(ol.shape)
    np.testing.assert_allclose(loss.detach().cpu().double().numpy(), ol.detach().numpy(), rtol=2e-6)
    w = torch.linspace(0.5, 1.5, loss.numel(), dtype=torch.float64).reshape(ol.shape)
    (loss * w.to(dev).float()).sum().backward()
    (ol * w).sum().backward()
    gx, gy = xt.grad.cpu().double().numpy(), yt.grad.cpu().double().numpy()
    np.testing.assert_allclose(gx, x64.grad.numpy(), rtol=1e-4, atol=1e-6 * np.abs(x64.grad.numpy()).max())
    np.testing.assert_allclose(gy, y64.grad.numpy(), rtol=1e-4, atol=1e-6 * np.abs(y64.grad.numpy()).max())
    for b in range(len(xl)):                                  # padded points: exactly zero gradient
        assert (gx[b, xl[b]:] == 0).all() and (gy[b, yl[b]:] == 0).all()


def test_chamfer_full_lengths_equal_the_dense_call(cuda_dev):
    x, y = _cloud(87, 3, 2000, 1500)
    dev = cuda_dev
    xt, yt = _t(x, dev), _t(y, dev)
    dense, _ = shim.chamfer_distance(xt, yt)
    ragged, _ = shim.chamfer_distance(xt, yt, x_lengths=torch.full((3,), 2000, device=dev), y_lengths=torch.full((3,), 1500, device=dev))
    assert abs(ragged.item() - dense.item()) <= 1e-6 * abs(dense.item())
    d = ops.chamfer(xt, yt)
    r = ops.chamfer_ragged(xt, yt)
    for a, b in zip(d[1:], r[1:]):
        assert torch.equal(a, b)


def test_chamfer_ragged_backward_direct(cuda_dev):
    """the bwd entry on its own: gsums scale each item, padded rows and -1 indices give nothing"""
    x, y, xl, yl = _chamfer_case(88)
    dev = cuda_dev
    xt, yt = _t(x, dev), _t(y, dev)
    xlt, ylt = torch.tensor(xl, device=dev), torch.tensor(yl, device=dev)
    _, dx, ix, dy, iy = ops.chamfer_ragged(xt, yt, xlt, ylt)
    gs = torch.tensor(np.random.default_rng(3).normal(size=(5, 2)), dtype=torch.float32, device=dev)
    gx, gy = torch.ops.b200pc.chamfer_ragged_bwd(xt, yt, ix, iy, xlt, ylt, gs)
    ex = np.zeros_like(x, np.float64); ey = np.zeros_like(y, np.float64)
    ixn, iyn, g = ix.cpu().numpy(), iy.cpu().numpy(), gs.cpu().numpy().astype(np.float64)
    for b in range(5):
        for i in range(xl[b]):
            j = ixn[b, i]
            if j >= 0:
                d = 2 * g[b, 0] * (x[b, i].astype(np.float64) - y[b, j]); ex[b, i] += d; ey[b, j] -= d
        for j in range(yl[b]):
            i = iyn[b, j]
            if i >= 0:
                d = 2 * g[b, 1] * (y[b, j].astype(np.float64) - x[b, i]); ey[b, j] += d; ex[b, i] -= d
    np.testing.assert_allclose(gx.cpu().numpy(), ex, rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(gy.cpu().numpy(), ey, rtol=1e-5, atol=1e-5)


# ---- the pytorch3d shim ------------------------------------------------------------------------------------------------
def test_shim_knn_points_and_knn_gather_with_lengths(cuda_dev):
    B, P1, P2, Kk = 6, 1200, 2000, 8
    p2, p1 = _cloud(89, B, P2, P1)
    l1, l2 = [1200, 0, 37, 1199, 600, 1], [2000, 5, 0, 513, 8, 1999]
    dev = cuda_dev
    l1t, l2t = torch.tensor(l1, device=dev), torch.tensor(l2, device=dev)
    knn = shim.knn_points(_t(p1, dev), _t(p2, dev), l1t, l2t, K=Kk, return_nn=True)
    oi, od = RO.knn(p2, p1, l2, l1, Kk, strict.FORM_DIRECT)
    pad = (np.arange(P1)[None, :, None] >= np.array(l1)[:, None, None]) | (np.arange(Kk)[None, None, :] >= np.array(l2)[:, None, None])
    np.testing.assert_array_equal(knn.idx.cpu().numpy(), np.where(pad, 0, oi))
    np.testing.assert_array_equal(_bits(knn.dists.cpu().numpy()), _bits(np.where(pad, np.float32(0), od)))
    want_nn = np.where(pad[..., None], np.float32(0), strict.index_points(p2, np.where(pad, 0, oi)))
    np.testing.assert_array_equal(knn.knn.cpu().numpy(), want_nn)
    g = shim.knn_gather(_t(p2, dev), knn.idx, l2t).cpu().numpy()
    kpad = np.arange(Kk)[None, None, :] >= np.array(l2)[:, None, None]
    np.testing.assert_array_equal(g, np.where(kpad[..., None], np.float32(0), strict.index_points(p2, np.where(pad, 0, oi))))
    # full lengths: the same results as the call without lengths
    full = shim.knn_points(_t(p1, dev), _t(p2, dev), torch.full((B,), P1, device=dev), torch.full((B,), P2, device=dev), K=Kk, return_nn=True)
    plain = shim.knn_points(_t(p1, dev), _t(p2, dev), K=Kk, return_nn=True)
    for a, b in zip(full, plain):
        assert torch.equal(a, b)


def test_shim_knn_points_gradients_with_lengths(cuda_dev):
    B, P1, P2, Kk = 3, 300, 400, 4
    p2, p1 = _cloud(90, B, P2, P1)
    l1, l2 = [300, 120, 0], [2, 400, 250]
    p1[1, 120:] = np.nan; p2[0, 2:] = np.nan                  # padding that must not poison the gradients
    dev = cuda_dev
    a = _t(p1, dev).requires_grad_(); b = _t(p2, dev).requires_grad_()
    knn = shim.knn_points(a, b, torch.tensor(l1, device=dev), torch.tensor(l2, device=dev), K=Kk, return_nn=True)
    w = torch.linspace(0.1, 2.0, knn.dists.numel(), device=dev).reshape(knn.dists.shape)
    ((knn.dists * w).sum() + knn.knn.sum()).backward()
    ga, gb = a.grad.cpu().numpy(), b.grad.cpu().numpy()
    assert np.isfinite(ga).all() and np.isfinite(gb).all()
    assert (ga[1, 120:] == 0).all() and (ga[2] == 0).all() and (gb[0, 2:] == 0).all()
    # float64 autograd of the same selection on the valid part
    idx = knn.idx.cpu().numpy()
    a64 = torch.from_numpy(np.nan_to_num(p1)).double().requires_grad_(); b64 = torch.from_numpy(np.nan_to_num(p2)).double().requires_grad_()
    loss = 0
    wn = w.cpu().double()
    for bi in range(B):
        n1, n2 = l1[bi], min(l2[bi], Kk)
        if n1 == 0 or n2 == 0:
            continue
        nn = b64[bi][torch.from_numpy(idx[bi, :n1, :n2])]
        d = ((a64[bi, :n1, None] - nn) ** 2).sum(-1)
        loss = loss + (d * wn[bi, :n1, :n2]).sum() + nn.sum()
    loss.backward()
    np.testing.assert_allclose(ga, a64.grad.numpy(), rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(gb, b64.grad.numpy(), rtol=1e-4, atol=1e-4)


# ---- bounds-checked build ----------------------------------------------------------------------------------------------
BOUNDS_SCRIPT = r"""
import sys; sys.path.insert(0, %(root)r); sys.path.insert(0, %(pkg)r)
import numpy as np, torch
from b200pc import _lib, ops, synth
assert _lib.LIB_PATH.endswith("libb200pc_bounds.so"), _lib.LIB_PATH
ops.TUNING_AUTORELOAD = True
import os
dev = torch.device("cuda:0")
for env in ({"B200PC_SMALL_PATH": "1"}, {"B200PC_SMALL_PATH": "0", "B200PC_GRID": "0", "B200PC_FORCE_SPLIT": "8"},
            {"B200PC_SMALL_PATH": "0", "B200PC_GRID": "2"}, {"B200PC_SMALL_PATH": "0", "B200PC_GRID": "3", "B200PC_FORCE_SPLIT": "3"},
            {"B200PC_SMALL_PATH": "0", "B200PC_GRID": "3", "B200PC_INTERLEAVE": "1"}, {"B200PC_SMALL_PATH": "0", "B200PC_FORCE_Q": "2"}):
    for k_ in ("B200PC_SMALL_PATH", "B200PC_GRID", "B200PC_FORCE_SPLIT", "B200PC_INTERLEAVE", "B200PC_FORCE_Q"):
        os.environ.pop(k_, None)
    os.environ.update(env)
    N = 1000 if env.get("B200PC_SMALL_PATH") == "1" else 5000
    a, b = synth.batch_pairs(3, 8, N)
    r = torch.from_numpy(a).to(dev); q = torch.from_numpy(b[:, :777].copy()).to(dev)
    rl = torch.tensor([-3, 0, 1, 15, 511, 513, N, N + 9], device=dev)
    ql = torch.tensor([777, 2 ** 40, -1, 0, 1, 33, 500, 776], device=dev)
    for k in (1, 16):
        ops.knn_ragged(r, q, k, 0, rl, ql, want_dist=True); ops.knn_ragged(r, q, k, 2, rl, None)
    x = r.clone().requires_grad_(); y = q.clone().requires_grad_()
    sums = ops.chamfer_ragged(x, y, rl, ql)[0]
    torch.where(torch.isfinite(sums), sums, torch.zeros_like(sums)).sum().backward()
    torch.cuda.synchronize()
print("ragged bounds ok")
"""


def test_ragged_entries_under_the_bounds_checked_build():
    lib = os.path.join(PKG, "b200pc", "libb200pc_bounds.so")
    assert os.path.exists(lib), "libb200pc_bounds.so is not built (make -C point-cloud-interpolation-_b200 bounds)"
    p = subprocess.run([sys.executable, "-c", BOUNDS_SCRIPT % {"root": ROOT, "pkg": PKG}], env=dict(os.environ, B200PC_LIBRARY="bounds"),
                       capture_output=True, text=True, timeout=600)
    out = p.stdout + p.stderr
    assert "device assert failed" not in out, out[-4000:]
    assert p.returncode == 0 and "ragged bounds ok" in out, out[-4000:]
