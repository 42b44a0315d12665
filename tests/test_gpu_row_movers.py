"""Every variant of the HBM row movers, bit-exact against oracle/strict.py:
  index_points       gather_flat / gather_rows<2|4|8> (B200PC_GATHER_FLAT, B200PC_GATHER_ROWS) / gather_scalar (misaligned)
  three_interpolate  interp_flat / interp_rows<1|2|4|8> (B200PC_INTERP_FLAT, B200PC_INTERP_ROWS) / interp_scalar (misaligned)
  group_points       the asynchronous-copy kernel (default and B200PC_BULK=1 shapes) / the register kernels
including shapes large enough that the warp-per-row kernels go round their grid-stride loop (their grid is capped at
16 CTAs of 8 warps per SM), where interp_rows prefetches the next group's (index, weight) before gathering the current one."""
import functools

import numpy as np
import pytest
import torch

from b200pc import ops, pointnet2_utils as P, synth
from oracle import strict


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _misaligned(a, dev):
    """contiguous copy on `dev` whose base is 4 bytes past a 16-byte boundary (the launchers then take the scalar kernels)"""
    a = np.ascontiguousarray(a, np.float32)
    t = torch.empty(a.size + 1, dtype=torch.float32, device=dev)[1:].view(a.shape)
    t.copy_(torch.from_numpy(a))
    assert t.data_ptr() % 16 == 4 and t.is_contiguous()
    return t


def _bits(a):
    return np.ascontiguousarray(a).view(np.int32)


def _assert_bits(got, want):
    assert got.shape == want.shape
    np.testing.assert_array_equal(_bits(got), _bits(want))


def _set_knobs(monkeypatch, **kw):
    for k, v in kw.items():
        monkeypatch.setenv("B200PC_" + k, str(v))
    ops.reload_tuning()


# ==========================================================================================
# index_points
# ==========================================================================================
GATHER_VARIANTS = [dict(GATHER_FLAT=f, GATHER_ROWS=r) for f in (0, 1) for r in (2, 4, 8)] + ["scalar"]
GATHER_IDS = ["flat%d-rows%d" % (v["GATHER_FLAT"], v["GATHER_ROWS"]) for v in GATHER_VARIANTS[:-1]] + ["scalar"]


def _gather(dev, monkeypatch, variant, pts, idx):
    if variant == "scalar":
        p = _misaligned(pts, dev)
    else:
        _set_knobs(monkeypatch, **variant)
        p = _t(pts, dev)
    return P.index_points(p, _t(idx, dev)).cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 8, 124, 128, 132, 256, 260])
@pytest.mark.parametrize("variant", GATHER_VARIANTS, ids=GATHER_IDS)
def test_index_points_variants_bit_exact(cuda_dev, monkeypatch, variant, C):
    B, N, R = 2, 1000, 333                                # 666 rows: not a multiple of 4 or 8
    rng = np.random.default_rng(C)
    pts = rng.normal(size=(B, N, C)).astype(np.float32)
    idx = rng.integers(-N, N, size=(B, R))
    _assert_bits(_gather(cuda_dev, monkeypatch, variant, pts, idx), strict.index_points(pts, idx))


@functools.lru_cache(maxsize=1)
def _big_gather_case():
    B, N, R, C = 2, 4096, 90000, 128                      # 180 000 rows: one pass of gather_rows<8> covers 151 552
    rng = np.random.default_rng(11)
    pts = rng.normal(size=(B, N, C)).astype(np.float32)
    idx = rng.integers(-N, N, size=(B, R))
    return pts, idx, strict.index_points(pts, idx)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", GATHER_VARIANTS, ids=GATHER_IDS)
def test_index_points_variants_grid_stride(cuda_dev, monkeypatch, variant):
    pts, idx, want = _big_gather_case()
    _assert_bits(_gather(cuda_dev, monkeypatch, variant, pts, idx), want)


# ==========================================================================================
# three_interpolate: (f0*w0 + f1*w1) + f2*w2 with separate roundings, like strict.c (built with -ffp-contract=off)
# ==========================================================================================
INTERP_VARIANTS = [dict(INTERP_FLAT=f, INTERP_ROWS=r) for f in (0, 1) for r in (1, 2, 4, 8)] + ["scalar"]
INTERP_IDS = ["flat%d-rows%d" % (v["INTERP_FLAT"], v["INTERP_ROWS"]) for v in INTERP_VARIANTS[:-1]] + ["scalar"]


def _interp(dev, monkeypatch, variant, feat, idx, w):
    if variant == "scalar":
        f = _misaligned(feat, dev)
    else:
        _set_knobs(monkeypatch, **variant)
        f = _t(feat, dev)
    return P.three_interpolate(f, _t(idx, dev), _t(w, dev)).cpu().numpy()


@functools.lru_cache(maxsize=1)
def _interp_geometry():
    a, _ = synth.batch_pairs(80, 2, 4099)                # 4 099 dense rows per cloud: ragged for every ROWS
    known = a[:, ::8].copy()
    dist, idx = strict.three_nn(a, known)
    return known.shape[1], dist, idx


@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 12, 64, 128, 256, 260])
@pytest.mark.parametrize("variant", INTERP_VARIANTS, ids=INTERP_IDS)
def test_three_interpolate_variants_bit_exact(cuda_dev, monkeypatch, variant, C):
    S, dist, idx = _interp_geometry()
    feat = np.random.default_rng(C).normal(size=(2, S, C)).astype(np.float32)
    for weights in (0, 1):
        w = strict.three_weights(dist, weights)
        _assert_bits(_interp(cuda_dev, monkeypatch, variant, feat, idx, w), strict.three_interpolate(feat, idx, w))


@functools.lru_cache(maxsize=1)
def _c3_interp_case():
    B, N, S, C = 16, 16384, 4096, 128                     # C3: 262 144 rows, ~7 grid-stride passes of interp_rows<2>
    rng = np.random.default_rng(12)
    feat = rng.normal(size=(B, S, C)).astype(np.float32)
    idx = rng.integers(0, S, size=(B, N, 3))
    w = strict.three_weights(rng.uniform(1e-3, 4.0, size=(B, N, 3)).astype(np.float32), 0)
    return feat, idx, w, strict.three_interpolate(feat, idx, w)


@pytest.mark.gpu
@pytest.mark.parametrize("variant", INTERP_VARIANTS, ids=INTERP_IDS)
def test_three_interpolate_variants_c3_size(cuda_dev, monkeypatch, variant):
    feat, idx, w, want = _c3_interp_case()
    _assert_bits(_interp(cuda_dev, monkeypatch, variant, feat, idx, w), want)


# ==========================================================================================
# group_points
# ==========================================================================================
def _group_ref(xyz, new, feat, idx, xyz_first):
    """strict.group_points with torch's wrap of negative indices; a slot still out of range reads as zeros
    (its xyz channels are 0 - centre), as the kernels document"""
    N = xyz.shape[1]
    w = np.where(idx < 0, idx + N, idx)
    ok = (w >= 0) & (w < N)
    out = strict.group_points(xyz, new, feat, np.where(ok, w, 0), xyz_first)
    D = 0 if feat is None else feat.shape[2]
    xoff, foff = (0, 3) if xyz_first else (D, 0)
    okT = ok.transpose(0, 2, 1)[:, None]                                           # [B,1,K,S]
    out[:, xoff:xoff + 3] = np.where(okT, out[:, xoff:xoff + 3], (np.float32(0) - new).transpose(0, 2, 1)[:, :, None, :])
    if D:
        out[:, foff:foff + D] = np.where(okT, out[:, foff:foff + D], np.float32(0))
    return out


def _group_case(B, N, S, K, D, seed):
    a, b = synth.batch_pairs(seed, B, max(N, S))
    rng = np.random.default_rng(seed)
    feat = rng.normal(size=(B, N, D)).astype(np.float32)
    idx = rng.integers(-N, N, size=(B, S, K))
    flat = idx.reshape(-1)
    flat[::23] = N                                         # the ball query's empty-ball sentinel
    flat[5::31] = -N - 1
    return a[:, :N].copy(), b[:, :S].copy(), feat, idx


def _check_group(dev, B, N, S, K, D, seed, misaligned=False):
    xyz, new, feat, idx = _group_case(B, N, S, K, D, seed)
    f = _misaligned(feat, dev) if misaligned else _t(feat, dev)
    for xyz_first in (True, False):
        out = P.group_points(_t(xyz, dev), _t(new, dev), f, _t(idx, dev), xyz_first)
        _assert_bits(out.cpu().numpy(), _group_ref(xyz, new, feat, idx, xyz_first))


# default plan (B200PC_BULK unset, D <= 64): K is cut into parts of kper > 1 slots that do not divide K evenly
BULK_DEFAULT_SHAPES = [(16, 4096, 10, 64), (16, 4096, 12, 32), (16, 4096, 20, 16), (8, 4096, 20, 16), (8, 4096, 24, 32),
                       (1, 16384, 48, 16)]                 # B, S, K, D
# B200PC_BULK=1: D = 132 is 33 chunks (warp_copy_row ends on a partial pass), 392 the widest row that still gets the 4 warps
# the forced plan needs, 396 falls back to the register kernel; the (1, 865, 256) and (1, 4000, 256) rows give kper = 2
BULK_FORCED_SHAPES = [(B, S, K, D) for D in (16, 32, 132, 392, 396) for (B, S, K) in ((3, 33, 1), (2, 777, 12), (1, 100, 256))] + \
                     [(1, 865, 256, 384), (1, 4000, 256, 16)]


def _bulk_plan(B, S, K, D, force, sms=148, fixed=True):
    """host restatement of group_bulk's planner (csrc/rowmove.cu) -> (ksplit, kper) or None when the shape is not served"""
    if (not force and B * S * K < 32768) or D < 16 or D % 4 or D > 1024 or K > 256 or (D < 128 and 32 % (D // 4)):
        return None
    tile = 32 * (D * 4 + (32 if (D >> 2) & 1 else 16))
    nwarps = 0
    for _ in range(2):
        base = B * ((S + 31) // 32)
        ksplit = 1
        while ksplit < K and base * ksplit < 6 * sms * (nwarps or 16):
            ksplit <<= 1
        ksplit = min(ksplit, K)
        kper = -(-K // ksplit)
        if fixed:
            ksplit = -(-K // kper)
        idx_bytes = (32 * (kper | 1) * 4 + 127) & ~127
        w1, w2 = 200 * 1024 // (idx_bytes + tile), 200 * 1024 // (idx_bytes + 2 * tile)
        nwarps = min(w2 if w2 >= 16 else w1, 16)
        if nwarps < 4 or (not force and nwarps < 16):
            return None
    return ksplit, kper


def test_bulk_shapes_cover_split_slots_cpu():
    """the shapes below reach what they are meant to on a 148-SM B200: parts of more than one slot (the unfixed planner
    numbered parts that started past K there), the forced path up to D = 392 and the fallback at D = 396"""
    for B, S, K, D in BULK_DEFAULT_SHAPES:
        ksplit, kper = _bulk_plan(B, S, K, D, False)
        old_split, _ = _bulk_plan(B, S, K, D, False, fixed=False)
        assert kper > 1 and (ksplit - 1) * kper < K <= ksplit * kper and (old_split - 1) * kper >= K
    assert _bulk_plan(1, 865, 256, 384, True)[1] == 2 and _bulk_plan(1, 4000, 256, 16, True)[1] == 2
    assert _bulk_plan(2, 777, 12, 392, True) is not None and _bulk_plan(2, 777, 12, 396, True) is None


@pytest.mark.gpu
@pytest.mark.parametrize("B,S,K,D", BULK_DEFAULT_SHAPES)
def test_group_points_default_bulk_plan(cuda_dev, B, S, K, D):
    _check_group(cuda_dev, B, 2048, S, K, D, seed=S + K + D)


@pytest.mark.gpu
@pytest.mark.parametrize("B,S,K,D", BULK_FORCED_SHAPES)
def test_group_points_forced_bulk(cuda_dev, monkeypatch, B, S, K, D):
    _set_knobs(monkeypatch, BULK=1)
    _check_group(cuda_dev, B, 600, S, K, D, seed=S + K + D)


@pytest.mark.gpu
@pytest.mark.parametrize("B,S,K,D", BULK_FORCED_SHAPES[:-2])
def test_group_points_forced_bulk_misaligned_features(cuda_dev, monkeypatch, B, S, K, D):
    """the asynchronous-copy kernel needs 16-byte rows: with a misaligned table it declines and the scalar kernel runs"""
    _set_knobs(monkeypatch, BULK=1)
    _check_group(cuda_dev, B, 600, S, K, D, seed=S + K + D + 1, misaligned=True)
