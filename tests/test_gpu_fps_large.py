"""Farthest point sampling of clouds beyond the registers of one cluster: the wide tier (fps_wide_kernel, csrc/fps.cu).

Clouds of 131 073 .. 262 144 points run on a cluster of 16 CTAs that keeps 8 192 points per CTA in registers and the rest
of its slice in shared memory; B200PC_FPS_CLUSTER=C sends a cloud of more than C * 8 192 points there at small N, where
the oracle is cheap.  Every case reads the plan line back (B200PC_DEBUG_PLAN) to prove which tier ran.

Bar: the picks bit-exact against oracle/strict (the reference's fp32 arithmetic and first arg-max).  The full-resolution
sweeps are those of the project's synthetic HDL-64 (b200pc/synth.py): 64 beams x 2 083 azimuth steps, 133 312 returns.
"""
import ctypes as C
import functools
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import guarded as G
from b200pc import _lib, io, ops, synth
from oracle import strict
from test_gpu_non_finite import _fps_cloud as _non_finite_cloud
from test_gpu_plans import FPS_PLAN, Knobs

gpu = pytest.mark.gpu

CTA_REGISTER_POINTS, MAX_N = 512 * 16, 262144          # fps.cu: FPS_T * FPS_WIDE_P, FPS_MAX_N
WIDE_PLAN = re.compile(FPS_PLAN.pattern + r"(?:, shared (?P<Q>\d+) points/thread)?\n")


class WideKnobs(Knobs):
    """Knobs whose run() also reads the shared-memory points per thread of the plan line (None: registers only)"""

    def run(self, fn):
        torch.cuda.synchronize()
        self.capfd.readouterr()
        out = fn()
        torch.cuda.synchronize()
        err = self.capfd.readouterr().err
        return out, [m.groupdict() for m in WIDE_PLAN.finditer(err)]


@pytest.fixture
def knobs(cuda_dev, monkeypatch, capfd):
    return WideKnobs(monkeypatch, capfd)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def wide_q(N, C):
    """shared-memory points per thread of the wide tier: the part of a ceil(N / C) slice beyond the registers, rounded
    up to a power of two"""
    extra = -(-N // C) - CTA_REGISTER_POINTS
    q = 1
    while 512 * q < extra:
        q *= 2
    return q


def expect_plan(plans, C, Q, n=1):
    assert len(plans) == n, plans
    for p in plans:
        if Q is None:
            assert (int(p["C"]), p["Q"]) == (C, None), p
        else:
            assert (int(p["C"]), int(p["P"]), p["exchange"], int(p["Q"])) == (C, 16, "two-level", Q), p


@functools.lru_cache(maxsize=None)
def full_sweeps(i):
    """both full-resolution sweeps of synthetic pair i (frame_pair(i, .) before its sub-sampling)"""
    rng = np.random.default_rng(1000 + i)
    walls, boxes = synth._scene(rng)
    f1 = synth._scan(walls, boxes, (0.0, 0.0, 0.0), rng)
    f2 = synth._scan(walls, boxes, (1.2, 0.0, np.deg2rad(1.0)), rng)
    return f1, f2


def test_full_sweep_is_above_the_register_capacity():
    """CPU: the synthetic HDL-64 sweep the loader must down-sample is larger than 16 CTAs x 8 192 points"""
    f1, f2 = full_sweeps(0)
    assert f1.shape == (133312, 3) and f1.shape[0] > 16 * CTA_REGISTER_POINTS
    assert f1.shape[0] + f2.shape[0] >= MAX_N


# ---- bit-exact against the oracle on the default plan -------------------------------------------------------------------
SIZES = [131072, 131073, 133312, 196608, 262144]


@functools.lru_cache(maxsize=None)
def _big_case(N):
    """three clouds of N points (crops of the two full sweeps of pairs 0..2 laid end to end; at 133 312 the full first
    sweep), starts 0, N - 1 and one in between; the oracle's first 4 096 picks"""
    clouds = []
    for i in range(3):
        f1, f2 = full_sweeps(i)
        clouds.append(f1 if N == f1.shape[0] else np.concatenate([f1, f2])[:N])
    a = np.ascontiguousarray(np.stack(clouds))
    start = np.array([0, N - 1, N // 2 + 17], np.int64)
    return a, start, strict.farthest_point_sample(a, 4096, start)


@gpu
@pytest.mark.parametrize("npoint", [37, 4096])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("N", SIZES)
def test_default_plan_matches_oracle(knobs, cuda_dev, N, B, npoint):
    a, start, want = _big_case(N)
    knobs.set(FPS_CLUSTER=None, FPS_FLAT=None)
    s = start[:B] if B > 1 else start[1:2]                      # B = 1 starts at N - 1
    w = want[:B] if B > 1 else want[1:2]
    out, plans = knobs.run(lambda: ops.fps(_t(a[:B] if B > 1 else a[1:2], cuda_dev), npoint, _t(s, cuda_dev)))
    expect_plan(plans, 16, None if N <= 16 * CTA_REGISTER_POINTS else wide_q(N, 16))
    np.testing.assert_array_equal(out.cpu().numpy(), w[:, :npoint])


def test_wide_q_of_the_default_plan():
    """CPU: a sweep just above the old limit puts one point per thread in shared memory, the largest cloud sixteen"""
    assert [wide_q(N, 16) for N in SIZES[1:]] == [1, 1, 8, 16]


# ---- the wide tier forced at small N ------------------------------------------------------------------------------------
FORCED = [(12000, 1), (20000, 2), (60000, 4), (100000, 8)]


@functools.lru_cache(maxsize=None)
def _forced_case(N):
    a, _ = synth.batch_pairs(90, 2, N)
    start = np.array([0, N - 1], np.int64)
    npoint = N if N <= 20000 else 2048                  # npoint = N: the final picks tie at min-dist 0
    return a, start, strict.farthest_point_sample(a, npoint, start)


@gpu
@pytest.mark.parametrize("N,C", FORCED)
def test_forced_cluster_runs_the_wide_tier(knobs, cuda_dev, N, C):
    a, start, want = _forced_case(N)
    assert C * CTA_REGISTER_POINTS < N <= 2 * C * CTA_REGISTER_POINTS
    knobs.set(FPS_CLUSTER=C, FPS_FLAT=None)
    x, s = _t(a, cuda_dev), _t(start, cuda_dev)
    for npoint in sorted({want.shape[1], 37}):
        out, plans = knobs.run(lambda: ops.fps(x, npoint, s))
        expect_plan(plans, C, wide_q(N, C))
        np.testing.assert_array_equal(out.cpu().numpy(), want[:, :npoint])


@gpu
def test_forced_flat_exchange_does_not_apply_to_the_wide_tier(knobs, cuda_dev):
    a, start, want = _forced_case(20000)
    knobs.set(FPS_CLUSTER=2, FPS_FLAT=1)
    out, plans = knobs.run(lambda: ops.fps(_t(a, cuda_dev), 300, _t(start, cuda_dev)))
    expect_plan(plans, 2, wide_q(20000, 2))
    np.testing.assert_array_equal(out.cpu().numpy(), want[:, :300])


@gpu
def test_cluster_values_valid_before_keep_their_plan(knobs, cuda_dev):
    """a forced cluster that holds the cloud in registers still runs the register kernels; one that cannot hold it even
    with the shared-memory tier is ignored (the default plan runs)"""
    a, start, want = _forced_case(20000)
    x, s = _t(a, cuda_dev), _t(start, cuda_dev)
    for C, plan in ((4, (4, None)), (3, (3, None)), (1, (8, None))):   # 3 x 8 192 >= 20 000; 1 x 16 384 < 20 000
        knobs.set(FPS_CLUSTER=C, FPS_FLAT=0)
        out, plans = knobs.run(lambda: ops.fps(x, 300, s))
        assert len(plans) == 1 and (int(plans[0]["C"]), plans[0]["Q"]) == plan, (C, plans)
        np.testing.assert_array_equal(out.cpu().numpy(), want[:, :300])


# ---- ties, padding, contraction ---------------------------------------------------------------------------------------
@gpu
def test_grid_snapped_ties(knobs, cuda_dev):
    """coordinates on a 2^-6 grid (all fp32 arithmetic exact, exact ties common): a wide cloud and one with many duplicates"""
    N = 140000
    a = np.concatenate([synth.grid_snapped(7, 1, N), synth.grid_snapped(8, 1, N, span=40)]).astype(np.float32)
    start = np.array([3, N - 1], np.int64)
    want = strict.farthest_point_sample(a, 1024, start)
    knobs.set(FPS_CLUSTER=None, FPS_FLAT=None)
    out, plans = knobs.run(lambda: ops.fps(_t(a, cuda_dev), 1024, _t(start, cuda_dev)))
    expect_plan(plans, 16, wide_q(N, 16))
    np.testing.assert_array_equal(out.cpu().numpy(), want)


@gpu
@pytest.mark.parametrize("real,C", [(10000, 1), (12000, 2)])
def test_padded_duplicates_first_argmax(knobs, cuda_dev, real, C):
    """a cloud followed by copies of its first half (the reference's loaders pad short frames by re-drawing points): once
    every real point is taken, the first arg-max must pick the original before its copies -- also across the register,
    shared-memory and CTA boundaries"""
    a, _ = synth.batch_pairs(71, 1, real)
    dup = np.concatenate([a, a[:, :real // 2]], 1)
    dup = np.ascontiguousarray(np.concatenate([dup, dup[:, ::-1]], 0))
    N = dup.shape[1]
    start = np.array([7, N - 1], np.int64)
    npoint = real + 1000
    want = strict.farthest_point_sample(dup, npoint, start)
    knobs.set(FPS_CLUSTER=C, FPS_FLAT=None)
    out, plans = knobs.run(lambda: ops.fps(_t(dup, cuda_dev), npoint, _t(start, cuda_dev)))
    expect_plan(plans, C, wide_q(N, C))
    np.testing.assert_array_equal(out.cpu().numpy(), want)


@gpu
@pytest.mark.parametrize("pairs,C", [(70000, None), (6000, 1), (9000, 2)])
def test_near_ties_no_fused_multiply_add(knobs, cuda_dev, pairs, C):
    """clouds whose first-round pick differs between the reference's (dx*dx + dy*dy) + dz*dz and a fused multiply-add
    (tests/adversarial.py): the wide tier must pick the unfused one"""
    from adversarial import first_round_pick, fps_rot90_cloud
    clouds = np.stack([fps_rot90_cloud(950 + i, pairs) for i in range(2)])
    N = clouds.shape[1]
    picks = []
    for c in clouds:
        unfused, fused = first_round_pick(c, False), first_round_pick(c, True)
        assert unfused != fused
        picks.append(unfused)
    start = np.zeros(2, np.int64)
    want = strict.farthest_point_sample(clouds, 64, start)
    knobs.set(FPS_CLUSTER=C, FPS_FLAT=None)
    out, plans = knobs.run(lambda: ops.fps(_t(clouds, cuda_dev), 64, _t(start, cuda_dev)))
    expect_plan(plans, C or 16, wide_q(N, C or 16))
    got = out.cpu().numpy()
    assert list(got[:, 1]) == picks
    np.testing.assert_array_equal(got, want)


def _sass_by_function():
    sass = subprocess.check_output(["cuobjdump", "-sass", _lib.LIB_PATH], text=True)
    out, name = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
        elif name is not None:
            out[name].append(line)
    return out


def test_wide_kernels_never_fuse_multiply_add():
    """CPU: the wide tier computes (dx*dx + dy*dy) + dz*dz with every product rounded on its own, like fps_kernel"""
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("library not built")
    funcs = {n: b for n, b in _sass_by_function().items() if "fps_wide_kernel" in n}
    assert len(funcs) == 5, sorted(funcs)           # Q = 1, 2, 4, 8, 16
    for name, body in funcs.items():
        text = "\n".join(body)
        for bad in ("FFMA2", "FMUL2", " FFMA ", "FFMA.", "DFMA"):
            assert bad not in text, "%s contains %s" % (name, bad.strip())
        assert " FMUL " in text and " FADD " in text


# ---- non-finite coordinates -----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("start_kind", ["finite", "non_finite"])
@pytest.mark.parametrize("N,C", [(140000, None), (20000, 2)])
def test_non_finite_coordinates(knobs, cuda_dev, N, C, start_kind):
    """+-1e30 points whose squared distances overflow, NaN and +-inf points, starts at a 1e30 or NaN point: the picks of
    tests/test_gpu_non_finite.py, where strict and the reference's own torch code agree"""
    cloud, start, want = _non_finite_cloud(N, start_kind)
    knobs.set(FPS_CLUSTER=C, FPS_FLAT=None)
    out, plans = knobs.run(lambda: ops.fps(_t(cloud, cuda_dev), 200, _t(start, cuda_dev)))
    expect_plan(plans, C or 16, wide_q(N, C or 16))
    np.testing.assert_array_equal(out.cpu().numpy(), want)


# ---- edges ---------------------------------------------------------------------------------------------------------------
@gpu
def test_above_the_limit_fails_cleanly(cuda_dev):
    x = torch.zeros(1, MAX_N + 1, 3, device=cuda_dev)
    s = torch.zeros(1, dtype=torch.long, device=cuda_dev)
    with pytest.raises(RuntimeError, match="262144"):
        ops.fps(x, 4, s)
    idx = torch.full((1, 4), -5, dtype=torch.long, device=cuda_dev)
    L = _lib.load()
    rc = L.b200pc_fps(x.data_ptr(), 1, MAX_N + 1, 4, s.data_ptr(), idx.data_ptr(), None, 0, None)
    torch.cuda.synchronize()
    assert rc == _lib.EINVAL and "262144" in _lib.last_error() and "262145" in _lib.last_error()
    assert (idx == -5).all()


# ---- guarded buffers -----------------------------------------------------------------------------------------------------
def _ok(rc):
    assert rc == 0, "rc %d: %s" % (rc, _lib.last_error())


def _st():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@functools.lru_cache(maxsize=None)
def _guarded_case(kind):
    if kind == "forced":                                # the wide tier on one CTA, every pick (the last ones tie at 0)
        a, _ = synth.batch_pairs(73, 2, 9001)
        start, npoint = np.array([17, 8999], np.int64), 9001
    else:                                               # a full sweep on the default plan
        a = np.ascontiguousarray(np.stack([full_sweeps(3)[0], full_sweeps(4)[0]]))
        start, npoint = np.array([0, 133311], np.int64), 300
    return a, start, npoint, strict.farthest_point_sample(a, npoint, start)


@gpu
@pytest.mark.parametrize("kind", ["forced", "default"])
@pytest.mark.parametrize("entry", ["fps", "fps_sample"])
def test_guarded_buffers(knobs, cuda_dev, entry, kind):
    """every output element written, nothing outside the outputs, the ignored workspace untouched (tests/guarded.py)"""
    cloud, start, npoint, want = _guarded_case(kind)
    B, N = cloud.shape[:2]
    C_ = 1 if kind == "forced" else 16
    knobs.set(FPS_CLUSTER=1 if kind == "forced" else None, FPS_FLAT=None)
    L = _lib.load()
    bufs = [G.inp("xyz", cloud), G.inp("start", start), G.out("idx", (B, npoint), torch.int64)]
    if entry == "fps":
        nws = L.b200pc_fps_workspace_bytes(B, N)
        bufs.append(G.inp("ws", np.random.default_rng(3).integers(0, 256, nws, dtype=np.uint8), align=16))

        def call(lay):
            _ok(L.b200pc_fps(lay.ptr("xyz"), B, N, npoint, lay.ptr("start"), lay.ptr("idx"), lay.ptr("ws"), nws, _st()))
    else:
        bufs.append(G.out("new_xyz", (B, npoint, 3), torch.float32))

        def call(lay):
            _ok(L.b200pc_fps_sample(lay.ptr("xyz"), B, N, npoint, lay.ptr("start"), lay.ptr("idx"), lay.ptr("new_xyz"), _st()))

    (res, _), plans = knobs.run(lambda: G.check_call(bufs, call, cuda_dev))
    expect_plan(plans, C_, wide_q(N, C_), n=len(G.POISONS) * len(G.ALIGNMENTS))
    np.testing.assert_array_equal(res["idx"], want)
    if entry == "fps_sample":
        np.testing.assert_array_equal(res["new_xyz"].view(np.int32), cloud[np.arange(B)[:, None], want].view(np.int32))


@gpu
def test_guarded_host_entry(cuda_dev):
    cloud, start, npoint, want = _guarded_case("default")
    B, N = cloud.shape[:2]
    H = dict(space="host")
    bufs = [G.inp("xyz", cloud, **H), G.inp("start", start, **H), G.out("idx", (B, npoint), torch.int64, **H)]
    L = _lib.load()
    ops.reload_tuning()

    def call(lay):
        _ok(L.b200pc_fps_host(lay.ptr("xyz"), B, N, npoint, lay.ptr("start"), lay.ptr("idx")))

    res, _ = G.check_call(bufs, call, cuda_dev)
    np.testing.assert_array_equal(res["idx"], want)


# ---- determinism -------------------------------------------------------------------------------------------------------
@gpu
def test_two_runs_agree_at_the_largest_cloud(cuda_dev):
    a, start, _ = _big_case(MAX_N)
    ops.reload_tuning()
    x, s = _t(a, cuda_dev), _t(start, cuda_dev)
    first = ops.fps(x, 4096, s).cpu()
    second = ops.fps(x, 4096, s).cpu()
    assert torch.equal(first, second)


# ---- the data loader -----------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _loader_case():
    f1 = full_sweeps(5)[0]
    both = np.ascontiguousarray(np.stack([f1, f1]))
    start = np.array([0, 70001], np.int64)
    return f1, start, strict.farthest_point_sample(both, 16384, start)


@gpu
def test_loader_samples_a_full_sweep(cuda_dev, monkeypatch):
    monkeypatch.delenv("B200PC_FPS_CLUSTER", raising=False)
    ops.reload_tuning()
    sweep, start, want = _loader_case()
    assert sweep.shape[0] == 133312
    for b, st in enumerate(("open3d", [int(start[1])])):
        pts, idx = io.sample_clouds([sweep], 16384, device=cuda_dev, start=st, return_index=True)
        np.testing.assert_array_equal(idx.cpu().numpy()[0], want[b])
        np.testing.assert_array_equal(pts.cpu().numpy()[0].view(np.int32), sweep[want[b]].view(np.int32))


@gpu
def test_loader_mixed_batch(cuda_dev, monkeypatch):
    """one full sweep and a 30 000-point sweep in one launch: the short one padded with copies of its point 0"""
    monkeypatch.delenv("B200PC_FPS_CLUSTER", raising=False)
    ops.reload_tuning()
    sweep, _, want_full = _loader_case()
    short = synth.frame_pair(6, 30000)[0]
    want_short = strict.farthest_point_sample(short[None], 4096, np.array([0], np.int64))
    pts, idx = io.sample_clouds([sweep, short], 4096, device=cuda_dev, return_index=True)
    idx = idx.cpu().numpy()
    np.testing.assert_array_equal(idx[0], want_full[0, :4096])
    np.testing.assert_array_equal(idx[1], want_short[0])
    np.testing.assert_array_equal(pts.cpu().numpy()[1].view(np.int32), short[want_short[0]].view(np.int32))
