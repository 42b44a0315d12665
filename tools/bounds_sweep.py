"""Every kernel family on small, ragged and awkward shapes -- meant to be run against the bounds-checked build
(B200PC_LIBRARY=bounds python tools/bounds_sweep.py): any index a kernel computes outside its array traps the launch
and this script dies with a CUDA error.  (compute-sanitizer is not available on the GPU pool.)"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "point-cloud-interpolation-_b200"))
import numpy as np
import torch
from b200pc import _lib, ops, pointnet2_utils as P, pytorch3d_shim as S3, synth
ops.TUNING_AUTORELOAD = True

dev = torch.device("cuda:0")
print("library:", os.path.basename(_lib.LIB_PATH), flush=True)
ENV = ("B200PC_GRID", "B200PC_SEED", "B200PC_INTERLEAVE", "B200PC_SMALL_PATH", "B200PC_FORCE_SPLIT", "B200PC_BULK", "B200PC_FPS_FLAT", "B200PC_FPS_CLUSTER",
       "B200PC_FORCE_WARPS", "B200PC_FORCE_Q", "B200PC_FILTER", "B200PC_NATURAL_ORDER")


def env(**kw):
    for k in ENV:
        os.environ.pop(k, None)
    for k, v in kw.items():
        os.environ["B200PC_" + k] = str(v)


def t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


rng = np.random.default_rng(3)
# ---- searches: every path (small / streaming / split), every grid variant, ragged sizes, ties, non-finite points
for B, N, S, k in ((2, 3000, 700, 16), (1, 513, 31, 3), (3, 1000, 777, 1), (1, 5, 9, 5), (1, 6000, 4100, 64), (2, 16384, 1024, 8), (1, 20000, 5000, 16)):
    a, b = synth.batch_pairs(11, B, max(N, S))
    ref, qry = t(a[:, :N]), t(b[:, :S])
    for kw in (dict(), dict(GRID=0, SMALL_PATH=0), dict(GRID=2, SMALL_PATH=0), dict(GRID=3, SMALL_PATH=0), dict(GRID=3, SMALL_PATH=0, INTERLEAVE=1, SEED=5),
               dict(GRID=3, SMALL_PATH=0, SEED=2, FORCE_SPLIT=3), dict(SMALL_PATH=1)):
        env(**kw)
        for form in (0, 1, 2):
            ops.knn_search(ref, qry, k, form, want_dist=True)
        ops.knn_search_i32(ref, qry, k, 0)
        P.query_ball_point(0.7, min(32, N), ref, qry)
    env()
bad_r, bad_q = a[:, :N].copy(), b[:, :S].copy()
bad_r[0, 7] = np.nan; bad_r[0, 99, 2] = np.inf; bad_q[0, 3] = np.nan
for kw in (dict(), dict(GRID=3, SMALL_PATH=0), dict(GRID=2, SMALL_PATH=0)):
    env(**kw); ops.knn_search(t(bad_r), t(bad_q), 16, 0, want_dist=True); P.query_ball_point(1.0, 16, t(bad_r), t(bad_q))
# k above the finite count on the small path (rows end in -1), and a split range (tile 1 of the strided order, 2 tiles)
# holding only non-finite refs; (+inf, 0, 0) is the query whose filter value is -inf for refs with x > 0
few = bad_r[:1, :900].copy(); few[0, 8:] = np.nan
half = bad_r[:1, :1000].copy(); half[0, 1::2] = np.inf
bq = bad_q[:1, :64].copy(); bq[0, 5] = [np.inf, 0.0, 0.0]
for kw, cloud in ((dict(SMALL_PATH=1), few), (dict(SMALL_PATH=0, GRID=0, FORCE_SPLIT=2), half), (dict(SMALL_PATH=0, GRID=3), half)):
    env(**kw)
    for form in (0, 1, 2):
        ops.knn_search(t(cloud), t(bq), 16, form, want_dist=True); ops.knn_search_i32(t(cloud), t(bq), 16, form)
    ops.chamfer(t(cloud), t(bq)); ops.fusion_group(t(bq), t(cloud), 16, t(cloud))
env()
same = np.repeat(np.array([[[1.5, -2.0, 0.25]]], np.float32), 900, axis=1)
env(GRID=3, SMALL_PATH=0); ops.knn_search(t(same), t(b[:1, :100]), 7, 0); env()
# forced plans (tests/test_gpu_plans.py): every split a range count can come from, short and ragged ranges, k above the refs
# of a range, warps per CTA with empty trailing warps, two queries per thread, the broadcast filter and the natural order
for (B, N, S, k), splits in (((1, 513, 77, 300), (2,)), ((2, 2048, 333, 600), (3, 4)), ((1, 5000, 700, 16), (3, 4, 5, 7, 8)),
                             ((1, 20000, 300, 64), (32, 40))):
    a, b = synth.batch_pairs(12, B, max(N, S))
    ref, qry = t(a[:, :N]), t(b[:, :S])
    for split in splits:
        for grid in (0, 2, 3):
            env(SMALL_PATH=0, GRID=grid, FORCE_SPLIT=split)
            for form in (0, 1, 2):
                ops.knn_search(ref, qry, k, form, want_dist=True)
            ops.knn_search_i32(ref, qry, k, 2)
        env(FORCE_SPLIT=split)
        P.query_ball_point(0.7, min(128, N), ref, qry); P.query_ball_point(100.0, 32, ref, qry)
a, b = synth.batch_pairs(13, 1, 4100)
for S in (33, 777, 4100):
    ref, qry = t(a[:, :3000]), t(b[:, :S])
    for q in (1, 2):
        for w in (1, 2, 5, 14):
            for kw in (dict(), dict(GRID=3, INTERLEAVE=1)):
                env(SMALL_PATH=0, FORCE_Q=q, FORCE_WARPS=w, **kw)
                ops.knn_search(ref, qry, 16, 0, want_dist=True); ops.knn_search_i32(ref, qry, 16, 2)
            env(FORCE_Q=q, FORCE_WARPS=w); P.query_ball_point(1.0, 32, ref, qry)
for kw in (dict(FILTER=0), dict(FILTER=0, FORCE_SPLIT=4), dict(NATURAL_ORDER=1), dict(NATURAL_ORDER=0, FORCE_SPLIT=4), dict(FORCE_Q=2, FORCE_SPLIT=4)):
    env(SMALL_PATH=0, GRID=0, **kw)
    for form in (0, 1, 2):
        ops.knn_search(ref, qry, 16, form, want_dist=True)
env()
torch.cuda.synchronize(); print("searches ok", flush=True)

# ---- FPS (single CTA, clusters, flat exchange), gather, group, interpolate, fusion, chamfer, polyfit, rebuild
a, b = synth.batch_pairs(2, 2, 16384)
big = t(a)
for kw in (dict(), dict(FPS_FLAT=1), dict(FPS_FLAT=0), dict(FPS_CLUSTER=2), dict(FPS_CLUSTER=16), dict(FPS_CLUSTER=16, FPS_FLAT=1),
           dict(FPS_CLUSTER=1, FPS_FLAT=1), dict(FPS_CLUSTER=8, FPS_FLAT=0)):
    env(**kw)
    for n, m in ((16384, 300), (12000, 64), (3000, 128), (40, 7)):
        ops.fps(big[:, :n].contiguous(), m, torch.tensor([1, n - 1], device=dev))
env()
ref = big[:, :3000].contiguous(); qry = t(b[:, :700])
fi = ops.fps(ref, 64, torch.tensor([1, 2], device=dev))
for C in (3, 32, 36, 128, 257):
    feats = torch.randn(2, 3000, C, device=dev, requires_grad=True)
    P.index_points(feats, fi).sum().backward()
    gi = P.knn_point(9, ref, qry)
    P.index_points(feats, gi)
    known = P.index_points(ref, fi); d, i3, w = P.three_nn_weights(ref, known)
    sf = torch.randn(2, 64, C, device=dev, requires_grad=True)
    P.three_interpolate(sf, i3, w.clone().requires_grad_(True)).sum().backward()
    P.feature_propagation(ref, known, sf.detach(), variant=C % 2)
for D in (0, 16, 20, 64, 128, 200):
    new_xyz = P.index_points(ref, fi)
    gi = P.knn_point(11, ref, new_xyz)
    fe = torch.randn(2, 3000, D, device=dev, requires_grad=True) if D else None
    for bulk in (0, 1):
        env(BULK=bulk)
        for xf in (True, False):
            out = P.group_points(ref, new_xyz, fe, gi, xyz_first=xf)
            if D: out.sum().backward()
    env()
gi = P.knn_point(16, big[:1], big[:1, :4096].contiguous())
env(BULK=1); P.group_points(big[:1], big[:1, :4096].contiguous(), torch.randn(1, 16384, 64, device=dev), gi, xyz_first=True); env()
# asynchronous grouping with K cut into parts of several slots that do not divide K (default plan, then forced), with
# sentinel and negative indices; feature gradients with D > 256 (the backward kernel loops over channel blocks)
for B, S, K, D, bulk in ((16, 4096, 10, 16, None), (16, 4096, 12, 32, None), (16, 4096, 20, 64, None), (8, 4096, 20, 16, None),
                         (8, 4096, 24, 32, None), (1, 16384, 48, 16, None), (1, 865, 256, 384, 1), (1, 4000, 256, 16, 1),
                         (2, 777, 12, 392, 1), (2, 777, 12, 132, 1)):
    env(**({} if bulk is None else dict(BULK=bulk)))
    gi = torch.randint(-2048, 2049, (B, S, K), device=dev)                  # 2048 = the empty-ball sentinel
    fe = torch.randn(B, 2048, D, device=dev)
    for xf in (True, False):
        P.group_points(big[:1, :2048].expand(B, -1, -1).contiguous(), big[:1, :S].expand(B, -1, -1).contiguous(), fe, gi, xyz_first=xf)
env()
for D in (257, 300, 520):
    gi = torch.randint(-1000, 1001, (2, 777, 16), device=dev)
    fe = torch.randn(2, 1000, D, device=dev, requires_grad=True)
    for xf in (True, False):
        P.group_points(ref[:, :1000].contiguous(), ref[:, :777].contiguous(), fe, gi, xyz_first=xf).sum().backward()
# interpolation gradients with negative and dropped neighbours
sf = torch.randn(2, 64, 12, device=dev, requires_grad=True)
i3 = torch.randint(-70, 70, (2, 5000, 3), device=dev)
P.three_interpolate(sf, i3, torch.rand(2, 5000, 3, device=dev, requires_grad=True)).sum().backward()
P.square_distance(ref[:, :100], qry[:, :33])
x = ref[:, :500].clone().requires_grad_(True); S3.chamfer_distance(x, qry)[0].backward()
ff = torch.randn(2, 3000, 13, device=dev)
P.fusion_group(qry, ref, 9, ff); P.fusion_group(qry, ref, 4, None)
ops.channel_max(torch.randn(5000, 128, device=dev)); ops.channel_max(torch.randn(77, 36, device=dev))
ops.unpack_rebuild(ops.rebuild_pack(ref, qry))
from b200pc import polypci
frames = [torch.randn(2, 3, 2000, device=dev) for _ in range(5)]
polypci.fit_and_predict(frames, [[0.0, 1.0, -1.0, 2.0, -2.0]] * 2, [0.5, -0.25], 3)
torch.cuda.synchronize(); print("row movers ok", flush=True)

# ---- the C entries at the smallest offsets the contract allows (tests/test_gpu_buffer_hygiene.py): fp32 / int32 buffers 4 bytes
# and int64 buffers 8 bytes past a 256-byte boundary, the search workspace and the 16-byte records 16 bytes past one, and the
# kernels that accumulate into a non-zero base
import ctypes as C
lib = _lib.load()


def off(a, align):
    """a device copy of `a` whose data starts `align` bytes past a 256-byte boundary"""
    a = torch.as_tensor(np.ascontiguousarray(a)) if isinstance(a, np.ndarray) else a
    n = a.numel() * a.element_size()
    raw = torch.empty(n + 512, dtype=torch.uint8, device=dev)
    s = (align - raw.data_ptr()) % 256
    v = raw[s:s + n].view(a.dtype).view(a.shape)
    v.copy_(a)
    return v


def f32(*shape):
    return off(torch.randn(*shape), 4)


def i64(a):
    return off(torch.as_tensor(np.asarray(a, np.int64)), 8)


def ok(rc):
    assert rc == 0, lib.b200pc_last_error()


def p(x):
    return x.data_ptr() if x is not None else None


st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
for (B, N, S, k), kw in (((2, 513, 77, 300), dict(SMALL_PATH=0, GRID=0, FORCE_SPLIT=2)), ((2, 5000, 700, 16), dict(SMALL_PATH=0, GRID=3, FORCE_SPLIT=3)),
                         ((2, 700, 333, 16), dict(SMALL_PATH=1)), ((2, 3000, 333, 16), dict(SMALL_PATH=0, FORCE_Q=2, GRID=0))):
    env(**kw); ops.reload_tuning()
    a, b = synth.batch_pairs(14, B, max(N, S))
    a[B - 1, 2:] = np.nan
    ref, qry = off(a[:, :N].copy(), 4), off(b[:, :S].copy(), 4)
    nws = lib.b200pc_search_workspace_bytes(B, N, S, k)
    ws = off(torch.empty(nws, dtype=torch.uint8), 16)
    ok(lib.b200pc_knn(p(ref), p(qry), B, N, S, k, 0, p(i64(np.zeros((B, S, k)))), p(f32(B, S, k)), p(ws), nws, st))
    ok(lib.b200pc_knn_i32(p(ref), p(qry), B, N, S, k, 2, p(off(torch.zeros(B, S, k, dtype=torch.int32), 4)), p(f32(B, S, k)), p(ws), nws, st))
    ok(lib.b200pc_ball_query(p(ref), p(qry), B, N, S, C.c_float(1.0), min(k, 64), p(i64(np.zeros((B, S, min(k, 64))))), p(ws), nws, st))
    nws3 = lib.b200pc_search_workspace_bytes(B, N, S, 3)
    ws3 = off(torch.empty(nws3, dtype=torch.uint8), 16)
    ok(lib.b200pc_three_nn(p(qry), p(ref), B, S, N, 0, p(f32(B, S, 3)), p(i64(np.zeros((B, S, 3)))), p(f32(B, S, 3)), p(ws3), nws3, st))
env(); ops.reload_tuning()
B, N, S, R = 2, 900, 123, 777
pts, new = f32(B, N, 64), f32(B, S, 3)
gidx = np.random.default_rng(5).integers(-N, N, size=(B, R)); gidx[:, ::37] = N
ok(lib.b200pc_gather(p(pts), p(i64(gidx)), B, N, 64, R, p(f32(B, R, 64)), p(off(torch.zeros(1, dtype=torch.int32), 4)), st))
ok(lib.b200pc_gather_bwd(p(f32(B, R, 64)), p(i64(gidx)), B, N, 64, R, p(f32(B, N, 64)), st))
i3 = np.random.default_rng(6).integers(-1, S, size=(B, N, 3))
ok(lib.b200pc_three_interpolate(p(f32(B, S, 12)), p(i64(i3)), p(f32(B, N, 3)), B, S, N, 12, p(f32(B, N, 12)), st))
ok(lib.b200pc_three_interpolate_bwd(p(f32(B, N, 12)), p(f32(B, S, 12)), p(i64(i3)), p(f32(B, N, 3)), B, S, N, 12, p(f32(B, S, 12)), p(f32(B, N, 3)), st))
gk = np.random.default_rng(7).integers(-N, N + 1, size=(B, S, 16))
for bulk in (0, 1):
    env(BULK=bulk); ops.reload_tuning()
    for xf in (0, 1):
        ok(lib.b200pc_group_points(p(pts[..., :3].contiguous()), p(new), p(pts), p(i64(gk)), B, N, S, 16, 64, xf, p(f32(B, 67, 16, S)), st))
        ok(lib.b200pc_group_points_bwd(p(f32(B, 67, 16, S)), p(i64(gk)), B, N, S, 16, 64, xf, p(f32(B, N, 64)), st))
env(); ops.reload_tuning()
ok(lib.b200pc_square_distance(p(f32(B, 77, 3)), p(f32(B, 1004, 3)), B, 77, 1004, p(f32(B, 77, 1004)), st))
ok(lib.b200pc_channel_max(p(off(torch.randn(1001, 4), 16)), 1001, 4, p(f32(1001)), st))
fr = [f32(3, 999) for _ in range(16)]
ok(lib.b200pc_poly_predict((C.c_void_p * 16)(*[p(f) for f in fr]), p(off(torch.randn(3, 16, dtype=torch.float64), 8)), 3, 16, 999, p(f32(3, 999)), st))
a, b = synth.batch_pairs(15, 2, 1200)
ref, qry = off(a, 4), off(b[:, :333].copy(), 4)
nws = lib.b200pc_search_workspace_bytes(2, 1200, 333, 16)
ws = off(torch.empty(nws, dtype=torch.uint8), 16)
ok(lib.b200pc_fusion_group(p(qry), p(ref), p(f32(2, 1200, 13)), 2, 1200, 333, 16, 13, p(f32(2, 4, 333, 16)), p(f32(2, 3, 333, 16)),
                           p(f32(2, 13, 333, 16)), p(i64(np.zeros((2, 333, 16)))), p(ws), nws, st))
ix, iy = i64(np.zeros((2, 333))), i64(np.zeros((2, 1200)))
nws = max(lib.b200pc_search_workspace_bytes(2, 1200, 333, 1), lib.b200pc_search_workspace_bytes(2, 333, 1200, 1))
ws = off(torch.empty(nws, dtype=torch.uint8), 16)
ok(lib.b200pc_chamfer_fwd(p(qry), p(ref), 2, 333, 1200, p(f32(2, 333)), p(ix), p(f32(2, 1200)), p(iy), p(f32(1)), p(ws), nws, st))
ok(lib.b200pc_chamfer_bwd(p(qry), p(ref), p(ix), p(iy), p(f32(1)), 2, 333, 1200, p(f32(2, 333, 3)), p(f32(2, 1200, 3)), st))
nws = lib.b200pc_rebuild_pack_workspace_bytes(2, 1200, 333)
ws = off(torch.empty(nws, dtype=torch.uint8), 16)
peers = [off(torch.randn(1500, 2, 4), 16) for _ in range(8)]
ok(lib.b200pc_rebuild_pack(p(ref), p(qry), 2, 1200, 333, 700, p(off(torch.zeros(333, 2, 4), 16)), (C.c_void_p * 8)(*[p(q) for q in peers]), 8,
                           p(ws), nws, st))
torch.cuda.synchronize(); print("bounds sweep ok", flush=True)
