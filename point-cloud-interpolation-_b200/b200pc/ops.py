"""Tensor-level entry points: torch CUDA tensors in, torch CUDA tensors out, via the C ABI.

Every compute entry of include/b200pc.h is registered as a PyTorch custom op `torch.ops.b200pc.<name>`
(`torch.library`): CUDA dispatch key ONLY -- a CPU tensor reaching the dispatcher has no kernel to run, there is
no fallback -- with fake (meta) kernels for shape inference and `register_autograd` formulas for gather,
group_points, three_interpolate and chamfer.  The op implementations do nothing but allocate outputs and call
libb200pc.so on the tensor's device and torch's current stream; torch is used for device memory, streams and autograd
bookkeeping only.  The public functions of this module validate / normalise their arguments the way the reference's
functions accept them (fp32 point-major [B,N,3] / [B,N,C], any integer index dtype, fresh contiguous outputs) and
then go through the dispatcher, so `b200pc.pointnet2_utils`, the pytorch3d shim and the drop-in all run the ops.
"""
import ctypes as C
import os

import torch

from . import _lib

FORM_REF_NORM_FIRST = 0
FORM_QRY_NORM_FIRST = 1
FORM_DIRECT = 2

# index_points bounds checking costs a device->host sync per call; the reference raises
# IndexError on out-of-range indices, so tests switch this on.  Off: bad rows come back as zeros.
CHECK_BOUNDS = os.environ.get("B200PC_CHECK_BOUNDS", "0") == "1"

launch_count = 0     # C-ABI compute calls issued (bench.py reports kernels from the plan below)

# The library reads its B200PC_* tuning variables once and caches them.  Probes that flip a knob between calls set this
# to True (or call reload_tuning() themselves): the cache is then refreshed before every C call.
TUNING_AUTORELOAD = False


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream(dev):
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _prep(t, name):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if not t.is_cuda:
        raise RuntimeError("b200pc: %s is on %s; this library has no CPU path (CUDA tensors only)" % (name, t.device))
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _idx64(idx, dev):
    if idx.device != dev:
        idx = idx.to(dev)
    if idx.dtype != torch.int64:
        idx = idx.long()
    return idx.contiguous()


def _workspace(nbytes, dev):
    return torch.empty(int(nbytes), dtype=torch.uint8, device=dev)


def _search_ws(lib, B, N, S, k):
    """workspace of a search call; sized under the SAME tuning state the call itself will see"""
    if TUNING_AUTORELOAD:
        lib.b200pc_tuning_reload()
    return lib.b200pc_search_workspace_bytes(B, N, S, k)


def _call(dev, fn, *args):
    """one C-ABI compute call on `dev` (current stream), error code -> exception"""
    global launch_count
    if TUNING_AUTORELOAD:
        _lib.load().b200pc_tuning_reload()
    if dev.index == torch.cuda.current_device():        # the common case: no device switch around the call
        _lib.check(fn(*args))
    else:
        with torch.cuda.device(dev):
            _lib.check(fn(*args))
    launch_count += 1


# ==========================================================================================
# torch.ops.b200pc.*: schemas, CUDA implementations (calls into libb200pc.so), fake kernels
# ==========================================================================================
try:
    _L = torch.library.Library("b200pc", "DEF")
except RuntimeError:                                    # the namespace already exists in this process (module re-import)
    _L = torch.library.Library("b200pc", "FRAGMENT")

OP_SCHEMAS = {
    # op name == C entry point without the b200pc_ prefix (tests/test_abi.py keeps the two lists in step)
    "square_distance": "(Tensor src, Tensor dst) -> Tensor",
    "knn": "(Tensor ref, Tensor qry, int k, int form, bool want_dist) -> (Tensor, Tensor)",
    "knn_ragged": "(Tensor ref, Tensor qry, Tensor? ref_len, Tensor? qry_len, int k, int form, bool want_dist) -> (Tensor, Tensor)",
    "knn_i32": "(Tensor ref, Tensor qry, int k, int form) -> Tensor",
    "ball_query": "(Tensor xyz, Tensor new_xyz, float r2, int nsample) -> Tensor",
    "fps": "(Tensor xyz, int npoint, Tensor start) -> Tensor",
    "fps_sample": "(Tensor xyz, int npoint, Tensor start) -> (Tensor, Tensor)",
    "gather": "(Tensor points, Tensor idx, bool check_bounds) -> Tensor",
    "gather_bwd": "(Tensor gout, Tensor idx, int N) -> Tensor",
    "group_points": "(Tensor xyz, Tensor new_xyz, Tensor? feat, Tensor idx, bool xyz_first) -> Tensor",
    "group_points_bwd": "(Tensor gout, Tensor idx, int N, int D, bool xyz_first) -> Tensor",
    "three_nn": "(Tensor unknown, Tensor known, int variant, bool want_weight) -> (Tensor, Tensor, Tensor)",
    "three_interpolate": "(Tensor feat, Tensor idx, Tensor weight) -> Tensor",
    "three_interpolate_bwd": "(Tensor gout, Tensor feat, Tensor idx, Tensor weight, bool want_gweight) -> (Tensor, Tensor)",
    "feature_propagation": "(Tensor unknown, Tensor known, Tensor feat, int variant) -> (Tensor, Tensor, Tensor)",
    "fusion_group": "(Tensor qry, Tensor ref, Tensor? feat, int k) -> (Tensor, Tensor, Tensor, Tensor)",
    "channel_max": "(Tensor x) -> Tensor",
    "rebuild_pack": "(Tensor ref, Tensor qry, int s_offset, int[] peer_ptrs) -> Tensor",
    "chamfer_fwd": "(Tensor x, Tensor y) -> (Tensor, Tensor, Tensor, Tensor, Tensor)",
    "chamfer_bwd": "(Tensor x, Tensor y, Tensor ix, Tensor iy, Tensor gloss) -> (Tensor, Tensor)",
    "chamfer_ragged_fwd": "(Tensor x, Tensor y, Tensor? x_len, Tensor? y_len) -> (Tensor, Tensor, Tensor, Tensor, Tensor)",
    "chamfer_ragged_bwd": "(Tensor x, Tensor y, Tensor ix, Tensor iy, Tensor? x_len, Tensor? y_len, Tensor gsums) -> (Tensor, Tensor)",
    "poly_predict": "(Tensor[] frames, Tensor weights) -> Tensor",
}
for _name, _schema in OP_SCHEMAS.items():
    _L.define(_name + _schema)


def _register(name, fake):
    def deco(fn):
        _L.impl(name, fn, "CUDA")
        torch.library.register_fake("b200pc::" + name, fake, lib=_L)
        return fn
    return deco


def _f32(*shape, like):
    return torch.empty(*shape, dtype=torch.float32, device=like.device)


def _i64(*shape, like):
    return torch.empty(*shape, dtype=torch.int64, device=like.device)


# ---- a1 ----------------------------------------------------------------------------------
@_register("square_distance", lambda src, dst: _f32(src.shape[0], src.shape[1], dst.shape[1], like=src))
def _square_distance(src, dst):
    B, N, _ = src.shape; M = dst.shape[1]
    out = _f32(B, N, M, like=src)
    _call(src.device, _lib.load().b200pc_square_distance, _ptr(src), _ptr(dst), B, N, M, _ptr(out), _stream(src.device))
    return out


# ---- a4 / a8 -----------------------------------------------------------------------------
def _knn_fake(ref, qry, k, form, want_dist):
    B, S = qry.shape[0], qry.shape[1]
    return _i64(B, S, k, like=ref), _f32(B, S, k if want_dist else 0, like=ref)


@_register("knn", _knn_fake)
def _knn(ref, qry, k, form, want_dist):
    B, N, _ = ref.shape; S = qry.shape[1]
    dev = ref.device
    idx = _i64(B, S, k, like=ref)
    dist = _f32(B, S, k, like=ref) if want_dist else None
    lib = _lib.load()
    nws = _search_ws(lib, B, N, S, k)
    ws = _workspace(nws, dev)
    _call(dev, lib.b200pc_knn, _ptr(ref), _ptr(qry), B, N, S, k, int(form), _ptr(idx), _ptr(dist), _ptr(ws), nws, _stream(dev))
    return idx, (dist if want_dist else _f32(B, S, 0, like=ref))


@_register("knn_ragged", lambda ref, qry, ref_len, qry_len, k, form, want_dist: _knn_fake(ref, qry, k, form, want_dist))
def _knn_ragged(ref, qry, ref_len, qry_len, k, form, want_dist):
    B, N, _ = ref.shape; S = qry.shape[1]
    dev = ref.device
    idx = _i64(B, S, k, like=ref)
    dist = _f32(B, S, k, like=ref) if want_dist else None
    lib = _lib.load()
    nws = _search_ws(lib, B, N, S, k)
    ws = _workspace(nws, dev)
    _call(dev, lib.b200pc_knn_ragged, _ptr(ref), _ptr(qry), _ptr(ref_len), _ptr(qry_len), B, N, S, k, int(form), _ptr(idx), _ptr(dist),
          _ptr(ws), nws, _stream(dev))
    return idx, (dist if want_dist else _f32(B, S, 0, like=ref))


@_register("knn_i32", lambda ref, qry, k, form: torch.empty(qry.shape[0], qry.shape[1], k, dtype=torch.int32, device=ref.device))
def _knn_i32(ref, qry, k, form):
    B, N, _ = ref.shape; S = qry.shape[1]
    dev = ref.device
    idx = torch.empty(B, S, k, dtype=torch.int32, device=dev)
    lib = _lib.load()
    nws = _search_ws(lib, B, N, S, k)
    ws = _workspace(nws, dev)
    _call(dev, lib.b200pc_knn_i32, _ptr(ref), _ptr(qry), B, N, S, k, int(form), _ptr(idx), C.c_void_p(0), _ptr(ws), nws, _stream(dev))
    return idx


# ---- a2 ----------------------------------------------------------------------------------
@_register("ball_query", lambda xyz, new_xyz, r2, nsample: _i64(new_xyz.shape[0], new_xyz.shape[1], nsample, like=xyz))
def _ball_query(xyz, new_xyz, r2, nsample):
    B, N, _ = xyz.shape; S = new_xyz.shape[1]
    dev = xyz.device
    idx = _i64(B, S, nsample, like=xyz)
    lib = _lib.load()
    nws = _search_ws(lib, B, N, S, nsample)
    ws = _workspace(nws, dev)
    _call(dev, lib.b200pc_ball_query, _ptr(xyz), _ptr(new_xyz), B, N, S, C.c_float(r2), nsample, _ptr(idx), _ptr(ws), nws, _stream(dev))
    return idx


# ---- a3 / a7 -----------------------------------------------------------------------------
@_register("fps", lambda xyz, npoint, start: _i64(xyz.shape[0], npoint, like=xyz))
def _fps(xyz, npoint, start):
    B, N, _ = xyz.shape
    idx = _i64(B, npoint, like=xyz)
    _call(xyz.device, _lib.load().b200pc_fps, _ptr(xyz), B, N, npoint, _ptr(start), _ptr(idx), C.c_void_p(0), 0, _stream(xyz.device))
    return idx


@_register("fps_sample", lambda xyz, npoint, start: (_i64(xyz.shape[0], npoint, like=xyz), _f32(xyz.shape[0], npoint, 3, like=xyz)))
def _fps_sample(xyz, npoint, start):
    B, N, _ = xyz.shape
    idx = _i64(B, npoint, like=xyz)
    new_xyz = _f32(B, npoint, 3, like=xyz)
    _call(xyz.device, _lib.load().b200pc_fps_sample, _ptr(xyz), B, N, npoint, _ptr(start), _ptr(idx), _ptr(new_xyz), _stream(xyz.device))
    return idx, new_xyz


# ---- a6 ----------------------------------------------------------------------------------
@_register("gather", lambda points, idx, check_bounds: _f32(points.shape[0], idx.shape[1], points.shape[2], like=points))
def _gather(points, idx, check_bounds):
    B, N, Cc = points.shape
    R = idx.shape[1]
    dev = points.device
    out = _f32(B, R, Cc, like=points)
    flag = torch.zeros(1, dtype=torch.int32, device=dev) if check_bounds else None
    _call(dev, _lib.load().b200pc_gather, _ptr(points), _ptr(idx), B, N, Cc, R, _ptr(out), _ptr(flag), _stream(dev))
    if flag is not None and int(flag.item()) != 0:
        raise IndexError("index out of range in index_points (valid range is [-%d, %d))" % (N, N))
    return out


@_register("gather_bwd", lambda gout, idx, N: _f32(gout.shape[0], N, gout.shape[2], like=gout))
def _gather_bwd(gout, idx, N):
    B, R, Cc = gout.shape
    gpts = torch.zeros(B, N, Cc, dtype=torch.float32, device=gout.device)
    _call(gout.device, _lib.load().b200pc_gather_bwd, _ptr(gout), _ptr(idx), B, N, Cc, R, _ptr(gpts), _stream(gout.device))
    return gpts


def _gather_setup(ctx, inputs, output):
    points, idx, _ = inputs
    ctx.save_for_backward(idx)
    ctx.N = points.shape[1]


def _gather_backward(ctx, gout):
    (idx,) = ctx.saved_tensors
    return torch.ops.b200pc.gather_bwd(gout.contiguous(), idx, ctx.N), None, None


torch.library.register_autograd("b200pc::gather", _gather_backward, setup_context=_gather_setup, lib=_L)


# ---- a7 / f1 -----------------------------------------------------------------------------
def _group_fake(xyz, new_xyz, feat, idx, xyz_first):
    D = 0 if feat is None else feat.shape[2]
    return _f32(xyz.shape[0], 3 + D, idx.shape[2], idx.shape[1], like=xyz)


@_register("group_points", _group_fake)
def _group_points(xyz, new_xyz, feat, idx, xyz_first):
    B, N, _ = xyz.shape
    S, K = idx.shape[1], idx.shape[2]
    D = 0 if feat is None else feat.shape[2]
    out = _f32(B, 3 + D, K, S, like=xyz)
    _call(xyz.device, _lib.load().b200pc_group_points, _ptr(xyz), _ptr(new_xyz), _ptr(feat if D else None), _ptr(idx), B, N, S, K,
          D, int(bool(xyz_first)), _ptr(out), _stream(xyz.device))
    return out


@_register("group_points_bwd", lambda gout, idx, N, D, xyz_first: _f32(gout.shape[0], N, D, like=gout))
def _group_points_bwd(gout, idx, N, D, xyz_first):
    B = gout.shape[0]
    S, K = idx.shape[1], idx.shape[2]
    gfeat = torch.zeros(B, N, D, dtype=torch.float32, device=gout.device)
    _call(gout.device, _lib.load().b200pc_group_points_bwd, _ptr(gout), _ptr(idx), B, N, S, K, D, int(bool(xyz_first)), _ptr(gfeat),
          _stream(gout.device))
    return gfeat


def _group_setup(ctx, inputs, output):
    xyz, new_xyz, feat, idx, xyz_first = inputs
    ctx.save_for_backward(idx)
    ctx.N = xyz.shape[1]
    ctx.D = 0 if feat is None else feat.shape[2]
    ctx.xyz_first = bool(xyz_first)


def _group_backward(ctx, gout):
    """differentiable in the features through the scatter kernel (what the reference's models train through); the
    coordinates get their gradient from the same three terms the unfused graph would produce, built with torch ops
    on the three xyz channels.  A slot whose index is still out of range after one wrap (the ball query's empty-ball
    sentinel N, for one) was filled with zeros by the forward pass: it gives xyz no gradient, while new_xyz still gets
    -gout there, because that output is 0 - centre."""
    (idx,) = ctx.saved_tensors
    N, D, xyz_first = ctx.N, ctx.D, ctx.xyz_first
    B, _, K, S = gout.shape
    gout = gout.contiguous()
    gxyz = gnew = gfeat = None
    if D and ctx.needs_input_grad[2]:
        gfeat = torch.ops.b200pc.group_points_bwd(gout, idx, N, D, xyz_first)
    if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
        gx = gout[:, 0:3] if xyz_first else gout[:, D:D + 3]              # [B,3,K,S]
        if ctx.needs_input_grad[1]:
            gnew = -gx.sum(dim=2).transpose(1, 2).contiguous()            # [B,S,3]
        if ctx.needs_input_grad[0]:
            rows = gx.permute(0, 3, 2, 1).reshape(B, S * K, 3)
            flat = torch.where(idx < 0, idx + N, idx).reshape(B, S * K, 1)
            flat = torch.where((flat >= 0) & (flat < N), flat, N).expand(-1, -1, 3)      # dropped slots land in spare row N
            gxyz = torch.zeros(B, N + 1, 3, dtype=torch.float32, device=gout.device).scatter_add_(1, flat, rows)[:, :N]
    return gxyz, gnew, gfeat, None, None


torch.library.register_autograd("b200pc::group_points", _group_backward, setup_context=_group_setup, lib=_L)


# ---- a5 ----------------------------------------------------------------------------------
def _three_nn_fake(unknown, known, variant, want_weight):
    B, N = unknown.shape[0], unknown.shape[1]
    return _f32(B, N, 3, like=unknown), _i64(B, N, 3, like=unknown), _f32(B, N, 3 if want_weight else 0, like=unknown)


@_register("three_nn", _three_nn_fake)
def _three_nn(unknown, known, variant, want_weight):
    B, N, _ = unknown.shape; S = known.shape[1]
    dev = unknown.device
    dist = _f32(B, N, 3, like=unknown)
    idx = _i64(B, N, 3, like=unknown)
    weight = _f32(B, N, 3, like=unknown) if want_weight else None
    lib = _lib.load()
    nws = _search_ws(lib, B, S, N, 3)
    ws = _workspace(nws, dev)
    _call(dev, lib.b200pc_three_nn, _ptr(unknown), _ptr(known), B, N, S, int(variant), _ptr(dist), _ptr(idx), _ptr(weight), _ptr(ws),
          nws, _stream(dev))
    return dist, idx, (weight if want_weight else _f32(B, N, 0, like=unknown))


@_register("three_interpolate", lambda feat, idx, weight: _f32(feat.shape[0], idx.shape[1], feat.shape[2], like=feat))
def _three_interpolate(feat, idx, weight):
    B, S, Cc = feat.shape; N = idx.shape[1]
    out = _f32(B, N, Cc, like=feat)
    _call(feat.device, _lib.load().b200pc_three_interpolate, _ptr(feat), _ptr(idx), _ptr(weight), B, S, N, Cc, _ptr(out),
          _stream(feat.device))
    return out


def _interp_bwd_fake(gout, feat, idx, weight, want_gweight):
    return torch.empty_like(feat), _f32(*(weight.shape if want_gweight else (0,)), like=feat)


@_register("three_interpolate_bwd", _interp_bwd_fake)
def _three_interpolate_bwd(gout, feat, idx, weight, want_gweight):
    B, S, Cc = feat.shape; N = idx.shape[1]
    gfeat = torch.zeros_like(feat)
    gw = torch.empty_like(weight) if want_gweight else None
    _call(gout.device, _lib.load().b200pc_three_interpolate_bwd, _ptr(gout), _ptr(feat), _ptr(idx), _ptr(weight), B, S, N, Cc,
          _ptr(gfeat), _ptr(gw), _stream(gout.device))
    return gfeat, (gw if want_gweight else _f32(0, like=feat))


def _interp_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _interp_backward(ctx, gout):
    feat, idx, weight = ctx.saved_tensors
    want = bool(ctx.needs_input_grad[2])
    gfeat, gw = torch.ops.b200pc.three_interpolate_bwd(gout.contiguous(), feat, idx, weight, want)
    return gfeat, None, (gw if want else None)


torch.library.register_autograd("b200pc::three_interpolate", _interp_backward, setup_context=_interp_setup, lib=_L)


def _fp_fake(unknown, known, feat, variant):
    B, N = unknown.shape[0], unknown.shape[1]
    return _f32(B, N, feat.shape[2], like=feat), _i64(B, N, 3, like=feat), _f32(B, N, 3, like=feat)


@_register("feature_propagation", _fp_fake)
def _feature_propagation(unknown, known, feat, variant):
    """three_nn -> weights -> three_interpolate behind ONE C call (the weights are also returned: the backward
    pass and the differentiable-coordinates path need them)"""
    B, N, _ = unknown.shape; S = known.shape[1]; Cc = feat.shape[2]
    dev = unknown.device
    out = _f32(B, N, Cc, like=feat)
    idx = _i64(B, N, 3, like=feat)
    weight = _f32(B, N, 3, like=feat)
    lib = _lib.load()
    nws = lib.b200pc_feature_propagation_workspace_bytes(B, N, S)
    ws = _workspace(nws, dev)
    _call(dev, lib.b200pc_feature_propagation, _ptr(unknown), _ptr(known), _ptr(feat), B, N, S, Cc, int(variant), _ptr(out),
          _ptr(idx), _ptr(weight), _ptr(ws), nws, _stream(dev))
    return out, idx, weight


def _fp_setup(ctx, inputs, output):
    _, _, feat, _ = inputs
    _, idx, weight = output
    ctx.save_for_backward(feat, idx, weight)


def _fp_backward(ctx, gout, _gidx, _gw):
    feat, idx, weight = ctx.saved_tensors
    gfeat, _ = torch.ops.b200pc.three_interpolate_bwd(gout.contiguous(), feat, idx, weight, False)
    return None, None, gfeat, None


torch.library.register_autograd("b200pc::feature_propagation", _fp_backward, setup_context=_fp_setup, lib=_L)


# ---- a8 / f2 -----------------------------------------------------------------------------
def _fusion_fake(qry, ref, feat, k):
    B, S = qry.shape[0], qry.shape[1]
    Cf = 0 if feat is None else feat.shape[2]
    return _f32(B, 4, S, k, like=qry), _f32(B, 3, S, k, like=qry), _f32(B, Cf, S, k, like=qry), _i64(B, S, k, like=qry)


@_register("fusion_group", _fusion_fake)
def _fusion_group(qry, ref, feat, k):
    """PointsFusion.knn_group / knn_group_withI: knn_points(return_nn) + resi + |resi| + cat + permute in one C call"""
    B, S, _ = qry.shape; N = ref.shape[1]
    Cf = 0 if feat is None else feat.shape[2]
    dev = qry.device
    resi = _f32(B, 4, S, k, like=qry)
    nn = _f32(B, 3, S, k, like=qry)
    gf = _f32(B, Cf, S, k, like=qry)
    idx = _i64(B, S, k, like=qry)
    lib = _lib.load()
    nws = _search_ws(lib, B, N, S, k)
    ws = _workspace(nws, dev)
    _call(dev, lib.b200pc_fusion_group, _ptr(qry), _ptr(ref), _ptr(feat if Cf else None), B, N, S, k, Cf, _ptr(resi), _ptr(nn),
          _ptr(gf if Cf else None), _ptr(idx), _ptr(ws), nws, _stream(dev))
    return resi, nn, gf, idx


@_register("channel_max", lambda x: _f32(x.shape[0], like=x))
def _channel_max(x):
    rows, Cc = x.shape
    out = _f32(rows, like=x)
    if x.data_ptr() % 16:       # the kernel reads each row as float4s: a view that starts between 16-byte boundaries
        x = x.clone()           # (a slice of a flat buffer) is copied into a fresh, aligned block first
    _call(x.device, _lib.load().b200pc_channel_max, _ptr(x), rows, Cc, _ptr(out), _stream(x.device))
    return out


@_register("rebuild_pack", lambda ref, qry, s_offset, peer_ptrs: _f32(qry.shape[1], qry.shape[0], 4, like=ref))
def _rebuild_pack(ref, qry, s_offset, peer_ptrs):
    """PolyPCI.rebuild for a query shard: K=1 search + (index, neighbour xyz) records [S_local,B,4]; the same kernel also
    stores the slab into every peer buffer (symmetric memory base pointers) -- the all-gather without a collective."""
    B, N, _ = ref.shape; S = qry.shape[1]
    dev = ref.device
    out = _f32(S, B, 4, like=ref)
    lib = _lib.load()
    nws = lib.b200pc_rebuild_pack_workspace_bytes(B, N, S)
    ws = _workspace(nws, dev)
    n = len(peer_ptrs)
    arr = (C.c_void_p * max(n, 1))(*[C.c_void_p(int(p)) for p in peer_ptrs])
    _call(dev, lib.b200pc_rebuild_pack, _ptr(ref), _ptr(qry), B, N, S, int(s_offset), _ptr(out), arr if n else C.c_void_p(0), n,
          _ptr(ws), nws, _stream(dev))
    return out


# ---- a9 ----------------------------------------------------------------------------------
def _chamfer_fake(x, y):
    B, N, M = x.shape[0], x.shape[1], y.shape[1]
    return _f32((), like=x), _f32(B, N, like=x), _i64(B, N, like=x), _f32(B, M, like=x), _i64(B, M, like=x)


@_register("chamfer_fwd", _chamfer_fake)
def _chamfer_fwd(x, y):
    B, N, _ = x.shape; M = y.shape[1]
    dev = x.device
    dx = _f32(B, N, like=x); ix = _i64(B, N, like=x)
    dy = _f32(B, M, like=x); iy = _i64(B, M, like=x)
    loss = _f32((), like=x)
    lib = _lib.load()
    nws = max(_search_ws(lib, B, M, N, 1), _search_ws(lib, B, N, M, 1))
    ws = _workspace(nws, dev)
    _call(dev, lib.b200pc_chamfer_fwd, _ptr(x), _ptr(y), B, N, M, _ptr(dx), _ptr(ix), _ptr(dy), _ptr(iy), _ptr(loss), _ptr(ws), nws,
          _stream(dev))
    return loss, dx, ix, dy, iy


@_register("chamfer_bwd", lambda x, y, ix, iy, gloss: (torch.empty_like(x), torch.empty_like(y)))
def _chamfer_bwd(x, y, ix, iy, gloss):
    B, N, _ = x.shape; M = y.shape[1]
    gx = torch.empty_like(x); gy = torch.empty_like(y)
    _call(x.device, _lib.load().b200pc_chamfer_bwd, _ptr(x), _ptr(y), _ptr(ix), _ptr(iy), _ptr(gloss), B, N, M, _ptr(gx), _ptr(gy),
          _stream(x.device))
    return gx, gy


def _chamfer_setup(ctx, inputs, output):
    x, y = inputs
    _, _, ix, _, iy = output
    ctx.save_for_backward(x, y, ix, iy)


def _chamfer_backward(ctx, gloss, *_):
    x, y, ix, iy = ctx.saved_tensors
    gx, gy = torch.ops.b200pc.chamfer_bwd(x, y, ix, iy, gloss.contiguous().float().view(1))
    return gx, gy


torch.library.register_autograd("b200pc::chamfer_fwd", _chamfer_backward, setup_context=_chamfer_setup, lib=_L)


def _chamfer_ragged_fake(x, y, x_len, y_len):
    B, N, M = x.shape[0], x.shape[1], y.shape[1]
    return _f32(B, 2, like=x), _f32(B, N, like=x), _i64(B, N, like=x), _f32(B, M, like=x), _i64(B, M, like=x)


@_register("chamfer_ragged_fwd", _chamfer_ragged_fake)
def _chamfer_ragged_fwd(x, y, x_len, y_len):
    B, N, _ = x.shape; M = y.shape[1]
    dev = x.device
    dx = _f32(B, N, like=x); ix = _i64(B, N, like=x)
    dy = _f32(B, M, like=x); iy = _i64(B, M, like=x)
    sums = _f32(B, 2, like=x)
    lib = _lib.load()
    nws = max(_search_ws(lib, B, M, N, 1), _search_ws(lib, B, N, M, 1))
    ws = _workspace(nws, dev)
    _call(dev, lib.b200pc_chamfer_ragged_fwd, _ptr(x), _ptr(y), _ptr(x_len), _ptr(y_len), B, N, M, _ptr(dx), _ptr(ix), _ptr(dy), _ptr(iy),
          _ptr(sums), _ptr(ws), nws, _stream(dev))
    return sums, dx, ix, dy, iy


@_register("chamfer_ragged_bwd", lambda x, y, ix, iy, x_len, y_len, gsums: (torch.empty_like(x), torch.empty_like(y)))
def _chamfer_ragged_bwd(x, y, ix, iy, x_len, y_len, gsums):
    B, N, _ = x.shape; M = y.shape[1]
    gx = torch.empty_like(x); gy = torch.empty_like(y)
    _call(x.device, _lib.load().b200pc_chamfer_ragged_bwd, _ptr(x), _ptr(y), _ptr(ix), _ptr(iy), _ptr(x_len), _ptr(y_len), _ptr(gsums),
          B, N, M, _ptr(gx), _ptr(gy), _stream(x.device))
    return gx, gy


def _chamfer_ragged_setup(ctx, inputs, output):
    x, y, x_len, y_len = inputs
    _, _, ix, _, iy = output
    ctx.save_for_backward(x, y, ix, iy, x_len, y_len)


def _chamfer_ragged_backward(ctx, gsums, *_):
    x, y, ix, iy, x_len, y_len = ctx.saved_tensors
    gx, gy = torch.ops.b200pc.chamfer_ragged_bwd(x, y, ix, iy, x_len, y_len, gsums.contiguous().float())
    return gx, gy, None, None


torch.library.register_autograd("b200pc::chamfer_ragged_fwd", _chamfer_ragged_backward, setup_context=_chamfer_ragged_setup, lib=_L)


# ---- f4 ----------------------------------------------------------------------------------
@_register("poly_predict", lambda frames, weights: torch.empty_like(frames[0]))
def _poly_predict(frames, weights):
    F = len(frames)
    B = frames[0].shape[0]
    per_batch = int(frames[0][0].numel())
    out = torch.empty_like(frames[0])
    ptrs = (C.c_void_p * F)(*[C.c_void_p(f.data_ptr()) for f in frames])
    dev = frames[0].device
    _call(dev, _lib.load().b200pc_poly_predict, ptrs, _ptr(weights), B, F, per_batch, _ptr(out), _stream(dev))
    return out


_O = torch.ops.b200pc


# ==========================================================================================
# public functions (argument normalisation like the reference's functions, then the ops)
# ==========================================================================================
def square_distance(src, dst):
    """Utils/Pointnet2Utils.py:20  [B,N,3],[B,M,3] -> [B,N,M], torch-CPU rounding order."""
    return _O.square_distance(_prep(src, "src"), _prep(dst, "dst"))


def knn_search(ref, qry, k, form, want_dist=False):
    """k nearest refs per query.  ref [B,N,3], qry [B,S,3] -> idx [B,S,k] int64 (, dist [B,S,k])."""
    ref = _prep(ref, "ref"); qry = _prep(qry, "qry")
    k = int(k)
    if k > ref.shape[1]:   # torch.topk raises RuntimeError("selected index k out of range")
        raise RuntimeError("selected index k out of range (k=%d > %d reference points)" % (k, ref.shape[1]))
    idx, dist = _O.knn(ref.detach(), qry.detach(), k, int(form), bool(want_dist))      # indices / raw distances carry no gradient
    return (idx, dist) if want_dist else idx


def _lengths(lengths, B, dev, name):
    """per-item lengths of a ragged batch: None (every item full) or int64 [B] on `dev`.  The values are NOT checked on
    the host (that would cost a device->host sync): the kernels clamp them to [0, padded size]."""
    if lengths is None:
        return None
    if not isinstance(lengths, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor or None" % name)
    if lengths.dtype.is_floating_point or lengths.dtype.is_complex or lengths.dtype == torch.bool:
        raise TypeError("%s must be an integer tensor, got %s" % (name, lengths.dtype))
    if tuple(lengths.shape) != (B,):
        raise ValueError("%s must have shape [%d], got %s" % (name, B, tuple(lengths.shape)))
    return _idx64(lengths, dev)


def knn_ragged(ref, qry, k, form, ref_len=None, qry_len=None, want_dist=False):
    """knn_search on a ragged batch: item b has ref_len[b] valid refs and qry_len[b] valid queries (int [B] tensors or None
    = full; clamped to [0, N] / [0, S] on the device).  Valid rows equal knn_search of qry[b, :s_b] against ref[b, :n_b] bit
    for bit; slots without a valid ref and padded rows are -1 / +inf.  k <= N; k > ref_len[b] is allowed."""
    ref = _prep(ref, "ref"); qry = _prep(qry, "qry")
    k = int(k)
    if k > ref.shape[1]:
        raise RuntimeError("selected index k out of range (k=%d > %d reference points)" % (k, ref.shape[1]))
    if ref.shape[0] != qry.shape[0]:
        raise ValueError("knn_ragged: ref and qry must have the same batch size")
    B = ref.shape[0]
    rl = _lengths(ref_len, B, ref.device, "ref_len"); ql = _lengths(qry_len, B, ref.device, "qry_len")
    idx, dist = _O.knn_ragged(ref.detach(), qry.detach(), rl, ql, k, int(form), bool(want_dist))
    return (idx, dist) if want_dist else idx


def knn_search_i32(ref, qry, k, form):
    """knn_search with int32 indices [B,S,k] (host-buffer callers: half the read-back bytes of the reference's int64)."""
    ref = _prep(ref, "ref"); qry = _prep(qry, "qry")
    k = int(k)
    if k > ref.shape[1]:
        raise RuntimeError("selected index k out of range (k=%d > %d reference points)" % (k, ref.shape[1]))
    return _O.knn_i32(ref.detach(), qry.detach(), k, int(form))


def ball_query(radius, nsample, xyz, new_xyz):
    """Utils/Pointnet2Utils.py:88  -> [B,S,nsample] int64 (N where the ball is empty)."""
    xyz = _prep(xyz, "xyz"); new_xyz = _prep(new_xyz, "new_xyz")
    # `sqrdists > radius ** 2`: python double squared, then compared against fp32 values
    r2 = torch.tensor(float(radius) ** 2, dtype=torch.float32).item()
    return _O.ball_query(xyz.detach(), new_xyz.detach(), r2, int(nsample))


def fps(xyz, npoint, start, want_xyz=False):
    """Utils/Pointnet2Utils.py:64  start [B] int64 (first centroid) -> [B,npoint] int64.
    want_xyz: also return the picks' coordinates [B,npoint,3] from the same C call (Sample.forward, Utils/Layers.py:23-27)."""
    xyz = _prep(xyz, "xyz")
    start = _idx64(start, xyz.device)
    if want_xyz:
        if torch.is_grad_enabled() and xyz.requires_grad:
            # index_points(points, fps_idx) is differentiable in the reference (Utils/Layers.py:25-26): the picks are
            # made on the detached cloud, the coordinates come from the differentiable gather
            idx = _O.fps(xyz.detach(), int(npoint), start)
            return idx, gather(xyz, idx)
        return _O.fps_sample(xyz, int(npoint), start)
    return _O.fps(xyz.detach(), int(npoint), start)


def gather(points, idx):
    """Utils/Pointnet2Utils.py:44  points [B,N,C], idx [B,...] -> [B,...,C]  (differentiable in points)."""
    points = _prep(points, "points")
    idx = _idx64(idx, points.device)
    B = points.shape[0]
    out_shape = tuple(idx.shape) + (points.shape[2],)
    if points.shape[2] == 0 or idx.numel() == 0:      # nothing to move (e.g. clouds without extra channels)
        return torch.empty(out_shape, dtype=torch.float32, device=points.device)
    return _O.gather(points, idx.reshape(B, -1), CHECK_BOUNDS).view(*out_shape)


def group_points(xyz, new_xyz, feat, idx, xyz_first=True):
    """Utils/Layers.py:57-66 (xyz_first) / Utils/Pointnet2Utils.py:243-253 (features first): xyz [B,N,3],
    new_xyz [B,S,3], feat [B,N,D] or None, idx [B,S,K] -> the Conv2d input [B,3+D,K,S] in one kernel."""
    xyz = _prep(xyz, "xyz"); new_xyz = _prep(new_xyz, "new_xyz")
    if feat is not None:
        feat = _prep(feat, "feat")
        if feat.shape[2] == 0:
            feat = None
    idx = _idx64(idx, xyz.device)
    if idx.dim() != 3 or idx.shape[0] != xyz.shape[0] or idx.shape[1] != new_xyz.shape[1]:
        raise ValueError("group_points: idx must be [B,S,K] with S = new_xyz.shape[1], got %s" % (tuple(idx.shape),))
    if feat is not None and (feat.shape[0] != xyz.shape[0] or feat.shape[1] != xyz.shape[1]):
        raise ValueError("group_points: feat must be [B,N,D] with the same B, N as xyz")
    N = xyz.shape[1]
    if CHECK_BOUNDS and idx.numel() and (int(idx.min()) < -N or int(idx.max()) >= N):
        raise IndexError("index out of range in group_points (valid range is [-%d, %d))" % (N, N))
    return _O.group_points(xyz, new_xyz, feat, idx, bool(xyz_first))


def three_nn(unknown, known, variant=0, want_weight=True):
    """three nearest `known` points for every `unknown` point.
    -> dist [B,N,3] (ascending raw expanded-form values), idx [B,N,3] int64, weight [B,N,3] (None unless want_weight)."""
    unknown = _prep(unknown, "unknown"); known = _prep(known, "known")
    dist, idx, weight = _O.three_nn(unknown.detach(), known.detach(), int(variant), bool(want_weight))
    return dist, idx, (weight if want_weight else None)


def three_nn_autograd(unknown, known, variant=0):
    """three_nn whose distances and weights are differentiable w.r.t. the coordinates, like the reference's
    `square_distance(...).sort()` + `1.0 / dists` (Utils/Layers.py:180-186, Utils/Pointnet2Utils.py:297-303; ISAPCInet
    trains through them, Models/New_Models0.py:164-172).  The search kernel picks the neighbours; the three distances
    are then rebuilt from the gathered neighbours with torch ops: VALUES stay the kernel's (bit-exact with the
    reference's expanded form), GRADIENTS are those of |u - k|^2, which is what autograd derives for the expanded form."""
    unknown = _prep(unknown, "unknown"); known = _prep(known, "known")
    dist, idx, _ = _O.three_nn(unknown.detach(), known.detach(), int(variant), False)
    diff = unknown.unsqueeze(2) - gather(known, idx)                      # [B,N,3,3], differentiable in both clouds
    d_torch = (diff * diff).sum(-1)
    d = dist + (d_torch - d_torch.detach())
    if int(variant) == 0:
        dd = torch.where(d < 1e-10, torch.full_like(d, 1e-10), d)         # dists[dists < 1e-10] = 1e-10 (no gradient there)
        inv = 1.0 / dd
    else:
        inv = 1.0 / (d + 1e-8)
    weight = inv / torch.sum(inv, dim=2, keepdim=True)
    return d, idx, weight


def three_interpolate(feat, idx, weight):
    """feat [B,S,C], idx [B,N,3], weight [B,N,3] -> [B,N,C] = (f0*w0 + f1*w1) + f2*w2."""
    feat = _prep(feat, "feat"); weight = _prep(weight, "weight")
    return _O.three_interpolate(feat, _idx64(idx, feat.device), weight)


def feature_propagation(unknown, known, feat, variant=0):
    """FeaturePropagation / PointNetFeaturePropagation interpolation (Utils/Layers.py:180-188, Utils/Pointnet2Utils.py:297-304):
    unknown [B,N,3] dense, known [B,S,3] sparse, feat [B,S,C] -> [B,N,C].  One C call (search -> weights -> mix) when
    the coordinates carry no gradient; otherwise the differentiable-weights path (three_nn_autograd)."""
    unknown = _prep(unknown, "unknown"); known = _prep(known, "known"); feat = _prep(feat, "feat")
    if torch.is_grad_enabled() and (unknown.requires_grad or known.requires_grad):
        _, idx, weight = three_nn_autograd(unknown, known, variant)
        return _O.three_interpolate(feat, idx, weight)
    return _O.feature_propagation(unknown, known, feat, int(variant))[0]


def fusion_group(qry, ref, k, feat=None):
    """PointsFusion.knn_group (Utils/Layers.py:207-226; upstream PointINet20230424/models/layers.py:346-368) and
    knn_group_withI (Utils/Layers.py:384-402) on point-major inputs: qry [B,S,3], ref [B,N,3], feat [B,N,Cf] or None
    -> (new_features [B,4,S,k] = (nn - q, |nn - q|), nn [B,3,S,k], grouped feat [B,Cf,S,k], idx [B,S,k])."""
    qry = _prep(qry, "qry"); ref = _prep(ref, "ref")
    k = min(int(k), ref.shape[1])
    if feat is not None:
        feat = _prep(feat, "feat")
        if feat.shape[2] == 0:
            feat = None
    return _O.fusion_group(qry, ref, feat, k)


def channel_max(x):
    """x [rows, C] (channels-last rows of PointsFusion's point-wise MLP) -> [rows] = max over the channels
    (`torch.max(new_features, dim=1)`, Utils/Layers.py:276).  Any storage offset: the op copies a view that is not
    16-byte aligned before its vector kernel reads it."""
    x = _prep(x, "x")
    if x.dim() != 2 or x.shape[1] % 4:
        return x.max(dim=1)[0]
    return _O.channel_max(x)


def rebuild_pack(ref, qry, s_offset=0, peer_ptrs=()):
    """PolyPCI.rebuild (PolyPCI/Models/Models_V1.py:102-114) on point-major inputs for a query shard: ref [B,N,3],
    qry [B,S_local,3] -> records [S_local,B,4] = {int32 index bits, nn x, y, z}; `peer_ptrs`: base addresses of the ranks'
    [S_total,B,4] symmetric buffers, written by the same kernel at row offset `s_offset`."""
    return _O.rebuild_pack(_prep(ref, "ref"), _prep(qry, "qry"), int(s_offset), [int(p) for p in peer_ptrs])


def unpack_rebuild(records):
    """records [S,B,4] -> (idx [B,S] int64, nn [B,S,3])"""
    idx = records[..., 0].contiguous().view(torch.int32).long().transpose(0, 1).contiguous()
    nn = records[..., 1:4].transpose(0, 1).contiguous()
    return idx, nn


def chamfer(x, y):
    """x [B,N,3], y [B,M,3] -> (loss scalar, dx [B,N], ix [B,N], dy [B,M], iy [B,M]); loss is differentiable."""
    return _O.chamfer_fwd(_prep(x, "x"), _prep(y, "y"))


def chamfer_ragged(x, y, x_len=None, y_len=None):
    """Chamfer terms of a ragged batch: x [B,N,3], y [B,M,3] padded, x_len / y_len int [B] tensors or None (full).
    -> (sums [B,2] = per-item sums of the valid points' minima in each direction, differentiable in x and y;
        dx [B,N], ix [B,N], dy [B,M], iy [B,M] with -1 / +inf for padded points).  The point / batch reductions are torch
    arithmetic on `sums` (chamfer_reduce)."""
    x = _prep(x, "x"); y = _prep(y, "y")
    if x.shape[0] != y.shape[0]:
        raise ValueError("chamfer_ragged: x and y must have the same batch size")
    B = x.shape[0]
    return _O.chamfer_ragged_fwd(x, y, _lengths(x_len, B, x.device, "x_len"), _lengths(y_len, B, x.device, "y_len"))


def chamfer_reduce(sums, x_len, y_len, N, M, point_reduction="mean", batch_reduction="mean"):
    """pytorch3d.loss.chamfer_distance's reductions of the per-item sums [B,2]: point_reduction "mean" divides each sum
    by max(length, 1) (the padded size when the lengths are None), "sum" keeps it; batch_reduction "mean" / "sum" / None
    (-> [B])."""
    if point_reduction not in ("mean", "sum"):
        raise ValueError('point_reduction must be "mean" or "sum", got %r' % (point_reduction,))
    if batch_reduction not in ("mean", "sum", None):
        raise ValueError('batch_reduction must be "mean", "sum" or None, got %r' % (batch_reduction,))
    B = sums.shape[0]
    cx, cy = sums[:, 0], sums[:, 1]
    if point_reduction == "mean":
        def div(lengths, full):
            if lengths is None:
                return torch.full((B,), float(max(full, 1)), dtype=sums.dtype, device=sums.device)
            return lengths.to(sums.device).clamp(0, full).clamp(min=1).to(sums.dtype)
        cx = cx / div(x_len, N)
        cy = cy / div(y_len, M)
    def batch(c):                  # per direction, then added, in pytorch3d's order
        if batch_reduction is None:
            return c
        return c.sum() / max(B, 1) if batch_reduction == "mean" else c.sum()
    return batch(cx) + batch(cy)


def poly_predict(frames, weights):
    """frames: list of F [B,...] fp32 CUDA tensors, weights [B,F] float64 on the device -> sum_f w[b,f] * frames[f][b]"""
    frames = [_prep(f, "frame") for f in frames]
    if not frames:
        raise ValueError("poly_predict: no frames")
    shape, dev = frames[0].shape, frames[0].device
    if any(f.shape != shape or f.device != dev for f in frames):
        raise ValueError("poly_predict: all frames must share shape and device")
    # the kernel reads B*F doubles from `weights`: anything else would read past the buffer or reinterpret its bits
    if not isinstance(weights, torch.Tensor) or weights.dtype != torch.float64 or weights.device != dev:
        raise ValueError("poly_predict: weights must be a float64 tensor on %s" % dev)
    if tuple(weights.shape) != (shape[0], len(frames)):
        raise ValueError("poly_predict: weights must be [B, F] = [%d, %d], got %s" % (shape[0], len(frames), tuple(weights.shape)))
    return _O.poly_predict(frames, weights.contiguous())


def reload_tuning():
    """re-read the B200PC_* tuning variables (the library caches them at its first launch); tests / probes only"""
    _lib.load().b200pc_tuning_reload()


def fma_peak(iters=4096):
    """sustained packed-FP32 FMA rate of the current device in TFLOP/s (roofline denominator)."""
    tf = C.c_double(0.0); ms = C.c_double(0.0)
    _lib.check(_lib.load().b200pc_fma_peak(int(iters), C.byref(tf), C.byref(ms), _stream(torch.cuda.current_device())))
    return tf.value, ms.value
