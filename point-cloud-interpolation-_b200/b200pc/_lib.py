"""ctypes binding of libb200pc.so (the C ABI declared in include/b200pc.h).

The library is the product; this module only loads it, declares argument types and turns error
codes into Python exceptions.  There is NO fallback: if the shared object is missing the import
of any compute entry point raises, loudly.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200PC_LIBRARY=bounds loads the bounds-checked build (make bounds: the same sources with device-side index asserts) --
# for the out-of-bounds test run only; it is slower and never the library a caller times or ships.
LIB_PATH = os.path.join(_HERE, "libb200pc_bounds.so" if os.environ.get("B200PC_LIBRARY") == "bounds" else "libb200pc.so")

OK, EINVAL, ECUDA, EWORKSPACE = 0, -1, -2, -3

_p = C.c_void_p
_i = C.c_int
_l = C.c_int64
_z = C.c_size_t
_f = C.c_float

# name -> (restype, argtypes); must list EVERY symbol include/b200pc.h declares
SIGNATURES = {
    "b200pc_last_error": (C.c_char_p, []),
    "b200pc_version": (_i, []),
    "b200pc_device_sm_count": (_i, []),
    "b200pc_tuning_reload": (None, []),
    "b200pc_search_workspace_bytes": (_z, [_i, _i, _i, _i]),
    "b200pc_fps_workspace_bytes": (_z, [_i, _i]),
    "b200pc_square_distance": (_i, [_p, _p, _i, _i, _i, _p, _p]),
    "b200pc_knn": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _z, _p]),
    "b200pc_knn_ragged": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _z, _p]),
    "b200pc_knn_i32": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _z, _p]),
    "b200pc_ball_query": (_i, [_p, _p, _i, _i, _i, _f, _i, _p, _p, _z, _p]),
    "b200pc_three_nn": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _z, _p]),
    "b200pc_three_interpolate": (_i, [_p, _p, _p, _i, _i, _i, _i, _p, _p]),
    "b200pc_three_interpolate_bwd": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "b200pc_feature_propagation_workspace_bytes": (_z, [_i, _i, _i]),
    "b200pc_feature_propagation": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _p, _z, _p]),
    "b200pc_fusion_group": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p, _z, _p]),
    "b200pc_channel_max": (_i, [_p, _l, _i, _p, _p]),
    "b200pc_rebuild_pack_workspace_bytes": (_z, [_i, _i, _i]),
    "b200pc_rebuild_pack": (_i, [_p, _p, _i, _i, _i, _i, _p, _p, _i, _p, _z, _p]),
    "b200pc_fps": (_i, [_p, _i, _i, _i, _p, _p, _p, _z, _p]),
    "b200pc_fps_sample": (_i, [_p, _i, _i, _i, _p, _p, _p, _p]),
    "b200pc_gather": (_i, [_p, _p, _i, _i, _i, _l, _p, _p, _p]),
    "b200pc_gather_bwd": (_i, [_p, _p, _i, _i, _i, _l, _p, _p]),
    "b200pc_group_points": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "b200pc_poly_predict": (_i, [_p, _p, _i, _i, _l, _p, _p]),
    "b200pc_group_points_bwd": (_i, [_p, _p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "b200pc_chamfer_fwd": (_i, [_p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _z, _p]),
    "b200pc_chamfer_bwd": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _p, _p, _p]),
    "b200pc_chamfer_ragged_fwd": (_i, [_p, _p, _p, _p, _i, _i, _i, _p, _p, _p, _p, _p, _p, _z, _p]),
    "b200pc_chamfer_ragged_bwd": (_i, [_p, _p, _p, _p, _p, _p, _p, _i, _i, _i, _p, _p, _p]),
    "b200pc_fma_peak": (_i, [_i, C.POINTER(C.c_double), C.POINTER(C.c_double), _p]),
    "b200pc_knn_host": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p]),
    "b200pc_ball_query_host": (_i, [_p, _p, _i, _i, _i, _f, _i, _p]),
    "b200pc_fps_host": (_i, [_p, _i, _i, _i, _p, _p]),
    "b200pc_knn_async_host_workspace_bytes": (_z, [_i, _i, _i, _i]),
    "b200pc_knn_async_host": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p, _p, _z, _p]),
}

_lib = None


class B200pcError(RuntimeError):
    pass


def load():
    """dlopen libb200pc.so (once) and declare every prototype.  Raises if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "libb200pc.so is not built (%s). Run `python __graft_entry__.py` or `make -C "
                "point-cloud-interpolation-_b200`. There is no CPU fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError here == header / library out of sync
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error():
    return load().b200pc_last_error().decode("utf-8", "replace")


def check(rc, exc_for_einval=RuntimeError):
    """0 -> ok; EINVAL -> the exception class the reference would have raised; else B200pcError."""
    if rc == OK:
        return
    msg = last_error()
    if rc == EINVAL:
        raise exc_for_einval(msg)
    raise B200pcError("b200pc error %d: %s" % (rc, msg))
