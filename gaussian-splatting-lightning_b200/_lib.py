"""ctypes binding of libb200gs.so (the C ABI declared in include/b200gs.h).

There is no fallback: if the shared library is missing or a call fails, this raises.  The product never routes
through ``oracle/`` or a torch re-implementation.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int32, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200gs.so")

MODE_VANILLA = 0
MODE_GSPLAT = 1
TILE = 16


class B200gsView(ctypes.Structure):
    _fields_ = [
        ("width", c_int32), ("height", c_int32), ("mode", c_int32), ("sh_degree", c_int32), ("sh_stride", c_int32),
        ("reserved0", c_int32),
        ("fx", c_float), ("fy", c_float), ("cx", c_float), ("cy", c_float),
        ("tanfovx", c_float), ("tanfovy", c_float), ("scale_modifier", c_float), ("eps2d", c_float),
        ("near_plane", c_float), ("reserved1", c_float),
        ("viewmatrix", c_float * 16), ("projmatrix", c_float * 16), ("campos", c_float * 3), ("reserved2", c_float),
    ]


class B200gsError(RuntimeError):
    pass


_lib = None

_P = c_void_p  # every device pointer is passed as an integer address

_SIGNATURES = {
    "b200gs_last_error": (c_char_p, []),
    "b200gs_version": (c_int32, []),
    "b200gs_launch_count": (c_int64, []),
    "b200gs_project_fwd": (c_int32, [POINTER(B200gsView), c_int64] + [_P] * 4 + [_P] * 9 + [_P]),
    "b200gs_project_bwd": (c_int32, [POINTER(B200gsView), c_int64] + [_P] * 4 + [_P] * 2 + [_P] * 5 + [_P] * 4 + [_P]),
    "b200gs_project_fwd_raw": (c_int32, [POINTER(B200gsView), c_int64] + [_P] * 6 + [c_int32] + [_P] * 9 + [_P]),
    "b200gs_selective_adam": (c_int32, [c_int64, c_int32, _P, _P, _P, _P, _P, c_float, c_float, c_float, c_float, _P]),
    "b200gs_densify_stats": (c_int32, [c_int64, _P, _P, _P, c_int32, c_float, c_float, _P, _P, _P, _P]),
    "b200gs_knn_workspace_bytes": (c_size_t, [c_int64]),
    "b200gs_knn_mean_dist2": (c_int32, [c_int64, _P, _P, _P, c_size_t, _P]),
    "b200gs_sh_fwd": (c_int32, [c_int32, c_int32, c_int64, _P, _P, _P, _P]),
    "b200gs_sh_bwd": (c_int32, [c_int32, c_int32, c_int64, _P, _P, _P, _P, _P, _P]),
    "b200gs_bin_count_workspace_bytes": (c_size_t, [c_int64]),
    "b200gs_bin_sort_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int32, c_int32]),
    "b200gs_bin_count": (c_int32, [c_int32, c_int32, c_int32, c_int64, _P, _P, _P, _P, _P, _P, c_size_t, _P, _P, c_int32, _P]),
    "b200gs_bin_sort": (c_int32, [c_int32, c_int32, c_int32, c_int64, c_int32, c_int64, c_int64, _P, _P, _P, c_size_t, _P, _P, _P, c_int32, _P]),
    "b200gs_loss_blocks": (c_int64, [c_int32, c_int32, c_int32]),
    "b200gs_loss_fwd": (c_int32, [c_int32, c_int32, c_int32, _P, _P, _P, _P, _P]),
    "b200gs_loss_bwd": (c_int32, [c_int32, c_int32, c_int32, _P, _P, _P, ctypes.c_float, _P, _P, _P]),
    "b200gs_publish_i64": (c_int32, [_P, _P, c_int32, _P]),
    "b200gs_blend_fwd": (c_int32, [c_int32] * 4 + [_P] * 7 + [_P, c_int64, c_int64, _P, _P, _P, _P]),
    "b200gs_blend_fwd_hits": (c_int32, [c_int32] * 4 + [_P] * 7 + [_P, c_int64, c_int64, _P, _P, _P, _P, _P]),
    "b200gs_blend_bwd": (c_int32, [c_int32] * 4 + [_P] * 7 + [_P, _P, _P, c_int64, c_int64, _P, c_float, c_float]
                         + [_P] * 5 + [_P]),
    "b200gs_project_bwd_rows": (c_int32, [POINTER(B200gsView), c_int64] + [_P] * 6 + [c_int32] + [_P] * 4 + [c_int32] + [_P] * 6 + [_P, c_int32] + [_P]),
    "b200gs_project_fwd_raw_multi": (c_int32, [POINTER(B200gsView), c_int32, c_int64] + [_P] * 6 + [c_int32] + [_P] * 7 + [_P]),
    "b200gs_project_bwd_rows_multi": (c_int32, [POINTER(B200gsView), c_int32, c_int64] + [_P] * 6 + [c_int32] + [_P] * 3 + [POINTER(c_void_p)] + [_P] * 6 + [_P]),
    "b200gs_ipc_alloc": (c_int32, [c_size_t, POINTER(c_void_p), ctypes.c_char_p]),
    "b200gs_ipc_open": (c_int32, [ctypes.c_char_p, POINTER(c_void_p)]),
    "b200gs_ipc_close": (c_int32, [c_void_p]),
    "b200gs_ipc_free": (c_int32, [c_void_p]),
    "b200gs_pack_rows_workspace_bytes": (c_size_t, [c_int64]),
    "b200gs_pack_rows": (c_int32, [c_int64, c_int64, c_int64] + [_P] * 7 + [_P, c_size_t, _P, _P, _P, _P]),
    "b200gs_bin_count_rows": (c_int32, [c_int32, c_int32, c_int32, c_int64, _P, c_int32, _P, c_size_t, _P, _P, c_int32, _P, _P, c_int64]),
    "b200gs_project_pack_workspace_bytes": (c_size_t, [c_int32, c_int64]),
    "b200gs_project_pack_multi": (c_int32, [POINTER(B200gsView), c_int32, c_int64] + [_P] * 6 + [c_int32] + [_P] * 4 + [POINTER(c_void_p), c_int64, _P, c_size_t, _P, _P]),
    "b200gs_blend_fwd_rows": (c_int32, [c_int32] * 3 + [_P] * 5 + [c_int64, c_int64, _P, _P, _P, _P]),
    "b200gs_blend_bwd_rows": (c_int32, [c_int32] * 3 + [_P] * 7 + [c_int64, c_int64, _P, ctypes.c_float, ctypes.c_float, _P, _P]),
    "b200gs_project_fwd_rows": (c_int32, [POINTER(B200gsView), c_int64] + [_P] * 6 + [c_int32] + [_P] * 4 + [_P]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES.keys())


def lib():
    """Load (once) and return the ctypes handle.  Raises B200gsError when the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B200gsError(
                f"{LIB_PATH} not found: build it with `python gaussian-splatting-lightning_b200/build.py` "
                "(or __graft_entry__.build()).  b200gs has no CPU / torch fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        msg = lib().b200gs_last_error().decode("utf-8", "replace")
        raise B200gsError(f"{what} failed (rc={rc}): {msg}")


def ptr(t):
    """Device address of a tensor (or None -> NULL)."""
    return None if t is None else t.data_ptr()
