"""ctypes binding of libsqloss.so (include/sqloss.h).  Fails loudly when the library is missing."""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_longlong, c_size_t, c_void_p, POINTER

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SQ_LIBSQLOSS") or os.path.join(HERE, "libsqloss.so")   # override: tuning builds only
SQ_F32, SQ_F64, SQ_U8 = 0, 1, 2

_lib = None

_PROTOS = {
    "sq_version": (c_char_p, []),
    "sq_error_string": (c_char_p, [c_int]),
    "sq_device_sm_count": (c_int, [c_int, POINTER(c_int)]),
    "sq_profile_events": (None, [c_void_p, c_void_p]),
    "sq_scratch_bytes": (c_size_t, [c_int, c_int]),
    "sq_scratch_init": (c_int, [c_void_p, c_size_t, c_void_p]),
    "sq_implicit_loss": (c_int, [c_void_p, c_int, c_int, c_int, c_double, c_double, c_void_p, c_longlong, c_void_p,
                                 c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_size_t, c_void_p]),
    "sq_implicit_loss_heads": (c_int, [c_void_p, c_int, c_int, c_int, c_double, c_double, c_void_p, c_longlong, c_void_p,
                                       c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_size_t, c_void_p]),
    "sq_depth_projection_vjp": (c_int, [c_void_p, c_int, c_int, c_int, c_double, c_double, c_float, c_float, c_void_p,
                                        c_void_p, c_void_p, c_size_t, c_void_p]),
    "sq_occupancy_vjp": (c_int, [c_void_p, c_int, c_int, c_int, c_double, c_double, c_float, c_void_p, c_void_p, c_void_p,
                                 c_size_t, c_void_p]),
    "sq_voxel_loss": (c_int, [c_void_p, c_int, c_float, c_void_p, c_int, c_int, c_int, c_double, c_double, c_float, c_float,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sq_explicit_loss": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_double, c_double, c_float, c_float,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sq_iou_counts": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_double, c_double, c_void_p, c_void_p,
                              c_void_p, c_size_t, c_void_p]),
    "sq_least_squares": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_longlong, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sq_points_scratch_bytes": (c_size_t, [c_int, c_longlong]),
    "sq_least_squares_points": (c_int, [c_void_p, c_int, c_int, c_void_p, c_longlong, c_void_p, c_longlong, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "sq_field": (c_int, [c_void_p, c_int, c_int, c_int, c_double, c_double, c_int, c_float, c_void_p, c_void_p,
                         c_size_t, c_void_p]),
    "sq_ctx_create": (c_int, [c_int, POINTER(c_void_p)]),
    "sq_ctx_destroy": (None, [c_void_p]),
    "sq_implicit_loss_host": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_float, c_float,
                                      c_void_p, c_void_p]),
    "sq_implicit_loss_host_submit": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_float,
                                             c_float, c_float, c_int]),
    "sq_implicit_loss_host_wait": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "sq_explicit_loss_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "sq_iou_counts_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
}

EXPORTS = tuple(_PROTOS)


def lib() -> ctypes.CDLL:
    """Load libsqloss.so once.  No fallback: a missing library is an error."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -m sq_recovery_b200.build` "
                "(nvcc, sm_100a).  sq_recovery_b200 has no CPU or PyTorch fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(handle, name)      # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().sq_error_string(rc)
        raise RuntimeError(f"{what} failed: CUDA error {rc} ({msg.decode() if msg else '?'})")
