"""ctypes binding of the TEST-ONLY library libsupcon_b200_test.so (csrc/supcon_debug.h): the product
library plus the tcgen05 one-tile diagnostic and the host-side plan introspection.  Loaded by tests/ and
tools/ only; the product package never touches it."""
import ctypes
import os
from ctypes import POINTER, c_int32, c_int64, c_void_p

from wav2vec_contr_loss_b200 import _cabi
from wav2vec_contr_loss_b200 import build as _build

_lib = None


def load():
    global _lib
    if _lib is None:
        _build.build()
        lib = ctypes.CDLL(_build.TEST_LIB_PATH)
        P = POINTER(_cabi.Problem)
        lib.supcon_debug_last_error.restype = ctypes.c_char_p
        lib.supcon_debug_tc_tile.restype = c_int32
        lib.supcon_debug_tc_tile.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p]
        lib.supcon_debug_plan.restype = c_int32
        lib.supcon_debug_plan.argtypes = [P, c_void_p, c_int32]
        lib.supcon_debug_ffma_plan.restype = c_int32
        lib.supcon_debug_ffma_plan.argtypes = [P, c_void_p, c_int32]
        lib.supcon_debug_route.restype = c_int32
        lib.supcon_debug_route.argtypes = [P, c_void_p, c_void_p, c_int32]
        lib.supcon_debug_sched.restype = c_int32
        lib.supcon_debug_sched.argtypes = [c_int32, c_int32, c_int64, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                           c_void_p]
        _lib = lib
    return _lib


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed (code {rc}): {load().supcon_debug_last_error().decode()}")


SMALL, MID, TENSOR, TILED = range(4)        # routes of supcon_debug_route
ROUTE_NAMES = ("small", "mid", "tensor", "tiled")


def route(prob, z):
    """supcon_debug_route of ``prob`` for rows at ``z`` (a tensor, or an address: only its alignment matters):
    dict(loss_and_grad, forward_rows, backward_rows, cluster, vec, fwd_class_sums, bwd_class_sums)"""
    out = (c_int32 * 7)()
    addr = z if isinstance(z, int) else z.data_ptr()
    check(load().supcon_debug_route(ctypes.byref(prob), c_void_p(addr), out, 7), "supcon_debug_route")
    keys = ("loss_and_grad", "forward_rows", "backward_rows", "cluster", "vec", "fwd_class_sums", "bwd_class_sums")
    return dict(zip(keys, list(out)))
