"""ctypes binding of libsupcon_b200.so (include/supcon_b200.h).

This is the stub a maintainer of the reference adds to bind the library
(INTEGRATION.md).  There is no fallback: if the shared object is missing the
import of the CUDA path raises, and every non-zero return code becomes a
``RuntimeError`` carrying ``supcon_last_error()``.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int32, c_size_t, c_uint32, c_void_p

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libsupcon_b200.so")

F32, BF16 = 0, 1
F16 = 2                 # a layer-mean store's element type only
COSINE, GEODESIC = 0, 1
FLAG_FORCE_EXACT, FLAG_FORCE_TENSOR, FLAG_NO_SMALL = 1, 2, 4
LABEL_I64, LABEL_F32, LABEL_F64 = 1, 2, 3
FLAG_UNIT_ROWS = 32
FLAG_PEER_EXCHANGE = 64
FLAG_CLASS_SUMS, FLAG_NO_CLASS_SUMS = 128, 256
FLAG_WS_FROM_FORWARD = 512
FLAG_MEMORY_COLUMNS = 1024
STATS_STRIDE = 8
N_PARTIALS = 8
P_SUM_FULL, P_CNT_FULL, P_SUM_MINED, P_CNT_MINED, P_SUM_W, P_GCNT_FULL, P_GCNT_MINED, P_FIXMAX = range(8)
ABI_VERSION = 3
ST_LSE, ST_LSE_M, ST_NPOS, ST_NNEG, ST_THR_VAL, ST_THR_IDX, ST_WSUM, ST_POS_MEAN = range(8)

EXPORTS = (
    "supcon_abi_version", "supcon_last_error", "supcon_workspace_bytes", "supcon_forward_rows",
    "supcon_finalize", "supcon_backward_rows", "supcon_loss_and_grad", "supcon_normalize_forward",
    "supcon_normalize_backward", "supcon_topk_indices", "supcon_forward_rows_local",
    "supcon_forward_rows_remote", "supcon_head_pool_forward", "supcon_head_pool_backward",
    "supcon_finalize_sets", "supcon_backward_rows_local", "supcon_backward_rows_remote",
    "supcon_peer_push", "supcon_peer_wait", "supcon_peer_end_step", "supcon_label_keys",
    "supcon_head_pool_forward_typed", "supcon_head_pool_backward_typed",
    "supcon_forward_rows_memory", "supcon_backward_rows_memory",
    "supcon_head_layer_mean_typed", "supcon_head_store_pool_forward", "supcon_head_sharded_store_pool_forward",
    "supcon_head_store_pool_forward_typed", "supcon_head_sharded_store_pool_forward_typed",
)


class Problem(ctypes.Structure):
    """struct supcon_problem (include/supcon_b200.h)."""
    _fields_ = [
        ("n_total", c_int32), ("row_offset", c_int32), ("n_rows", c_int32), ("d", c_int32),
        ("z_dtype", c_int32), ("similarity", c_int32), ("topk", c_int32), ("flags", c_uint32),
        ("tau", c_float), ("alpha", c_float), ("lambda_uni", c_float), ("uni_t", c_float),
    ]


class Peer(ctypes.Structure):
    """struct supcon_peer (include/supcon_b200.h)."""
    _fields_ = [("rank", c_int32), ("world", c_int32), ("peer_bases", c_void_p), ("off_flags", ctypes.c_uint64),
                ("epoch", c_void_p), ("mc_base", ctypes.c_uint64)]


PEER_FLAG_Z, PEER_FLAG_STATS, PEER_FLAG_DONE, PEER_NFLAGS = 0, 1, 2, 3


def peer_flag_bytes(world: int) -> int:
    return (PEER_NFLAGS * world + 4) * 4


_lib = None


def lib_path() -> str:
    return _LIB_PATH


def load():
    """Load the shared library once; raise loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(_LIB_PATH):
        raise RuntimeError(
            f"{_LIB_PATH} is missing: the CUDA extension has not been built "
            "(run `python -m wav2vec_contr_loss_b200.build`). There is no CPU fallback.")
    lib = ctypes.CDLL(_LIB_PATH)
    P = POINTER(Problem)
    lib.supcon_abi_version.restype = c_int32
    lib.supcon_abi_version.argtypes = []
    lib.supcon_last_error.restype = c_char_p
    lib.supcon_last_error.argtypes = []
    lib.supcon_workspace_bytes.restype = c_int32
    lib.supcon_workspace_bytes.argtypes = [P, POINTER(c_size_t)]
    lib.supcon_forward_rows.restype = c_int32
    lib.supcon_forward_rows.argtypes = [P, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_size_t, c_void_p]
    lib.supcon_forward_rows_memory.restype = c_int32
    lib.supcon_forward_rows_memory.argtypes = [P, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                               c_void_p, c_size_t, c_void_p]
    lib.supcon_forward_rows_local.restype = c_int32
    lib.supcon_forward_rows_local.argtypes = [P, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    lib.supcon_forward_rows_remote.restype = c_int32
    lib.supcon_forward_rows_remote.argtypes = [P, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    lib.supcon_finalize.restype = c_int32
    lib.supcon_finalize.argtypes = [P, c_void_p, c_void_p, c_void_p]
    lib.supcon_backward_rows.restype = c_int32
    lib.supcon_backward_rows.argtypes = [P, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_int32, c_void_p, c_size_t, c_void_p]
    lib.supcon_backward_rows_memory.restype = c_int32
    lib.supcon_backward_rows_memory.argtypes = [P, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_void_p, c_int32, c_void_p, c_size_t, c_void_p]
    lib.supcon_loss_and_grad.restype = c_int32
    lib.supcon_loss_and_grad.argtypes = [P, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_void_p,
                                         c_void_p, c_void_p, c_size_t, c_void_p]
    lib.supcon_normalize_forward.restype = c_int32
    lib.supcon_normalize_forward.argtypes = [c_void_p, c_int32, c_int32, c_void_p, c_int32, c_void_p, c_void_p]
    lib.supcon_normalize_backward.restype = c_int32
    lib.supcon_normalize_backward.argtypes = [c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_int32,
                                              c_int32, c_void_p, c_void_p]
    lib.supcon_topk_indices.restype = c_int32
    lib.supcon_topk_indices.argtypes = [P, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.supcon_finalize_sets.restype = c_int32
    lib.supcon_finalize_sets.argtypes = [P, c_void_p, c_int32, c_void_p, c_void_p, c_void_p]
    lib.supcon_backward_rows_local.restype = c_int32
    lib.supcon_backward_rows_local.argtypes = [P, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
    lib.supcon_backward_rows_remote.restype = c_int32
    lib.supcon_backward_rows_remote.argtypes = [P, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_int32, c_void_p, c_size_t, c_void_p]
    lib.supcon_head_pool_forward.restype = c_int32
    lib.supcon_head_pool_forward.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_float, c_float,
                                             c_void_p, c_void_p, c_void_p]
    lib.supcon_head_pool_backward.restype = c_int32
    lib.supcon_head_pool_backward.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_float, c_float,
                                              c_void_p, c_void_p, c_void_p, c_void_p]
    lib.supcon_head_pool_forward_typed.restype = c_int32
    lib.supcon_head_pool_forward_typed.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_float,
                                                   c_float, c_void_p, c_void_p, c_void_p]
    lib.supcon_head_pool_backward_typed.restype = c_int32
    lib.supcon_head_pool_backward_typed.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_float,
                                                    c_float, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.supcon_head_layer_mean_typed.restype = c_int32
    lib.supcon_head_layer_mean_typed.argtypes = [c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                                 c_void_p]
    lib.supcon_head_store_pool_forward.restype = c_int32
    lib.supcon_head_store_pool_forward.argtypes = [c_void_p, ctypes.c_int64, c_int32, c_int32, c_void_p, c_int32,
                                                   c_float, c_float, c_void_p, c_void_p, c_void_p]
    lib.supcon_head_sharded_store_pool_forward.restype = c_int32
    lib.supcon_head_sharded_store_pool_forward.argtypes = [c_void_p, c_int32, ctypes.c_int64, c_int32, c_int32,
                                                           c_void_p, c_int32, c_float, c_float, c_void_p, c_void_p,
                                                           c_void_p]
    lib.supcon_head_store_pool_forward_typed.restype = c_int32
    lib.supcon_head_store_pool_forward_typed.argtypes = [c_void_p, c_int32, ctypes.c_int64, c_int32, c_int32,
                                                         c_void_p, c_int32, c_float, c_float, c_void_p, c_void_p,
                                                         c_void_p]
    lib.supcon_head_sharded_store_pool_forward_typed.restype = c_int32
    lib.supcon_head_sharded_store_pool_forward_typed.argtypes = [c_void_p, c_int32, c_int32, ctypes.c_int64,
                                                                 c_int32, c_int32, c_void_p, c_int32, c_float,
                                                                 c_float, c_void_p, c_void_p, c_void_p]
    lib.supcon_label_keys.restype = c_int32
    lib.supcon_label_keys.argtypes = [c_void_p, c_int32, c_int32, c_void_p, c_void_p]
    PP = POINTER(Peer)
    lib.supcon_peer_push.restype = c_int32
    lib.supcon_peer_push.argtypes = [PP, c_void_p, c_size_t, ctypes.c_uint64, c_void_p, c_size_t, ctypes.c_uint64,
                                     c_int32, c_int32, c_int32, c_void_p]
    lib.supcon_peer_wait.restype = c_int32
    lib.supcon_peer_wait.argtypes = [PP, c_int32, c_void_p]
    lib.supcon_peer_end_step.restype = c_int32
    lib.supcon_peer_end_step.argtypes = [PP, c_int32, c_void_p]
    if lib.supcon_abi_version() != ABI_VERSION:
        raise RuntimeError("libsupcon_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().supcon_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")
