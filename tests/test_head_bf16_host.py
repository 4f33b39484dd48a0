"""CPU: argument checks of the typed entry points of the fused compression head (bf16 or fp32 hs,
supcon_head_pool_forward_typed / supcon_head_pool_backward_typed).  Every rejected call returns before any CUDA work,
so these run without a device."""
import ctypes

import pytest

from wav2vec_contr_loss_b200 import _cabi


@pytest.fixture()
def lib_and_buf(lib_built):
    buf = (ctypes.c_float * 16)()
    return _cabi.load(), ctypes.cast(buf, ctypes.c_void_p)


def test_typed_entries_reject_unknown_hs_dtype(lib_and_buf):
    lib, p = lib_and_buf
    fwd, bwd = lib.supcon_head_pool_forward_typed, lib.supcon_head_pool_backward_typed
    for dtype in (2, -1):
        assert fwd(p, dtype, 2, 3, 4, 5, 0.0, 0.01, None, p, None) == -1
        msg = lib.supcon_last_error()
        assert b"supcon_head_pool_forward_typed" in msg and b"hs_dtype" in msg
        assert bwd(p, dtype, 2, 3, 4, 5, 0.0, 0.01, None, p, p, None) == -1
        msg = lib.supcon_last_error()
        assert b"supcon_head_pool_backward_typed" in msg and b"hs_dtype" in msg


@pytest.mark.parametrize("dtype", [_cabi.F32, _cabi.BF16])
def test_typed_entries_reject_bad_arguments(lib_and_buf, dtype):
    lib, p = lib_and_buf
    fwd, bwd = lib.supcon_head_pool_forward_typed, lib.supcon_head_pool_backward_typed
    assert fwd(None, dtype, 2, 3, 4, 5, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == b"NULL buffer passed to supcon_head_pool_forward_typed"
    assert bwd(None, dtype, 2, 3, 4, 5, 0.0, 0.01, None, p, p, None) == -1
    assert lib.supcon_last_error() == b"NULL buffer passed to supcon_head_pool_backward_typed"
    assert fwd(p, dtype, 2, 3, 4, 5, 0.0, 0.01, None, None, None) == -1
    assert bwd(p, dtype, 2, 3, 4, 5, 0.0, 0.01, None, p, None, None) == -1
    assert bwd(p, dtype, 2, 3, 4, 5, 0.0, 0.01, None, None, p, None) == -1
    assert b"dpooled" in lib.supcon_last_error() and b"backward_typed" in lib.supcon_last_error()
    assert fwd(p, dtype, 2, 0, 4, 5, 0.0, 0.01, None, p, None) == -1 and b"bad shape" in lib.supcon_last_error()
    assert fwd(p, dtype, 2, 3, 4, 5, 1.0, 0.01, None, p, None) == -1 and b"dropout_p" in lib.supcon_last_error()
    assert fwd(p, dtype, 70000, 3, 4, 5, 0.0, 0.01, None, p, None) == -2 and b"65535" in lib.supcon_last_error()
    assert fwd(p, dtype, 2, 3, 4, 12289, 0.0, 0.01, None, p, None) == -2 and b"frames" in lib.supcon_last_error()
    with pytest.raises(RuntimeError, match="supcon_head_pool_forward_typed failed"):
        _cabi.check(fwd(None, dtype, 2, 3, 4, 5, 0.0, 0.01, None, p, None), "supcon_head_pool_forward_typed")


def test_untyped_entries_still_name_themselves(lib_and_buf):
    """the fp32 entry points are the SUPCON_F32 case of the typed ones, and their messages are their own"""
    lib, p = lib_and_buf
    assert lib.supcon_head_pool_forward(None, 2, 3, 4, 5, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == b"NULL buffer passed to supcon_head_pool_forward"
    assert lib.supcon_head_pool_backward(p, 2, 3, 4, 5, 0.0, 0.01, None, None, p, None) == -1
    assert lib.supcon_last_error() == b"NULL dpooled passed to supcon_head_pool_backward"
