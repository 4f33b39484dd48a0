"""CPU: host side of the fused compression head (wav2vec_contr_loss_b200.head) - parameter names compatible with
the reference's CompressionModule checkpoints, no CPU path, launch-geometry rules of csrc/supcon_head.cu."""
import pytest
import torch

from wav2vec_contr_loss_b200 import FusedCompressionHead, layer_time_pool


def test_parameters_are_the_reference_modules():
    head = FusedCompressionHead(1024, 256, 0.1)
    assert list(head.state_dict().keys()) == ["mlp3.weight", "mlp3.bias"]     # compression_module.py:30-32
    assert head.mlp3.weight.shape == (256, 1024) and head.dropout_head.p == 0.1
    assert head.activation_head.negative_slope == 0.01
    assert "rng_state" not in head.state_dict() and head.rng_state.dtype == torch.int64


def test_dropout_stream_follows_manual_seed():
    torch.manual_seed(11)
    a = FusedCompressionHead(8, 4)
    torch.manual_seed(12)
    b = FusedCompressionHead(8, 4)
    assert a.rng_state.tolist() == [11, 0] and b.rng_state.tolist() == [12, 0]


def test_dropout_stream_can_be_reseeded_per_rank_and_checkpointed():
    """ADVICE r01: the stream is seeded at construction (documented), reseed() follows a later manual_seed and
    mixes a per-rank stream id, and its position survives a checkpoint without touching state_dict()."""
    torch.manual_seed(3)
    head = FusedCompressionHead(8, 4)
    torch.manual_seed(99)
    assert head.rng_state.tolist() == [3, 0]            # construction-time seed: manual_seed afterwards is inert ...
    head.reseed()
    assert head.rng_state.tolist() == [99, 0]           # ... until reseed()
    keys = set()
    for rank in range(4):
        head.reseed(seed=1337, stream=rank)
        keys.add(head.rng_state.tolist()[0])
    assert len(keys) == 4                               # same torch seed on every rank, different masks
    head.rng_state[1] = 41
    saved = head.dropout_stream_state()
    other = FusedCompressionHead(8, 4)
    other.load_dropout_stream_state(saved)
    assert other.rng_state.tolist() == head.rng_state.tolist() and saved[1] == 41
    assert list(head.state_dict().keys()) == ["mlp3.weight", "mlp3.bias"]


def test_no_cpu_path():
    head = FusedCompressionHead(8, 4, 0.0)
    hs = torch.randn(2, 3, 8, 5)
    for call in (lambda: head(hs), lambda: head.embed(hs), lambda: layer_time_pool(hs)):
        with pytest.raises((RuntimeError, ValueError, OSError)):
            call()


def test_c_abi_argument_validation_without_gpu(lib_built):
    """every rejected call returns before any CUDA work, so this runs on the CPU-only box"""
    import ctypes
    from wav2vec_contr_loss_b200 import _cabi
    lib = _cabi.load()
    buf = (ctypes.c_float * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    fwd, bwd = lib.supcon_head_pool_forward, lib.supcon_head_pool_backward
    assert fwd(None, 2, 3, 4, 5, 0.0, 0.01, None, p, None) == -1 and b"NULL" in lib.supcon_last_error()
    assert fwd(p, 2, 3, 4, 5, 0.0, 0.01, None, None, None) == -1
    assert fwd(p, 0, 3, 4, 5, 0.0, 0.01, None, p, None) == -1 and b"bad shape" in lib.supcon_last_error()
    assert fwd(p, 2, 3, 4, 5, 1.0, 0.01, None, p, None) == -1 and b"dropout_p" in lib.supcon_last_error()
    assert fwd(p, 2, 3, 4, 5, -0.1, 0.01, None, p, None) == -1
    assert fwd(p, 70000, 3, 4, 5, 0.0, 0.01, None, p, None) == -2 and b"65535" in lib.supcon_last_error()
    assert fwd(p, 2, 3, 4, 12289, 0.0, 0.01, None, p, None) == -2 and b"frames" in lib.supcon_last_error()
    assert bwd(p, 2, 3, 4, 5, 0.0, 0.01, None, None, p, None) == -1 and b"dpooled" in lib.supcon_last_error()
    assert bwd(p, 2, 3, 4, 5, 0.0, 0.01, None, p, None, None) == -1
    with pytest.raises(RuntimeError, match="supcon_head_pool_forward failed"):
        _cabi.check(fwd(None, 2, 3, 4, 5, 0.0, 0.01, None, p, None), "supcon_head_pool_forward")
