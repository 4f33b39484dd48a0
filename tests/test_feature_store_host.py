"""CPU: the layer-mean store (wav2vec_contr_loss_b200.feature_store, supcon_head_layer_mean_typed /
supcon_head_store_pool_forward): declarations and exports, argument checks that return before any CUDA work, the
store's slot / shape / label bookkeeping and the epoch functions' refusal of a stale store."""
import ctypes
import os
from types import SimpleNamespace

import pytest
import torch

from wav2vec_contr_loss_b200 import _cabi

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "supcon_b200.h")
NEW = ("supcon_head_layer_mean_typed", "supcon_head_store_pool_forward")


@pytest.fixture()
def lib_and_buf(lib_built):
    buf = (ctypes.c_float * 16)()
    return _cabi.load(), ctypes.cast(buf, ctypes.c_void_p)


def test_entries_declared_exported_and_abi_unchanged(lib_built):
    text = open(HEADER).read()
    lib = _cabi.load()
    for name in NEW:
        assert f"int {name}(" in text
        assert name in _cabi.EXPORTS
        assert hasattr(lib, name)
    assert lib.supcon_abi_version() == _cabi.ABI_VERSION == 3


def test_layer_mean_rejects_bad_arguments(lib_and_buf):
    lib, p = lib_and_buf
    fn = lib.supcon_head_layer_mean_typed
    who = b"supcon_head_layer_mean_typed"
    assert fn(None, _cabi.F32, 2, 3, 4, 5, p, None) == -1
    assert lib.supcon_last_error() == b"NULL buffer passed to " + who
    assert fn(p, _cabi.BF16, 2, 3, 4, 5, None, None) == -1
    assert lib.supcon_last_error() == b"NULL buffer passed to " + who
    for dtype in (2, -1):
        assert fn(p, dtype, 2, 3, 4, 5, p, None) == -1
        assert who in lib.supcon_last_error() and b"hs_dtype" in lib.supcon_last_error()
    for shape in ((0, 3, 4, 5), (2, 0, 4, 5), (2, 3, 0, 5), (2, 3, 4, 0)):
        assert fn(p, _cabi.F32, *shape, p, None) == -1
        assert lib.supcon_last_error() == who + b": bad shape (%d, %d, %d, %d)" % shape
    assert fn(p, _cabi.F32, 70000, 3, 4, 5, p, None) == -2 and b"65535" in lib.supcon_last_error()
    assert fn(p, _cabi.F32, 2, 3, 4, 12289, p, None) == -2 and b"frames" in lib.supcon_last_error()
    with pytest.raises(RuntimeError, match="supcon_head_layer_mean_typed failed"):
        _cabi.check(fn(None, _cabi.F32, 2, 3, 4, 5, p, None), "supcon_head_layer_mean_typed")


def test_store_pool_rejects_bad_arguments(lib_and_buf):
    lib, p = lib_and_buf
    fn = lib.supcon_head_store_pool_forward
    who = b"supcon_head_store_pool_forward"
    #        store, n_store, F, T, idx, B, p, slope, rng, pooled, stream
    assert fn(None, 10, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == b"NULL buffer passed to " + who
    assert fn(p, 10, 4, 5, p, 2, 0.0, 0.01, None, None, None) == -1
    assert lib.supcon_last_error() == b"NULL buffer passed to " + who
    assert fn(p, 10, 4, 5, None, 2, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == b"NULL idx passed to " + who
    assert fn(p, 0, 4, 5, p, 2, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == who + b": bad store size 0"
    assert fn(p, 10, 4, 5, p, 0, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == who + b": bad shape (0, 1, 4, 5)"
    assert fn(p, 10, 0, 5, p, 2, 0.0, 0.01, None, p, None) == -1 and b"bad shape" in lib.supcon_last_error()
    for bad_p in (1.0, -0.1, float("nan")):
        assert fn(p, 10, 4, 5, p, 2, bad_p, 0.01, None, p, None) == -1
        assert lib.supcon_last_error() == who + b": dropout_p must be in [0, 1)"
    assert fn(p, 10, 4, 5, p, 70000, 0.0, 0.01, None, p, None) == -2 and b"65535" in lib.supcon_last_error()
    assert fn(p, 10, 4, 12289, p, 2, 0.0, 0.01, None, p, None) == -2 and b"frames" in lib.supcon_last_error()
    # n_store is 64-bit: a count past 2^31 is not truncated into a "bad store size"
    assert fn(p, 2 ** 33, 4, 5, p, 0, 0.0, 0.01, None, p, None) == -1
    assert lib.supcon_last_error() == who + b": bad shape (0, 1, 4, 5)"


def test_store_bookkeeping():
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore, store_bytes
    s = LayerMeanStore(6, 8, 5, "cpu")
    assert (s.n, s.feat, s.frames, s.filled) == (6, 8, 5, 0)
    assert s.rows.shape == (6, 8, 5) and s.rows.dtype == torch.float32
    assert s.labels.shape == (6,) and s.labels.dtype == torch.int64 and s.labels.tolist() == [-1] * 6
    assert store_bytes(6, 8, 5) == 6 * 8 * 5 * 4 + 6 * 8
    assert store_bytes(25000, 1024, 199) > 2 ** 31 * 4        # 64-bit sizes: about 20 GB of rows
    with pytest.raises(ValueError, match="bad store shape"):
        LayerMeanStore(0, 8, 5, "cpu")
    # every shape check comes before the device check, so a wrong clip is named even off the GPU
    with pytest.raises(ValueError, match=r"\(F, T\) = \(8, 6\), the store holds \(8, 5\)"):
        s.append(torch.zeros(2, 3, 8, 6), torch.zeros(2))
    with pytest.raises(ValueError, match="labels must be"):
        s.append(torch.zeros(2, 3, 8, 5), torch.zeros(3))
    with pytest.raises(ValueError, match="no room for 7 more"):
        s.append(torch.zeros(7, 3, 8, 5), torch.zeros(7))
    with pytest.raises(ValueError, match="batch, layers, feat, frames"):
        s.append(torch.zeros(3, 8, 5), torch.zeros(3))
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        s.append(torch.zeros(2, 3, 8, 5), torch.zeros(2))
    assert s.filled == 0
    # the slots [0, filled) are the valid ones: the label gather clamps into them
    s.labels[:3] = torch.tensor([1, 0, 1])
    s.filled = 3
    assert s.labels_of(torch.tensor([2, 0, -4, 9])).tolist() == [1, 1, 1, 1]
    assert s.labels_of(torch.tensor([1])).tolist() == [0]


def test_store_that_does_not_fit_is_refused(monkeypatch):
    from wav2vec_contr_loss_b200.feature_store import LayerMeanStore
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (10 ** 9, 180 * 10 ** 9))
    with pytest.raises(MemoryError, match="takes 20.38 GB; 1.00 GB are free"):
        LayerMeanStore(25000, 1024, 199, "cuda:0")


def test_epoch_functions_refuse_a_stale_store():
    from wav2vec_contr_loss_b200 import stage1 as S
    base = dict(topk_neg=3, warmup_epochs=0, alpha_ramp_epochs=1, alpha_end=1.0)
    fine = SimpleNamespace(finetune_encoder=True, use_rawboost=False, **base)
    boost = SimpleNamespace(finetune_encoder=False, use_rawboost=True, **base)
    for cfg, what in ((fine, "finetune_encoder"), (boost, "use_rawboost")):
        with pytest.raises(ValueError, match=what):
            S.train_one_epoch_from_store(None, None, None, [[0, 1]], None, "cpu", 1, cfg)
    with pytest.raises(ValueError, match="finetune_encoder"):
        S.evaluate_from_store(None, None, None, [[0, 1]], "cpu", fine)


def test_store_batches_outside_the_store_are_refused():
    from wav2vec_contr_loss_b200 import stage1 as S
    store = SimpleNamespace(filled=4)
    assert S._store_indices(store, [3, 0, 2], "cpu").tolist() == [3, 0, 2]
    for bad in ([0, 4], [-1, 2]):
        with pytest.raises(IndexError, match=r"\[0, 4\)"):
            S._store_indices(store, bad, "cpu")
