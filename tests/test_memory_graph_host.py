"""CPU: the entry points that read a memory's fill level from device memory (supcon_forward_rows_memory /
supcon_backward_rows_memory) in the header and the binding, their argument checks, and the device copy of the ring
state of CrossBatchMemory."""
import ctypes
import os
import re

import pytest
import torch

from conftest import ROOT

ENTRY_POINTS = ("supcon_forward_rows_memory", "supcon_backward_rows_memory")


def test_memory_entry_points_in_header_and_binding(lib_built):
    from wav2vec_contr_loss_b200 import _cabi
    text = open(os.path.join(ROOT, "include", "supcon_b200.h")).read()
    for name in ENTRY_POINTS:
        assert re.search(r"\bint\s+%s\s*\(" % name, text), name
        assert name in _cabi.EXPORTS
        assert hasattr(_cabi.load(), name)
    assert _cabi.ABI_VERSION == 3 and _cabi.load().supcon_abi_version() == 3


def _call(lib, name, prob, mem_filled):
    """every buffer is a bogus non-NULL pointer: a call that reached the device would fault, not return -1"""
    bogus = ctypes.c_void_p(16)
    if name == "supcon_forward_rows_memory":
        return lib.supcon_forward_rows_memory(ctypes.byref(prob), bogus, bogus, mem_filled, bogus, bogus, bogus,
                                              bogus, 1 << 30, None)
    return lib.supcon_backward_rows_memory(ctypes.byref(prob), bogus, bogus, mem_filled, bogus, bogus, None, bogus,
                                           0, bogus, 1 << 30, None)


@pytest.mark.parametrize("name", ENTRY_POINTS)
@pytest.mark.parametrize("dtype_id", [0, 1])
def test_memory_entry_points_need_the_memory_flag(lib_built, name, dtype_id):
    from wav2vec_contr_loss_b200 import _cabi
    from wav2vec_contr_loss_b200.functional import make_problem
    lib = _cabi.load()
    plain = make_problem(64 + 4096, 256, dtype_id, tau=0.07, similarity=_cabi.COSINE, n_rows=64,
                         flags=_cabi.FLAG_UNIT_ROWS)
    for mem_filled in (None, ctypes.c_void_p(16)):
        assert _call(lib, name, plain, mem_filled) == -1
        assert b"SUPCON_FLAG_MEMORY_COLUMNS" in lib.supcon_last_error()
    # with the flag, the problem is validated as for the plain calls (row_offset must be 0)
    bad = make_problem(64 + 4096, 256, dtype_id, tau=0.07, similarity=_cabi.COSINE, row_offset=64, n_rows=64,
                       flags=_cabi.FLAG_MEMORY_COLUMNS)
    assert _call(lib, name, bad, None) == -1 and b"row_offset" in lib.supcon_last_error()


def test_null_fill_level_is_a_full_memory(lib_built):
    """mem_filled == NULL is accepted: the call is the plain one.  A NULL z reaches the plain call's NULL check
    (its message names the memory entry point), before any device work."""
    from wav2vec_contr_loss_b200 import _cabi
    from wav2vec_contr_loss_b200.functional import make_problem
    lib = _cabi.load()
    prob = make_problem(64 + 4096, 256, 1, tau=0.07, similarity=_cabi.COSINE, n_rows=64,
                        flags=_cabi.FLAG_MEMORY_COLUMNS | _cabi.FLAG_UNIT_ROWS)
    bogus = ctypes.c_void_p(16)
    rc = lib.supcon_forward_rows_memory(ctypes.byref(prob), None, bogus, None, bogus, bogus, bogus, bogus, 1 << 30,
                                        None)
    assert rc == -1 and b"NULL buffer passed to supcon_forward_rows_memory" in lib.supcon_last_error()
    rc = lib.supcon_backward_rows_memory(ctypes.byref(prob), None, bogus, None, bogus, bogus, None, bogus, 0, bogus,
                                         1 << 30, None)
    assert rc == -1 and b"NULL buffer passed to supcon_backward_rows_memory" in lib.supcon_last_error()


def _check_state(mem):
    assert mem.state.dtype == torch.int32
    assert mem.state.tolist() == [mem.head, mem.filled]


@pytest.mark.parametrize("size", [0, 1, 7, 40])
def test_device_state_follows_the_host_state_on_cpu(size):
    from wav2vec_contr_loss_b200.memory import CrossBatchMemory
    mem = CrossBatchMemory(size)
    g = torch.Generator().manual_seed(size)
    ring, head, filled = [None] * size, 0, 0          # the slots the host-side bookkeeping names
    for n in (3, 16, 1, 45, size + 5, 2, 0, 9):       # batches smaller and larger than the ring, and empty
        z = torch.randn(n, 5, generator=g)
        y = torch.randint(0, 3, (n,), generator=g)
        mem.enqueue(z, y)
        _check_state(mem)
        if size:
            rows = list(zip(z, y.tolist()))[-size:]   # a batch larger than the ring: its newest rows, from head on
            for k, r in enumerate(rows):
                ring[(head + k) % size] = r
            head, filled = (head + len(rows)) % size, min(filled + len(rows), size)
        assert (mem.head, mem.filled) == (head, filled)
        if filled:
            assert torch.equal(mem.embeddings, torch.stack([r for r, _ in ring[:filled]]))
            assert mem.keys.tolist() == [y for _, y in ring[:filled]]
    mem.reset()
    _check_state(mem)
    assert mem.state.tolist() == [0, 0]


def test_buffers_are_zero_filled_and_snapshot_restores_state():
    from wav2vec_contr_loss_b200.memory import CrossBatchMemory
    mem = CrossBatchMemory(10)
    mem.enqueue(torch.ones(4, 3), torch.zeros(4, dtype=torch.int64))
    assert torch.equal(mem._z[mem._slots + 4:], torch.zeros(6, 3))   # absent slots: finite
    snap = mem.snapshot()
    emb = mem.embeddings.clone()
    for _ in range(3):
        mem.enqueue(torch.full((4, 3), 2.0), torch.ones(4, dtype=torch.int64))
    assert (mem.filled, mem.head) == (10, 6)
    mem.restore(snap)
    assert (mem.filled, mem.head) == (4, 4)
    _check_state(mem)
    assert torch.equal(mem.embeddings, emb) and mem.keys.tolist() == [0] * 4
