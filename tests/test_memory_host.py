"""CPU: the cross-batch memory flag in the C ABI, its validation, the ring bookkeeping of CrossBatchMemory, and the
fp64 reference of the loss with a memory (tests/memory_ref.py) against the oracle."""
import ctypes
import os
import re

import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT
from memory_ref import memory_loss
from oracle import supcon_oracle as O


def test_memory_flag_in_header_and_binding():
    from wav2vec_contr_loss_b200 import _cabi
    text = open(os.path.join(ROOT, "include", "supcon_b200.h")).read()
    m = re.search(r"#define\s+SUPCON_FLAG_MEMORY_COLUMNS\s+(\d+)u", text)
    assert m and int(m.group(1)) == 1024 == _cabi.FLAG_MEMORY_COLUMNS
    assert re.search(r"#define\s+SUPCON_ABI_VERSION\s+3\b", text) and _cabi.ABI_VERSION == 3


def _ws(lib, prob):
    nbytes = ctypes.c_size_t(0)
    rc = lib.supcon_workspace_bytes(ctypes.byref(prob), ctypes.byref(nbytes))
    return rc, nbytes.value


@pytest.mark.parametrize("dtype_id", [0, 1])
def test_memory_problem_validation_without_gpu(lib_built, dtype_id):
    from wav2vec_contr_loss_b200 import _cabi
    from wav2vec_contr_loss_b200.functional import make_problem
    lib = _cabi.load()
    mem = _cabi.FLAG_MEMORY_COLUMNS | _cabi.FLAG_UNIT_ROWS
    ok = make_problem(64 + 4096, 256, dtype_id, tau=0.07, similarity=_cabi.COSINE, n_rows=64, flags=mem,
                      lambda_uni=0.2, uni_t=2.0)
    rc, n = _ws(lib, ok)
    assert rc == 0 and n >= 256
    bad = make_problem(64 + 4096, 256, dtype_id, tau=0.07, similarity=_cabi.COSINE, row_offset=64, n_rows=64,
                       flags=mem)
    assert _ws(lib, bad)[0] == -1 and b"row_offset" in lib.supcon_last_error()
    bad = make_problem(64 + 4096, 256, dtype_id, tau=0.07, similarity=_cabi.COSINE, n_rows=64, flags=mem,
                       lambda_uni=0.2, uni_t=0.0)
    assert _ws(lib, bad)[0] == -1 and b"uni_t" in lib.supcon_last_error()
    # the same shape without the flag is a plain row block (a rank's share): valid as before
    plain = make_problem(64 + 4096, 256, dtype_id, tau=0.07, similarity=_cabi.COSINE, row_offset=64, n_rows=64)
    assert _ws(lib, plain)[0] == 0


def test_memory_is_single_rank(lib_built):
    """finalize_sets of several ranks' partials is refused before any device work (the buffer pointers are
    never dereferenced)"""
    from wav2vec_contr_loss_b200 import _cabi
    from wav2vec_contr_loss_b200.functional import make_problem
    lib = _cabi.load()
    prob = make_problem(1088, 256, 1, tau=0.07, similarity=0, n_rows=64, flags=_cabi.FLAG_MEMORY_COLUMNS)
    rc = lib.supcon_finalize_sets(ctypes.byref(prob), ctypes.c_void_p(16), 2, ctypes.c_void_p(16), None, None)
    assert rc == -2 and b"single-rank" in lib.supcon_last_error()


def _simulate(size, batches):
    """expected ring contents (slot order) after enqueueing ``batches`` one by one"""
    ring, head, filled = [None] * size, 0, 0
    for rows in batches:
        rows = rows[-size:] if size else []
        for r in rows:
            ring[head] = r
            head = (head + 1) % size
            filled = min(filled + 1, size)
    return ring[:filled], head, filled


@pytest.mark.parametrize("size,b", [(10, 4), (7, 3), (5, 8), (0, 4)])
def test_ring_bookkeeping_on_cpu(size, b):
    from wav2vec_contr_loss_b200.memory import CrossBatchMemory
    mem = CrossBatchMemory(size)
    g = torch.Generator().manual_seed(size * 100 + b)
    batches, labs = [], []
    for step in range(5):
        z = torch.randn(b, 6, generator=g)
        y = torch.randint(0, 3, (b,), generator=g)
        mem.enqueue(z, y)
        batches.append(list(range(step * b, (step + 1) * b)))
        labs.append((z, y))
        want, head, filled = _simulate(size, batches)
        assert (mem.filled, mem.head) == (filled, head)
        all_z = torch.cat([z for z, _ in labs])
        all_y = torch.cat([y for _, y in labs])
        assert mem.embeddings.shape == (filled, 6)
        if filled:
            assert torch.equal(mem.embeddings, all_z[want])
            assert torch.equal(mem.keys, all_y[want].to(torch.int32))
    mem.reset()
    assert (mem.filled, mem.head, mem.label_dtype) == (0, 0, None) and mem.embeddings.shape == (0, 6)


def test_label_dtype_change_raises():
    from wav2vec_contr_loss_b200.memory import CrossBatchMemory
    mem = CrossBatchMemory(8)
    mem.enqueue(torch.randn(3, 4), torch.tensor([0, 1, 1]))
    with pytest.raises(ValueError, match="dtype"):
        mem.enqueue(torch.randn(3, 4), torch.tensor([0.0, 1.0, 1.0]))
    assert mem.filled == 3
    mem.reset()
    mem.enqueue(torch.randn(3, 4), torch.tensor([0.0, 1.0, 1.0]))   # an empty memory takes any dtype
    assert mem.label_dtype == torch.float32
    with pytest.raises(ValueError, match="width"):
        mem.enqueue(torch.randn(3, 5), torch.tensor([0.0, 1.0, 1.0]))


def test_module_without_grad_on_cpu_is_the_plain_loss():
    """evaluation (no graph) never touches the memory; like SupConBinaryLoss there is no CPU path"""
    from wav2vec_contr_loss_b200.memory import MemorySupConLoss
    m = MemorySupConLoss(0.07, "cosine", 0.2, memory_size=16)
    assert (m.tau, m.similarity, m.lambda_uni, m.uni_t, m.memory.size) == (0.07, "cosine", 0.2, 2.0, 16)
    assert m.kernel_flags == 0 and m.assume_unit_rows is None
    out = m(torch.randn(1, 8), torch.tensor([1]))
    assert out.item() == 0.0
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.randn(4, 8, requires_grad=True), torch.tensor([0, 1, 0, 1]))
    assert m.memory.filled == 0


CASES = [
    # sim, lam, K, alpha, classes
    ("cosine", 0.0, 15, 0.0, 2),
    ("cosine", 0.2, 15, 0.5, 2),
    ("geodesic", 0.2, 32, 1.0, 2),
    ("geodesic", 0.0, 4, 0.5, 3),
    ("cosine", 0.3, 0, 0.5, 5),
]


@pytest.mark.parametrize("sim,lam,k,alpha,classes", CASES)
def test_reference_without_memory_is_the_oracle(sim, lam, k, alpha, classes):
    x, y = O.make_inputs(48, 32, "iso", classes=classes, seed=7)
    z = F.normalize(x, dim=1).double()
    ref = memory_loss(z, y, tau=0.1, similarity=sim, lam=lam, t=2.0, topk=k, alpha=alpha)
    want = O.closed_form(z, y, temperature=0.1, similarity=sim, uniformity_weight=lam, uniformity_t=2.0,
                         topk_neg=k, alpha=alpha)
    assert abs(ref["loss"] - want["loss"]) < 1e-10
    assert float((ref["dz"] - want["dz"]).abs().max()) < 1e-10


@pytest.mark.parametrize("sim,k,classes,m", [("cosine", 15, 2, 100), ("geodesic", 32, 3, 77), ("cosine", 4, 2, 5)])
def test_reference_anchor_rows_match_the_oracle_row_block(sim, k, classes, m):
    """with a memory (lambda = 0) the anchors' statistics are those of rows [0, B) against the concatenated
    columns, and the loss follows from their partial sums"""
    b = 40
    x, y = O.make_inputs(b + m, 32, "clustered", classes=classes, seed=11)
    z = F.normalize(x, dim=1).double()
    ref = memory_loss(z[:b], y[:b], z[b:], y[b:], tau=0.1, similarity=sim, topk=k, alpha=0.5)
    sid = O.sim_id(sim)
    stats, partials = O.rowblock_forward(z, y, 0, b, tau=0.1, similarity=sid, topk=k)
    assert float((ref["lse"] - stats["lse"]).abs().max()) < 1e-10
    assert torch.equal(ref["npos"], stats["npos"]) and torch.equal(ref["nneg"], stats["nneg"])
    assert torch.equal(ref["thr_val"], stats["thr_val"]) and torch.equal(ref["thr_idx"], stats["thr_idx"])
    loss, _ = O.loss_from_partials(partials, b + m, alpha=0.5, lambda_uni=0.0)
    assert abs(ref["loss"] - loss) < 1e-10
