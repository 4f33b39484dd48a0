"""GPU: SupCon with a cross-batch memory (SUPCON_FLAG_MEMORY_COLUMNS, MemorySupConLoss) against the fp64 autograd
reference of tests/memory_ref.py: exact fp32 path 1e-5, bf16 tensor-core path 2e-3, hard-negative index sets exact."""
import pytest
import torch
import torch.nn.functional as F

import gpu_util as G
from memory_ref import memory_loss
from oracle import supcon_oracle as O

pytestmark = pytest.mark.gpu

TOL_F32 = 1e-5
TOL_BF16 = 2e-3


def _inputs(b, m, d=256, classes=2, seed=0):
    g = torch.Generator().manual_seed(seed)
    z = F.normalize(torch.randn(b + m, d, generator=g), dim=1)
    if classes == 2:
        y = torch.cat([torch.arange(b) % 2, torch.randint(0, 2, (m,), generator=g)])
    else:
        y = torch.randint(0, classes, (b + m,), generator=g)
    return z[:b], y[:b], z[b:], y[b:]


def _kernel(zb, yb, zm, ym, *, dtype, flags, tau, sim, lam, k, alpha, t=2.0, want_idx=False):
    """forward_rows + backward_rows (+ topk_indices) of the batch rows against batch + memory, via the C ABI"""
    from wav2vec_contr_loss_b200 import _cabi
    from wav2vec_contr_loss_b200 import functional as Fn
    dev = torch.device("cuda:0")
    z_all = torch.cat([zb, zm]).to(dev, dtype).contiguous()
    n, d = z_all.shape
    y_all = Fn.canonical_labels(torch.cat([yb, ym]).to(dev), n)
    prob = Fn.make_problem(n, d, Fn._dtype_id(z_all), tau=tau, similarity=Fn.similarity_id(sim), lambda_uni=lam,
                           uni_t=t, topk=k, alpha=alpha, n_rows=zb.size(0), flags=flags | _cabi.FLAG_MEMORY_COLUMNS)
    stats, partials, loss = Fn.forward_rows(z_all, y_all, prob, want_loss=True)
    dz = Fn.backward_rows(z_all, y_all, stats, partials, None, prob, out_dtype=torch.float32)
    idx = Fn.topk_indices(z_all, y_all, stats, prob) if want_idx else None
    torch.cuda.synchronize()
    return dict(loss=float(loss), dz=dz.double().cpu(), stats=stats.cpu(), partials=partials.cpu(),
                idx=None if idx is None else idx.cpu(), prob=prob)


def _index_sets(member, k):
    out = torch.full((member.size(0), k), -1, dtype=torch.int64)
    for i in range(member.size(0)):
        cols = torch.nonzero(member[i]).view(-1)[:k]
        out[i, :cols.numel()] = cols
    return out


# K > 32 runs only on the exact path: 64 keeps one top-K list per column split and merges them (M >= 1000), 129
# takes two selection rounds over one sweep
EXACT_PATH_MEMORY, EXACT_PATH_TOPK = [0, 1000, 4096], [15, 32, 64, 129]


@pytest.mark.parametrize("m", EXACT_PATH_MEMORY)
@pytest.mark.parametrize("sim", ["cosine", "geodesic"])
@pytest.mark.parametrize("lam", [0.0, 0.2])
@pytest.mark.parametrize("k", EXACT_PATH_TOPK)
@pytest.mark.parametrize("alpha", [0.0, 0.5, 1.0])
def test_exact_path_fp32(cuda_device, m, sim, lam, k, alpha):
    zb, yb, zm, ym = _inputs(64, m, seed=m + k)
    kw = dict(tau=0.07, sim=sim, lam=lam, k=k, alpha=alpha)
    out = _kernel(zb, yb, zm, ym, dtype=torch.float32, flags=0, want_idx=alpha > 0, **kw)
    ref = memory_loss(zb, yb, zm, ym, tau=0.07, similarity=sim, lam=lam, t=2.0, topk=k, alpha=alpha)
    assert out["loss"] == pytest.approx(ref["loss"], rel=TOL_F32)
    assert G.rel_err(out["dz"], ref["dz"]) < TOL_F32
    st = out["stats"].view(torch.int32)
    assert torch.equal(st[:, 2].long(), ref["npos"]) and torch.equal(st[:, 3].long(), ref["nneg"])
    if alpha > 0:
        assert torch.equal(out["idx"].long(), _index_sets(ref["member"], k))   # memory indices included


def test_exact_path_fp32_ragged(cuda_device):
    """B = 37 anchors of width 200 (no vector loads, partial tiles everywhere)"""
    zb, yb, zm, ym = _inputs(37, 1000, d=200, seed=5)
    kw = dict(tau=0.07, sim="cosine", lam=0.2, k=15, alpha=0.5)
    out = _kernel(zb, yb, zm, ym, dtype=torch.float32, flags=0, want_idx=True, **kw)
    ref = memory_loss(zb, yb, zm, ym, tau=0.07, similarity="cosine", lam=0.2, t=2.0, topk=15, alpha=0.5)
    assert out["loss"] == pytest.approx(ref["loss"], rel=TOL_F32)
    assert G.rel_err(out["dz"], ref["dz"]) < TOL_F32
    assert torch.equal(out["idx"].long(), _index_sets(ref["member"], 15))


TC_CASES = [(b, m, c) for b in (64, 300) for m in (1024, 8192) for c in (2, 40)]


@pytest.mark.parametrize("b,m,classes", TC_CASES)
@pytest.mark.parametrize("lam", [0.0, 0.2])
@pytest.mark.parametrize("class_sums", [False, True])
def test_tensor_path_bf16(cuda_device, b, m, classes, lam, class_sums):
    """FORCE_TENSOR | UNIT_ROWS; CLASS_SUMS pins the forward's class-sum route (its per-pair twin with 40 classes);
    the backward always takes the per-pair sweep with a memory"""
    from wav2vec_contr_loss_b200 import _cabi
    zb, yb, zm, ym = _inputs(b, m, classes=classes, seed=b + m + classes)
    zb, zm = zb.to(torch.bfloat16).float(), zm.to(torch.bfloat16).float()
    flags = _cabi.FLAG_FORCE_TENSOR | _cabi.FLAG_UNIT_ROWS | (_cabi.FLAG_CLASS_SUMS if class_sums else 0)
    out = _kernel(zb, yb, zm, ym, dtype=torch.bfloat16, flags=flags, tau=0.07, sim="cosine", lam=lam, k=15, alpha=0.0)
    ref = memory_loss(zb, yb, zm, ym, tau=0.07, similarity="cosine", lam=lam, t=2.0, topk=15, alpha=0.0)
    assert out["loss"] == pytest.approx(ref["loss"], rel=TOL_BF16)
    assert G.rel_err(out["dz"], ref["dz"]) < TOL_BF16
    assert torch.equal(out["stats"].view(torch.int32)[:, 2].long(), ref["npos"])
    p = out["partials"]
    assert p[5] == p[1] and p[6] == p[3]      # SUPCON_P_GCNT_* count the anchors, as SUPCON_P_CNT_* do


@pytest.mark.parametrize("b,m,classes,sim,lam,k,alpha", [
    (64, 8192, 2, "cosine", 0.0, 15, 0.5),
    (300, 1024, 40, "cosine", 0.2, 32, 1.0),
    (64, 4096, 2, "geodesic", 0.2, 15, 0.5),
])
def test_tensor_path_bf16_mining(cuda_device, b, m, classes, sim, lam, k, alpha):
    from wav2vec_contr_loss_b200 import _cabi
    zb, yb, zm, ym = _inputs(b, m, classes=classes, seed=7 * b + m)
    zb, zm = zb.to(torch.bfloat16).float(), zm.to(torch.bfloat16).float()
    flags = _cabi.FLAG_FORCE_TENSOR | _cabi.FLAG_UNIT_ROWS
    out = _kernel(zb, yb, zm, ym, dtype=torch.bfloat16, flags=flags, tau=0.07, sim=sim, lam=lam, k=k, alpha=alpha)
    ref = memory_loss(zb, yb, zm, ym, tau=0.07, similarity=sim, lam=lam, t=2.0, topk=k, alpha=alpha)
    assert out["loss"] == pytest.approx(ref["loss"], rel=TOL_BF16)
    assert G.rel_err(out["dz"], ref["dz"]) < TOL_BF16


def _expected_ring(size, rows):
    """slot contents after enqueueing ``rows`` in order, in batches no larger than the ring"""
    ring, head = [None] * size, 0
    for r in rows:
        ring[head] = r
        head = (head + 1) % size
    return ring[:min(len(rows), size)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_module_three_steps(cuda_device, dtype):
    """each step equals the reference on the batch + the memory as it was before the call; after each step the
    memory holds the previous batches; evaluation leaves it alone; forward, forward, backward raises"""
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    from wav2vec_contr_loss_b200.memory import MemorySupConLoss
    dev = torch.device("cuda:0")
    b, size = 64, 1150                                   # 1150 % 64 != 0: the third step wraps around
    kw = dict(topk_neg=15, alpha=0.5)
    mod = MemorySupConLoss(0.07, "cosine", 0.2, 2.0, memory_size=size)
    tol = TOL_F32 if dtype == torch.float32 else TOL_BF16
    history = []                                         # (z row, label) of every sample that entered the memory
    if dtype == torch.bfloat16:
        mod.assume_unit_rows = True                      # batch + memory >= 256 rows: the tensor-core path
        z0, y0, _, _ = _inputs(1000, 0, seed=99)
        mod.memory.enqueue(z0.to(dev, dtype), y0.to(dev), unit_rows=True)
        history += [(z0[i].to(dtype).float(), int(y0[i])) for i in range(1000)]
    for step in range(3):
        zb, yb, _, _ = _inputs(b, 0, seed=step)
        snap_z = mod.memory.embeddings.float().cpu().clone() if mod.memory.filled else zb[:0]
        snap_y = mod.memory.keys.long().cpu().clone() if mod.memory.filled else yb[:0]
        z = zb.to(dev, dtype).requires_grad_(True)
        loss = mod(z, yb.to(dev), **kw)
        loss.backward()
        ref = memory_loss(z.detach().float().cpu(), yb, snap_z, snap_y, tau=0.07, similarity="cosine", lam=0.2,
                          t=2.0, topk=15, alpha=0.5)
        assert float(loss) == pytest.approx(ref["loss"], rel=tol)
        assert G.rel_err(z.grad.double().cpu(), ref["dz"]) < (tol if dtype == torch.float32 else 2 * tol)
        history += [(z.detach()[i].float().cpu(), int(yb[i])) for i in range(b)]
        want = _expected_ring(size, history)
        assert mod.memory.filled == len(want) == min(size, len(history))
        assert torch.equal(mod.memory.embeddings.float().cpu(), torch.stack([r for r, _ in want]))
        assert mod.memory.keys.long().cpu().tolist() == [y for _, y in want]

    zb, yb, _, _ = _inputs(b, 0, seed=10)
    z = zb.to(dev, dtype).requires_grad_(True)
    before = (mod.memory.filled, mod.memory.head, mod.memory.embeddings.clone())
    with torch.no_grad():
        ev = mod(z, yb.to(dev), **kw)
        plain = SupConBinaryLoss(0.07, "cosine", 0.2, 2.0)
        plain.assume_unit_rows = mod.assume_unit_rows
        assert float(ev) == float(plain(z, yb.to(dev), **kw))
    assert (mod.memory.filled, mod.memory.head) == before[:2] and torch.equal(mod.memory.embeddings, before[2])

    l1 = mod(z, yb.to(dev), **kw)
    zb2, yb2, _, _ = _inputs(b, 0, seed=11)
    l2 = mod(zb2.to(dev, dtype).requires_grad_(True), yb2.to(dev), **kw)
    with pytest.raises(RuntimeError):
        l1.backward()                    # its memory view was rewritten by the second call
    l2.backward()                        # the second call is intact and enqueues its batch
    assert mod.memory.filled == min(size, before[0] + b)
