"""GPU: a memory problem run at its capacity with the fill level read from device memory
(supcon_forward_rows_memory / supcon_backward_rows_memory) against the compacted problem and the fp64 reference of
tests/memory_ref.py, and GraphedHeadStep replays with a MemorySupConLoss against the same steps run eagerly."""
import copy

import pytest
import torch
import torch.nn.functional as F

import gpu_util as G
from memory_ref import memory_loss
from oracle.gen_host_golden import TinyHead

pytestmark = pytest.mark.gpu

TOL_F32 = 1e-5
TOL_BF16 = 2e-3
B, M = 64, 1100                        # capacity B + M = 1164
FILLS = [0, 1, B - 1, 1000, M]


def _setup(seed, dtype):
    """anchors, a full memory's rows, and the same labels everywhere; rows a call must treat as absent are made
    large (finite) and carry the anchors' labels, so any absent column that is counted moves the results"""
    g = torch.Generator().manual_seed(seed)
    z = F.normalize(torch.randn(B + M, 256, generator=g), dim=1).to(dtype).float()
    y = torch.cat([torch.arange(B) % 2, torch.randint(0, 2, (M,), generator=g)])
    junk = 30.0 * torch.randn(M, 256, generator=g)
    return z, y, junk


def _run(z_all, y_all, prob, mem_filled):
    from wav2vec_contr_loss_b200 import functional as Fn
    stats, partials, loss = Fn.forward_rows(z_all, y_all, prob, want_loss=True, mem_filled=mem_filled)
    dz = Fn.backward_rows(z_all, y_all, stats, partials, None, prob, out_dtype=torch.float32, mem_filled=mem_filled)
    torch.cuda.synchronize()
    return dict(loss=float(loss), dz=dz.double().cpu(), stats=stats.cpu())


def _problem(n_total, dtype, flags, sim, lam, k, alpha):
    from wav2vec_contr_loss_b200 import _cabi
    from wav2vec_contr_loss_b200 import functional as Fn
    return Fn.make_problem(n_total, 256, Fn._dtype_id(torch.empty(0, dtype=dtype)), tau=0.07,
                           similarity=Fn.similarity_id(sim), lambda_uni=lam, uni_t=2.0, topk=k, alpha=alpha, n_rows=B,
                           flags=flags | _cabi.FLAG_MEMORY_COLUMNS)


def _routes():
    from wav2vec_contr_loss_b200 import _cabi
    return {"exact_fp32": (torch.float32, _cabi.FLAG_FORCE_EXACT, TOL_F32),
            "tensor_bf16": (torch.bfloat16, _cabi.FLAG_FORCE_TENSOR | _cabi.FLAG_UNIT_ROWS, TOL_BF16)}


@pytest.mark.parametrize("route", ["exact_fp32", "tensor_bf16"])
@pytest.mark.parametrize("sim", ["cosine", "geodesic"])
@pytest.mark.parametrize("lam", [0.0, 0.2])
@pytest.mark.parametrize("k", [0, 15, 32])
@pytest.mark.parametrize("alpha", [0.0, 0.5, 1.0])
def test_fill_level_equals_compacted_problem(cuda_device, route, sim, lam, k, alpha):
    dtype, flags, tol = _routes()[route]
    dev = cuda_device
    from wav2vec_contr_loss_b200 import functional as Fn
    z, y, junk = _setup(len(route) + 3 * len(sim) + int(10 * lam) + 7 * k + int(4 * alpha), dtype)
    cap = _problem(B + M, dtype, flags, sim, lam, k, alpha)
    for f in FILLS:
        zc, yc = z.clone(), y.clone()
        zc[B + f:] = junk[f:]
        yc[B + f:] = y[torch.arange(B + f, B + M) % B]
        z_all = zc.to(dev, dtype).contiguous()
        y_all = Fn.canonical_labels(yc.to(dev), B + M)
        filled = torch.tensor([f], dtype=torch.int32, device=dev)
        got = _run(z_all, y_all, cap, filled)
        ref = memory_loss(zc[:B], yc[:B], zc[B:B + f], yc[B:B + f], tau=0.07, similarity=sim, lam=lam, t=2.0,
                          topk=k, alpha=alpha)
        assert got["loss"] == pytest.approx(ref["loss"], rel=tol), f
        assert G.rel_err(got["dz"], ref["dz"]) < tol, f
        st = got["stats"].view(torch.int32)
        assert torch.equal(st[:, 2].long(), ref["npos"]) and torch.equal(st[:, 3].long(), ref["nneg"]), f
        if dtype == torch.bfloat16 and B + f < 256:
            continue                                   # the compacted problem is below the tensor path's minimum
        want = _run(z_all[:B + f].contiguous(), y_all[:B + f].contiguous(),
                    _problem(B + f, dtype, flags, sim, lam, k, alpha), None)
        gs, ws = got["stats"], want["stats"]
        for col in (2, 3, 5):                          # npos, nneg, thr_idx: exactly
            assert torch.equal(gs.view(torch.int32)[:, col], ws.view(torch.int32)[:, col]), (f, col)
        assert torch.equal(gs[:, 4], ws[:, 4]), f      # thr_val: exactly
        assert G.rel_err(gs[:, 0].double(), ws[:, 0].double()) < 1e-5, f
        assert got["loss"] == pytest.approx(want["loss"], rel=1e-5), f
        assert G.rel_err(got["dz"], want["dz"]) < 1e-5, f


@pytest.mark.parametrize("route", ["exact_fp32", "tensor_bf16"])
def test_fill_level_out_of_range_is_nan(cuda_device, route):
    dtype, flags, tol = _routes()[route]
    from wav2vec_contr_loss_b200 import functional as Fn
    z, y, _ = _setup(3, dtype)
    z_all = z.to(cuda_device, dtype).contiguous()
    y_all = Fn.canonical_labels(y.to(cuda_device), B + M)
    for sim, alpha in (("cosine", 0.5), ("geodesic", 0.0)):
        cap = _problem(B + M, dtype, flags, sim, 0.2, 15, alpha)
        for f in (-1, M + 1, -(2 ** 31)):
            got = _run(z_all, y_all, cap, torch.tensor([f], dtype=torch.int32, device=cuda_device))
            assert got["loss"] != got["loss"], (sim, f)
            assert torch.isnan(got["dz"]).all(), (sim, f)
        ok = _run(z_all, y_all, cap, torch.tensor([M], dtype=torch.int32, device=cuda_device))   # device still fine
        full = _run(z_all, y_all, cap, None)
        assert ok["loss"] == pytest.approx(full["loss"], rel=1e-6) and G.rel_err(ok["dz"], full["dz"]) < 1e-5


def _step_problem(device, batch, dim, steps, seed=5):
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    head = TinyHead(feat=32, dim=dim).to(device)
    hs = torch.randn(steps, batch, 3, 32, 10, generator=g)
    y = torch.stack([torch.randperm(batch, generator=g) % 2 for _ in range(steps)])
    hs = hs + 0.5 * (2.0 * y.view(steps, batch, 1, 1, 1) - 1.0)
    return head, hs.to(device), y.to(device)


def _flat(module):
    return torch.cat([p.detach().reshape(-1) for p in module.parameters()]).double().cpu()


def _mem_state(mem):
    return (mem.filled, mem.head, mem.embeddings.float().cpu().clone(), mem.keys.cpu().clone())


def _twins(device, batch, dim, size, steps, dtype, sim):
    from wav2vec_contr_loss_b200 import functional as Fn
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.memory import MemorySupConLoss
    head_e, hs, y = _step_problem(device, batch, dim, steps)
    head_g = copy.deepcopy(head_e)
    loss_e = MemorySupConLoss(0.1, sim, 0.1, 2.0, memory_size=size)
    loss_g = MemorySupConLoss(0.1, sim, 0.1, 2.0, memory_size=size)
    normalize = (lambda x: Fn.l2_normalize(x, dtype)) if dtype != torch.float32 else None
    # AdamW moves every weight by about lr whatever the gradient's size: where the bf16 tensor path and the eager
    # twin's exact path differ in a gradient's sign, the weights differ by up to 2 lr.  bf16 takes a small lr.
    lr = 5e-3 if dtype == torch.float32 else 1e-5
    opt_e = torch.optim.AdamW(head_e.parameters(), lr=lr, weight_decay=3e-3, capturable=True)
    opt_g = torch.optim.AdamW(head_g.parameters(), lr=lr, weight_decay=3e-3, capturable=True)

    def eager(s, alpha):
        z = S.embed(head_e, hs[s], normalize)
        loss = loss_e(z, y[s], topk_neg=7, alpha=alpha)
        opt_e.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(head_e.parameters(), 5.0)
        opt_e.step()
        return float(loss)

    step = S.GraphedHeadStep(head_g, loss_g, opt_g, hs[0], y[0], topk_neg=7, normalize=normalize)
    return head_e, head_g, loss_e, loss_g, hs, y, eager, step


@pytest.mark.parametrize("dtype,batch,dim,size,tol", [
    (torch.float32, 16, 16, 40, TOL_F32),             # empty, filling, full, wrapping: 16 + 16 + 8 | 8 + ...
    (torch.bfloat16, 64, 256, 300, TOL_BF16),         # capacity 364 >= 256: the replays take the tensor path
])
@pytest.mark.parametrize("sim", ["cosine", "geodesic"])
def test_graphed_memory_steps_equal_eager_steps(cuda_device, dtype, batch, dim, size, tol, sim):
    steps = 7
    head_e, head_g, loss_e, loss_g, hs, y, eager, step = _twins(cuda_device, batch, dim, size, steps, dtype, sim)
    alphas = [0.0, 0.5, 0.5, 0.0, 0.5, 0.5, 0.5]
    for s, alpha in enumerate(alphas):
        want = eager(s, alpha)
        got = float(step(hs[s], y[s], alpha))
        assert got == pytest.approx(want, rel=tol), s
        assert torch.allclose(_flat(head_g), _flat(head_e), rtol=1e-4 if dtype == torch.float32 else tol,
                              atol=1e-6 if dtype == torch.float32 else 1e-5), s
        ge, ee = _mem_state(loss_g.memory), _mem_state(loss_e.memory)
        assert ge[:2] == ee[:2] == (min((s + 1) * batch, size), (s + 1) * batch % size), s
        assert loss_g.memory.state.tolist() == [ge[1], ge[0]], s
        assert torch.equal(ge[3], ee[3]), s
        assert G.rel_err(ge[2].double(), ee[2].double()) < (TOL_F32 if dtype == torch.float32 else tol), s


def test_capture_leaves_the_memory_as_it_was(cuda_device):
    from wav2vec_contr_loss_b200 import stage1 as S
    from wav2vec_contr_loss_b200.memory import MemorySupConLoss
    head, hs, y = _step_problem(cuda_device, 16, 16, 3)
    loss_fn = MemorySupConLoss(0.1, "cosine", memory_size=40)
    opt = torch.optim.AdamW(head.parameters(), lr=5e-3, capturable=True)
    step = S.GraphedHeadStep(head, loss_fn, opt, hs[0], y[0], topk_neg=7)
    step._graphs[0.0] = step._capture(0.0)         # empty memory: warm-up and capture enqueue nothing that stays
    assert (loss_fn.memory.filled, loss_fn.memory.head) == (0, 0)
    assert loss_fn.memory.state.tolist() == [0, 0]
    step(hs[0], y[0], 0.0)
    before = _mem_state(loss_fn.memory)
    params = _flat(head)
    step._graphs[0.5] = step._capture(0.5)         # a partly filled memory, contents included
    after = _mem_state(loss_fn.memory)
    assert before[:2] == after[:2] == (16, 16) and loss_fn.memory.state.tolist() == [16, 16]
    assert torch.equal(before[2], after[2]) and torch.equal(before[3], after[3])
    assert torch.equal(_flat(head), params)


def test_two_alphas_share_one_memory(cuda_device):
    """graphs of alpha 0 and 0.5 replayed alternately enqueue into one ring, in replay order"""
    head_e, head_g, loss_e, loss_g, hs, y, eager, step = _twins(cuda_device, 16, 16, 40, 6, torch.float32, "cosine")
    for s in range(6):
        alpha = 0.5 * (s % 2)
        want = eager(s, alpha)
        assert float(step(hs[s], y[s], alpha)) == pytest.approx(want, rel=TOL_F32), s
    assert len(step._graphs) == 2
    ge, ee = _mem_state(loss_g.memory), _mem_state(loss_e.memory)
    assert ge[:2] == ee[:2] == (40, 96 % 40)
    assert torch.equal(ge[3], ee[3]) and G.rel_err(ge[2].double(), ee[2].double()) < TOL_F32
