"""GPU: the fused compression head on bf16 encoder output (csrc/supcon_head.cu, head.py), read as it is.

bf16 elements are widened to fp32 exactly and the kernel's arithmetic after the load is the fp32 one, so the bf16
route must give bit for bit the fp32 route's pooled values on ``hs.float()``, and its d loss / d hs must be the fp32
route's rounded to bf16 - on the vector path and on every shape that takes the scalar one.  Through the module it is
checked against the reference's op chain (``reference_chain`` of test_head_gpu.py) on ``hs.float()``, for the absence
of an fp32 copy of hs, and inside a CUDA-graph step."""
import copy

import pytest
import torch

from test_head_gpu import TOL, make_head, reference_chain, rel
from wav2vec_contr_loss_b200 import _cabi
from wav2vec_contr_loss_b200 import functional as Fn

pytestmark = pytest.mark.gpu

CASES = [           # batch, layers, feat, frames, base pointer offset (elements); "vector" = 16-byte loads of 8 bf16
    (64, 25, 1024, 199, 0),    # the Stage-1 batch: vector
    (2, 3, 7, 13, 0),          # odd F and odd T: scalar
    (2, 2, 18, 199, 0),        # ragged last block of rows: scalar
    (2, 4, 24, 999, 0),        # T > 768, odd: 8 rows per block for bf16 (12 for fp32), vector
    (2, 3, 10, 1001, 0),       # T > 768, odd, plane not a multiple of 8: scalar
    (1, 2, 6, 3000, 0),        # long clip: 4 rows per block, vector
    (1, 2, 5, 3001, 0),        # long clip, odd: scalar
    (3, 5, 40, 64, 1),         # base pointer one element past a 16-byte boundary: scalar
    (4, 1, 256, 199, 0),       # K = 1 (layer-mean features)
    (1, 25, 1024, 199, 0),     # B = 1
]


def case_id(c):
    return "x".join(map(str, c[:4])) + (f"+{c[4]}" if c[4] else "")


def bf16_hs(shape, offset, device, seed=1):
    """bf16 (B, K, F, T) starting `offset` elements into its allocation"""
    n = 1
    for s in shape:
        n *= s
    flat = torch.randn(n + offset, generator=torch.Generator().manual_seed(seed)).to(device, torch.bfloat16)
    hs = flat[offset:].view(shape)
    assert hs.data_ptr() % 16 == 2 * (offset % 8)
    return hs


def pool_fwd(lib, hs, dtype, p, rng):
    b, k, f, t = hs.shape
    pooled = torch.empty((b, f), dtype=torch.float32, device=hs.device)
    if dtype == _cabi.F32:
        rc = lib.supcon_head_pool_forward(Fn._p(hs), b, k, f, t, p, 0.01, Fn._p(rng), Fn._p(pooled),
                                          Fn._stream(hs.device))
    else:
        rc = lib.supcon_head_pool_forward_typed(Fn._p(hs), dtype, b, k, f, t, p, 0.01, Fn._p(rng), Fn._p(pooled),
                                                Fn._stream(hs.device))
    _cabi.check(rc, "head pool forward")
    return pooled


def pool_bwd(lib, hs, dtype, p, rng, dpooled):
    b, k, f, t = hs.shape
    dhs = torch.empty_like(hs)
    if dtype == _cabi.F32:
        rc = lib.supcon_head_pool_backward(Fn._p(hs), b, k, f, t, p, 0.01, Fn._p(rng), Fn._p(dpooled), Fn._p(dhs),
                                           Fn._stream(hs.device))
    else:
        rc = lib.supcon_head_pool_backward_typed(Fn._p(hs), dtype, b, k, f, t, p, 0.01, Fn._p(rng), Fn._p(dpooled),
                                                 Fn._p(dhs), Fn._stream(hs.device))
    _cabi.check(rc, "head pool backward")
    return dhs


@pytest.mark.parametrize("p", [0.0, 0.1], ids=["eval", "dropout"])
@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_bf16_entry_is_bit_identical_to_fp32_entry_on_widened_hs(cuda_device, case, p):
    lib = _cabi.load()
    b, k, f, t, offset = case
    hs = bf16_hs((b, k, f, t), offset, cuda_device)
    wide = hs.float()
    rng = torch.tensor([987654321, 5], dtype=torch.int64, device=cuda_device) if p > 0 else None
    dpooled = torch.randn(b, f, generator=torch.Generator().manual_seed(2)).to(cuda_device)

    pooled = pool_fwd(lib, hs, _cabi.BF16, p, rng)
    pooled_ref = pool_fwd(lib, wide, _cabi.F32, p, rng)
    assert torch.equal(pooled, pooled_ref)

    dhs = pool_bwd(lib, hs, _cabi.BF16, p, rng, dpooled)
    dhs_ref = pool_bwd(lib, wide, _cabi.F32, p, rng, dpooled)
    assert dhs.dtype == torch.bfloat16
    assert torch.equal(dhs.view(torch.int16), dhs_ref.to(torch.bfloat16).view(torch.int16))
    if p > 0:     # the dropout really dropped: some (b, f, t) have a zero gradient in every layer
        assert bool((dhs_ref[:, 0] == 0).any())
    torch.cuda.synchronize()


def test_typed_f32_entry_equals_fp32_entry(cuda_device):
    lib = _cabi.load()
    hs = torch.randn(3, 5, 40, 64, generator=torch.Generator().manual_seed(4)).to(cuda_device)
    rng = torch.tensor([11, 3], dtype=torch.int64, device=cuda_device)
    dpooled = torch.randn(3, 40, device=cuda_device)
    b, k, f, t = hs.shape
    pooled = torch.empty((b, f), device=cuda_device)
    _cabi.check(lib.supcon_head_pool_forward_typed(Fn._p(hs), _cabi.F32, b, k, f, t, 0.1, 0.01, Fn._p(rng),
                                                   Fn._p(pooled), Fn._stream(cuda_device)), "fwd")
    dhs = torch.empty_like(hs)
    _cabi.check(lib.supcon_head_pool_backward_typed(Fn._p(hs), _cabi.F32, b, k, f, t, 0.1, 0.01, Fn._p(rng),
                                                    Fn._p(dpooled), Fn._p(dhs), Fn._stream(cuda_device)), "bwd")
    assert torch.equal(pooled, pool_fwd(lib, hs, _cabi.F32, 0.1, rng))
    assert torch.equal(dhs, pool_bwd(lib, hs, _cabi.F32, 0.1, rng, dpooled))


def bf16_ulps(a, b):
    """distance in bf16 steps between two bf16 tensors of one sign pattern (int16 bit patterns are monotone per sign)"""
    return (a.view(torch.int16).int() - b.view(torch.int16).int()).abs()


@pytest.mark.parametrize("shape", [(3, 25, 256, 199), (2, 3, 7, 13), (2, 5, 40, 50)], ids=lambda s: "x".join(map(str, s)))
def test_module_on_bf16_hs_equals_reference_ops(cuda_device, shape):
    """FusedCompressionHead on a bf16 hs (encoder fine-tuned, so d hs is computed) against the reference op chain in
    fp32 on hs.float(): values, d W and d b to test_head_gpu.py's 2e-5.  d hs comes back in bf16 and is compared with
    the reference's fp32 d hs rounded to bf16: the fp32 values differ in the last bits (sums reordered), which
    rounding to bf16 turns into a one-step difference where a value lies at a rounding boundary - so every element
    must be within one bf16 step and all but a sliver equal."""
    b, k, f, t = shape
    head = make_head(f, 16, 0.1, cuda_device).eval()
    hs = bf16_hs(shape, 0, cuda_device)
    w = torch.randn(b, 16, generator=torch.Generator().manual_seed(2)).to(cuda_device)

    hs_a = hs.clone().requires_grad_(True)
    feats = head.pooled_features(hs_a)
    seq1 = head(hs_a)
    z = head.embed(hs_a)
    (z * w).sum().backward()
    dhs = hs_a.grad
    grads = [head.mlp3.weight.grad.clone(), head.mlp3.bias.grad.clone()]
    head.zero_grad()
    assert dhs.dtype == torch.bfloat16 and dhs.shape == hs.shape

    hs_r = hs.float().requires_grad_(True)
    feats_r, pooled_r, z_r = reference_chain(hs_r, head.mlp3.weight, head.mlp3.bias)
    (z_r * w).sum().backward()
    assert rel(feats, feats_r) < TOL
    assert rel(seq1.mean(dim=-1), pooled_r) < TOL
    assert rel(z, z_r) < TOL
    assert rel(grads[0], head.mlp3.weight.grad) < TOL
    assert rel(grads[1], head.mlp3.bias.grad) < TOL
    ref = hs_r.grad.to(torch.bfloat16)
    same_sign = (dhs.float() * ref.float() > 0) | ((dhs.float() == 0) & (ref.float() == 0))
    assert bool(same_sign.all())
    ulps = bf16_ulps(dhs, ref)
    assert int(ulps.max()) <= 1 and float((ulps > 0).float().mean()) < 1e-3
    assert rel(dhs.float(), ref.float()) < 2.0 ** -8


def test_bf16_forward_makes_no_copy_of_hs(cuda_device):
    """at the Stage-1 shape, frozen encoder: the forward allocates O(B F), not O(B K F T); fine-tuned: it keeps hs
    itself for the backward, and the backward allocates one bf16 d hs"""
    head = make_head(1024, 256, 0.1, cuda_device).train()
    hs = bf16_hs((64, 25, 1024, 199), 0, cuda_device)
    warm = hs.detach().requires_grad_(True)          # library workspaces (cuBLAS, ...) are allocated here, once
    head.embed(warm).sum().backward()
    del warm
    head.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    for finetune in (False, True):
        x = hs.detach().requires_grad_(finetune)
        base = torch.cuda.memory_allocated(cuda_device)
        torch.cuda.reset_peak_memory_stats(cuda_device)
        z = head.embed(x)
        torch.cuda.synchronize()
        assert torch.cuda.max_memory_allocated(cuda_device) - base < 0.1 * hs.nbytes
        if finetune:
            torch.cuda.reset_peak_memory_stats(cuda_device)
            z.sum().backward()
            torch.cuda.synchronize()
            assert x.grad.dtype == torch.bfloat16
            assert torch.cuda.max_memory_allocated(cuda_device) - base < 1.1 * hs.nbytes
        del z
        head.zero_grad(set_to_none=True)


def test_graphed_step_on_bf16_hs_equals_eager_steps(cuda_device):
    """GraphedHeadStep captured on a bf16 example, dropout on: the replays follow the eager steps on the same bf16
    hs, with the tolerances of test_graphed_step_with_fused_head_and_dropout"""
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    from wav2vec_contr_loss_b200 import stage1 as S
    head = make_head(64, 32, 0.1, cuda_device).train()
    g = torch.Generator().manual_seed(3)
    y = (torch.randperm(64, generator=g) % 2).to(cuda_device)
    hs = (torch.randn(64, 3, 64, 20, generator=g).to(cuda_device)
          + 0.6 * (2.0 * y.view(-1, 1, 1, 1) - 1.0)).to(torch.bfloat16)
    opt = torch.optim.AdamW(head.parameters(), lr=1e-2, capturable=True)
    head_e = copy.deepcopy(head)
    opt_e = torch.optim.AdamW(head_e.parameters(), lr=1e-2, capturable=True)
    twin = S.GraphedHeadStep(head_e, SupConBinaryLoss(0.1, "cosine"), opt_e, hs, y, topk_neg=7)
    step = S.GraphedHeadStep(head, SupConBinaryLoss(0.1, "cosine"), opt, hs, y, topk_neg=7)
    assert step.hs.dtype == torch.bfloat16
    before = torch.cat([p.detach().reshape(-1) for p in head.parameters()]).clone()
    losses = [float(step(hs, y, 0.0)) for _ in range(25)]
    assert head.rng_state.tolist()[1] == 25
    assert all(l == l for l in losses) and sum(losses[-5:]) < sum(losses[:5]) - 0.01
    eager = [float(twin._eager(0.0)) for _ in range(25)]
    assert head_e.rng_state.tolist() == head.rng_state.tolist()
    assert losses == pytest.approx(eager, rel=1e-4)
    flat_g = torch.cat([p.detach().reshape(-1) for p in head.parameters()])
    flat_e = torch.cat([p.detach().reshape(-1) for p in head_e.parameters()])
    assert not torch.equal(flat_g, before)
    assert torch.allclose(flat_g, flat_e, rtol=1e-3, atol=1e-5)
