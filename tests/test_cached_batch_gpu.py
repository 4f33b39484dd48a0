"""GPU: the cached-embedding step (wav2vec_contr_loss_b200.cached_batch) with the product defaults, against plain
autograd through all k micro-batch forwards at once (same dropout offsets, same RNG states), on a tiny conv + dropout
encoder: loss 1e-6, head and encoder gradients and the weights after three steps 1e-5 (fp32) / 2e-3 (bf16), the loss
of the concatenated batch against the fp64 oracle, the cross-batch memory, and peak memory against a k = 1 step."""
import copy

import pytest
import torch
import torch.nn as nn

import gpu_util as G
from oracle import supcon_oracle as O

pytestmark = pytest.mark.gpu

B, D = 64, 256


class ConvEncoder(nn.Module):
    """(B, L) waveforms -> (B, K, F, T): strided conv, dropout, tanh."""

    def __init__(self, layers=3, feat=64, hop=16, p=0.1):
        super().__init__()
        self.layers, self.feat = layers, feat
        self.conv = nn.Conv1d(1, layers * feat, hop, stride=hop)
        self.drop = nn.Dropout(p)

    def forward(self, waveforms, attention_mask=None):
        x = (waveforms * attention_mask.to(waveforms.dtype)).unsqueeze(1)
        h = torch.tanh(self.drop(self.conv(x)))
        return h.view(h.size(0), self.layers, self.feat, -1)


class TorchHead(nn.Module):
    """the reference CompressionModule's op chain: layer mean -> Dropout -> LeakyReLU -> Linear per frame."""

    def __init__(self, feat=64, dim=D, p=0.1):
        super().__init__()
        self.drop, self.act, self.fc = nn.Dropout(p), nn.LeakyReLU(), nn.Linear(feat, dim)

    def forward(self, hs):
        x = self.act(self.drop(hs.mean(dim=1)))
        return self.fc(x.transpose(1, 2)).transpose(1, 2)


class Recording(nn.Module):
    """loss_fn wrapper that keeps what the step handed the loss"""

    def __init__(self, inner):
        super().__init__()
        self.inner = inner
        self.takes_mining_args = getattr(inner, "takes_mining_args", True)
        self.seen = []

    def forward(self, z, labels, **kw):
        from wav2vec_contr_loss_b200 import functional as Fn
        self.seen.append((z.detach().clone(), labels.clone(), bool(getattr(z, Fn.UNIT_ROWS_TAG, False))))
        return self.inner(z, labels, **kw)


def _models(head_kind, finetune, device, seed=0):
    from wav2vec_contr_loss_b200 import FusedCompressionHead
    torch.manual_seed(seed)
    enc = ConvEncoder().to(device).train(finetune)
    head = (FusedCompressionHead(64, D, 0.1) if head_kind == "fused" else TorchHead()).to(device).train()
    return enc, head


def _micro(k, device, seed=0, length=1600, classes=2):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(k):
        y = torch.randperm(B, generator=g) % classes
        w = torch.randn(B, length, generator=g) + 0.3 * (2.0 * y.view(-1, 1).float() - 1.0)
        w[:, length * 3 // 4:] *= (torch.rand(B, 1, generator=g) < 0.5).float()          # padded tails
        out.append((w.to(device), y.to(device)))
    return out


def _normalize(dtype):
    from wav2vec_contr_loss_b200 import functional as Fn
    return None if dtype == torch.float32 else (lambda x: Fn.l2_normalize(x, dtype))


def _reference_step(enc, head, loss_fn, opt, micro, topk, alpha, finetune, normalize):
    from wav2vec_contr_loss_b200 import functional as Fn
    from wav2vec_contr_loss_b200 import stage1 as S
    opt.zero_grad(set_to_none=True)
    zs = []
    for w, _ in micro:
        with torch.set_grad_enabled(finetune):
            hs = enc(w, attention_mask=(w != 0).long())
        zs.append(S.embed(head, hs, normalize))
    z = Fn.mark_unit_rows(torch.cat(zs))          # every row came from l2_normalize
    loss = S.call_loss(loss_fn, z, torch.cat([y for _, y in micro]), topk, alpha)
    loss.backward()
    torch.nn.utils.clip_grad_norm_(head.parameters(), 5.0)
    opt.step()
    return loss.detach()


def _grads(module):
    gs = [p.grad.reshape(-1) for p in module.parameters() if p.grad is not None]
    return torch.cat(gs).double().cpu() if gs else None


def _flat(module):
    return torch.cat([p.detach().reshape(-1) for p in module.parameters()]).double().cpu()


def _run_twins(device, *, k, head_kind, finetune, make_loss, alpha=0.0, dtype=torch.float32,
               steps=3, classes=2):
    """three cached steps and three reference steps from the same weights and RNG states; returns both sides'
    per-step losses, gradients and the final weights (and the loss objects)"""
    from wav2vec_contr_loss_b200.cached_batch import CachedBatchStep
    enc, head = _models(head_kind, finetune, device)
    enc2, head2 = copy.deepcopy(enc), copy.deepcopy(head)
    params = lambda h, e: list(h.parameters()) + (list(e.parameters()) if finetune else [])  # noqa: E731
    opt = torch.optim.SGD(params(head, enc), lr=0.05, momentum=0.9)
    opt2 = torch.optim.SGD(params(head2, enc2), lr=0.05, momentum=0.9)
    loss_a, loss_b = make_loss(), make_loss()
    normalize = _normalize(dtype)
    step = CachedBatchStep(enc, head, loss_a, opt, micro_batches=k, normalize=normalize, finetune_encoder=finetune,
                           check_replay=True)
    start = (_flat(head), _flat(enc))
    out = []
    for s in range(steps):
        micro = _micro(k, device, seed=100 + s, classes=classes)
        rng0 = torch.cuda.get_rng_state(device)
        got = float(step(micro, 15, alpha))
        rng_after = torch.cuda.get_rng_state(device)
        grads = (_grads(head), _grads(enc))
        torch.cuda.set_rng_state(rng0, device)
        want = float(_reference_step(enc2, head2, loss_b, opt2, micro, 15, alpha, finetune, normalize))
        assert torch.equal(torch.cuda.get_rng_state(device), rng_after)      # both streams continue alike
        if head_kind == "fused":
            assert torch.equal(head.rng_state, head2.rng_state)
        out.append((got, want, grads, (_grads(head2), _grads(enc2))))
    return out, (head, enc, start), (head2, enc2), loss_a, loss_b


def _check(out, models, models_ref, tol, finetune):
    """per step: loss, and the head's and encoder's gradients; at the end: the weights' updates"""
    for got, want, (gh, ge), (wh, we) in out:
        assert got == pytest.approx(want, rel=1e-6)
        assert G.rel_err(gh, wh) < tol
        if finetune:
            assert G.rel_err(ge, we) < tol
        else:
            assert ge is None and we is None
    head, enc, start = models
    for m, m2, w0 in zip((head, enc), models_ref, start):
        assert G.rel_err(_flat(m) - w0, _flat(m2) - w0) < tol


FP32_CASES = [(k, sim, alpha) for k in (1, 2, 4, 8) for sim in ("cosine", "geodesic") for alpha in (0.0, 0.5)]


@pytest.mark.parametrize("head_kind", ["fused", "torch"])
@pytest.mark.parametrize("finetune", [False, True], ids=["frozen", "finetune"])
@pytest.mark.parametrize("k,sim,alpha", FP32_CASES)
def test_fp32_equals_autograd_over_all_micro_batches(cuda_device, head_kind, finetune, k, sim, alpha):
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    out, models, models_ref, _, _ = _run_twins(cuda_device, k=k, head_kind=head_kind, finetune=finetune, alpha=alpha,
                                               make_loss=lambda: SupConBinaryLoss(0.1, sim, 0.05))
    _check(out, models, models_ref, 1e-5, finetune)


@pytest.mark.parametrize("head_kind", ["fused", "torch"])
@pytest.mark.parametrize("finetune", [False, True], ids=["frozen", "finetune"])
@pytest.mark.parametrize("k,sim,alpha", [(4, "cosine", 0.0), (4, "geodesic", 0.5), (8, "cosine", 0.5),
                                         (8, "geodesic", 0.0)])
def test_bf16_unit_rows_tensor_path(cuda_device, head_kind, finetune, k, sim, alpha):
    """bf16 z of unit rows, N = k B >= 256: the loss gets the unit-rows tag on the whole batch (tensor-core path)."""
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    out, models, models_ref, loss_a, loss_b = _run_twins(
        cuda_device, k=k, head_kind=head_kind, finetune=finetune, alpha=alpha, dtype=torch.bfloat16,
        make_loss=lambda: Recording(SupConBinaryLoss(0.1, sim)))
    _check(out, models, models_ref, 2e-3, finetune)
    for s, ((z, _, tagged), (z2, _, _)) in enumerate(zip(loss_a.seen, loss_b.seen)):
        assert z.dtype == torch.bfloat16 and z.shape == (k * B, D) and tagged
        # step 0 starts from the same weights: the two passes recompute plain autograd's rows bit for bit.  One Linear
        # over the k B cached pooled rows (frozen fused head) and the weights after a step (the k gradient
        # contributions are summed in another order) round differently, within bf16 rounding.
        if s == 0 and (finetune or head_kind == "torch"):
            assert torch.equal(z, z2)
        else:
            assert G.rel_err(z.float(), z2.float()) < 2e-3


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 2e-3)])
def test_loss_of_the_global_batch_against_the_oracle(cuda_device, dtype, tol):
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    out, _, _, loss_a, _ = _run_twins(cuda_device, k=4, head_kind="fused", finetune=True, alpha=0.5, dtype=dtype,
                                      steps=1, make_loss=lambda: Recording(SupConBinaryLoss(0.07, "cosine", 0.05)))
    (z, y, _), = loss_a.seen
    ref = O.closed_form(z.double().cpu(), y.cpu(), temperature=0.07, similarity="cosine", uniformity_weight=0.05,
                        topk_neg=15, alpha=0.5, want_grad=False)
    assert out[0][0] == pytest.approx(ref["loss"], rel=tol)


@pytest.mark.parametrize("head_kind,finetune", [("fused", False), ("torch", True)])
def test_multiclass_loss(cuda_device, head_kind, finetune):
    from wav2vec_contr_loss_b200 import SupConMultiClassLoss
    out, models, models_ref, _, _ = _run_twins(cuda_device, k=4, head_kind=head_kind, finetune=finetune, classes=5,
                                               make_loss=lambda: SupConMultiClassLoss(0.1))
    _check(out, models, models_ref, 1e-5, finetune)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, 1e-5), (torch.bfloat16, 2e-3)])
@pytest.mark.parametrize("head_kind,finetune", [("fused", False), ("fused", True), ("torch", False)])
def test_memory_loss_takes_the_global_batch(cuda_device, dtype, tol, head_kind, finetune):
    """MemorySupConLoss: the k B rows are the batch, and all of them enter the memory after the backward."""
    from wav2vec_contr_loss_b200.memory import MemorySupConLoss
    k = 4

    def make():
        return Recording(MemorySupConLoss(0.1, "cosine", 0.05, memory_size=1024))

    out, models, models_ref, loss_a, loss_b = _run_twins(cuda_device, k=k, head_kind=head_kind, finetune=finetune,
                                                         alpha=0.5, dtype=dtype, make_loss=make)
    _check(out, models, models_ref, tol, finetune)
    mem, mem2 = loss_a.inner.memory, loss_b.inner.memory
    assert mem.filled == mem2.filled == 3 * k * B
    for s, (z, _, _) in enumerate(loss_a.seen):
        assert torch.equal(mem.embeddings[s * k * B:(s + 1) * k * B], z)
    # the twin's rows differ from step 1 on by the rounding of the weights (the gradient sums' order), and the frozen
    # fused head's by that of one Linear over k B rows: the same rows within the step's tolerance, the same labels
    assert G.rel_err(mem.embeddings.float(), mem2.embeddings.float()) < tol and torch.equal(mem.keys, mem2.keys)


@pytest.mark.parametrize("head_kind,finetune", [("fused", False), ("fused", True), ("torch", False),
                                                ("torch", True)], ids=lambda v: str(v))
def test_peak_memory_of_a_step_does_not_grow_with_k(cuda_device, head_kind, finetune):
    """peak allocation of a k = 8 step <= that of a k = 1 step + the step's caches (z_all, dz_all, pooled) + 10 %."""
    from wav2vec_contr_loss_b200.cached_batch import CachedBatchStep
    from wav2vec_contr_loss_b200 import SupConBinaryLoss
    length = 32000                                   # hs of one micro-batch: 64 x 3 x 64 x 2000 fp32 = 98 MB
    enc, head = _models(head_kind, finetune, cuda_device)
    params = list(head.parameters()) + (list(enc.parameters()) if finetune else [])
    opt = torch.optim.SGD(params, lr=0.01, momentum=0.9)
    micro = _micro(8, cuda_device, length=length)

    def peak(k):
        step = CachedBatchStep(enc, head, SupConBinaryLoss(0.1, "cosine"), opt, micro_batches=k,
                               finetune_encoder=finetune)
        step(micro[:k], 15, 0.0)                     # warm: gradients and momentum exist before the measured call
        torch.cuda.synchronize(cuda_device)
        torch.cuda.reset_peak_memory_stats(cuda_device)
        base = torch.cuda.memory_allocated(cuda_device)
        step(micro[:k], 15, 0.0)
        torch.cuda.synchronize(cuda_device)
        return torch.cuda.max_memory_allocated(cuda_device) - base

    p1, p8 = peak(1), peak(8)
    caches = 8 * B * D * 4 * 2 + 8 * B * 4 + (8 * B * 64 * 4 if head_kind == "fused" and not finetune else 0)
    assert p1 > 50e6                                 # the activations dominate what is measured
    assert p8 <= p1 + caches + 0.1 * p1, (p1, p8, caches)
