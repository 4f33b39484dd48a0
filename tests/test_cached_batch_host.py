"""Host side of the cached-embedding step (wav2vec_contr_loss_b200.cached_batch) on the CPU: the loss is the oracle
port and the normalisation is torch's, injected through the keyword hooks, and the fused head's kernel is replaced by
a torch stand-in with a counter-keyed dropout.  Checked: grouping of loader batches, the RNG replay of pass 2, the
encoder runs per route, and two gloo ranks against one process on the concatenated global batch."""
import copy
import os
import socket
from types import SimpleNamespace

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn
import torch.nn.functional as F

from oracle import supcon_oracle as O
from oracle.gen_host_golden import TinyHead
from wav2vec_contr_loss_b200 import stage1 as S
from wav2vec_contr_loss_b200.cached_batch import CachedBatchStep, train_one_epoch_cached
from wav2vec_contr_loss_b200.head import FusedCompressionHead


def torch_normalize(x):
    return F.normalize(x, p=2, dim=1)


class OracleLoss:
    def __init__(self, temperature, similarity, uniformity_weight=0.0, uniformity_t=2.0):
        self.kw = dict(temperature=temperature, similarity=similarity, uniformity_weight=uniformity_weight,
                       uniformity_t=uniformity_t)
        self.calls = []

    def __call__(self, z, labels, topk_neg=32, alpha=0.0):
        self.calls.append(labels.clone())
        return O.anchor_loop_loss(z, labels, topk_neg=topk_neg, alpha=alpha, **self.kw)


class OracleMultiClass:
    takes_mining_args = False

    def __init__(self, temperature):
        self.tau = temperature

    def __call__(self, z, labels):
        return O.anchor_loop_multiclass(z, labels, temperature=self.tau)


class DropoutEncoder(nn.Module):
    """(B, L) waveforms -> (B, K, F, T), with dropout drawn from the global generator; counts its forward calls."""

    def __init__(self, layers=3, feat=12, hop=16, p=0.3):
        super().__init__()
        self.layers, self.hop = layers, hop
        self.proj = nn.Linear(hop, layers * feat)
        self.drop = nn.Dropout(p)
        self.calls = 0

    def forward(self, waveforms, attention_mask=None):
        self.calls += 1
        b = waveforms.size(0)
        frames = (waveforms * attention_mask.to(waveforms.dtype)).view(b, -1, self.hop)
        hs = torch.tanh(self.drop(self.proj(frames))).view(b, frames.size(1), self.layers, -1)
        return hs.permute(0, 2, 3, 1).contiguous()


class DropoutTorchHead(TinyHead):
    """layer mean -> Dropout -> LeakyReLU -> Linear per frame (the reference CompressionModule's order)."""

    def __init__(self, feat=12, dim=8, p=0.2):
        super().__init__(feat, dim)
        self.drop = nn.Dropout(p)

    def forward(self, hs):
        x = self.act(self.drop(hs.mean(dim=1)))
        return self.fc(x.transpose(1, 2)).transpose(1, 2)


class CpuFusedHead(FusedCompressionHead):
    """FusedCompressionHead whose pooling kernel is replaced by torch ops; the dropout mask is a function of
    ``rng_state`` = {seed, offset}, which advances by one per call like the kernel's stream."""

    def pooled_features(self, hs):
        x = hs.mean(dim=1)
        p = self.dropout_head.p if self.training else 0.0
        if p > 0.0:
            seed, offset = (int(v) for v in self.rng_state.tolist())
            g = torch.Generator().manual_seed((seed * 1000003 + offset) % (2 ** 62))
            x = x * (torch.rand(x.shape, generator=g) >= p).to(x.dtype) / (1.0 - p)
            self.rng_state[1] += 1
        return F.leaky_relu(x, self.activation_head.negative_slope).mean(dim=-1)


class Unreproducible(DropoutEncoder):
    """an encoder whose output changes from call to call under the same RNG state"""

    def forward(self, waveforms, attention_mask=None):
        return super().forward(waveforms, attention_mask) + 1e-3 * self.calls


def _batches(count, bsz, seed=0, classes=None):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(count):
        y = torch.randperm(bsz, generator=g) % 2
        wave = torch.randn(bsz, 64, generator=g) + 0.75 * (2.0 * y.view(-1, 1) - 1.0)
        wave[:, 48:] *= torch.where(torch.rand(bsz, 1, generator=g) < 0.5, 0.0, 1.0)      # padding
        extra = torch.randint(0, classes or 2, (bsz,), generator=g)
        out.append((wave, y, extra))
    return out


def _cfg(finetune, **kw):
    return SimpleNamespace(**{**dict(finetune_encoder=finetune, use_rawboost=False, topk_neg=3, warmup_epochs=0,
                                     alpha_ramp_epochs=2, alpha_end=1.0), **kw})


def _flat(*modules):
    return torch.cat([p.detach().reshape(-1) for m in modules for p in m.parameters()]).double()


def _reference_step(enc, head, loss_fn, opt, micro, topk, alpha, finetune, max_grad_norm=5.0):
    """plain autograd through the k micro-batch forwards at once: the step the cached one must equal"""
    opt.zero_grad(set_to_none=True)
    zs = []
    for w, _ in micro:
        with torch.set_grad_enabled(finetune):
            hs = enc(w, attention_mask=(w != 0).long())
        zs.append(S.embed(head, hs, torch_normalize))
    loss = S.call_loss(loss_fn, torch.cat(zs), torch.cat([y for _, y in micro]), topk, alpha)
    loss.backward()
    torch.nn.utils.clip_grad_norm_(head.parameters(), max_grad_norm)
    opt.step()
    return loss.detach()


# --------------------------------------------------------------------------------------------------- grouping

@pytest.mark.parametrize("k,steps,dropped", [(1, 7, 0), (2, 3, 1), (3, 2, 1), (7, 1, 0), (8, 0, 7)])
def test_groups_of_k_consecutive_batches_and_the_dropped_tail(k, steps, dropped):
    torch.manual_seed(0)
    enc, head = DropoutEncoder(p=0.0), TinyHead()
    loader = _batches(7, 6)
    loss_fn = OracleLoss(0.2, "cosine")
    opt = torch.optim.SGD(head.parameters(), lr=0.1)
    avg, alpha, n_dropped = train_one_epoch_cached(enc, head, loss_fn, loader, opt, torch.device("cpu"), 1,
                                                   _cfg(False), micro_batches=k, normalize=torch_normalize)
    assert n_dropped == dropped and alpha == 0.5
    assert len(loss_fn.calls) == steps
    for s, labels in enumerate(loss_fn.calls):                     # step s sees batches [s k, (s + 1) k), in order
        assert torch.equal(labels, torch.cat([loader[s * k + i][1] for i in range(k)]))
    if steps == 0:
        assert avg == 0.0


def test_epoch_equals_train_one_epoch_on_merged_batches():
    """frozen encoder, torch head: k = 3 groups of the loader train exactly like train_one_epoch on batches that ARE
    those groups (loss per step, alpha, weights)."""
    torch.manual_seed(1)
    enc, head = DropoutEncoder(p=0.0), TinyHead()
    enc2, head2 = copy.deepcopy(enc), copy.deepcopy(head)
    loader = _batches(7, 6, seed=3)
    merged = [tuple(torch.cat([b[j] for b in loader[s * 3:(s + 1) * 3]]) for j in range(3)) for s in range(2)]
    cfg, cpu = _cfg(False), torch.device("cpu")
    opt = torch.optim.AdamW(head.parameters(), lr=5e-3, weight_decay=3e-3)
    opt2 = torch.optim.AdamW(head2.parameters(), lr=5e-3, weight_decay=3e-3)
    for epoch in (1, 2, 3):
        got, a, dropped = train_one_epoch_cached(enc, head, OracleLoss(0.1, "geodesic", 0.1), loader, opt, cpu,
                                                 epoch, cfg, micro_batches=3, normalize=torch_normalize)
        want, b = S.train_one_epoch(enc2, head2, OracleLoss(0.1, "geodesic", 0.1), merged, opt2, cpu, epoch, cfg,
                                    normalize=torch_normalize)
        assert dropped == 1 and a == b and got == pytest.approx(want, rel=1e-6)
    assert torch.allclose(_flat(head), _flat(head2), rtol=1e-5, atol=1e-7)


def test_multiclass_labels_column():
    torch.manual_seed(2)
    enc, head = DropoutEncoder(p=0.0), TinyHead()
    head2 = copy.deepcopy(head)
    loader = _batches(4, 6, seed=4, classes=3)
    merged = [tuple(torch.cat([b[j] for b in loader[s * 2:(s + 1) * 2]]) for j in range(3)) for s in range(2)]
    cpu = torch.device("cpu")
    opt, opt2 = torch.optim.SGD(head.parameters(), lr=0.1), torch.optim.SGD(head2.parameters(), lr=0.1)
    got, _, _ = train_one_epoch_cached(enc, head, OracleMultiClass(0.1), loader, opt, cpu, 1, _cfg(False),
                                       micro_batches=2, normalize=torch_normalize, label_index=2)
    want, _ = S.train_one_epoch(enc, head2, OracleMultiClass(0.1), merged, opt2, cpu, 1, _cfg(False),
                                normalize=torch_normalize, label_index=2)
    assert got == pytest.approx(want, rel=1e-6)
    assert torch.allclose(_flat(head), _flat(head2), rtol=1e-5, atol=1e-7)


def test_rawboost_runs_once_per_micro_batch_and_pass_2_reuses_it():
    torch.manual_seed(3)
    enc, head = DropoutEncoder(p=0.0), TinyHead()
    seen = []

    def augment(w, cfg):
        seen.append(w)
        return w + 0.05 * torch.randn_like(w)      # a fresh draw per call: a second call would give other waveforms

    cfg = _cfg(True, use_rawboost=True)
    with pytest.raises(ValueError, match="augment"):
        train_one_epoch_cached(enc, head, OracleLoss(0.2, "cosine"), _batches(4, 6), torch.optim.SGD(
            head.parameters(), lr=0.1), torch.device("cpu"), 1, cfg, micro_batches=2, normalize=torch_normalize)
    params = list(head.parameters()) + list(enc.parameters())
    _, _, dropped = train_one_epoch_cached(enc, head, OracleLoss(0.2, "cosine"), _batches(5, 6), torch.optim.SGD(
        params, lr=0.1), torch.device("cpu"), 1, cfg, micro_batches=2, normalize=torch_normalize, augment=augment,
        check_replay=True)
    assert len(seen) == 4 and dropped == 1       # the dropped batch is not augmented either
    assert enc.calls == 8                        # pass 1 + pass 2, and check_replay found the same rows


# ---------------------------------------------------------------------------------------------- RNG replay

@pytest.mark.parametrize("head_kind", ["fused", "torch"])
def test_pass_2_replays_pass_1_bit_for_bit(head_kind):
    """fine-tuned dropout encoder (global generator) and a dropout head (the fused head's {seed, offset} counter, or
    nn.Dropout on the global generator): pass 2 recomputes the pass-1 rows bit for bit, the step equals plain
    autograd through the k forwards, and both RNG streams end where k plain forwards leave them."""
    torch.manual_seed(4)
    enc = DropoutEncoder(p=0.3)
    head = CpuFusedHead(12, 8, 0.2) if head_kind == "fused" else DropoutTorchHead(p=0.2)
    enc2, head2 = copy.deepcopy(enc), copy.deepcopy(head)
    for m in (enc, head, enc2, head2):
        m.train()
    loss_fn = OracleLoss(0.1, "cosine", 0.05)
    opt = torch.optim.SGD(list(head.parameters()) + list(enc.parameters()), lr=0.05, momentum=0.9)
    opt2 = torch.optim.SGD(list(head2.parameters()) + list(enc2.parameters()), lr=0.05, momentum=0.9)
    step = CachedBatchStep(enc, head, loss_fn, opt, micro_batches=4, normalize=torch_normalize,
                           finetune_encoder=True, check_replay=True)
    loader = _batches(12, 6, seed=5)
    for s in range(3):
        micro = [(w, y) for w, y, _ in loader[4 * s:4 * s + 4]]
        rng0 = torch.get_rng_state()
        got = step(micro, 3, 0.5)
        rng_cached = torch.get_rng_state()
        torch.set_rng_state(rng0)
        want = _reference_step(enc2, head2, loss_fn, opt2, micro, 3, 0.5, True)
        assert torch.equal(torch.get_rng_state(), rng_cached)
        assert float(got) == float(want)                    # the same rows: the same loss, bit for bit
        if head_kind == "fused":
            assert torch.equal(head.rng_state, head2.rng_state) and int(head.rng_state[1]) == 4 * (s + 1)
        assert torch.allclose(_flat(head, enc), _flat(head2, enc2), rtol=1e-5, atol=1e-7)
    assert enc.calls == 2 * 12


def test_check_replay_catches_an_unreproducible_encoder():
    torch.manual_seed(5)
    enc, head = Unreproducible(p=0.0), TinyHead()
    step = CachedBatchStep(enc, head, OracleLoss(0.2, "cosine"), torch.optim.SGD(head.parameters(), lr=0.1),
                           micro_batches=2, normalize=torch_normalize, finetune_encoder=True, check_replay=True)
    with pytest.raises(RuntimeError, match="micro-batch 0"):
        step([(w, y) for w, y, _ in _batches(2, 6)], 3, 0.0)


def test_step_argument_checks():
    enc, head = DropoutEncoder(), TinyHead()
    opt = torch.optim.SGD(head.parameters(), lr=0.1)
    with pytest.raises(ValueError, match="micro_batches"):
        CachedBatchStep(enc, head, OracleLoss(0.2, "cosine"), opt, micro_batches=0)
    step = CachedBatchStep(enc, head, OracleLoss(0.2, "cosine"), opt, micro_batches=3, normalize=torch_normalize)
    with pytest.raises(ValueError, match="built for 3"):
        step([(w, y) for w, y, _ in _batches(2, 6)], 3, 0.0)


# ------------------------------------------------------------------------------------- encoder runs per route

@pytest.mark.parametrize("head_kind,finetune,runs", [("fused", False, 1), ("torch", False, 2), ("fused", True, 2),
                                                     ("torch", True, 2)])
def test_encoder_runs_per_sample(head_kind, finetune, runs):
    """frozen encoder + fused head: pooled features are cached, the encoder runs once per sample; every other route
    runs it twice (pass 1 and pass 2).  Each route equals plain autograd through the k forwards."""
    torch.manual_seed(6)
    enc = DropoutEncoder(p=0.3)
    head = CpuFusedHead(12, 8, 0.2) if head_kind == "fused" else DropoutTorchHead(p=0.2)
    enc2, head2 = copy.deepcopy(enc), copy.deepcopy(head)
    for e in (enc, enc2):
        e.train(finetune)
    params = lambda h, e: list(h.parameters()) + (list(e.parameters()) if finetune else [])  # noqa: E731
    opt = torch.optim.SGD(params(head, enc), lr=0.05)
    opt2 = torch.optim.SGD(params(head2, enc2), lr=0.05)
    loss_fn = OracleLoss(0.2, "geodesic")
    step = CachedBatchStep(enc, head, loss_fn, opt, micro_batches=3, normalize=torch_normalize,
                           finetune_encoder=finetune)
    micro = [(w, y) for w, y, _ in _batches(3, 6, seed=7)]
    rng0 = torch.get_rng_state()
    got = step(micro, 3, 1.0)
    torch.set_rng_state(rng0)
    enc2.calls = 0
    want = _reference_step(enc2, head2, loss_fn, opt2, micro, 3, 1.0, finetune)
    assert enc.calls == runs * 3 and enc2.calls == 3
    assert float(got) == float(want)
    assert torch.allclose(_flat(head, enc), _flat(head2, enc2), rtol=1e-5, atol=1e-7)
    if not finetune:
        assert all(p.grad is None for p in enc.parameters())


# --------------------------------------------------------------- two ranks: ShardedSupConLoss + GradSync (gloo)

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


N_LOCAL, K_MICRO = 6, 2


def _problem():
    g = torch.Generator().manual_seed(7)
    torch.manual_seed(7)
    head = DropoutTorchHead(feat=6, dim=8, p=0.0)
    labels = [int(v) for v in (torch.rand(90, generator=g) < 0.45)]
    feats = torch.randn(90, 2, 6, 5, generator=g) + torch.tensor(labels).view(-1, 1, 1, 1) * 0.8
    dataset = SimpleNamespace(data=[(f"utt{i}", lab) for i, lab in enumerate(labels)])
    return head, feats, torch.tensor(labels), dataset


def _loader(sampler, feats, labels):
    return [(feats[idx], labels[idx]) for idx in map(torch.tensor, sampler)]


class _Identity(nn.Module):
    def forward(self, x, attention_mask=None):
        return x


_CFG = dict(finetune_encoder=False, use_rawboost=False, topk_neg=3, warmup_epochs=0, alpha_ramp_epochs=2,
            alpha_end=1.0)


def _rank_main(rank, world, port, out):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from oracle_kernels import OracleKernels
    from wav2vec_contr_loss_b200.distributed import ShardedSupConLoss
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    assert S.setup_distributed(backend="gloo") == (True, rank, world, rank)
    try:
        head, feats, labels, dataset = _problem()
        sampler = S.BalancedBatchSampler(dataset, N_LOCAL, seed=5, rank=rank, world_size=world)
        loss_fn = ShardedSupConLoss(0.2, "cosine", 0.05, 2.0, kernels=OracleKernels)
        opt = torch.optim.SGD(head.parameters(), lr=0.5)
        history = []
        for epoch in (1, 2):
            sampler.set_epoch(epoch)
            loader = _loader(sampler, feats, labels)
            avg, alpha, dropped = train_one_epoch_cached(_Identity(), head, loss_fn, loader, opt,
                                                         torch.device("cpu"), epoch, SimpleNamespace(**_CFG),
                                                         micro_batches=K_MICRO, normalize=torch_normalize,
                                                         grad_sync=S.GradSync(head.parameters()))
            history.append((len(loader) // K_MICRO, avg, alpha, dropped))
        out[rank] = (history, _flat(head))
    finally:
        dist.destroy_process_group()


def test_two_ranks_train_like_one_process_on_the_global_batch():
    """each rank groups K_MICRO of its own loader batches; ShardedSupConLoss contrasts the R * K_MICRO * B rows and
    GradSync sums the head's gradients: the trajectory of ONE process whose batch at step s is rank 0's micro-batches
    then rank 1's."""
    world = 2
    out = mp.Manager().dict()
    mp.spawn(_rank_main, args=(world, _free_port(), out), nprocs=world, join=True)

    head, feats, labels, dataset = _problem()
    sampler = S.BalancedBatchSampler(dataset, N_LOCAL, seed=5)
    opt = torch.optim.SGD(head.parameters(), lr=0.5)
    want = []
    for epoch in (1, 2):
        sampler.set_epoch(epoch)
        batches = list(sampler)
        per_rank = [batches[r:len(batches) - len(batches) % world:world] for r in range(world)]
        steps = len(per_rank[0]) // K_MICRO
        merged = [sum((per_rank[r][s * K_MICRO + i] for r in range(world) for i in range(K_MICRO)), [])
                  for s in range(steps)]
        avg, alpha = S.train_one_epoch(_Identity(), head, OracleLoss(0.2, "cosine", 0.05, 2.0),
                                       _loader(merged, feats, labels), opt, torch.device("cpu"), epoch,
                                       SimpleNamespace(**_CFG), normalize=torch_normalize)
        want.append((steps, avg, alpha, len(per_rank[0]) % K_MICRO))
    assert want[0][0] >= 2
    want_w = _flat(head)
    for rank in range(world):
        history, got_w = out[rank]
        for (steps, avg, alpha, dropped), (w_steps, w_avg, w_alpha, w_dropped) in zip(history, want):
            assert (steps, alpha, dropped) == (w_steps, w_alpha, w_dropped)
            assert avg == pytest.approx(w_avg, rel=1e-5)
        assert torch.allclose(got_w, want_w, rtol=1e-4, atol=1e-6)
    assert torch.equal(out[0][1], out[1][1])
