"""Stage-1 steps on a global batch of k micro-batches: the exact gradient of a batch the encoder cannot hold at once.

The loss of a batch of N rows is cheap on this library's kernels; what limits a fine-tuned Stage-1 step is the memory
of the encoder's activations.  The loss's backward hands back ``d loss / d z`` for every row, N x d numbers, so the
global batch splits into micro-batches (gradient caching, Gao et al., "Scaling Deep Contrastive Learning Batch Size
under Memory Limited Setup", 2021):

  pass 1   each micro-batch: encoder -> head -> normalise without a graph, rows written into ``z_all``;
  loss     ``call_loss`` once over all k * B rows, ``dz_all = d loss / d z_all``;
  pass 2   each micro-batch again with a graph, ``z_i.backward(dz_all[rows_i])``: the parameter gradients add up
           over the micro-batches and only one micro-batch's activations are alive at a time.

Dropout draws the same masks in both passes: before a micro-batch's pass 1 the step records the RNG state of the
input's device (the encoder's and a torch head's dropout) and ``FusedCompressionHead.rng_state`` (its in-kernel
dropout), and pass 2 restores both.  After pass 2 both streams are put back where pass 1 left them, so the next step
draws new masks, exactly as k plain forwards would have.

Frozen encoder: with ``FusedCompressionHead`` the only parameters are the Linear layer's and only the pooled features
feed it, so pass 1 keeps ``pooled`` (k B x F fp32) and the step runs Linear -> normalise -> loss -> backward once with a
graph; the encoder runs once per sample.  Any other head is recomputed in pass 2 from a second encoder run without a
graph (its input, the encoder output, is too large to keep: 1.3 GB per micro-batch of 64 at Stage-1 size), so the
encoder runs twice per sample.
"""
from typing import Callable, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

from . import functional as Fn
from .head import FusedCompressionHead
from .stage1 import (RunningLoss, _check_augment, _to_device, alpha_for_epoch, call_loss, embed)

__all__ = ["CachedBatchStep", "train_one_epoch_cached"]


def _rng_state(device: torch.device) -> torch.Tensor:
    return torch.cuda.get_rng_state(device) if device.type == "cuda" else torch.get_rng_state()


def _set_rng_state(device: torch.device, state: torch.Tensor) -> None:
    if device.type == "cuda":
        torch.cuda.set_rng_state(state, device)
    else:
        torch.set_rng_state(state)


class CachedBatchStep:
    """One optimizer step on the loss of the concatenation of k micro-batches (see the module docstring).

        step = CachedBatchStep(encoder, head, loss_fn, optimizer, micro_batches=k, finetune_encoder=True)
        loss = step([(waveforms_0, labels_0), ..., (waveforms_k-1, labels_k-1)], topk_neg, alpha)

    A call is the step of ``train_one_epoch`` on the global batch: zero_grad, the two passes, ``grad_sync``, clipping
    of the head's parameters to ``max_grad_norm``, one ``optimizer.step()``.  It returns the loss of the whole batch
    (detached).  Waveforms are zero-padded (the attention mask is ``waveforms != 0``); micro-batches may differ in
    size.  The caller sets the train / eval modes of ``encoder`` and ``head``.

    ``loss_fn`` is anything ``call_loss`` takes: ``SupConBinaryLoss``, ``SupConMultiClassLoss``, ``MemorySupConLoss``
    (the k B rows are the batch, and they enter the memory when the loss's backward has run) or ``ShardedSupConLoss``
    (each rank passes its k micro-batches, the loss is over the R k B rows of all ranks; pass ``grad_sync``).

    ``check_replay``: pass 2 compares every recomputed row with its pass-1 row and raises if one differs in any bit
    (one host sync per micro-batch; for debugging an encoder whose forward is not reproducible)."""

    def __init__(self, encoder, head, loss_fn, optimizer, micro_batches: int, *, normalize: Optional[Callable] = None,
                 grad_sync: Optional[Callable] = None, max_grad_norm: float = 5.0, finetune_encoder: bool = False,
                 check_replay: bool = False):
        if int(micro_batches) < 1:
            raise ValueError(f"micro_batches must be >= 1, got {micro_batches}")
        self.encoder, self.head, self.loss_fn, self.optimizer = encoder, head, loss_fn, optimizer
        self.micro_batches = int(micro_batches)
        self.normalize, self.grad_sync = normalize, grad_sync
        self.max_grad_norm = float(max_grad_norm)
        self.finetune = bool(finetune_encoder)
        self.check_replay = bool(check_replay)
        # frozen encoder + fused head: the pooled features are all the step needs to keep (module docstring)
        self.cache_pooled = not self.finetune and isinstance(head, FusedCompressionHead)

    def _encode(self, waveforms: torch.Tensor) -> torch.Tensor:
        return self.encoder(waveforms, attention_mask=(waveforms != 0.0).long())

    def __call__(self, micro: Sequence[Tuple[torch.Tensor, torch.Tensor]], topk_neg: int = 32,
                 alpha: float = 0.0) -> torch.Tensor:
        if len(micro) != self.micro_batches:
            raise ValueError(f"CachedBatchStep was built for {self.micro_batches} micro-batches, got {len(micro)}")
        sizes = [int(w.size(0)) for w, _ in micro]
        bounds = [0]
        for s in sizes:
            bounds.append(bounds[-1] + s)
        labels_all = torch.cat([y.reshape(-1) for _, y in micro])
        self.optimizer.zero_grad(set_to_none=True)
        if self.cache_pooled:
            loss = self._frozen_fused(micro, bounds, labels_all, topk_neg, alpha)
        else:
            loss = self._two_pass(micro, bounds, labels_all, topk_neg, alpha)
        if self.grad_sync is not None:
            self.grad_sync()
        torch.nn.utils.clip_grad_norm_(self.head.parameters(), self.max_grad_norm)
        self.optimizer.step()
        return loss.detach()

    def _frozen_fused(self, micro, bounds, labels_all, topk_neg, alpha):
        pooled_all = None
        with torch.no_grad():
            for i, (w, _) in enumerate(micro):
                pooled = self.head.pooled_features(self._encode(w))
                if pooled_all is None:
                    pooled_all = torch.empty((bounds[-1], pooled.size(1)), dtype=pooled.dtype, device=pooled.device)
                pooled_all[bounds[i]:bounds[i + 1]].copy_(pooled)
        z = (self.normalize or Fn.l2_normalize)(F.linear(pooled_all, self.head.mlp3.weight, self.head.mlp3.bias))
        loss = call_loss(self.loss_fn, z, labels_all, topk_neg, alpha)
        loss.backward()
        return loss

    def _embed(self, waveforms: torch.Tensor, with_graph: bool) -> torch.Tensor:
        """encoder -> head -> normalise; the encoder keeps a graph only when it is fine-tuned."""
        with torch.set_grad_enabled(with_graph and self.finetune):
            hs = self._encode(waveforms)
        with torch.set_grad_enabled(with_graph):
            return embed(self.head, hs, self.normalize)

    def _two_pass(self, micro, bounds, labels_all, topk_neg, alpha):
        dev = micro[0][0].device
        head_rng = self.head.rng_state if isinstance(self.head, FusedCompressionHead) else None
        saved = []
        z_all, unit_rows = None, True
        # pass 1: no graph; the RNG states each micro-batch starts from are kept for pass 2
        for i, (w, _) in enumerate(micro):
            saved.append((_rng_state(dev), None if head_rng is None else head_rng.clone()))
            z = self._embed(w, with_graph=False)
            if z_all is None:
                z_all = torch.empty((bounds[-1], z.size(1)), dtype=z.dtype, device=z.device)
            z_all[bounds[i]:bounds[i + 1]].copy_(z)
            unit_rows = unit_rows and bool(getattr(z, Fn.UNIT_ROWS_TAG, False))
        after = (_rng_state(dev), None if head_rng is None else head_rng.clone())
        if unit_rows:                       # every row came from l2_normalize: the loss may take the unit-rows route
            Fn.mark_unit_rows(z_all)
        z_all.requires_grad_(True)
        loss = call_loss(self.loss_fn, z_all, labels_all, topk_neg, alpha)
        (dz_all,) = torch.autograd.grad(loss, z_all, allow_unused=True)
        if dz_all is None:                  # a batch without pairs: the loss is the constant 0
            dz_all = torch.zeros_like(z_all)
        # pass 2: the same masks, now with a graph, one micro-batch at a time
        for i, (w, _) in enumerate(micro):
            _set_rng_state(dev, saved[i][0])
            if head_rng is not None:
                head_rng.copy_(saved[i][1])
            z = self._embed(w, with_graph=True)
            rows = slice(bounds[i], bounds[i + 1])
            if self.check_replay and not torch.equal(z.detach(), z_all[rows].detach()):
                raise RuntimeError(f"micro-batch {i}: the recomputed rows differ from pass 1 (the encoder or head "
                                   f"forward is not reproducible under the same RNG state)")
            z.backward(dz_all[rows])
        _set_rng_state(dev, after[0])
        if head_rng is not None:
            head_rng.copy_(after[1])
        return loss


def train_one_epoch_cached(encoder, head, loss_fn, loader, optimizer, device, epoch, cfg, *, micro_batches: int,
                           normalize: Optional[Callable] = None, augment: Optional[Callable] = None,
                           grad_sync: Optional[Callable] = None, max_grad_norm: float = 5.0, label_index: int = 1,
                           check_replay: bool = False):
    """``train_one_epoch`` with one optimizer step per ``micro_batches`` consecutive loader batches
    (``CachedBatchStep``).  Returns ``(mean loss over global steps and ranks, alpha, dropped)``: ``dropped`` is the
    number of trailing loader batches that did not fill a last group and were not trained on.

    Batches of ``BalancedBatchSampler`` are balanced, so a group of them is too.  RawBoost (``augment``) runs once
    per micro-batch before pass 1, and pass 2 recomputes from those same augmented waveforms."""
    _check_augment(cfg, augment)
    finetune = bool(cfg.finetune_encoder)
    encoder.train(finetune)
    head.train()
    alpha = alpha_for_epoch(epoch, cfg)
    running = RunningLoss(device)
    step = CachedBatchStep(encoder, head, loss_fn, optimizer, micro_batches, normalize=normalize,
                           grad_sync=grad_sync, max_grad_norm=max_grad_norm, finetune_encoder=finetune,
                           check_replay=check_replay)
    rawboost = augment is not None and getattr(cfg, "use_rawboost", False)
    group: List = []
    for batch in loader:
        group.append(batch)
        if len(group) < step.micro_batches:
            continue
        micro = []
        for b in group:
            waveforms, labels = _to_device(b[0], b[label_index], device)
            if rawboost:
                waveforms = augment(waveforms, cfg)
            micro.append((waveforms, labels))
        group = []
        running.add(step(micro, cfg.topk_neg, alpha))
    return running.average(), alpha, len(group)
