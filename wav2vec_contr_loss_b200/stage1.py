"""Host side of the Stage-1 step either side of the loss (SURVEY.md §8 rows a1, a9 and "next" N2-N4).

What the reference keeps in ``stage1_utils.py`` around ``loss_fn(z, labels, topk_neg=..., alpha=...)``:

  alpha_for_epoch        hard-negative blend schedule          stage1_utils.py:84-88
  BalancedBatchSampler   half bonafide / half spoof batches    stage1_utils.py:22-53
  train_one_epoch        encoder -> head -> normalise -> loss  stage1_utils.py:101-134
  evaluate               the same without grad, alpha = 0      stage1_utils.py:137-153
  setup_distributed      torchrun / SLURM rendezvous           stage1_utils.py:156-172
  export_embeddings      (N, 256) fp32 .npy for Stage 2        extract_stage1_embeddings.py:148-163,220-231
  GraphedHeadStep        head+loss+optimizer step, one CUDA graph replay (no reference counterpart)
  train_one_epoch_from_store / evaluate_from_store
                         the epoch functions for a frozen encoder whose layer means are held in a
                         feature_store.LayerMeanStore (train_stage1_from_emb.py trains from disk features)

Same names, positional arguments and return values, so a caller that does
``from stage1_utils import train_one_epoch`` can import it from here instead.  What differs, on purpose:

* the row normalisation runs through this library's CUDA kernel (``functional.l2_normalize``), not
  ``F.normalize``;
* the running loss is accumulated on the device (fp64) and read back ONCE per epoch instead of one
  ``loss.item()`` host sync per step (stage1_utils.py:132) - the value returned is bit-identical, the sum
  is over the same fp32 numbers in the same order;
* with several ranks every rank takes the SAME number of steps (the reference's ``__len__`` differs across
  ranks when the batch count is not a multiple of the world size, which is what hung its DDP attempt,
  train_stage1_log/supcon-38897091.log:57); the loss of the step is the loss of the GLOBAL batch
  (``distributed.ShardedSupConLoss``), and ``GradSync`` sums the head's parameter gradients over ranks;
* RawBoost augmentation (stage1_utils.py:56-81, CPU numpy) is outside this package: pass it as ``augment=``.

Nothing here falls back to a CPU loss: the defaults need CUDA tensors and raise otherwise.  The keyword-only
``normalize=`` hook exists so the host logic can be exercised without a GPU in tests.
"""
import os
import random
from typing import Callable, Iterator, List, Optional, Sequence

import torch
import torch.distributed as dist
from torch.utils.data import Sampler

from . import functional as Fn

__all__ = ["alpha_for_epoch", "BalancedBatchSampler", "RunningLoss", "GradSync", "embed", "call_loss",
           "normalized_supcon_loss",
           "train_one_epoch", "evaluate", "setup_distributed", "export_embeddings", "GraphedHeadStep",
           "CachedBatchStep", "train_one_epoch_cached", "train_one_epoch_from_store", "evaluate_from_store"]

_CACHED_BATCH = ("CachedBatchStep", "train_one_epoch_cached")


def __getattr__(name):
    """Re-export of ``cached_batch`` (global batches of k micro-batches), which itself builds on this module."""
    if name in _CACHED_BATCH:
        from . import cached_batch
        return getattr(cached_batch, name)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")


# ------------------------------------------------------------------------------------------------ schedule

def alpha_for_epoch(epoch: int, cfg) -> float:
    """Weight of the mined (top-K hard negative) term for this epoch: 0 through the warm-up, then a linear
    ramp of ``alpha_ramp_epochs`` epochs up to ``alpha_end`` (reference stage1_utils.py:84-88; the module-level
    copy at train_stage1_from_emb.py:108-111 is the same formula over constants).  The value goes to the
    kernels as a plain fp32 argument."""
    past_warmup = epoch - cfg.warmup_epochs
    if past_warmup <= 0:
        return 0.0
    ramp = min(1.0, past_warmup / max(1, cfg.alpha_ramp_epochs))
    return ramp * cfg.alpha_end


# ------------------------------------------------------------------------------------------------- sampler

class BalancedBatchSampler(Sampler[List[int]]):
    """Batches of ``batch_size // 2`` bonafide (label 1) + ``batch_size // 2`` spoof (label 0) indices,
    shuffled inside the batch (reference stage1_utils.py:22-53; ``dataset.data[i][1]`` is the label).

    Single process: the batches are the reference's, index for index, for the same ``seed`` and the same
    sequence of ``set_epoch`` / iteration calls (same ``random.Random(seed + epoch)`` draws in the same order;
    like the reference the two index pools are shuffled in place, so an epoch's order depends on the epochs
    iterated before it).

    Several ranks: global step ``s`` gives rank ``r`` batch ``s * world_size + r`` of that same sequence (the
    reference's ``b % world_size == rank`` assignment), and the tail ``num_batches % world_size`` batches
    are dropped so ``len()`` is equal on every rank - each step ends in collectives.  ``equal_steps=False``
    restores the reference's uneven lengths.
    """

    def __init__(self, dataset, batch_size: int, seed: int = 0, rank: int = 0, world_size: int = 1,
                 equal_steps: bool = True):
        if batch_size <= 0 or batch_size % 2:
            raise ValueError(f"batch_size must be positive and even, got {batch_size}")
        if not 0 <= rank < world_size:
            raise ValueError(f"rank {rank} outside world of {world_size}")
        self.batch_size = batch_size
        self.per_class = batch_size // 2
        self.data = dataset.data
        self.real: List[int] = []
        self.fake: List[int] = []
        for index, item in enumerate(self.data):
            if item[1] == 1:
                self.real.append(index)
            elif item[1] == 0:
                self.fake.append(index)
        self.num_batches = min(len(self.real), len(self.fake)) // self.per_class
        self.seed, self.epoch = seed, 0
        self.rank, self.world_size, self.equal_steps = rank, world_size, equal_steps

    def set_epoch(self, epoch: int) -> None:
        self.epoch = epoch

    def _usable_batches(self) -> int:
        if self.equal_steps:
            return self.num_batches - self.num_batches % self.world_size
        return self.num_batches

    def __len__(self) -> int:
        usable = self._usable_batches()
        return len(range(self.rank, usable, self.world_size))

    def __iter__(self) -> Iterator[List[int]]:
        rng = random.Random(self.seed + self.epoch)
        rng.shuffle(self.real)
        rng.shuffle(self.fake)
        usable, half = self._usable_batches(), self.per_class
        for b in range(self.num_batches):
            batch = self.real[b * half:(b + 1) * half] + self.fake[b * half:(b + 1) * half]
            rng.shuffle(batch)            # drawn for every batch on every rank: the streams stay aligned
            if b < usable and b % self.world_size == self.rank:
                yield batch


# --------------------------------------------------------------------------------------- epoch bookkeeping

class RunningLoss:
    """Sum of the per-step losses kept on the device (fp64), read back once: replaces the per-step
    ``total += loss.item()`` of stage1_utils.py:132,151 and ``_reduce_avg`` (stage1_utils.py:91-98)."""

    def __init__(self, device):
        self.total = torch.zeros((), dtype=torch.float64, device=device)
        self.steps = 0

    def add(self, loss: torch.Tensor) -> None:
        self.total += loss.detach().to(torch.float64)
        self.steps += 1

    def average(self, group=None) -> float:
        """mean over the steps of every rank (one collective, one host sync)."""
        if dist.is_available() and dist.is_initialized():
            both = torch.stack([self.total, torch.tensor(float(self.steps), dtype=torch.float64,
                                                         device=self.total.device)])
            dist.all_reduce(both, op=dist.ReduceOp.SUM, group=group)
            total, steps = both.tolist()
            return total / max(1.0, steps)
        return float(self.total) / max(1, self.steps)


class GradSync:
    """Sum of the parameter gradients over ranks, one flat all-reduce.

    With ``ShardedSupConLoss`` every rank back-propagates d(global loss)/d(z_local) through its own copy of the
    head, so each rank holds the part of d(global loss)/d(theta) that flows through its rows: the full
    gradient is the SUM over ranks (not DDP's mean).  Call between ``loss.backward()`` and the clip/step."""

    def __init__(self, params: Sequence[torch.nn.Parameter], group=None):
        self.params = [p for p in params if p.requires_grad]
        self.group = group

    def __call__(self) -> None:
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(self.group) == 1:
            return
        grads = []
        for p in self.params:
            if p.grad is None:            # a rank whose rows did not reach p still has to join the collective
                p.grad = torch.zeros_like(p)
            grads.append(p.grad)
        flat = torch.cat([g.reshape(-1) for g in grads])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group)
        offset = 0
        for g in grads:
            g.copy_(flat[offset:offset + g.numel()].view_as(g))
            offset += g.numel()


# ------------------------------------------------------------------------------------------------ the step

def embed(head, hs: torch.Tensor, normalize: Optional[Callable] = None) -> torch.Tensor:
    """``F.normalize(head(hs).mean(dim=-1), p=2, dim=1)`` of stage1_utils.py:122-123,148-149 with the row
    normalisation on this library's kernel (forward and backward)."""
    fused = getattr(head, "pooled_embedding", None)          # head.FusedCompressionHead: one pass over hs
    pooled = fused(hs) if fused is not None else head(hs).mean(dim=-1)
    return (normalize or Fn.l2_normalize)(pooled)


def normalized_supcon_loss(x: torch.Tensor, labels: torch.Tensor, loss_fn, topk_neg: int = 32, alpha: float = 0.0,
                           normalize: Optional[Callable] = None) -> torch.Tensor:
    """normalise + loss in one call (SURVEY §8 a1): ``x`` are the un-normalised pooled features (N, d)."""
    return call_loss(loss_fn, (normalize or Fn.l2_normalize)(x), labels, topk_neg, alpha)


def call_loss(loss_fn, z, labels, topk_neg: int, alpha: float) -> torch.Tensor:
    """``loss_fn(z, labels, topk_neg=..., alpha=...)`` (stage1_utils.py:125), or ``loss_fn(z, labels)`` for a loss
    without mining arguments such as ``SupConMultiClassLoss`` (train_multiclass_con.py:162,210)."""
    if getattr(loss_fn, "takes_mining_args", True):
        return loss_fn(z, labels, topk_neg=topk_neg, alpha=alpha)
    return loss_fn(z, labels)


def _to_device(waveforms, labels, device):
    return waveforms.to(device, non_blocking=True), labels.to(device, non_blocking=True).long()


def _check_augment(cfg, augment):
    if getattr(cfg, "use_rawboost", False) and augment is None:
        raise ValueError("cfg.use_rawboost is set but RawBoost lives outside this package: pass "
                         "augment=<callable(waveforms, cfg)> (e.g. the reference's apply_rawboost_batch)")


def train_one_epoch(encoder, head, loss_fn, loader, optimizer, device, epoch, cfg, *,
                    normalize: Optional[Callable] = None, augment: Optional[Callable] = None,
                    grad_sync: Optional[Callable] = None, max_grad_norm: float = 5.0, label_index: int = 1):
    """One training epoch; returns ``(mean loss over steps and ranks, alpha)`` like stage1_utils.py:101-134.

    ``loader`` yields ``(waveforms, labels, *rest)``; zero samples are padding (``attention_mask``).  The encoder
    runs without grad unless ``cfg.finetune_encoder``.  ``grad_sync`` (e.g. ``GradSync(head.parameters())``) runs
    after ``backward`` when the loss is the sharded global-batch loss.  ``label_index`` picks the label column
    of the batch tuple: 1 = bonafide/spoof, 2 = the multi-class ids of train_multiclass_con.py:147."""
    _check_augment(cfg, augment)
    finetune = bool(cfg.finetune_encoder)
    encoder.train(finetune)
    head.train()
    alpha = alpha_for_epoch(epoch, cfg)
    running = RunningLoss(device)
    for batch in loader:
        waveforms, labels = _to_device(batch[0], batch[label_index], device)
        if augment is not None and getattr(cfg, "use_rawboost", False):
            waveforms = augment(waveforms, cfg)
        mask = (waveforms != 0.0).long()
        with torch.set_grad_enabled(finetune):
            hs = encoder(waveforms, attention_mask=mask)
        z = embed(head, hs, normalize)
        loss = call_loss(loss_fn, z, labels, cfg.topk_neg, alpha)

        optimizer.zero_grad(set_to_none=True)
        loss.backward()
        if grad_sync is not None:
            grad_sync()
        torch.nn.utils.clip_grad_norm_(head.parameters(), max_grad_norm)
        optimizer.step()
        running.add(loss)
    return running.average(), alpha


@torch.no_grad()
def evaluate(encoder, head, loss_fn, loader, device, cfg, *, normalize: Optional[Callable] = None,
             label_index: int = 1):
    """Mean loss over a loader with alpha = 0 and no graph (stage1_utils.py:137-153)."""
    encoder.eval()
    head.eval()
    running = RunningLoss(device)
    for batch in loader:
        waveforms, labels = _to_device(batch[0], batch[label_index], device)
        hs = encoder(waveforms, attention_mask=(waveforms != 0.0).long())
        running.add(call_loss(loss_fn, embed(head, hs, normalize), labels, cfg.topk_neg, 0.0))
    return running.average()


# ------------------------------------------------------------------ epochs from a store of layer means

def _check_store_cfg(cfg, training: bool) -> None:
    if getattr(cfg, "finetune_encoder", False):
        raise ValueError("cfg.finetune_encoder is set: the encoder's output changes every step, so a store of its "
                         "layer means would be stale; train with train_one_epoch")
    if training and getattr(cfg, "use_rawboost", False):
        raise ValueError("cfg.use_rawboost is set: augmented waveforms give new hidden states every epoch, so a store "
                         "of layer means would be stale; train with train_one_epoch")


def _store_indices(store, batch, device) -> torch.Tensor:
    rows = [int(i) for i in batch]
    if rows and not (0 <= min(rows) and max(rows) < store.filled):
        raise IndexError(f"batch indices must lie in [0, {store.filled}), the clips in the store")
    return torch.tensor(rows, dtype=torch.int64).to(device, non_blocking=True)


def _store_embed(head, store, idx: torch.Tensor, normalize: Optional[Callable] = None) -> torch.Tensor:
    return (normalize or Fn.l2_normalize)(head.pooled_embedding_from_store(store, idx))


def train_one_epoch_from_store(head, loss_fn, store, batches, optimizer, device, epoch, cfg, *,
                               normalize: Optional[Callable] = None, grad_sync: Optional[Callable] = None,
                               max_grad_norm: float = 5.0):
    """``train_one_epoch`` for a frozen encoder whose layer means are in ``store``
    (``feature_store.build_layer_mean_store``): no encoder call.  ``batches`` are index lists into the store, e.g.
    the batches of the same ``BalancedBatchSampler``; labels are gathered from the store on the device.  ``head`` is
    a ``FusedCompressionHead``.  With the same batches, seeds and dropout stream the epoch is ``train_one_epoch``'s
    whenever the encoder's output for a clip does not depend on its batch mates.  Returns ``(mean loss, alpha)``.
    On several ranks (a ``feature_store.ShardedLayerMeanStore``, ``BalancedBatchSampler(rank=, world_size=)`` batches,
    ``ShardedSupConLoss``) pass ``grad_sync=GradSync(head.parameters())``: it runs after ``backward`` as in
    ``train_one_epoch``.  Raises when ``cfg.finetune_encoder`` or ``cfg.use_rawboost`` is set: the store would be stale."""
    _check_store_cfg(cfg, training=True)
    head.train()
    alpha = alpha_for_epoch(epoch, cfg)
    running = RunningLoss(device)
    for batch in batches:
        idx = _store_indices(store, batch, device)
        z = _store_embed(head, store, idx, normalize)
        loss = call_loss(loss_fn, z, store.labels_of(idx), cfg.topk_neg, alpha)

        optimizer.zero_grad(set_to_none=True)
        loss.backward()
        if grad_sync is not None:
            grad_sync()
        torch.nn.utils.clip_grad_norm_(head.parameters(), max_grad_norm)
        optimizer.step()
        running.add(loss)
    return running.average(), alpha


@torch.no_grad()
def evaluate_from_store(head, loss_fn, store, batches, device, cfg, *, normalize: Optional[Callable] = None):
    """``evaluate`` over index lists into a store of layer means (alpha = 0, no graph).  Raises when
    ``cfg.finetune_encoder`` is set."""
    _check_store_cfg(cfg, training=False)
    head.eval()
    running = RunningLoss(device)
    for batch in batches:
        idx = _store_indices(store, batch, device)
        running.add(call_loss(loss_fn, _store_embed(head, store, idx, normalize), store.labels_of(idx),
                              cfg.topk_neg, 0.0))
    return running.average()


# --------------------------------------------------------------------------------------------- rendezvous

def setup_distributed(backend: str = "nccl"):
    """``(is_distributed, rank, world_size, local_rank)`` from torchrun's or SLURM's environment; initialises the
    process group when there is more than one rank (stage1_utils.py:156-172)."""
    env = os.environ
    if "RANK" in env and "WORLD_SIZE" in env:
        rank, world, local = int(env["RANK"]), int(env["WORLD_SIZE"]), int(env.get("LOCAL_RANK", 0))
    elif "SLURM_PROCID" in env:
        rank, world, local = int(env["SLURM_PROCID"]), int(env.get("SLURM_NTASKS", "1")), int(env.get("SLURM_LOCALID", "0"))
    else:
        return False, 0, 1, 0
    if world <= 1:
        return False, 0, 1, 0
    if backend == "nccl":
        torch.cuda.set_device(local)
    if not dist.is_initialized():
        dist.init_process_group(backend=backend, init_method="env://", rank=rank, world_size=world)
    return True, rank, world, local


# -------------------------------------------------------------------------------------- Stage-2 hand-over

@torch.no_grad()
def export_embeddings(encoder, head, loader, device, out_dir: str, split_name: str, *,
                      normalize: Optional[Callable] = None, overwrite: bool = False):
    """Write ``{split}_embeddings.npy`` (N, d) float32 and ``{split}_labels.npy`` (N,) - the files
    train_stage2_classifier.py:29-37 loads - from a frozen encoder + head
    (extract_stage1_embeddings.py:148-163,170-231).  Existing files are kept unless ``overwrite``.
    Returns ``(emb_path, lab_path, n)``; ``n`` is None when the files were already there, 0 for an empty loader
    (nothing is written, as in the reference)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    emb_path = os.path.join(out_dir, f"{split_name}_embeddings.npy")
    lab_path = os.path.join(out_dir, f"{split_name}_labels.npy")
    if not overwrite and os.path.exists(emb_path) and os.path.exists(lab_path):
        return emb_path, lab_path, None
    encoder.eval()
    head.eval()
    z_parts, y_parts = [], []
    for waveforms, labels, *_ in loader:
        waveforms = waveforms.to(device, non_blocking=True)
        hs = encoder(waveforms, attention_mask=(waveforms != 0.0).long())
        z_parts.append(embed(head, hs, normalize).float().to("cpu", non_blocking=True))
        y_parts.append(torch.as_tensor(labels).to("cpu"))
    if not z_parts:
        return emb_path, lab_path, 0
    if torch.device(device).type == "cuda":
        torch.cuda.synchronize(device)
    z_all = torch.cat(z_parts).numpy()
    y_all = torch.cat(y_parts).numpy()
    np.save(emb_path, z_all)
    np.save(lab_path, y_all)
    return emb_path, lab_path, int(z_all.shape[0])


# ------------------------------------------------------------------------ one CUDA-graph replay per step

class GraphedHeadStep:
    """head -> time mean -> normalise -> loss -> backward -> (grad sync) -> clip -> optimizer step as ONE CUDA
    graph replay per training step (SURVEY §8 f-N2): the step of stage1_utils.py:121-130 for a frozen encoder,
    with no host sync and no per-kernel launch cost.  Measured at batch 64 on the (64, 25, 1024, 199) fp32
    encoder output (tools/graphed_step_bench.py, profiles/r01_graphed_head_step.json): 1.07 ms eager ->
    0.86 ms per replay, of which the layer mean over the 1.3 GB input is 0.21 ms (6.3 TB/s, HBM-bound).

        step = GraphedHeadStep(head, loss_fn, optimizer, hs_example, labels_example, topk_neg=cfg.topk_neg)
        for hs, labels in batches:                      # hs = encoder output (B, K, F, T), computed without grad
            loss = step(hs, labels, alpha)              # device scalar, overwritten by the next call
            running.add(loss)

    Requirements: CUDA tensors of the example's shape every step; an optimizer constructed with
    ``capturable=True`` (Adam/AdamW) so its step counter lives on the device.  ``alpha`` and ``topk_neg`` are
    plain kernel arguments, so one graph is captured per distinct alpha (one per epoch on the reference's
    schedule) and kept.  The warm-up iterations torch needs before a capture run on the example batch; the
    parameters and the optimizer state are put back afterwards, in place, so constructing the object does not
    train.  ``grad_sync`` (``GradSync``) is captured into the graph when given (NCCL collectives capture).
    Inputs are copied into the static buffers ``step.hs`` / ``step.labels`` unless they ARE those buffers (an
    encoder that writes its output there saves the copy).

    A ``loss_fn`` with a cross-batch ``memory`` (``MemorySupConLoss``) is captured at the memory's capacity and reads
    its fill level and ring head on the device, so one graph serves the memory while it fills, once it is full and
    as it wraps.  Construction and capture leave the memory's contents and state as they were (the warm-up and
    the captured step enqueue nothing that stays).  Each replay enqueues its batch on the device and advances the
    host ``filled`` / ``head`` by B, so ``memory.embeddings`` / ``memory.keys`` describe what the device holds.
    The graphs of different alphas share that one memory.  Eager calls of the loss between replays stay valid as
    long as the batch size does not grow (a larger batch reallocates the buffers the graphs use).

    ``store=`` (a ``feature_store.LayerMeanStore`` or ``ShardedLayerMeanStore``, head = ``FusedCompressionHead``) captures the step of
    ``train_one_epoch_from_store`` instead: the graph gathers and pools the store rows ``step.idx`` and their labels,
    so the static input is the (B,) int64 index vector.  Pass an index example in place of ``hs_example``, no
    labels, and call ``step(idx, alpha=alpha)``: a replay copies ``idx`` and runs."""

    def __init__(self, head, loss_fn, optimizer, hs_example: torch.Tensor, labels_example: Optional[torch.Tensor] = None,
                 *, topk_neg: int = 32, max_grad_norm: float = 5.0, normalize: Optional[Callable] = None,
                 grad_sync: Optional[Callable] = None, warmup: int = 3, store=None):
        if hs_example.device.type != "cuda":
            raise RuntimeError("GraphedHeadStep needs CUDA tensors (there is no CPU path)")
        for group in optimizer.param_groups:
            if not group.get("capturable", False):
                raise ValueError("GraphedHeadStep needs an optimizer built with capturable=True")
        self.head, self.loss_fn, self.optimizer = head, loss_fn, optimizer
        self.topk_neg, self.max_grad_norm = int(topk_neg), float(max_grad_norm)
        self.normalize, self.grad_sync, self.warmup = normalize, grad_sync, max(1, int(warmup))
        self.store = store
        if store is not None:
            if labels_example is not None:
                raise ValueError("with store= the labels come from the store: pass no labels_example")
            if hs_example.dim() != 1 or hs_example.dtype != torch.int64:
                raise ValueError("with store= the example is the (B,) int64 vector of store rows")
            self.idx = hs_example.detach().clone()
            self.hs = self.labels = None
        else:
            if labels_example is None:
                raise ValueError("GraphedHeadStep needs labels_example (or store=)")
            self.hs = hs_example.detach().clone()
            self.labels = labels_example.detach().clone().long()
        self.memory = getattr(loss_fn, "memory", None)
        self._graphs = {}

    def _eager(self, alpha: float) -> torch.Tensor:
        if self.store is not None:
            z = _store_embed(self.head, self.store, self.idx, self.normalize)
            labels = self.store.labels_of(self.idx)
        else:
            z = embed(self.head, self.hs, self.normalize)
            labels = self.labels
        loss = call_loss(self.loss_fn, z, labels, self.topk_neg, alpha)
        self.optimizer.zero_grad(set_to_none=True)
        loss.backward()
        if self.grad_sync is not None:
            self.grad_sync()
        torch.nn.utils.clip_grad_norm_(self.head.parameters(), self.max_grad_norm)
        self.optimizer.step()
        return loss.detach()

    def _snapshot(self):
        params = [p.detach().clone() for p in self.head.parameters()]
        buffers = [b.detach().clone() for b in self.head.buffers()]
        state = {p: {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in st.items()}
                 for p, st in self.optimizer.state.items()}
        memory = self.memory.snapshot() if self.memory is not None else None
        return params, buffers, state, memory

    def _restore(self, snap) -> None:
        params, buffers, state, memory = snap
        if self.memory is not None:
            self.memory.restore(memory)
        with torch.no_grad():
            for p, saved in zip(self.head.parameters(), params):
                p.copy_(saved)
            for b, saved in zip(self.head.buffers(), buffers):
                b.copy_(saved)
            for p, st in self.optimizer.state.items():
                before = state.get(p)
                for k, v in st.items():
                    if not torch.is_tensor(v):
                        continue
                    if before is not None and k in before:
                        v.copy_(before[k])
                    else:
                        v.zero_()                   # state created by the warm-up: back to its initial zeros

    def _capture(self, alpha: float):
        dev = (self.idx if self.store is not None else self.hs).device
        snap = self._snapshot()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(self.warmup):
                self._eager(alpha)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        graph = torch.cuda.CUDAGraph()
        self.optimizer.zero_grad(set_to_none=True)
        with torch.cuda.graph(graph, capture_error_mode="thread_local"):
            loss = self._eager(alpha)
        push = self.memory.last_push if self.memory is not None else None   # what each replay enqueues
        self._restore(snap)
        return graph, loss, push

    def __call__(self, hs: torch.Tensor, labels: Optional[torch.Tensor] = None, alpha: float = 0.0) -> torch.Tensor:
        if self.store is not None:
            if labels is not None or hs.shape != self.idx.shape or hs.dtype != torch.int64:
                raise ValueError(f"GraphedHeadStep was captured for store rows of shape {tuple(self.idx.shape)} "
                                 f"(int64, no labels), got {hs.dtype} {tuple(hs.shape)}"
                                 + (" and labels" if labels is not None else ""))
        elif labels is None or hs.shape != self.hs.shape or labels.shape != self.labels.shape:
            raise ValueError(f"GraphedHeadStep was captured for hs {tuple(self.hs.shape)} / labels "
                             f"{tuple(self.labels.shape)}, got {tuple(hs.shape)} / "
                             f"{tuple(labels.shape) if labels is not None else None}")
        key = float(alpha)
        if key not in self._graphs:
            self._graphs[key] = self._capture(key)
        graph, loss, push = self._graphs[key]
        if self.store is not None:
            if hs.data_ptr() != self.idx.data_ptr():
                self.idx.copy_(hs, non_blocking=True)
        else:
            if hs.data_ptr() != self.hs.data_ptr():     # producers may write straight into step.hs / step.labels
                self.hs.copy_(hs, non_blocking=True)
            if labels.data_ptr() != self.labels.data_ptr():
                self.labels.copy_(labels, non_blocking=True)
        graph.replay()
        if push is not None:
            self.memory.advance_host(*push)
        return loss
