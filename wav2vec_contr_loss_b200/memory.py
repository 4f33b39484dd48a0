"""Cross-batch memory (XBM, Wang et al., CVPR 2020): contrast each batch against the embeddings of earlier batches.

At the Stage-1 batch size (64 per GPU, half of it per class) an anchor sees about 32 negatives, so hard-negative
mining has little to choose from.  ``MemorySupConLoss`` keeps the embeddings and labels of the last ``memory_size``
training samples in a ring buffer on the device and adds them as extra COLUMNS of every anchor's row: the
log-sum-exp, the positives, the negatives and the mined top-K run over batch + memory.  The memory is a constant: it
gets no gradient, costs no encoder work, and the uniformity term stays over the batch's own pairs.  The kernels run
the problem as rows [0, B) against columns [0, B + filled) with SUPCON_FLAG_MEMORY_COLUMNS (include/supcon_b200.h).

A training call (grad enabled, ``z.requires_grad``) uses the memory as it is when the call starts; its batch enters
the memory when its backward has run.  A second training call before the first one's backward rewrites the buffer
that the first backward needs, and that backward then raises (autograd's version check) instead of computing a
gradient against a memory its forward did not see.  Under ``torch.no_grad()`` the loss is ``SupConBinaryLoss`` of
the batch alone and the memory is left as it is, so dev losses stay comparable with runs without a memory.

The ring keeps its ``(head, filled)`` twice: as host ints, and in a device int32 tensor that the enqueue advances
with graph-capturable ops.  A call captured into a CUDA graph (``stage1.GraphedHeadStep``) runs the problem at the
memory's capacity, ``B + memory_size`` columns, and the kernels read the fill level from the device
(``supcon_forward_rows_memory``), so every replay contrasts against the memory as it is at that replay and enqueues
at the current head.  Eager calls keep the ``B + filled`` problem.
"""
from typing import Optional

import torch

from . import _cabi
from . import functional as Fn
from .loss import SupConBinaryLoss


class CrossBatchMemory:
    """Ring buffer of the embeddings and int32 label keys (``canonical_labels``) of the last ``size`` samples.

    One buffer ``[slots + size, d]`` holds ``slots`` batch slots followed by the ring, and the same for the keys: a
    batch of B rows is staged in the last B batch slots, so that one pointer spans batch + memory.  The ring always
    fills slots ``[0, filled)``; ``head`` is where the next row goes.  The buffers are allocated on first use,
    zero-filled (the slots a replay at full capacity reads before they are filled hold finite values), and grow
    only when a larger batch arrives: a step allocates nothing of size O(size * d).  ``state`` is the device copy of
    ``(head, filled)`` (int32, on the buffers' device); the enqueue advances both copies by the same rule.
    """

    def __init__(self, size: int):
        if int(size) < 0:
            raise ValueError(f"memory size must be >= 0, got {size}")
        self.size = int(size)
        self.filled = 0
        self.head = 0
        self.label_dtype: Optional[torch.dtype] = None   # dtype of the labels in memory: keys of int and float labels differ
        self.unit_rows = True                            # every enqueued batch carried the unit-rows promise
        self.state: Optional[torch.Tensor] = None         # device [head, filled], int32
        self._z: Optional[torch.Tensor] = None
        self._keys: Optional[torch.Tensor] = None
        self._arange: Optional[torch.Tensor] = None       # 0 .. size-1 (int64): ring offsets of a batch
        self._slots = 0
        self.last_push = None                             # (rows, unit_rows, label_dtype) of the last enqueue

    def reset(self):
        """Empty the memory (the buffers are kept)."""
        self.filled = 0
        self.head = 0
        self.label_dtype = None
        self.unit_rows = True
        if self.state is not None:
            self.state.zero_()

    @property
    def embeddings(self) -> Optional[torch.Tensor]:
        """The filled slots ``[filled, d]`` in slot order (a view), or None before first use."""
        return None if self._z is None else self._z[self._slots:self._slots + self.filled]

    @property
    def keys(self) -> Optional[torch.Tensor]:
        """int32 label keys of the filled slots (a view), or None before first use."""
        return None if self._keys is None else self._keys[self._slots:self._slots + self.filled]

    def check_labels(self, labels: torch.Tensor):
        if self.label_dtype is not None and labels.dtype != self.label_dtype:
            raise ValueError(f"labels of dtype {labels.dtype} cannot be compared with the memory's labels of dtype "
                             f"{self.label_dtype}: their class keys differ; reset() the memory first")

    def enqueue(self, z: torch.Tensor, labels: torch.Tensor, unit_rows: bool = False):
        """Append a batch (detached); the oldest rows are overwritten once the memory is full.  ``unit_rows``: the
        rows are L2-normalised (the tensor-core path needs that promise for every row it sees)."""
        self.check_labels(labels)
        zc = Fn.canonical_z(z.detach())
        keys = Fn.canonical_labels(labels, zc.size(0))
        self._reserve(0, zc)
        self._push(zc, keys, unit_rows, labels.dtype)

    # ---- used by MemorySupConLoss ----
    def stage(self, zc: torch.Tensor, keys: torch.Tensor, capacity: bool = False):
        """Copy a batch into the batch slots in front of the ring.  Returns ``(z_all, keys_all)``: views spanning
        the batch (rows [0, B)) and the filled memory (rows [B, B + filled)), or with ``capacity`` the whole ring
        (rows [B, B + size))."""
        b = zc.size(0)
        self._reserve(b, zc)
        lo, hi = self._slots - b, self._slots + (self.size if capacity else self.filled)
        with torch.no_grad():
            self._z[lo:self._slots].copy_(zc)
            self._keys[lo:self._slots].copy_(keys)
        return self._z[lo:hi], self._keys[lo:hi]

    def _reserve(self, batch: int, zc: torch.Tensor):
        d, dtype, dev = zc.size(1), zc.dtype, zc.device
        if self._z is not None:
            if (self._z.size(1), self._z.dtype, self._z.device) != (d, dtype, dev):
                raise ValueError(f"batch of width {d}, {dtype} on {dev} does not match the memory's "
                                 f"{self._z.size(1)}, {self._z.dtype} on {self._z.device}")
            if batch <= self._slots:
                return
        slots = max(batch, self._slots)
        z = torch.zeros((slots + self.size, d), dtype=dtype, device=dev)
        keys = torch.zeros(slots + self.size, dtype=torch.int32, device=dev)
        if self._z is not None and self.filled:
            z[slots:slots + self.filled].copy_(self.embeddings)
            keys[slots:slots + self.filled].copy_(self.keys)
        if self.state is None:
            self.state = torch.tensor([self.head, self.filled], dtype=torch.int32, device=dev)
            self._arange = torch.arange(self.size, dtype=torch.int64, device=dev)
        self._z, self._keys, self._slots = z, keys, slots

    def _push(self, rows: torch.Tensor, keys: torch.Tensor, unit_rows: bool, label_dtype: torch.dtype):
        """Enqueue at the DEVICE head and advance both copies of the state: the same slots as the host state
        names, and capturable into a CUDA graph: each replay enqueues at the head as it is at that replay."""
        n, m = rows.size(0), self.size
        self.last_push = (n, bool(unit_rows), label_dtype)
        if m and n:
            if n > m:   # only the newest m rows survive
                rows, keys, n = rows[n - m:], keys[n - m:], m
            with torch.no_grad():
                slots = (self._arange[:n] + self.state[0]).remainder_(m)
                self._z[self._slots:].index_copy_(0, slots, rows)
                self._keys[self._slots:].index_copy_(0, slots, keys)
                self.state.add_(n)
                self.state[0].remainder_(m)
                self.state[1].clamp_(max=m)
        self.advance_host(*self.last_push)

    def advance_host(self, n: int, unit_rows: bool, label_dtype: torch.dtype):
        """The host half of an enqueue of ``n`` rows (a graph replay has done the device half)."""
        self.label_dtype = label_dtype
        self.unit_rows = self.unit_rows and bool(unit_rows)
        m = self.size
        if m == 0 or n == 0:
            return
        n = min(n, m)
        self.head = (self.head + n) % m
        self.filled = min(self.filled + n, m)

    def snapshot(self):
        """Contents and both copies of the state, for ``restore``."""
        if self._z is None:
            return None
        return (self.embeddings.clone(), self.keys.clone(), self.head, self.filled, self.label_dtype,
                self.unit_rows)

    def restore(self, snap):
        """Put back what ``snapshot`` saved, in place (the buffers a captured graph uses stay where they are)."""
        if self._z is None:
            return
        if snap is None:
            self.reset()
            return
        z, keys, self.head, self.filled, self.label_dtype, self.unit_rows = snap
        with torch.no_grad():
            self._z[self._slots:self._slots + self.filled].copy_(z)
            self._keys[self._slots:self._slots + self.filled].copy_(keys)
            self.state.copy_(torch.tensor([self.head, self.filled], dtype=torch.int32))


class _MemorySupConFunction(torch.autograd.Function):
    """SupCon of the batch rows against batch + memory columns; the gradient flows to the batch rows only."""

    @staticmethod
    def forward(ctx, z, z_all, keys_all, prob, memory, unit_rows, label_dtype, mem_filled):
        stats, partials, loss = Fn.forward_rows(z_all, keys_all, prob, want_loss=True, mem_filled=mem_filled)
        # z_all / keys_all are views of the memory's buffers: any later write to them (the next call's staging,
        # this batch's enqueue) bumps their version, and unpacking them in backward() then raises
        ctx.save_for_backward(z_all, keys_all, stats, partials)
        ctx.prob, ctx.memory, ctx.unit_rows, ctx.label_dtype = prob, memory, unit_rows, label_dtype
        ctx.mem_filled = mem_filled
        ctx.in_dtype = z.dtype
        return Fn._loss_dtype(loss, z.dtype)

    @staticmethod
    def backward(ctx, grad_out):
        z_all, keys_all, stats, partials = ctx.saved_tensors
        dz = Fn.backward_rows(z_all, keys_all, stats, partials, grad_out, ctx.prob, out_dtype=z_all.dtype,
                              mem_filled=ctx.mem_filled)
        b = ctx.prob.n_rows
        ctx.memory._push(z_all[:b], keys_all[:b], ctx.unit_rows, ctx.label_dtype)   # the batch enters the memory
        return dz.to(ctx.in_dtype), None, None, None, None, None, None, None


class MemorySupConLoss(SupConBinaryLoss):
    """``SupConBinaryLoss`` whose anchors are also contrasted against a memory of the last ``memory_size`` training
    samples (see the module docstring).  Same ``forward(z, labels, topk_neg=32, alpha=0.0)``, ``kernel_flags`` and
    ``assume_unit_rows``, so it can be the ``loss_fn`` of ``stage1.train_one_epoch`` as it is.  Single GPU only."""

    def __init__(self, temperature: float = 0.2, similarity: str = "geodesic",
                 uniformity_weight: float = 0.0, uniformity_t: float = 2.0, memory_size: int = 4096):
        super().__init__(temperature, similarity, uniformity_weight, uniformity_t)
        self.memory = CrossBatchMemory(memory_size)

    def forward(self, z: torch.Tensor, labels: torch.Tensor, topk_neg: int = 32,
                alpha: float = 0.0) -> torch.Tensor:
        if not (torch.is_grad_enabled() and z.requires_grad):
            return super().forward(z, labels, topk_neg=topk_neg, alpha=alpha)   # evaluation: the batch alone
        Fn._require_cuda(z, "z")
        mem = self.memory
        mem.check_labels(labels)
        zc = Fn.canonical_z(z.detach())
        b, d = zc.shape
        keys = Fn.canonical_labels(labels, b)
        sim_id = Fn.similarity_id(self.similarity)
        unit = bool(Fn.unit_rows_flag(z, sim_id, self.assume_unit_rows))
        # captured into a CUDA graph: the problem at capacity, the fill level read on the device at each replay
        capturing = torch.cuda.is_current_stream_capturing()
        n_total = b + (mem.size if capturing else mem.filled)
        if n_total < 2:
            # reference loss.py:138-139,149: no anchor has a positive and there is no pair; nothing to backward
            mem._reserve(0, zc)
            mem._push(zc, keys, unit, labels.dtype)
            return torch.tensor(0.0, device=z.device, requires_grad=True)
        z_all, keys_all = mem.stage(zc, keys, capacity=capturing)
        flags = int(self.kernel_flags) | _cabi.FLAG_MEMORY_COLUMNS
        if unit and mem.unit_rows:
            flags |= _cabi.FLAG_UNIT_ROWS
        prob = Fn.make_problem(n_total, d, Fn._dtype_id(zc), tau=float(self.tau), similarity=sim_id,
                               lambda_uni=self.lambda_uni, uni_t=self.uni_t, topk=int(topk_neg), alpha=float(alpha),
                               n_rows=b, flags=flags)
        mem_filled = mem.state[1:] if capturing else None
        return _MemorySupConFunction.apply(z, z_all, keys_all, prob, mem, unit, labels.dtype, mem_filled)


__all__ = ["CrossBatchMemory", "MemorySupConLoss"]
