"""Device-resident store of a frozen encoder's layer-averaged hidden states, for training the Stage-1 head without
running the encoder every epoch.

The head's first operation is the mean over the encoder's K layers (compression_module.py:48-65), which is linear
and comes before Dropout.  With a frozen encoder and no waveform augmentation that mean is the same for a clip in
every epoch, so

    m[c] = (1/K) sum_k hs[c, k]          (F, T) fp32 per clip

is all an epoch needs: Dropout (fresh masks), LeakyReLU, the time mean and ``mlp3`` are recomputed from it.  At
F = 1024, T = 199 a clip takes 815 KB, so about 25 k clips fit a B200 in 21 GB.

``build_layer_mean_store`` runs the encoder once over a loader and writes each clip's mean with
``supcon_head_layer_mean_typed``; ``LayerMeanStore.pool`` is ``supcon_head_store_pool_forward``, which gathers
the rows of a batch and pools them with the arithmetic and the dropout masks of ``head.layer_time_pool`` on the
same batch read from hs.  Training from the store therefore walks the trajectory of ``stage1.train_one_epoch``
whenever the encoder's output for a clip does not depend on the other clips of its batch.

``ShardedLayerMeanStore`` / ``build_sharded_layer_mean_store`` split the store over the GPUs of one node: slot i
lives on rank i % R, each rank encodes only its own clips, and ``pool`` reads the other ranks' rows through peer
memory (``supcon_head_sharded_store_pool_forward``), with the same bits as ``LayerMeanStore.pool``.

Preconditions: frozen encoder, no waveform augmentation, the same crop / pad of each clip in every epoch.  The rows
are fp32 by default, which keeps that equality (a rounded mean would lose it).  ``dtype=torch.float16`` keeps them
in fp16 instead, at half the bytes: twice the clips per GPU.  Each layer mean is then rounded once, to nearest even
(``rows32.half()``), and the kernel widens it back exactly, so pooling an fp16 store gives bit for bit what pooling
an fp32 store of the same widened values gives.  A finite mean beyond fp16's range (|m| >= 65520 rounds to inf) is
an error: the build and a load raise naming the slot, and ``save`` refuses.  There is no backward: the store is a
constant.

On disk a store is a directory of two ``.npy`` files, ``rows.npy`` (n, F, T) in C order, fp32 (``<f4``) or for an
fp16 store ``<f2``, and ``labels.npy`` (n,) int64, in slot order whatever the number of ranks that wrote it: the
layout of the reference's layer-mean feature memmap (extract_encoder_embeddings.py).  ``save`` / ``load_layer_mean_store`` /
``load_sharded_layer_mean_store`` stream the rows between the file and the device through two pinned staging
buffers, so the host never holds the array.
"""
import io
import mmap
import os
import shutil
import socket

import numpy as np
import torch
import torch.distributed as dist

from . import _cabi
from . import functional as Fn

__all__ = ["LayerMeanStore", "build_layer_mean_store", "ShardedLayerMeanStore", "build_sharded_layer_mean_store",
           "shard_slots", "load_layer_mean_store", "load_sharded_layer_mean_store"]

ROWS_FILE, LABELS_FILE = "rows.npy", "labels.npy"
STAGE_BYTES = 64 << 20      # each of the two pinned staging buffers of a save or load
# the element types of a store's rows: C-ABI store_dtype, .npy descr, name
_STORE_DTYPES = {torch.float32: (_cabi.F32, "<f4", "fp32"), torch.float16: (_cabi.F16, "<f2", "fp16")}


def _store_dtype(dtype) -> torch.dtype:
    if dtype not in _STORE_DTYPES:
        raise ValueError(f"the store dtype must be torch.float32 or torch.float16, got {dtype}")
    return dtype


class LayerMeanStore:
    """``rows`` (n, F, T) of ``dtype`` (fp32, or fp16 at half the bytes: module docstring) and ``labels`` (n,)
    int64, both on one device; slots ``[0, filled)`` are written.

    ``append`` writes the layer means of a batch of hidden states at the next ``B`` slots.  ``pool`` and
    ``labels_of`` take a device int64 index vector, so both can be captured in a CUDA graph and fed new indices
    every replay.  An index outside ``[0, filled)`` gives a NaN pooled row (the loss turns NaN) instead of a fault."""

    def __init__(self, n: int, feat: int, frames: int, device, dtype=torch.float32):
        if n < 1 or feat < 1 or frames < 1:
            raise ValueError(f"bad store shape ({n}, {feat}, {frames})")
        dtype = _store_dtype(dtype)
        device = torch.device(device)
        too_big = _fit_error(n, feat, frames, device, store_bytes(n, feat, frames, dtype), dtype)
        if too_big:
            raise MemoryError(too_big)
        self.rows = torch.empty((n, feat, frames), dtype=dtype, device=device)
        self.labels = torch.full((n,), -1, dtype=torch.int64, device=device)
        self.filled = 0
        self._rounding = _Rounding(self.rows)

    @property
    def n(self) -> int:
        return self.rows.shape[0]

    @property
    def feat(self) -> int:
        return self.rows.shape[1]

    @property
    def frames(self) -> int:
        return self.rows.shape[2]

    @property
    def device(self) -> torch.device:
        return self.rows.device

    @property
    def dtype(self) -> torch.dtype:
        return self.rows.dtype

    def append(self, hs: torch.Tensor, labels: torch.Tensor) -> int:
        """Write ``mean_k hs[b, k]`` (hs = (B, K, F, T), fp32 or bf16; other dtypes through an fp32 copy) and
        ``labels[b]`` at slot ``filled + b``; returns the first slot written.  An fp16 store rounds the fp32 mean to
        nearest even and notes, on the device, a finite mean that became inf (``build_layer_mean_store`` and
        ``save`` raise on it)."""
        b = _check_hs(hs, self.feat, self.frames, self.filled)
        if tuple(labels.shape) != (b,):
            raise ValueError(f"labels must be ({b},), got {tuple(labels.shape)}")
        if self.filled + b > self.n:
            raise ValueError(f"the store holds {self.n} clips: no room for {b} more after {self.filled}")
        slot0 = self.filled
        self._rounding.write_means(slot0, hs)
        self.labels[slot0:slot0 + b].copy_(labels.detach().long(), non_blocking=True)
        self.filled += b
        return slot0

    def labels_of(self, idx: torch.Tensor) -> torch.Tensor:
        """labels of the slots ``idx`` (device int64).  Indices are clamped into range for this gather only: the
        pooled row of a bad index is already NaN, and the gather must not fault before the NaN reaches the loss."""
        return self.labels.index_select(0, idx.clamp(0, max(self.filled, 1) - 1))

    def pool(self, idx: torch.Tensor, dropout_p: float = 0.0, negative_slope: float = 0.01,
             rng_state=None) -> torch.Tensor:
        """(B, F) fp32: ``LeakyReLU(Dropout(rows[idx])).mean(-1)``, equal bit for bit to ``head.layer_time_pool``
        on the hs of those clips with the same ``rng_state`` {seed, offset}.  No host sync."""
        idx, rng = _pool_args(self.rows, idx, dropout_p, rng_state)
        with torch.cuda.device(self.device):
            pooled = torch.empty((idx.shape[0], self.feat), dtype=torch.float32, device=self.device)
            _cabi.check(_cabi.load().supcon_head_store_pool_forward_typed(
                Fn._p(self.rows), _STORE_DTYPES[self.dtype][0], self.filled, self.feat, self.frames, Fn._p(idx),
                idx.shape[0], float(dropout_p), float(negative_slope), Fn._p(rng), Fn._p(pooled),
                Fn._stream(self.device)), "supcon_head_store_pool_forward_typed")
        return pooled

    def save(self, path, overwrite: bool = False):
        """Write slots ``[0, filled)`` to the directory ``path`` (``rows.npy``, ``labels.npy``; module docstring).
        The files are written into ``<path>.partial``, fsynced and then renamed to ``path``, so a save that dies
        leaves nothing that loads.  An existing ``path`` is kept unless ``overwrite`` (as ``export_embeddings``
        keeps its files): returns None then, else the number of clips written.  Raises on an empty store and on an
        fp16 store holding a mean that rounded to inf."""
        path = os.fspath(path)
        if self.filled < 1:
            raise ValueError("the store is empty: nothing to save")
        bad = self._rounding.first_overflow()
        if bad is not None:
            raise ValueError(_overflow_message(bad) + ": not saved")
        if os.path.exists(path) and not overwrite:
            return None
        partial = path + ".partial"
        try:
            header = _create_rows_file(partial, (self.filled, self.feat, self.frames), _STORE_DTYPES[self.dtype][1])
            _write_rows(self.rows, range(self.filled), partial, header)
            _finish_save(partial, path, self.labels[:self.filled])
        except BaseException:
            _discard(partial)
            raise
        return self.filled

    @classmethod
    def from_arrays(cls, rows, labels, device, dtype=torch.float32) -> "LayerMeanStore":
        """A store of ``n == filled`` clips from host arrays: ``rows`` (n, F, T) float32 or float16 as a numpy
        array, memmap or CPU tensor, ``labels`` (n,) integers.  Into the default fp32 store float32 is copied bit
        for bit and float16 widened exactly; into an fp16 store (``dtype=torch.float16``) float16 is copied bit for
        bit and float32 rounded to nearest even on the store's device (``rows.half()``).  A memmap of a whole
        ``.npy`` file is read from the file in chunks, any other array copied in chunks; either way through the
        pinned staging buffers, never as a whole.  Raises on another dtype (float64 would round), another rank,
        labels that are not (n,) integers and a float32 value that rounds to inf in fp16 (naming the file and the
        slot)."""
        src = _RowSource(rows)
        lab = _label_tensor(labels, src.n)
        store = cls(src.n, src.feat, src.frames, device, dtype)
        _read_rows(src, range(src.n), store._rounding)
        bad = store._rounding.first_overflow()
        if bad is not None:
            raise ValueError(f"{src.name}: {_overflow_message(bad)}")
        store.labels.copy_(lab)
        store.filled = src.n
        return store


def load_layer_mean_store(path, device, dtype=torch.float32) -> LayerMeanStore:
    """The store that ``LayerMeanStore.save`` or ``ShardedLayerMeanStore.save`` (any number of ranks) wrote to
    ``path``, or layer means extracted elsewhere in that layout, on ``device``: ``n == filled ==`` the file's row
    count; ``dtype`` the store's (``from_arrays``), whatever the file's.  Raises FileNotFoundError on a missing store
    and ValueError naming the file on a truncated or unreadable one, besides the checks of
    ``LayerMeanStore.from_arrays``."""
    return LayerMeanStore.from_arrays(*_open_store(path), device, dtype)


def store_bytes(n: int, feat: int, frames: int, dtype=torch.float32) -> int:
    """device bytes of a store of n clips: rows of ``dtype`` (4 or 2 bytes an element) and int64 labels"""
    return n * feat * frames * _store_dtype(dtype).itemsize + n * 8


def _fit_error(n: int, feat: int, frames: int, device: torch.device, need: int, dtype=torch.float32) -> str:
    """why ``need`` bytes for a store of n clips do not fit the free memory of ``device`` ("" when they do)"""
    if device.type != "cuda":
        return ""
    free, _ = torch.cuda.mem_get_info(device)
    if need <= free:
        return ""
    return (f"a store of {n} clips x ({feat}, {frames}) {_STORE_DTYPES[dtype][2]} takes {need / 1e9:.2f} GB; "
            f"{free / 1e9:.2f} GB are free on {device}")


def _overflow_message(slot: int) -> str:
    return (f"slot {slot}: a finite layer mean rounds to inf in fp16 (largest finite value 65504); "
            f"keep this store in fp32")


class _Rounding:
    """Writes fp32 values into the rows of a store.  An fp32 store takes them as they are; an fp16 store rounds them
    to nearest even (torch's ``copy_``, so the rows equal ``rows32.half()``) and keeps on the device the first
    element where a finite value became inf: no host sync until ``first_overflow``.  Shared by ``append``, the
    sharded build and the loads."""
    NONE = 1 << 62

    def __init__(self, rows: torch.Tensor):
        self.rows = rows
        self.row = rows.shape[1] * rows.shape[2]
        self.scratch = None                                  # fp16: (B, F, T) fp32 layer means, kept between calls
        self.first = (torch.full((), self.NONE, dtype=torch.int64, device=rows.device)
                      if rows.dtype == torch.float16 else None)

    def write_means(self, row0: int, hs: torch.Tensor) -> None:
        """``rows[row0 + b] = mean_k hs[b, k]`` with ``write_layer_means``: in place, or for fp16 through the fp32
        scratch and ``put``"""
        if self.first is None:
            write_layer_means(self.rows, row0, hs)
            return
        b = hs.shape[0]
        if self.scratch is None or self.scratch.shape[0] < b:
            self.scratch = torch.empty((b,) + tuple(self.rows.shape[1:]), dtype=torch.float32,
                                       device=self.rows.device)
        write_layer_means(self.scratch, 0, hs)
        self.put(row0 * self.row, self.scratch[:b].view(-1))

    def put(self, offset: int, src: torch.Tensor) -> None:
        """the rows' flat elements ``[offset, offset + src.numel())`` = ``src`` (fp32, on the rows' device),
        rounded to the store dtype, in the current stream"""
        dst = self.rows.view(-1)[offset:offset + src.numel()]
        dst.copy_(src)
        if self.first is None:
            return
        hit, i = (dst.isinf() & src.isfinite()).to(torch.uint8).max(0)       # i: the first hit, if any
        torch.minimum(self.first, torch.where(hit.bool(), i + offset, self.NONE), out=self.first)

    def first_overflow(self):
        """the first row holding a finite value rounded to inf, or None (always None for fp32; syncs for fp16)"""
        if self.first is None:
            return None
        first = int(self.first)
        return None if first == self.NONE else first // self.row


def _check_hs(hs: torch.Tensor, feat: int, frames: int, slot0: int) -> int:
    """the batch size of hidden states (B, K, F, T) that fit a store of (feat, frames) rows"""
    if hs.dim() != 4:
        raise ValueError(f"hs must be (batch, layers, feat, frames), got {tuple(hs.shape)}")
    b, _, f, t = hs.shape
    if (f, t) != (feat, frames):
        raise ValueError(f"clips {slot0}..{slot0 + b - 1}: hidden states of (F, T) = ({f}, {t}), "
                         f"the store holds ({feat}, {frames})")
    return b


def write_layer_means(rows: torch.Tensor, slot0: int, hs: torch.Tensor) -> None:
    """``rows[slot0 + b] = mean_k hs[b, k]`` with ``supcon_head_layer_mean_typed`` (hs fp32 or bf16; other dtypes
    through an fp32 copy); the caller has checked the shape and the room"""
    Fn._require_cuda(hs, "hs")
    if hs.device != rows.device:
        raise ValueError(f"hs is on {hs.device}, the store on {rows.device}")
    x = hs.detach()
    if x.dtype not in (torch.float32, torch.bfloat16):
        x = x.float()
    x = x.contiguous()
    b, k, f, t = x.shape
    with torch.cuda.device(rows.device):
        _cabi.check(_cabi.load().supcon_head_layer_mean_typed(
            Fn._p(x), _cabi.BF16 if x.dtype == torch.bfloat16 else _cabi.F32, b, k, f, t,
            Fn._p(rows[slot0]), Fn._stream(rows.device)), "supcon_head_layer_mean_typed")


def _pool_args(rows: torch.Tensor, idx: torch.Tensor, dropout_p: float, rng_state):
    """(contiguous idx, rng_state or None) of a pool call on a store whose rows are on ``rows.device``"""
    device = rows.device
    if idx.dim() != 1 or idx.dtype != torch.int64 or idx.device != device:
        raise ValueError(f"idx must be a 1-D int64 tensor on {device}, got {idx.dtype} "
                         f"{tuple(idx.shape)} on {idx.device}")
    Fn._require_cuda(rows, "the store")
    rng = None
    if dropout_p > 0.0:
        if (rng_state is None or rng_state.dtype != torch.int64 or rng_state.numel() != 2
                or rng_state.device != device):
            raise ValueError("dropout needs rng_state = int64 tensor {seed, offset} on the store's device")
        rng = rng_state
    return idx.contiguous(), rng


def _labels_of(labels: torch.Tensor, filled: int, idx: torch.Tensor) -> torch.Tensor:
    return labels.index_select(0, idx.clamp(0, max(filled, 1) - 1))


@torch.no_grad()
def build_layer_mean_store(encoder, loader, device, *, label_index: int = 1, n=None,
                           dtype=torch.float32) -> LayerMeanStore:
    """Run ``encoder`` once over ``loader`` as ``stage1.train_one_epoch`` runs a frozen one (eval mode, no grad,
    ``attention_mask = (waveforms != 0).long()``) and store each clip's layer mean.  Slot i holds the loader's i-th
    clip, so a sequential loader over the dataset gives slot = dataset index.  ``n`` (default
    ``len(loader.dataset)``) is the number of clips to allocate for; a loader that yields fewer leaves the store
    ``filled`` short of ``n``.  Raises on a clip whose (F, T) differs from the first one, on more clips than ``n``
    and on a store that does not fit the device's free memory.  ``label_index`` picks the label column of the batch
    tuple, as in ``train_one_epoch``.  ``dtype`` is the store's (``LayerMeanStore``); an fp16 store raises at the
    end, naming the first slot, when a finite layer mean rounded to inf."""
    from .stage1 import _to_device
    if n is None:
        dataset = getattr(loader, "dataset", None)
        if dataset is None:
            raise ValueError("pass n= (the number of clips) for a loader without a .dataset")
        n = len(dataset)
    encoder.eval()
    store = None
    for batch in loader:
        waveforms, labels = _to_device(batch[0], batch[label_index], device)
        hs = encoder(waveforms, attention_mask=(waveforms != 0.0).long())
        if store is None:
            store = LayerMeanStore(n, hs.shape[-2], hs.shape[-1], device, dtype)
        store.append(hs, labels)
    if store is None:
        raise ValueError("the loader yielded no clips")
    bad = store._rounding.first_overflow()
    if bad is not None:
        raise ValueError(_overflow_message(bad))
    return store


# ---------------------------------------------------------------------- the store sharded over one node's GPUs

def shard_slots(n: int, rank: int, world: int) -> range:
    """the dataset indices (slots) rank ``rank`` of ``world`` holds, in the order of its local rows: slot i lives on
    rank i % world at local row i // world.  ``build_sharded_layer_mean_store``'s loader yields these clips."""
    return range(rank, n, world)


def _agree(problem, group) -> None:
    """Every rank passes its own failed check (an exception, or None); raises the same error on every rank when any
    rank has one.  Checks that can fail on one rank alone go through here, so that no rank is left waiting in a
    collective that the failing rank never joins."""
    got = [None] * dist.get_world_size(group)
    dist.all_gather_object(got, None if problem is None else (type(problem).__name__, str(problem)), group=group)
    bad = [(r, p) for r, p in enumerate(got) if p is not None]
    if bad:
        kind = {"MemoryError": MemoryError, "RuntimeError": RuntimeError}.get(bad[0][1][0], ValueError)
        raise kind("; ".join(f"rank {r}: {msg}" for r, (_, msg) in bad))


class _SymmetricShard:
    """This rank's (rows, F, T) shard of ``dtype`` in symmetric memory (``torch.distributed._symmetric_memory``, as
    the peer exchange of ``distributed.py`` allocates its buffers): the same size on every rank and mapped into every
    process, so ``bases[r]`` is rank r's shard as seen from this one."""

    def __init__(self, rows: int, feat: int, frames: int, device, group, *, dtype=torch.float32):
        import torch.distributed._symmetric_memory as symm
        problem = None
        try:
            self.buf = symm.empty(rows * feat * frames, dtype=dtype, device=device)
        except Exception as exc:  # noqa: BLE001  (refused by the allocator: every rank must hear of it)
            self.buf, problem = None, RuntimeError(f"symmetric allocation of {rows} x ({feat}, {frames}) "
                                                   f"{_STORE_DTYPES[dtype][2]}: {exc}")
        _agree(problem, group)
        self.handle = symm.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        self.rows = self.buf.view(rows, feat, frames)
        self.bases = [int(p) for p in self.handle.buffer_ptrs]

    def write(self, row0: int, hs: torch.Tensor) -> None:
        """fp32 shards: ``rows[row0 + b] = mean_k hs[b, k]`` (the store writes an fp16 shard itself)"""
        write_layer_means(self.rows, row0, hs)

    def close(self) -> None:
        self.rows = self.buf = self.handle = None


class ShardedLayerMeanStore:
    """A ``LayerMeanStore`` of n clips split over the R ranks of ``group`` on one node: slot i is row i // R of the
    shard of rank i % R.  Every rank allocates ceil(n / R) rows; ``rows`` is this rank's shard, ``labels`` (n,) a
    full copy on every rank.  ``pool`` gathers any slot, reading the other ranks' rows through peer memory over
    NVLink, with the values and dropout masks of ``LayerMeanStore.pool`` bit for bit; ``labels_of`` is a local
    gather.  It offers the interface the Stage-1 code calls on a ``LayerMeanStore`` (``pool``, ``labels_of``,
    ``filled``, ``n``, ``feat``, ``frames``, ``device``), so ``FusedCompressionHead.pooled_features_from_store``,
    ``train_one_epoch_from_store``, ``evaluate_from_store`` and ``GraphedHeadStep(store=)`` take it unchanged.

    Construction is collective: every rank passes the same (n, feat, frames) with its own device.  The checks --
    n >= R, the same shape on every rank, the shard fits free memory, one host, every pair of GPUs peer-capable --
    are agreed on first and raise on every rank.  ``close()`` (collective) releases the mapping; call it before
    ``destroy_process_group``.  ``allocate`` replaces the symmetric allocation (tests without a GPU): it is called
    as ``allocate(local_rows, feat, frames, device, group)``, with ``dtype=torch.float16`` added for an fp16 store.
    ``dtype`` (the same on every rank) is the rows' element type, as in ``LayerMeanStore``."""

    def __init__(self, n: int, feat: int, frames: int, device, group=None, *, allocate=None, dtype=torch.float32):
        self.group = group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        device = torch.device(device)
        self.n, self.feat, self.frames = n, feat, frames
        self.local_rows = -(-n // self.world) if n > 0 else 0
        where = [None] * self.world
        dist.all_gather_object(where, ((n, feat, frames), socket.gethostname(), device.index, str(dtype)),
                               group=group)
        _agree(self._local_problem(device, where, dtype), group)
        self.dtype = dtype
        alloc = allocate or _SymmetricShard
        kw = {} if dtype == torch.float32 else {"dtype": dtype}
        self._shard = alloc(self.local_rows, feat, frames, device, group, **kw)
        self.rows = self._shard.rows
        self._rounding = _Rounding(self.rows)
        self.bases = torch.tensor(self._shard.bases, dtype=torch.int64, device=device)
        self.labels = torch.full((n,), -1, dtype=torch.int64, device=device)
        self.filled = 0

    @property
    def device(self) -> torch.device:
        return self.labels.device

    def _local_problem(self, device, where, dtype):
        """this rank's failed precondition, or None; ``where`` = every rank's ((n, F, T), host, device index,
        dtype)"""
        if self.n < self.world:
            return ValueError(f"a store sharded over {self.world} ranks needs at least {self.world} clips, "
                              f"got {self.n}")
        shapes = [w[0] for w in where]
        if len(set(shapes)) != 1:
            return ValueError("the ranks disagree on the store's (n, F, T): " +
                              ", ".join(f"rank {r} {s}" for r, s in enumerate(shapes)))
        kinds = [w[3] for w in where]
        if len(set(kinds)) != 1:
            return ValueError("the ranks disagree on the store dtype: " +
                              ", ".join(f"rank {r} {k}" for r, k in enumerate(kinds)))
        try:
            _store_dtype(dtype)
        except ValueError as exc:
            return exc
        if self.feat < 1 or self.frames < 1:
            return ValueError(f"bad store shape ({self.n}, {self.feat}, {self.frames})")
        too_big = _fit_error(self.local_rows, self.feat, self.frames, device,
                             store_bytes(self.local_rows, self.feat, self.frames, dtype) + self.n * 8, dtype)
        if too_big:
            return MemoryError(f"the shard of {too_big}")
        if device.type != "cuda":
            return None
        # the shards are read over NVLink: one host, and this GPU reaches every other rank's
        alone = "; a sharded store needs the GPUs of one node with peer access: use feature_store.LayerMeanStore"
        if len({w[1] for w in where}) != 1:
            return RuntimeError("the ranks run on several hosts" + alone)
        blocked = [r for r, (_, _, d, _) in enumerate(where)
                   if d != device.index and not torch.cuda.can_device_access_peer(device.index, d)]
        if blocked:
            return RuntimeError(f"cuda:{device.index} has no peer access to the GPU of rank(s) {blocked}" + alone)
        return None

    def labels_of(self, idx: torch.Tensor) -> torch.Tensor:
        """labels of the slots ``idx`` (device int64), from this rank's full copy (clamped as in
        ``LayerMeanStore.labels_of``)"""
        return _labels_of(self.labels, self.filled, idx)

    def pool(self, idx: torch.Tensor, dropout_p: float = 0.0, negative_slope: float = 0.01,
             rng_state=None) -> torch.Tensor:
        """(B, F) fp32, ``LayerMeanStore.pool`` of the slots ``idx`` wherever they live.  No host sync, no
        collective: the other ranks' shards are read in place."""
        if self._shard is None:
            raise RuntimeError("the sharded store is closed")
        idx, rng = _pool_args(self.rows, idx, dropout_p, rng_state)
        with torch.cuda.device(self.device):
            pooled = torch.empty((idx.shape[0], self.feat), dtype=torch.float32, device=self.device)
            _cabi.check(_cabi.load().supcon_head_sharded_store_pool_forward_typed(
                Fn._p(self.bases), self.world, _STORE_DTYPES[self.dtype][0], self.filled, self.feat, self.frames,
                Fn._p(idx), idx.shape[0], float(dropout_p), float(negative_slope), Fn._p(rng), Fn._p(pooled),
                Fn._stream(self.device)), "supcon_head_sharded_store_pool_forward_typed")
        return pooled

    def _write(self, row0: int, hs: torch.Tensor) -> None:
        """local rows ``row0 + b`` = the layer means of hs: through the allocation's own ``write`` for fp32, through
        ``_Rounding`` (as ``LayerMeanStore.append``) for fp16"""
        if self.dtype == torch.float32:
            self._shard.write(row0, hs)
        else:
            self._rounding.write_means(row0, hs)

    def _overflow_problem(self, where: str = ""):
        """a ValueError naming the first slot of this rank whose fp16 row holds a finite value rounded to inf, or
        None"""
        bad = self._rounding.first_overflow()
        return None if bad is None else ValueError(where + _overflow_message(self.rank + bad * self.world))

    def gather_labels(self, local_labels: torch.Tensor) -> None:
        """``labels`` = every rank's ``local_labels`` (ceil(n / R),) in slot order, through one all-gather"""
        parts = [torch.empty_like(local_labels) for _ in range(self.world)]
        dist.all_gather(parts, local_labels.contiguous(), group=self.group)
        self.labels.copy_(torch.stack(parts, dim=1).reshape(-1)[:self.n])

    def close(self) -> None:
        """Release this rank's shard and its mapping of the others' (collective: waits until no rank still reads a
        shard).  The store cannot pool afterwards."""
        if self._shard is None:
            return
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)
        self._shard.close()
        self._shard = self.rows = None

    def save(self, path, overwrite: bool = False):
        """``LayerMeanStore.save`` of slots ``[0, filled)`` (collective), in the same format: the file does not
        depend on R.  Rank 0 creates and sizes ``<path>.partial/rows.npy``; then every rank writes its own rows at
        their slots (local row j is slot rank + j R) and fsyncs; then rank 0 writes ``labels.npy`` and renames.  A
        failure on any rank raises on every rank and removes the partial directory.  Whether ``path`` exists is
        rank 0's view."""
        if self._shard is None:
            raise RuntimeError("the sharded store is closed")
        path = os.fspath(path)
        if self.filled < 1:
            raise ValueError("the store is empty: nothing to save")
        problem = self._overflow_problem()
        _agree(problem and ValueError(f"{problem}: not saved"), self.group)
        seen = [None] * self.world
        dist.all_gather_object(seen, os.path.exists(path), group=self.group)
        if seen[0] and not overwrite:
            return None
        partial, lead = path + ".partial", self.rank == 0
        descr = _STORE_DTYPES[self.dtype][1]
        header = len(_npy_header((self.filled, self.feat, self.frames), descr))

        def step(fn):
            problem = None
            try:
                fn()
            except (OSError, ValueError, RuntimeError) as exc:
                problem = exc
            try:
                _agree(problem, self.group)
            except Exception:
                if lead:
                    _discard(partial)
                raise

        step(lambda: _create_rows_file(partial, (self.filled, self.feat, self.frames), descr) if lead else None)
        step(lambda: _write_rows(self.rows, shard_slots(self.filled, self.rank, self.world), partial, header))
        step(lambda: _finish_save(partial, path, self.labels[:self.filled]) if lead else None)
        return self.filled

    @classmethod
    def from_arrays(cls, rows, labels, device, group=None, *, allocate=None,
                    dtype=torch.float32) -> "ShardedLayerMeanStore":
        """``LayerMeanStore.from_arrays`` split over the ranks of ``group`` (collective): every rank passes the
        whole (n, F, T) array (typically a memmap of the same file) and reads only its slots
        ``shard_slots(n, rank, R)`` into its shard, in place; ``dtype`` is the store's.  Besides ``from_arrays``'
        checks and the constructor's, the ranks must agree on the rows' dtype; every check raises on every rank."""
        src, lab, problem = None, None, None
        try:
            src = _RowSource(rows)
            lab = _label_tensor(labels, src.n)
        except ValueError as exc:
            problem = exc
        _agree(problem, group)
        kinds = [None] * dist.get_world_size(group)
        dist.all_gather_object(kinds, str(src.rows.dtype), group=group)
        if len(set(kinds)) != 1:
            raise ValueError("the ranks disagree on the rows' dtype: " +
                             ", ".join(f"rank {r} {k}" for r, k in enumerate(kinds)))
        store = cls(src.n, src.feat, src.frames, device, group, allocate=allocate, dtype=dtype)
        problem = None
        try:
            _read_rows(src, shard_slots(store.n, store.rank, store.world), store._rounding)
            problem = store._overflow_problem(f"{src.name}: ")
            store.labels.copy_(lab)
        except (OSError, ValueError, RuntimeError) as exc:
            problem = exc
        try:
            _agree(problem, group)                  # also the barrier before any rank reads a peer's shard
        except Exception:
            store.close()
            raise
        store.filled = store.n
        return store


@torch.no_grad()
def build_sharded_layer_mean_store(encoder, loader, device, *, n: int, group=None, label_index: int = 1,
                                   allocate=None, dtype=torch.float32) -> ShardedLayerMeanStore:
    """``build_layer_mean_store`` split over the ranks of ``group`` (collective): each rank runs ``encoder`` on its
    own share of the n clips, so the build takes 1 / R of the time and the node holds R times the clips.
    ``loader`` yields this rank's clips in the order ``shard_slots(n, rank, R)`` lists them (e.g. a
    ``DataLoader(Subset(dataset, shard_slots(...)), shuffle=False)``); the encoder is called as
    ``build_layer_mean_store`` calls it.  Raises on every rank when the ranks' (F, T) differ, a shard does not fit
    free memory, a rank's loader yields more or fewer clips than its share, n < R, or the GPUs cannot reach each
    other's memory, and, for an fp16 store (``dtype``, the same on every rank), when a finite layer mean rounded to
    inf (naming the first such slot of each rank).  Afterwards ``filled == n`` and ``labels`` holds every slot's
    label on every rank."""
    from .stage1 import _to_device
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    encoder.eval()

    def encoded(batch):
        waveforms, labels = _to_device(batch[0], batch[label_index], device)
        return encoder(waveforms, attention_mask=(waveforms != 0.0).long()), labels

    batches = iter(loader)
    first = next(batches, None)
    hs, labels = encoded(first) if first is not None else (None, None)
    shape = tuple(hs.shape[-2:]) if hs is not None else (0, 0)
    store = ShardedLayerMeanStore(n, *shape, device, group, allocate=allocate, dtype=dtype)
    share = len(shard_slots(n, rank, world))
    local_labels = torch.full((store.local_rows,), -1, dtype=torch.int64, device=store.device)
    filled, problem = 0, None
    try:
        while hs is not None:
            b = _check_hs(hs, store.feat, store.frames, filled)
            if tuple(labels.shape) != (b,):
                raise ValueError(f"labels must be ({b},), got {tuple(labels.shape)}")
            if filled + b > share:
                raise ValueError(f"the loader yields more than this rank's {share} clips of {n}")
            store._write(filled, hs)
            local_labels[filled:filled + b].copy_(labels.detach().long(), non_blocking=True)
            filled += b
            batch = next(batches, None)
            hs, labels = encoded(batch) if batch is not None else (None, None)
        if filled != share:
            raise ValueError(f"the loader yielded {filled} clips, this rank's share of {n} is {share}")
        problem = store._overflow_problem()
    except ValueError as exc:
        problem = exc
    try:
        _agree(problem, group)
    except Exception:
        store.close()
        raise
    store.gather_labels(local_labels)
    store.filled = n
    return store


def load_sharded_layer_mean_store(path, device, group=None, *, allocate=None,
                                  dtype=torch.float32) -> ShardedLayerMeanStore:
    """``load_layer_mean_store`` into a store sharded over the ranks of ``group`` (collective): the file may have
    been written by any number of ranks, one included, and rank r reads only its own slots.  A missing, truncated
    or unreadable file on any rank raises on every rank, as do the checks of ``ShardedLayerMeanStore.from_arrays``.
    ``allocate`` and ``dtype`` as in ``ShardedLayerMeanStore``."""
    arrays, problem = None, None
    try:
        arrays = _open_store(path)
    except (OSError, ValueError) as exc:
        problem = exc
    _agree(problem, group)
    return ShardedLayerMeanStore.from_arrays(*arrays, device, group, allocate=allocate, dtype=dtype)


# ---------------------------------------------------------------------------------- the store on disk

def _open_store(path):
    """(rows, labels) memmaps of the store directory ``path``; np.load checks each header against the file's size"""
    path = os.fspath(path)
    if not os.path.isdir(path):
        raise FileNotFoundError(f"no layer-mean store at {path}")
    arrays = []
    for name in (ROWS_FILE, LABELS_FILE):
        file = os.path.join(path, name)
        try:
            arrays.append(np.load(file, mmap_mode="r"))
        except FileNotFoundError:
            raise
        except (OSError, ValueError) as exc:
            raise ValueError(f"{file} is not a readable .npy array: {exc}") from exc
    return arrays


class _RowSource:
    """(n, F, T) float32 or float16 rows from the host: a memmap of a whole file (what np.load returns) is read from
    the file with preadv, which keeps its pages out of this process; any other array is copied row by row."""

    def __init__(self, rows):
        if isinstance(rows, torch.Tensor):
            if rows.device.type != "cpu" or rows.dtype not in (torch.float32, torch.float16):
                raise ValueError(f"rows must be a float32 or float16 CPU tensor, got {rows.dtype} on {rows.device}")
            rows = rows.detach().numpy()
        if not isinstance(rows, np.ndarray):
            raise ValueError(f"rows must be a numpy array or a CPU tensor, got {type(rows).__name__}")
        if rows.dtype not in (np.dtype(np.float32), np.dtype(np.float16)):
            raise ValueError(f"rows must be float32 or float16 (another dtype would be rounded), got {rows.dtype}")
        if rows.ndim != 3:
            raise ValueError(f"rows must be (n, F, T), got {rows.shape}")
        self.rows = rows
        self.n, self.feat, self.frames = rows.shape
        self.row = self.feat * self.frames
        self.file = self.offset = None
        if (isinstance(rows, np.memmap) and isinstance(rows.base, mmap.mmap) and rows.flags.c_contiguous
                and rows.filename):
            self.file, self.offset = rows.filename, rows.offset
        self.name = self.file or "rows"
        # a float16 source bound for a float32 staging buffer is read here and widened (exact)
        self.raw = np.empty(0, rows.dtype)

    def fill(self, out: np.ndarray, pieces, fd) -> None:
        """``out`` (m,) = the source's elements ``pieces`` [(flat offset, count), ...] in order: ``out`` has the
        source's dtype, or is float32 for a float16 source"""
        widen = out.dtype != self.rows.dtype
        if widen and self.raw.size < out.size:
            self.raw = np.empty(out.size, self.rows.dtype)
        dst = self.raw[:out.size] if widen else out
        pos = 0
        for start, count in pieces:
            if fd is not None:
                _read_exactly(fd, dst[pos:pos + count], self.offset + start * dst.itemsize, self.file)
            else:
                done = 0
                while done < count:                         # rows, so that a strided array is never copied whole
                    i, lo = divmod(start + done, self.row)
                    k = min(self.row - lo, count - done)
                    np.copyto(dst[pos + done:pos + done + k], self.rows[i].reshape(-1)[lo:lo + k])
                    done += k
            pos += count
        if widen:
            np.copyto(out, dst)


def _read_exactly(fd: int, out: np.ndarray, offset: int, file: str) -> None:
    view = memoryview(out).cast("B")
    while view.nbytes:
        got = os.preadv(fd, [view], offset)
        if got == 0:
            raise ValueError(f"{file} ends at byte {offset}, before the rows its header declares")
        view, offset = view[got:], offset + got


def _write_all(fd: int, data: np.ndarray, offset: int) -> None:
    view = memoryview(data).cast("B")
    while view.nbytes:
        put = os.pwrite(fd, view, offset)
        view, offset = view[put:], offset + put


def _label_tensor(labels, n: int) -> torch.Tensor:
    """(n,) int64 CPU tensor of labels given as integers of any width (numpy array, memmap or tensor)"""
    lab = labels.detach().cpu().numpy() if isinstance(labels, torch.Tensor) else np.asarray(labels)
    if lab.shape != (n,) or lab.dtype.kind not in "iu":
        raise ValueError(f"labels must be ({n},) integers, got {lab.dtype} {lab.shape}")
    return torch.from_numpy(lab.astype(np.int64))


def _chunks(slots, row: int, chunk: int):
    """(device element offset, [(file element offset, count), ...]) of at most ``chunk`` elements each, in order:
    the device tensor's local row j is slot ``slots[j]`` of the file.  A chunk may split a row."""
    runs = ([(slots.start * row, len(slots) * row)] if isinstance(slots, range) and slots.step == 1
            else [(s * row, row) for s in slots])
    d0, pieces, size = 0, [], 0
    for f0, count in runs:
        while count:
            k = min(count, chunk - size)
            pieces.append((f0, k))
            size, f0, count = size + k, f0 + k, count - k
            if size == chunk:
                yield d0, pieces
                d0, pieces, size = d0 + size, [], 0
    if pieces:
        yield d0, pieces


class _Staging:
    """Two host byte buffers of ``STAGE_BYTES`` (pinned when the store is on a GPU), each holding a chunk of
    elements of ``dtype``, and a side stream for their copies to and from the device, each a ``cudaMemcpyAsync``;
    an event per buffer guards its reuse, so the file I/O of one chunk overlaps the copy of the other.  ``rounded``
    adds a device fp32 buffer per host buffer, for chunks that ``round`` puts into an fp16 store."""

    def __init__(self, device, dtype=torch.float32, rounded: bool = False):
        self.dtype = dtype
        self.chunk = max(STAGE_BYTES // dtype.itemsize, 1)
        self.cuda = device.type == "cuda"
        self.bufs = [torch.empty(self.chunk * dtype.itemsize, dtype=torch.uint8, pin_memory=self.cuda)
                     for _ in range(2)]
        self.dev = ([torch.empty(self.chunk, dtype=torch.float32, device=device) for _ in range(2)]
                    if rounded and self.cuda else None)
        self.events = [None, None]
        if self.cuda:
            self.stream = torch.cuda.Stream(device)
            self.stream.wait_stream(torch.cuda.current_stream(device))

    def host(self, c: int) -> torch.Tensor:
        """the buffer of chunk c, once the last copy into or out of it has completed"""
        if self.events[c % 2] is not None:
            self.events[c % 2].synchronize()
        return self.bufs[c % 2].view(self.dtype)

    def copy(self, c: int, dst: torch.Tensor, src: torch.Tensor) -> None:
        if not self.cuda:
            dst.copy_(src)
            return
        with torch.cuda.stream(self.stream):
            dst.copy_(src, non_blocking=True)
            self.events[c % 2] = torch.cuda.Event()
            self.events[c % 2].record(self.stream)

    def round(self, c: int, rounding: "_Rounding", offset: int, src: torch.Tensor) -> None:
        """``rounding.put(offset, src)`` of the host fp32 chunk ``src``, on the device"""
        if not self.cuda:
            rounding.put(offset, src)
            return
        with torch.cuda.stream(self.stream):
            dev = self.dev[c % 2][:src.numel()]
            dev.copy_(src, non_blocking=True)
            rounding.put(offset, dev)
            self.events[c % 2] = torch.cuda.Event()
            self.events[c % 2].record(self.stream)

    def finish(self) -> None:
        if self.cuda:
            self.stream.synchronize()


def _read_rows(src: _RowSource, slots, rounding: "_Rounding") -> None:
    """``rows[j] = src[slots[j]]`` for the rows of ``rounding`` (contiguous, on a GPU or the CPU); returns when the
    copies are done.  The chunks travel in the source's dtype, except a float16 source for an fp32 store (widened on
    the host, exactly); a float32 source for an fp16 store is rounded on the device by ``rounding.put``."""
    dst = rounding.rows.view(-1)
    rounded = rounding.rows.dtype == torch.float16 and src.rows.dtype == np.float32
    wire = torch.float16 if rounding.rows.dtype == torch.float16 and not rounded else torch.float32
    st = _Staging(dst.device, wire, rounded)
    fd = os.open(src.file, os.O_RDONLY) if src.file else None
    try:
        for c, (d0, pieces) in enumerate(_chunks(slots, src.row, st.chunk)):
            m = sum(k for _, k in pieces)
            buf = st.host(c)[:m]
            src.fill(buf.numpy(), pieces, fd)
            if rounded:
                st.round(c, rounding, d0, buf)
            else:
                st.copy(c, dst[d0:d0 + m], buf)
        st.finish()
    finally:
        if fd is not None:
            os.close(fd)


def _write_rows(rows: torch.Tensor, slots, partial: str, header: int) -> None:
    """write ``rows[j]`` at slot ``slots[j]`` of ``<partial>/rows.npy`` (sized by ``_create_rows_file``; its data
    starts at byte ``header``) and fsync it"""
    row = rows.shape[1] * rows.shape[2]
    src = rows.view(-1)
    st = _Staging(rows.device, rows.dtype)
    chunks = list(_chunks(slots, row, st.chunk))
    sizes = [sum(k for _, k in pieces) for _, pieces in chunks]

    def issue(c):
        st.copy(c, st.host(c)[:sizes[c]], src[chunks[c][0]:chunks[c][0] + sizes[c]])

    fd = os.open(os.path.join(partial, ROWS_FILE), os.O_WRONLY)
    try:
        if chunks:
            issue(0)
        for c, (_, pieces) in enumerate(chunks):
            if c + 1 < len(chunks):
                issue(c + 1)                                # its buffer was written to the file one chunk ago
            buf, pos = st.host(c).numpy(), 0
            for f0, k in pieces:
                _write_all(fd, buf[pos:pos + k], header + rows.element_size() * f0)
                pos += k
        st.finish()
        os.fsync(fd)
    finally:
        os.close(fd)


def _npy_header(shape, descr: str = "<f4") -> bytes:
    """the .npy header of a C-order array of ``shape`` and ``descr`` (``<f4`` or ``<f2``): the same bytes on every
    rank"""
    out = io.BytesIO()
    np.lib.format.write_array_header_1_0(out, {"descr": descr, "fortran_order": False, "shape": tuple(shape)})
    return out.getvalue()


def _create_rows_file(partial: str, shape, descr: str = "<f4") -> int:
    """a fresh ``<partial>/rows.npy`` of ``shape`` and ``descr`` (header written, data sized, not yet filled);
    returns the header's length.  A ``partial`` left by a save that died is removed first."""
    _discard(partial)
    os.makedirs(partial)
    header = _npy_header(shape, descr)
    with open(os.path.join(partial, ROWS_FILE), "wb") as fh:
        fh.write(header)
        fh.truncate(len(header) + np.dtype(descr).itemsize * int(np.prod(shape)))
    return len(header)


def _fsync_dir(path: str) -> None:
    fd = os.open(path, os.O_RDONLY)
    try:
        os.fsync(fd)
    finally:
        os.close(fd)


def _finish_save(partial: str, path: str, labels: torch.Tensor) -> None:
    """write ``labels.npy``, fsync, and rename ``partial`` to ``path`` (replacing what is there)"""
    with open(os.path.join(partial, LABELS_FILE), "wb") as fh:
        np.save(fh, labels.detach().cpu().numpy().astype(np.int64))
        fh.flush()
        os.fsync(fh.fileno())
    _fsync_dir(partial)
    old = None
    if os.path.lexists(path):
        old = path + ".old"
        _discard(old)
        os.rename(path, old)
    os.rename(partial, path)
    _fsync_dir(os.path.dirname(os.path.abspath(path)))
    if old is not None:
        _discard(old)


def _discard(path: str) -> None:
    if os.path.isdir(path) and not os.path.islink(path):
        shutil.rmtree(path)
    elif os.path.lexists(path):
        os.remove(path)
