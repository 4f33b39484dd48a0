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

Preconditions: frozen encoder, no waveform augmentation, the same crop / pad of each clip in every epoch.  The rows
are fp32 (a bf16 store would round the mean and lose that equality).  There is no backward: the store is a constant.
"""
import torch

from . import _cabi
from . import functional as Fn

__all__ = ["LayerMeanStore", "build_layer_mean_store"]


class LayerMeanStore:
    """``rows`` (n, F, T) fp32 and ``labels`` (n,) int64, both on one device; slots ``[0, filled)`` are written.

    ``append`` writes the layer means of a batch of hidden states at the next ``B`` slots.  ``pool`` and
    ``labels_of`` take a device int64 index vector, so both can be captured in a CUDA graph and fed new indices
    every replay.  An index outside ``[0, filled)`` gives a NaN pooled row (the loss turns NaN) instead of a fault."""

    def __init__(self, n: int, feat: int, frames: int, device):
        if n < 1 or feat < 1 or frames < 1:
            raise ValueError(f"bad store shape ({n}, {feat}, {frames})")
        device = torch.device(device)
        need = store_bytes(n, feat, frames)
        if device.type == "cuda":
            free, _ = torch.cuda.mem_get_info(device)
            if need > free:
                raise MemoryError(f"a store of {n} clips x ({feat}, {frames}) fp32 takes {need / 1e9:.2f} GB; "
                                  f"{free / 1e9:.2f} GB are free on {device}")
        self.rows = torch.empty((n, feat, frames), dtype=torch.float32, device=device)
        self.labels = torch.full((n,), -1, dtype=torch.int64, device=device)
        self.filled = 0

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

    def append(self, hs: torch.Tensor, labels: torch.Tensor) -> int:
        """Write ``mean_k hs[b, k]`` (hs = (B, K, F, T), fp32 or bf16; other dtypes through an fp32 copy) and
        ``labels[b]`` at slot ``filled + b``; returns the first slot written."""
        if hs.dim() != 4:
            raise ValueError(f"hs must be (batch, layers, feat, frames), got {tuple(hs.shape)}")
        b, k, f, t = hs.shape
        if (f, t) != (self.feat, self.frames):
            raise ValueError(f"clips {self.filled}..{self.filled + b - 1}: hidden states of (F, T) = ({f}, {t}), "
                             f"the store holds ({self.feat}, {self.frames})")
        if tuple(labels.shape) != (b,):
            raise ValueError(f"labels must be ({b},), got {tuple(labels.shape)}")
        if self.filled + b > self.n:
            raise ValueError(f"the store holds {self.n} clips: no room for {b} more after {self.filled}")
        Fn._require_cuda(hs, "hs")
        if hs.device != self.device:
            raise ValueError(f"hs is on {hs.device}, the store on {self.device}")
        x = hs.detach()
        if x.dtype not in (torch.float32, torch.bfloat16):
            x = x.float()
        x = x.contiguous()
        slot0 = self.filled
        with torch.cuda.device(self.device):
            _cabi.check(_cabi.load().supcon_head_layer_mean_typed(
                Fn._p(x), _cabi.BF16 if x.dtype == torch.bfloat16 else _cabi.F32, b, k, f, t,
                Fn._p(self.rows[slot0]), Fn._stream(self.device)), "supcon_head_layer_mean_typed")
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
        if idx.dim() != 1 or idx.dtype != torch.int64 or idx.device != self.device:
            raise ValueError(f"idx must be a 1-D int64 tensor on {self.device}, got {idx.dtype} "
                             f"{tuple(idx.shape)} on {idx.device}")
        Fn._require_cuda(self.rows, "the store")
        rng = None
        if dropout_p > 0.0:
            if (rng_state is None or rng_state.dtype != torch.int64 or rng_state.numel() != 2
                    or rng_state.device != self.device):
                raise ValueError("dropout needs rng_state = int64 tensor {seed, offset} on the store's device")
            rng = rng_state
        idx = idx.contiguous()
        with torch.cuda.device(self.device):
            pooled = torch.empty((idx.shape[0], self.feat), dtype=torch.float32, device=self.device)
            _cabi.check(_cabi.load().supcon_head_store_pool_forward(
                Fn._p(self.rows), self.filled, self.feat, self.frames, Fn._p(idx), idx.shape[0], float(dropout_p),
                float(negative_slope), Fn._p(rng), Fn._p(pooled), Fn._stream(self.device)),
                "supcon_head_store_pool_forward")
        return pooled


def store_bytes(n: int, feat: int, frames: int) -> int:
    """device bytes of a store of n clips: fp32 rows and int64 labels"""
    return n * feat * frames * 4 + n * 8


@torch.no_grad()
def build_layer_mean_store(encoder, loader, device, *, label_index: int = 1, n=None) -> LayerMeanStore:
    """Run ``encoder`` once over ``loader`` as ``stage1.train_one_epoch`` runs a frozen one (eval mode, no grad,
    ``attention_mask = (waveforms != 0).long()``) and store each clip's layer mean.  Slot i holds the loader's i-th
    clip, so a sequential loader over the dataset gives slot = dataset index.  ``n`` (default
    ``len(loader.dataset)``) is the number of clips to allocate for; a loader that yields fewer leaves the store
    ``filled`` short of ``n``.  Raises on a clip whose (F, T) differs from the first one, on more clips than ``n``
    and on a store that does not fit the device's free memory.  ``label_index`` picks the label column of the batch
    tuple, as in ``train_one_epoch``."""
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
            store = LayerMeanStore(n, hs.shape[-2], hs.shape[-1], device)
        store.append(hs, labels)
    if store is None:
        raise ValueError("the loader yielded no clips")
    return store
