"""Fused compression head: the producer of the loss's input (SURVEY §8 f-N1).

The reference builds z as (compression_module.py:48-65, stage1_utils.py:122-123)

    x   = LeakyReLU(Dropout(hs.mean(dim=1)))          (B, F, T)     hs = encoder output (B, K, F, T)
    seq = mlp3(x.transpose(1, 2)).transpose(1, 2)     (B, D, T)
    z   = F.normalize(seq.mean(dim=-1), p=2, dim=1)   (B, D)

``mlp3`` and the time mean are both linear, so ``seq.mean(-1) == mlp3(x.mean(-1))``: the per-frame GEMM over
B*T rows collapses to one over B rows and everything left of it is a single pass over ``hs``, which is what
``supcon_head_pool_forward_typed`` (csrc/supcon_head.cu) does - hs read once, (B, F) floats written.  ``hs`` is read
in its own dtype when that is fp32 or bf16 (the output of an encoder run in bf16: no fp32 copy, and d loss / d hs comes
back in bf16); other dtypes are converted to fp32 first.  The (B, F) x (F, D) product that remains is a plain library GEMM (``F.linear``: autograd gives the weight/bias gradients), and the row
normalisation is this library's kernel.

``FusedCompressionHead`` has the reference module's parameters under the same names (``mlp3.weight``,
``mlp3.bias``), so Stage-1 checkpoints (``compression_state_dict``) load into it unchanged.  ``forward(hs)`` returns
the sequence ALREADY averaged over time, shape (B, D, 1): the unchanged caller's ``seq.mean(dim=-1)`` then yields
exactly the pooled embedding.  ``embed(hs)`` goes all the way to the normalised z.  In train mode the dropout mask
comes from a counter-based generator inside the kernel (Bernoulli(1 - p), scaled by 1/(1-p), like ``nn.Dropout``;
the stream differs from torch's, as it would between two torch versions).  There is no CPU path.

One process per GPU: do not wrap this module in ``nn.DataParallel`` for training - replicas are rebuilt from the
master copy every step and their buffer updates are discarded, so the dropout offset would never advance.
"""

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _cabi
from . import functional as Fn


class _LayerTimePool(torch.autograd.Function):
    """pooled[b, f] = mean_t LeakyReLU(Dropout(mean_k hs[b, k, f, t])).  fp32 and bf16 hs go to the kernel as they
    are (bf16 is widened exactly inside it, and dhs is returned in bf16); other dtypes through an fp32 copy."""

    @staticmethod
    def forward(ctx, hs, dropout_p, negative_slope, rng_state):
        Fn._require_cuda(hs, "hs")
        if hs.dim() != 4:
            raise ValueError(f"hs must be (batch, layers, feat, frames), got {tuple(hs.shape)}")
        lib = _cabi.load()
        x = hs.detach()
        if x.dtype not in (torch.float32, torch.bfloat16):
            x = x.float()
        x = x.contiguous()
        dtype_code = _cabi.BF16 if x.dtype == torch.bfloat16 else _cabi.F32
        b, k, f, t = x.shape
        dev = x.device
        rng = None
        if dropout_p > 0.0:
            if rng_state is None or rng_state.dtype != torch.int64 or rng_state.numel() != 2 or rng_state.device != dev:
                raise ValueError("dropout needs rng_state = int64 tensor {seed, offset} on hs's device")
            rng = rng_state.clone()                    # the backward must see the values this forward used
        with torch.cuda.device(dev):
            pooled = torch.empty((b, f), dtype=torch.float32, device=dev)
            _cabi.check(lib.supcon_head_pool_forward_typed(Fn._p(x), dtype_code, b, k, f, t, float(dropout_p),
                                                           float(negative_slope), Fn._p(rng), Fn._p(pooled),
                                                           Fn._stream(dev)),
                        "supcon_head_pool_forward_typed")
        if ctx.needs_input_grad[0]:
            ctx.save_for_backward(x, rng if rng is not None else torch.empty(0, device=dev))
            ctx.cfg = (float(dropout_p), float(negative_slope), rng is not None, hs.dtype, dtype_code)
        return pooled

    @staticmethod
    def backward(ctx, dpooled):
        x, rng = ctx.saved_tensors
        dropout_p, negative_slope, has_rng, in_dtype, dtype_code = ctx.cfg
        lib = _cabi.load()
        b, k, f, t = x.shape
        dev = x.device
        g = dpooled.detach().float().contiguous()
        with torch.cuda.device(dev):
            dhs = torch.empty_like(x)                  # in x's dtype: the kernel writes bf16 for a bf16 hs
            _cabi.check(lib.supcon_head_pool_backward_typed(Fn._p(x), dtype_code, b, k, f, t, dropout_p,
                                                            negative_slope, Fn._p(rng) if has_rng else None,
                                                            Fn._p(g), Fn._p(dhs), Fn._stream(dev)),
                        "supcon_head_pool_backward_typed")
        return dhs.to(in_dtype), None, None, None


def layer_time_pool(hs: torch.Tensor, dropout_p: float = 0.0, negative_slope: float = 0.01, rng_state=None):
    """One pass over hs (B, K, F, T): ``LeakyReLU(Dropout(hs.mean(1))).mean(-1)`` -> (B, F) fp32.  hs may be fp32 or
    bf16 (read natively, with the layer sum in fp32); any other dtype is converted to fp32 first."""
    return _LayerTimePool.apply(hs, float(dropout_p), float(negative_slope), rng_state)


class FusedCompressionHead(nn.Module):
    """``CompressionModule(input_dim, hidden_dim, dropout_rate)`` (compression_module.py:7-32) with the layer mean,
    Dropout, LeakyReLU and the time mean fused into one kernel in front of ``mlp3``."""

    def __init__(self, input_dim: int = 1024, hidden_dim: int = 256, dropout_rate: float = 0.1):
        super().__init__()
        self.dropout_head = nn.Dropout(p=dropout_rate)
        self.activation_head = nn.LeakyReLU()
        self.mlp3 = nn.Linear(input_dim, hidden_dim)
        # {seed, offset} of the dropout stream, on the device so that CUDA-graph replays draw fresh masks.
        # Seeded HERE, at construction, from torch.initial_seed() (a later torch.manual_seed() does not move it:
        # call reseed()).  dropout_stream_state() / load_dropout_stream_state() let a resumed run continue the
        # stream instead of replaying the masks from offset 0.
        self.register_buffer("rng_state", torch.tensor([0, 0], dtype=torch.int64), persistent=False)
        self.reseed()

    def reseed(self, seed=None, stream=None) -> None:
        """Restart the dropout stream.  ``seed`` defaults to ``torch.initial_seed()``; ``stream`` (default: this
        process's rank in the default process group, 0 without one) is mixed into the key so that the ranks of a
        data-parallel job -- which the reference's set_seed() gives the SAME torch seed -- draw different masks."""
        if seed is None:
            seed = torch.initial_seed()
        if stream is None:
            import torch.distributed as dist
            stream = dist.get_rank() if (dist.is_available() and dist.is_initialized()) else 0
        key = (int(seed) ^ (int(stream) * 0x9E3779B97F4A7C15)) & 0x7FFFFFFFFFFFFFFF
        with torch.no_grad():
            self.rng_state.copy_(torch.tensor([key, 0], dtype=torch.int64))

    # -- checkpointing.  state_dict() stays exactly the reference module's (mlp3.weight, mlp3.bias) so that
    #    checkpoints move both ways between this class and compression_module.CompressionModule with strict=True;
    #    the position of the dropout stream is saved NEXT to it, like an optimizer's state:
    #        ckpt = {"compression_state_dict": head.state_dict(), "dropout_stream": head.dropout_stream_state()}
    def dropout_stream_state(self):
        """{seed key, offset} of the dropout stream as Python ints (one device read)."""
        return [int(v) for v in self.rng_state.tolist()]

    def load_dropout_stream_state(self, state) -> None:
        """Continue the stream of a saved run instead of replaying its masks from offset 0."""
        with torch.no_grad():
            self.rng_state.copy_(torch.tensor([int(state[0]), int(state[1])], dtype=torch.int64))

    def pooled_features(self, hs: torch.Tensor) -> torch.Tensor:
        """(B, F): mean over time of the activated layer mean."""
        p = self.dropout_head.p if self.training else 0.0
        if p > 0.0:
            out = layer_time_pool(hs, p, self.activation_head.negative_slope, self.rng_state)
            self.rng_state[1] += 1                # in-stream: the next call (or graph replay) uses a new mask
            return out
        return layer_time_pool(hs, 0.0, self.activation_head.negative_slope, None)

    def pooled_embedding(self, hs: torch.Tensor) -> torch.Tensor:
        """(B, D) == ``CompressionModule(hs).mean(dim=-1)`` of the reference."""
        return F.linear(self.pooled_features(hs), self.mlp3.weight, self.mlp3.bias)

    def pooled_features_from_store(self, store, idx: torch.Tensor) -> torch.Tensor:
        """``pooled_features`` of the clips in slots ``idx`` (device int64) of a ``feature_store.LayerMeanStore`` (or ``ShardedLayerMeanStore``):
        the same values, bit for bit, and the same dropout stream (one offset per call in train mode)."""
        p = self.dropout_head.p if self.training else 0.0
        if p > 0.0:
            out = store.pool(idx, p, self.activation_head.negative_slope, self.rng_state)
            self.rng_state[1] += 1
            return out
        return store.pool(idx, 0.0, self.activation_head.negative_slope, None)

    def pooled_embedding_from_store(self, store, idx: torch.Tensor) -> torch.Tensor:
        """(B, D) == ``pooled_embedding`` of the clips in slots ``idx`` of the store."""
        return F.linear(self.pooled_features_from_store(store, idx), self.mlp3.weight, self.mlp3.bias)

    def forward(self, hs: torch.Tensor) -> torch.Tensor:
        """(B, D, 1): the reference's (B, D, T) sequence already averaged over T, so that the unchanged caller's
        ``seq.mean(dim=-1)`` (stage1_utils.py:123) is the pooled embedding."""
        return self.pooled_embedding(hs).unsqueeze(-1)

    def embed(self, hs: torch.Tensor, out_dtype=torch.float32) -> torch.Tensor:
        """L2-normalised z (B, D) = ``F.normalize(head(hs).mean(-1), p=2, dim=1)``; ``out_dtype=torch.bfloat16``
        feeds the tensor-core loss path directly."""
        return Fn.l2_normalize(self.pooled_embedding(hs), out_dtype)
