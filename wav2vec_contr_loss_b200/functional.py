"""Torch-facing wrappers around the C-ABI: tensors in, tensors out.

PyTorch is plumbing here (device memory, streams, autograd hook-up).  Every
number is produced by libsupcon_b200.so; there is no eager/CPU fallback and a
non-CUDA tensor is rejected.
"""
import ctypes
from typing import Optional, Tuple

import torch

from . import _cabi

_SIM = {"cosine": _cabi.COSINE, "geodesic": _cabi.GEODESIC}


def similarity_id(similarity: str) -> int:
    key = similarity.lower()
    if key not in _SIM:
        # same text as reference loss.py:32
        raise ValueError(f"Unknown similarity: {similarity}")
    return _SIM[key]


def _p(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream(dev) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


class _NoSwitch:
    """Stand-in for torch.cuda.device(dev) when dev already is the current device (the usual case: one process per
    GPU): entering torch's context manager costs ~8 us per call, more than a whole launch at the native batch."""
    __slots__ = ()

    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NO_SWITCH = _NoSwitch()


def _on(dev):
    """Context in which ``dev`` is the current CUDA device."""
    idx = dev.index
    if idx is None or idx == torch.cuda.current_device():
        return _NO_SWITCH
    return torch.cuda.device(dev)


def _dtype_id(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return _cabi.F32
    if t.dtype == torch.bfloat16:
        return _cabi.BF16
    raise TypeError(f"unsupported element type {t.dtype}")


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError(
            f"{what} must be a CUDA tensor: the B200 SupCon path has no CPU fallback "
            f"(got device {t.device})")


def canonical_z(z: torch.Tensor) -> torch.Tensor:
    """Contiguous fp32 or bf16 view/copy of the embeddings."""
    if z.dim() != 2:
        raise ValueError(f"z must be (B, D), got shape {tuple(z.shape)}")
    if z.dtype not in (torch.float32, torch.bfloat16):
        z = z.float()
    return z.contiguous()


def canonical_labels(labels: torch.Tensor, n: int) -> torch.Tensor:
    """int32 class keys: equal labels <-> equal keys (reference compares with ==, loss.py:123-124; any dtype,
    shape (B,) or (B,1)).  Wide labels (int64 as the callers pass them, float32/64) go through ONE kernel of the
    library (supcon_label_keys) that also guards the narrowing: a label 32 bits cannot hold losslessly is a loud
    device fault, never two classes silently merged; NaN labels match nothing, as in the reference."""
    lab = labels.reshape(-1)
    if lab.numel() != n:
        raise ValueError(f"labels must have {n} elements, got {lab.numel()}")
    if lab.dtype == torch.int32:
        return lab.contiguous()
    if lab.dtype in (torch.int8, torch.int16, torch.uint8, torch.bool):
        return lab.to(torch.int32).contiguous()                     # lossless
    if lab.dtype in (torch.float16, torch.bfloat16):
        lab = lab.float()                                           # lossless
    code = {torch.int64: _cabi.LABEL_I64, torch.float32: _cabi.LABEL_F32, torch.float64: _cabi.LABEL_F64}.get(lab.dtype)
    if code is None:
        raise TypeError(f"unsupported label dtype {lab.dtype}")
    lab = lab.contiguous()
    if not lab.is_cuda:   # host tensors only occur with the CPU stand-in kernels of the tests: same rules, eagerly
        if lab.dtype == torch.int64:
            if n and (int(lab.max()) > 2**31 - 1 or int(lab.min()) < -2**31):
                raise ValueError("integer labels do not fit 32 bits; relabel the classes densely")
            return lab.to(torch.int32)
        f = lab.float()
        if lab.dtype == torch.float64 and not bool(((f.double() == lab) | lab.isnan()).all()):
            raise ValueError("float64 labels are not exactly float32 values; relabel the classes")
        keys = (f + 0.0).view(torch.int32).clone()
        nan = f.isnan()
        keys[nan] = 0x7fc00000 | (torch.arange(n, dtype=torch.int32)[nan] & 0x3fffff)
        return keys
    lib = _cabi.load()
    dev = lab.device
    with _on(dev):
        keys = torch.empty(n, dtype=torch.int32, device=dev)
        _cabi.check(lib.supcon_label_keys(_p(lab), code, n, _p(keys), _stream(dev)), "supcon_label_keys")
    return keys


_PROBLEMS = {}          # argument tuple -> Problem (host structs are immutable once built: safe to share)
_WORKSPACE_BYTES = {}   # (problem fields, device index) -> bytes: the size is asked of the library once per shape


def make_problem(n_total, d, z_dtype_id, *, tau, similarity, lambda_uni=0.0, uni_t=2.0, topk=32,
                 alpha=0.0, row_offset=0, n_rows=None, flags=0) -> _cabi.Problem:
    key = (n_total, d, z_dtype_id, tau, similarity, lambda_uni, uni_t, topk, alpha, row_offset, n_rows, flags)
    prob = _PROBLEMS.get(key)
    if prob is None:
        k = max(0, min(int(topk), 2**31 - 1))
        prob = _cabi.Problem(
            n_total=int(n_total), row_offset=int(row_offset),
            n_rows=int(n_total if n_rows is None else n_rows), d=int(d), z_dtype=int(z_dtype_id),
            similarity=int(similarity), topk=k, flags=int(flags), tau=float(tau), alpha=float(alpha),
            lambda_uni=float(lambda_uni), uni_t=float(uni_t))
        if len(_PROBLEMS) > 4096:   # alpha changes every epoch: bound the cache
            _PROBLEMS.clear()
        _PROBLEMS[key] = prob
    return prob


def _problem_key(prob: _cabi.Problem):
    return (prob.n_total, prob.row_offset, prob.n_rows, prob.d, prob.z_dtype, prob.similarity, prob.topk, prob.flags,
            prob.tau, prob.alpha, prob.lambda_uni, prob.uni_t)


def workspace_bytes(prob: _cabi.Problem, device) -> int:
    """Scratch bytes the library wants for this problem on this device (asked once per shape and cached: the
    plan depends on the device's SM count)."""
    key = (_problem_key(prob), getattr(device, "index", None))
    n = _WORKSPACE_BYTES.get(key)
    if n is None:
        lib = _cabi.load()
        nbytes = ctypes.c_size_t(0)
        import contextlib
        on_gpu = getattr(device, "type", None) == "cuda"
        with (torch.cuda.device(device) if on_gpu else contextlib.nullcontext()):   # the plan uses this device's SMs
            _cabi.check(lib.supcon_workspace_bytes(ctypes.byref(prob), ctypes.byref(nbytes)), "supcon_workspace_bytes")
        n = max(int(nbytes.value), 256)
        if len(_WORKSPACE_BYTES) > 4096:
            _WORKSPACE_BYTES.clear()
        _WORKSPACE_BYTES[key] = n
    return n


def workspace_for(prob: _cabi.Problem, device) -> torch.Tensor:
    return torch.empty(workspace_bytes(prob, device), dtype=torch.uint8, device=device)


def _stats_buffers(n_rows: int, dev, want_loss: bool = True):
    """row statistics [n_rows, 8] f32 + partial sums [8] f64 + the scalar loss in ONE allocation."""
    words = n_rows * _cabi.STATS_STRIDE
    buf = torch.empty(words + 2 * _cabi.N_PARTIALS + 2, dtype=torch.float32, device=dev)
    stats = buf[:words].view(n_rows, _cabi.STATS_STRIDE)
    partials = buf[words:words + 2 * _cabi.N_PARTIALS].view(torch.float64)   # byte offset 32 n_rows: 8-aligned
    loss = buf[words + 2 * _cabi.N_PARTIALS] if want_loss else None
    return stats, partials, loss


_WITH_FLAGS = {}


def with_flags(prob: _cabi.Problem, extra: int) -> _cabi.Problem:
    """The same problem with ``extra`` OR-ed into its flags (cached: host structs are immutable once built)."""
    key = (_problem_key(prob), int(extra))
    out = _WITH_FLAGS.get(key)
    if out is None:
        out = _cabi.Problem(n_total=prob.n_total, row_offset=prob.row_offset, n_rows=prob.n_rows, d=prob.d,
                            z_dtype=prob.z_dtype, similarity=prob.similarity, topk=prob.topk,
                            flags=prob.flags | int(extra), tau=prob.tau, alpha=prob.alpha,
                            lambda_uni=prob.lambda_uni, uni_t=prob.uni_t)
        if len(_WITH_FLAGS) > 4096:
            _WITH_FLAGS.clear()
        _WITH_FLAGS[key] = out
    return out


def forward_rows(z_all: torch.Tensor, labels_i32: torch.Tensor, prob: _cabi.Problem, want_loss: bool,
                 keep_ws: bool = False, mem_filled: Optional[torch.Tensor] = None):
    """Row-block forward. Returns (row_stats [n_rows,8] f32, partials [8] f64, loss or None) and, with
    ``keep_ws``, the workspace as a fourth item: handed to backward_rows(ws=...) untouched, it lets the backward
    reuse the label table and class sums the forward built (SUPCON_FLAG_WS_FROM_FORWARD).
    ``mem_filled``: a one-element int32 CUDA tensor, the fill level of a memory problem's columns
    (supcon_forward_rows_memory); ``prob.n_total`` is then the capacity."""
    _require_cuda(z_all, "z")
    lib = _cabi.load()
    dev = z_all.device
    with _on(dev):
        stats, partials, loss = _stats_buffers(prob.n_rows, dev, want_loss)
        ws = workspace_for(prob, dev)
        if mem_filled is None:
            _cabi.check(lib.supcon_forward_rows(ctypes.byref(prob), _p(z_all), _p(labels_i32), _p(stats),
                                                _p(partials), _p(loss), _p(ws), ws.numel(), _stream(dev)),
                        "supcon_forward_rows")
        else:
            _cabi.check(lib.supcon_forward_rows_memory(ctypes.byref(prob), _p(z_all), _p(labels_i32), _p(mem_filled),
                                                       _p(stats), _p(partials), _p(loss), _p(ws), ws.numel(),
                                                       _stream(dev)),
                        "supcon_forward_rows_memory")
    if keep_ws:
        return stats, partials, loss, ws
    return stats, partials, loss


def loss_and_grad(z: torch.Tensor, labels_i32: torch.Tensor, prob: _cabi.Problem, want_grad: bool = True,
                  out_dtype=torch.float32):
    """Whole batch on one GPU through supcon_loss_and_grad (one launch for small batches).
    Returns (loss, dz or None, row_stats, partials); dz is d loss / d z for grad_out = 1."""
    _require_cuda(z, "z")
    lib = _cabi.load()
    dev = z.device
    with _on(dev):
        stats, partials, loss = _stats_buffers(prob.n_rows, dev, True)
        dz = torch.empty((prob.n_rows, prob.d), dtype=out_dtype, device=dev) if want_grad else None
        ws = workspace_for(prob, dev)
        _cabi.check(lib.supcon_loss_and_grad(ctypes.byref(prob), _p(z), _p(labels_i32), _p(loss), _p(dz),
                                             _dtype_id(dz) if dz is not None else 0, _p(stats), _p(partials),
                                             _p(ws), ws.numel(), _stream(dev)),
                    "supcon_loss_and_grad")
    return loss, dz, stats, partials


SMALL_BATCH_MAX = 320   # supcon_small.cu (N <= 160) and supcon_mid.cu (N <= 320): forward + backward in one launch


def forward_rows_local(z_all, labels_i32, prob: _cabi.Problem) -> torch.Tensor:
    """Phase 1 of the two-phase row-block forward: sweep this rank's own columns.  Only rows
    [row_offset, row_offset + n_rows) of z_all / labels need to be valid.  Returns the workspace that
    forward_rows_remote must be given."""
    _require_cuda(z_all, "z")
    lib = _cabi.load()
    dev = z_all.device
    with _on(dev):
        ws = workspace_for(prob, dev)
        _cabi.check(lib.supcon_forward_rows_local(ctypes.byref(prob), _p(z_all), _p(labels_i32), _p(ws), ws.numel(),
                                                  _stream(dev)), "supcon_forward_rows_local")
    return ws


def forward_rows_remote(z_all, labels_i32, prob: _cabi.Problem, ws: torch.Tensor):
    """Phase 2: all other columns + merge. Returns (row_stats, partials) like forward_rows."""
    lib = _cabi.load()
    dev = z_all.device
    with _on(dev):
        stats, partials, _ = _stats_buffers(prob.n_rows, dev, False)
        _cabi.check(lib.supcon_forward_rows_remote(ctypes.byref(prob), _p(z_all), _p(labels_i32), _p(stats),
                                                   _p(partials), _p(ws), ws.numel(), _stream(dev)),
                    "supcon_forward_rows_remote")
    return stats, partials


def finalize(prob: _cabi.Problem, partials_global: torch.Tensor) -> torch.Tensor:
    lib = _cabi.load()
    dev = partials_global.device
    with _on(dev):
        loss = torch.empty((), dtype=torch.float32, device=dev)
        _cabi.check(lib.supcon_finalize(ctypes.byref(prob), _p(partials_global), _p(loss), _stream(dev)),
                    "supcon_finalize")
    return loss


def finalize_sets(prob: _cabi.Problem, partial_sets: torch.Tensor):
    """Rank-ordered sum of every rank's partial sums [R, 8] f64 + the scalar loss, one launch.
    Returns (partials_global [8] f64, loss)."""
    lib = _cabi.load()
    dev = partial_sets.device
    with _on(dev):
        out = torch.empty(_cabi.N_PARTIALS + 1, dtype=torch.float64, device=dev)
        partials, loss = out[:_cabi.N_PARTIALS], out[_cabi.N_PARTIALS:].view(torch.float32)[0]
        _cabi.check(lib.supcon_finalize_sets(ctypes.byref(prob), _p(partial_sets), partial_sets.numel() // _cabi.N_PARTIALS,
                                             _p(partials), _p(loss), _stream(dev)), "supcon_finalize_sets")
    return partials, loss


def peer_push(desc: _cabi.Peer, src0: torch.Tensor, dst_off0: int, src1, dst_off1: int, flag_id: int,
              wait_flag_id: int = -1, include_self: bool = False):
    """supcon_peer_push: src0 (and src1) -> the same byte offsets of every peer's exchange buffer, then the flag."""
    lib = _cabi.load()
    dev = src0.device
    with _on(dev):
        _cabi.check(lib.supcon_peer_push(ctypes.byref(desc), _p(src0), src0.numel() * src0.element_size(), int(dst_off0),
                                         _p(src1), 0 if src1 is None else src1.numel() * src1.element_size(),
                                         int(dst_off1), int(flag_id), int(wait_flag_id), 1 if include_self else 0,
                                         _stream(dev)), "supcon_peer_push")


def peer_wait(desc: _cabi.Peer, flag_id: int, device):
    """Block the stream until the flag of every rank carries the current step."""
    lib = _cabi.load()
    with _on(device):
        _cabi.check(lib.supcon_peer_wait(ctypes.byref(desc), int(flag_id), _stream(device)), "supcon_peer_wait")


def peer_end_step(desc: _cabi.Peer, flag_id: int, device):
    lib = _cabi.load()
    with _on(device):
        _cabi.check(lib.supcon_peer_end_step(ctypes.byref(desc), int(flag_id), _stream(device)), "supcon_peer_end_step")


def backward_rows_local(z_all, labels_i32, stats_local, partials_local, prob: _cabi.Problem) -> torch.Tensor:
    """Phase 1 of the two-phase row-block backward: the rank's own columns, from its own statistics only
    (no exchange needed yet, no grad_out needed yet).  Returns the workspace backward_rows_remote must be given."""
    lib = _cabi.load()
    dev = z_all.device
    with _on(dev):
        ws = workspace_for(prob, dev)
        _cabi.check(lib.supcon_backward_rows_local(ctypes.byref(prob), _p(z_all), _p(labels_i32), _p(stats_local),
                                                   _p(partials_local), _p(ws), ws.numel(), _stream(dev)),
                    "supcon_backward_rows_local")
    return ws


def backward_rows_remote(z_all, labels_i32, stats_all, partials_global, grad_out, prob: _cabi.Problem, ws,
                         out_dtype=torch.float32) -> torch.Tensor:
    """Phase 2: all other columns + sum of both phases, scaled by grad_out."""
    lib = _cabi.load()
    dev = z_all.device
    with _on(dev):
        dz = torch.empty((prob.n_rows, prob.d), dtype=out_dtype, device=dev)
        g = None
        if grad_out is not None:
            g = grad_out.detach().reshape(()).to(device=dev, dtype=torch.float32)
        _cabi.check(lib.supcon_backward_rows_remote(ctypes.byref(prob), _p(z_all), _p(labels_i32), _p(stats_all),
                                                    _p(partials_global), _p(g), _p(dz), _dtype_id(dz), _p(ws),
                                                    ws.numel(), _stream(dev)),
                    "supcon_backward_rows_remote")
    return dz


def backward_rows(z_all, labels_i32, stats_all, partials_global, grad_out, prob: _cabi.Problem,
                  out_dtype=torch.float32, ws: Optional[torch.Tensor] = None,
                  mem_filled: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``ws``: the workspace forward_rows(..., keep_ws=True) returned for the SAME problem, untouched since (the
    backward then reuses what the forward built there); None = a fresh one.  ``mem_filled``: as in forward_rows
    (supcon_backward_rows_memory)."""
    lib = _cabi.load()
    dev = z_all.device
    with _on(dev):
        dz = torch.empty((prob.n_rows, prob.d), dtype=out_dtype, device=dev)
        if ws is None:
            ws = workspace_for(prob, dev)
        else:
            prob = with_flags(prob, _cabi.FLAG_WS_FROM_FORWARD)
        g = None
        if grad_out is not None:
            g = grad_out.detach().reshape(()).to(device=dev, dtype=torch.float32)
        if mem_filled is None:
            _cabi.check(lib.supcon_backward_rows(ctypes.byref(prob), _p(z_all), _p(labels_i32), _p(stats_all),
                                                 _p(partials_global), _p(g), _p(dz), _dtype_id(dz), _p(ws),
                                                 ws.numel(), _stream(dev)),
                        "supcon_backward_rows")
        else:
            _cabi.check(lib.supcon_backward_rows_memory(ctypes.byref(prob), _p(z_all), _p(labels_i32), _p(mem_filled),
                                                        _p(stats_all), _p(partials_global), _p(g), _p(dz),
                                                        _dtype_id(dz), _p(ws), ws.numel(), _stream(dev)),
                        "supcon_backward_rows_memory")
    return dz


def topk_indices(z_all, labels_i32, row_stats, prob: _cabi.Problem) -> torch.Tensor:
    lib = _cabi.load()
    dev = z_all.device
    with _on(dev):
        idx = torch.empty((prob.n_rows, prob.topk), dtype=torch.int32, device=dev)
        _cabi.check(lib.supcon_topk_indices(ctypes.byref(prob), _p(z_all), _p(labels_i32), _p(row_stats),
                                            _p(idx), _stream(dev)), "supcon_topk_indices")
    return idx


def _loss_dtype(loss: torch.Tensor, z_dtype) -> torch.Tensor:
    """The reference returns the loss in z's dtype (fp32 in every shipped run).
    For 16-bit z the scalar stays fp32: rounding it to bf16 would by itself
    cost 2e-3 relative, the whole bf16 error budget."""
    return loss.to(z_dtype) if z_dtype in (torch.float32, torch.float64) else loss


class SupConFunction(torch.autograd.Function):
    """loss = SupCon(z, labels): forward keeps O(N) row statistics, backward
    recomputes the similarity tiles (replaces autograd through reference
    loss.py:96-153)."""

    @staticmethod
    def forward(ctx, z, labels_i32, tau, sim_id, lambda_uni, uni_t, topk, alpha, flags):
        _require_cuda(z, "z")
        zc = canonical_z(z.detach())
        n, d = zc.shape
        prob = make_problem(n, d, _dtype_id(zc), tau=tau, similarity=sim_id, lambda_uni=lambda_uni,
                            uni_t=uni_t, topk=topk, alpha=alpha, flags=flags)
        ctx.fused = False
        if ctx.needs_input_grad[0] and n <= SMALL_BATCH_MAX and not (flags & (_cabi.FLAG_NO_SMALL | _cabi.FLAG_FORCE_TENSOR)):
            # small batch: forward and backward in ONE launch; backward() only scales by grad_out
            loss, dz, _, _ = loss_and_grad(zc, labels_i32, prob, want_grad=True, out_dtype=zc.dtype)
            ctx.save_for_backward(dz)
            ctx.fused = True
            ctx.in_dtype = z.dtype
            return _loss_dtype(loss, z.dtype)
        if ctx.needs_input_grad[0]:
            # the workspace stays alive until the backward, which reuses the label table / class sums left in it
            stats, partials, loss, ws = forward_rows(zc, labels_i32, prob, want_loss=True, keep_ws=True)
            ctx.save_for_backward(zc, labels_i32, stats, partials, ws)
            ctx.prob = prob
            ctx.in_dtype = z.dtype
        else:
            stats, partials, loss = forward_rows(zc, labels_i32, prob, want_loss=True)
        return _loss_dtype(loss, z.dtype)

    @staticmethod
    def backward(ctx, grad_out):
        if ctx.fused:
            (dz,) = ctx.saved_tensors
            return (dz * grad_out.to(dz.dtype)).to(ctx.in_dtype), None, None, None, None, None, None, None, None
        zc, labels_i32, stats, partials, ws = ctx.saved_tensors
        out_dtype = zc.dtype
        dz = backward_rows(zc, labels_i32, stats, partials, grad_out, ctx.prob, out_dtype=out_dtype, ws=ws)
        return dz.to(ctx.in_dtype), None, None, None, None, None, None, None, None


UNIT_ROWS_TAG = "_supcon_unit_rows"   # set on tensors produced by this library's row normalisation
_warned_untagged = False


def mark_unit_rows(z: torch.Tensor) -> torch.Tensor:
    """Tag ``z`` as having L2-normalised rows (done by l2_normalize / FusedCompressionHead.embed).  The tag is a
    plain attribute of this tensor object: views, casts and copies do not carry it."""
    setattr(z, UNIT_ROWS_TAG, True)
    return z


def unit_rows_flag(z: torch.Tensor, similarity_id_: int, unit_rows) -> int:
    """SUPCON_FLAG_UNIT_ROWS when the caller promises (unit_rows=True) or the tensor carries this library's tag
    (unit_rows=None).  Only a bf16, d = 256, cosine problem is affected: it reaches the tensor-core path under
    the promise and the exact path (z taken as given, any norms) without it."""
    global _warned_untagged
    if unit_rows is None:
        unit_rows = bool(getattr(z, UNIT_ROWS_TAG, False))
        if (not unit_rows and not _warned_untagged and z.dtype == torch.bfloat16 and z.dim() == 2
                and z.size(1) == 256 and z.size(0) >= 256 and similarity_id_ == _cabi.COSINE):
            _warned_untagged = True
            import warnings
            warnings.warn("SupCon: bf16 z of width 256 that was not produced by l2_normalize()/embed() is taken as "
                          "given on the exact fp32 path (any row norms).  If its rows are L2-normalised, set "
                          "loss.assume_unit_rows = True (or pass unit_rows=True) to use the tensor-core path.",
                          stacklevel=3)
    return _cabi.FLAG_UNIT_ROWS if unit_rows else 0


def supcon_loss(z, labels, *, temperature, similarity="cosine", uniformity_weight=0.0, uniformity_t=2.0,
                topk_neg=32, alpha=0.0, flags=0, unit_rows=None) -> torch.Tensor:
    """Functional form of SupConBinaryLoss.forward (reference loss.py:110-153).  ``unit_rows``: None = rows are
    known to be L2-normalised only if ``z`` came from this library's l2_normalize / embed; True = the caller
    promises it (checked on the device: a broken promise gives NaN, never a silently wrong number)."""
    sim_id = similarity_id(similarity) if isinstance(similarity, str) else int(similarity)
    n = z.size(0)
    if n < 2:
        # reference loss.py:138-139,149: no anchor has a positive and the uniformity term needs B > 1
        return torch.tensor(0.0, device=z.device, requires_grad=True)
    lab = canonical_labels(labels, n)
    flags = int(flags) | unit_rows_flag(z, sim_id, unit_rows)
    return SupConFunction.apply(z, lab, float(temperature), sim_id, float(uniformity_weight),
                                float(uniformity_t), int(topk_neg), float(alpha), int(flags))


class _NormalizeFunction(torch.autograd.Function):
    """F.normalize(x, p=2, dim=1) (reference stage1_utils.py:123) on the library's kernels."""

    @staticmethod
    def forward(ctx, x, out_dtype):
        _require_cuda(x, "x")
        lib = _cabi.load()
        xc = x.detach().float().contiguous()
        n, d = xc.shape
        dev = xc.device
        with _on(dev):
            z = torch.empty((n, d), dtype=out_dtype, device=dev)
            norms = torch.empty(n, dtype=torch.float32, device=dev)
            _cabi.check(lib.supcon_normalize_forward(_p(xc), n, d, _p(z), _dtype_id(z), _p(norms), _stream(dev)),
                        "supcon_normalize_forward")
        ctx.save_for_backward(z, norms)
        ctx.in_dtype = x.dtype
        return z

    @staticmethod
    def backward(ctx, dz):
        lib = _cabi.load()
        z, norms = ctx.saved_tensors
        if dz.dtype not in (torch.float32, torch.bfloat16):
            dz = dz.float()
        dz = dz.contiguous()
        n, d = z.shape
        dev = z.device
        with _on(dev):
            dx = torch.empty((n, d), dtype=torch.float32, device=dev)
            _cabi.check(lib.supcon_normalize_backward(_p(z), _dtype_id(z), _p(norms), _p(dz), _dtype_id(dz),
                                                      n, d, _p(dx), _stream(dev)),
                        "supcon_normalize_backward")
        return dx.to(ctx.in_dtype), None


def l2_normalize(x: torch.Tensor, out_dtype=torch.float32) -> torch.Tensor:
    return mark_unit_rows(_NormalizeFunction.apply(x, out_dtype))
