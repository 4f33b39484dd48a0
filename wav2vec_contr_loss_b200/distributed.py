"""Row-sharded SupCon over several GPUs (one process per GPU, NCCL).

Rank r holds the embeddings/labels of its local batch = rows
[r*n_local, (r+1)*n_local) of the global N x N similarity matrix:

  forward   all_gather(z) + all_gather(labels)          (one coalesced NCCL launch over NVLink, on a side
            stream) WHILE the forward kernel sweeps the rank's own columns; then the other columns
            -> row stats + 8 partial sums
            all_gather(partial sums) + all_gather(row stats, N x 32 B)   (one coalesced launch on the side
            stream; one kernel sums the partials in rank order on every rank -- deterministic -- and writes
            the scalar loss, identical on every rank) WHILE the backward kernel already sweeps the rank's own
            columns, which need only its own statistics (the global anchor counts come from the gathered
            labels).  This speculative part of the backward is issued from forward() when z needs a gradient.
  backward  the other columns of the row-block backward: dz_i = sum_j (G_ij + G_ji) z_j for the
            owned rows, recomputing the tiles, + the sum of both phases scaled by grad_out.  Because the
            similarity matrix is symmetric the column-side term G_ji only needs the *statistics*
            of row j, so no N x d reduce-scatter of column partials is needed
            (deviation from the north_star plan, SURVEY H4/H6: the exchange is
            N x 32 B of statistics instead of N x d x 4 B of gradients).

Every rank must hold the SAME number of local rows (checked once per distinct local size with an all-reduce of
min/max; ragged shards raise instead of hanging NCCL).

The result equals the single-GPU loss on the concatenated batch (what the
reference's nn.DataParallel computes, train_stage1.py:82-84).  The returned
gradient is d(global loss)/d(z_local).

``kernels`` is the object providing forward_rows / finalize / backward_rows
(default: the CUDA C-ABI wrappers).  The CPU gloo tests inject an oracle-backed
stand-in to exercise this host logic without a GPU; the product default has no
CPU path.
"""
from typing import Optional

import torch
import torch.distributed as dist

from . import functional as Fn


class _CudaKernels:
    name = "cuda"

    @staticmethod
    def forward_rows(z_all, labels_all, prob):
        stats, partials, _ = Fn.forward_rows(z_all, labels_all, prob, want_loss=False)
        return stats, partials

    finalize = staticmethod(Fn.finalize)

    @staticmethod
    def backward_rows(z_all, labels_all, stats_all, partials, grad_out, prob, out_dtype):
        return Fn.backward_rows(z_all, labels_all, stats_all, partials, grad_out, prob, out_dtype=out_dtype)

    # two-phase forward: own columns while the all-gather is in flight, then the rest
    forward_rows_local = staticmethod(Fn.forward_rows_local)
    forward_rows_remote = staticmethod(Fn.forward_rows_remote)
    # two-phase backward: own columns while the statistics are exchanged, then the rest
    backward_rows_local = staticmethod(Fn.backward_rows_local)
    backward_rows_remote = staticmethod(Fn.backward_rows_remote)
    finalize_sets = staticmethod(Fn.finalize_sets)


_COMM_STREAMS = {}


def _comm_stream(device) -> "torch.cuda.Stream":
    key = (device.type, device.index)
    if key not in _COMM_STREAMS:
        _COMM_STREAMS[key] = torch.cuda.Stream(device=device, priority=-1)
    return _COMM_STREAMS[key]


class PeerExchange:
    """Exchange buffer of one (group, local rows, width, dtype) shape in SYMMETRIC memory: every rank maps every
    other rank's buffer (torch.distributed._symmetric_memory over NVLink / NVSwitch), and the library's own kernels
    write into the peers' buffers directly (csrc/supcon_peer.cu) -- no NCCL call inside a step.

    Layout per rank (byte offsets, 256-aligned): z_all [N, d] | labels_all [N] i32 | stats_all [N, 8] f32 |
    partial_sets [world, 8] f64 | flags.  Rank r only ever writes block r of each region (in every buffer).
    One step = forward (+ its backward); a second forward before the pending backward is refused, because the
    buffers are what the backward reads."""

    def __init__(self, group, n_local: int, d: int, z_dtype, device):
        import torch.distributed._symmetric_memory as symm
        from . import _cabi
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.n_local, self.d, self.device = n_local, d, device
        n = n_local * self.world
        esz = torch.empty((), dtype=z_dtype).element_size()
        self.row_bytes = d * esz

        def al(x):
            return (x + 255) // 256 * 256
        self.off_z = 0
        self.off_labels = al(n * d * esz)
        self.off_stats = self.off_labels + al(n * 4)
        self.off_partials = self.off_stats + al(n * 4 * _cabi.STATS_STRIDE)
        self.off_flags = self.off_partials + al(self.world * 8 * _cabi.N_PARTIALS)
        total = self.off_flags + al(_cabi.peer_flag_bytes(self.world))
        self.buf = symm.empty(total, dtype=torch.uint8, device=device)
        self.buf.zero_()
        self.handle = symm.rendezvous(self.buf, self.group)
        torch.cuda.synchronize(device)
        dist.barrier(group)                       # every buffer is zeroed before anybody pushes into it
        self.peer_bases = torch.tensor([int(p) for p in self.handle.buffer_ptrs], dtype=torch.int64, device=device)
        self.epoch = torch.ones(1, dtype=torch.int32, device=device)
        b = self.buf
        self.z_all = b[self.off_z:self.off_z + n * d * esz].view(z_dtype).view(n, d)
        self.labels_all = b[self.off_labels:self.off_labels + n * 4].view(torch.int32)
        self.stats_all = b[self.off_stats:self.off_stats + n * 4 * _cabi.STATS_STRIDE].view(torch.float32).view(
            n, _cabi.STATS_STRIDE)
        self.partial_sets = b[self.off_partials:self.off_partials + self.world * 8 * _cabi.N_PARTIALS].view(
            torch.float64).view(self.world, _cabi.N_PARTIALS)
        # NVSwitch multicast mapping of the same buffers, when the fabric offers one: a single store per 16 bytes
        # reaches every rank (multimem.st), so a rank's egress is its block, not (world - 1) copies of it
        try:
            mc = int(getattr(self.handle, "multicast_ptr", 0) or 0)
        except Exception:  # noqa: BLE001
            mc = 0
        self.multicast = mc != 0
        self.desc = _cabi.Peer(rank=self.rank, world=self.world, peer_bases=self.peer_bases.data_ptr(),
                               off_flags=self.off_flags, epoch=self.epoch.data_ptr(), mc_base=mc)
        self.pending = False                      # a forward whose backward has not run yet

    def forward(self, zc, labels_local, prob, kernels, want_grad: bool):
        """push rows | own-column forward -> wait -> other columns -> push statistics -> wait -> loss."""
        from . import _cabi
        if self.pending:
            raise RuntimeError("ShardedSupConLoss (peer exchange): forward() called again before the backward of the "
                               "previous call; the exchange buffers hold what that backward reads")
        r, nl, dev = self.rank, self.n_local, self.device
        cur, comm = torch.cuda.current_stream(dev), _comm_stream(dev)
        zb, yb = self.z_all[r * nl:(r + 1) * nl], self.labels_all[r * nl:(r + 1) * nl]
        zb.copy_(zc)                               # own block of the own buffer: only this rank's kernels read it
        yb.copy_(labels_local)
        comm.wait_stream(cur)
        with torch.cuda.stream(comm):              # rows + labels to every peer, beside the own-column forward
            Fn.peer_push(self.desc, zb, self.off_z + r * nl * self.row_bytes, yb, self.off_labels + r * nl * 4,
                         _cabi.PEER_FLAG_Z, wait_flag_id=_cabi.PEER_FLAG_DONE, include_self=False)
        ws = kernels.forward_rows_local(self.z_all, self.labels_all, prob)
        cur.wait_stream(comm)
        Fn.peer_wait(self.desc, _cabi.PEER_FLAG_Z, dev)
        stats, partials = kernels.forward_rows_remote(self.z_all, self.labels_all, prob, ws)
        return self._finish_forward(stats, partials, prob, kernels, want_grad)

    def _finish_forward(self, stats, partials, prob, kernels, want_grad):
        """statistics + partial sums to every rank, wait for everybody's, loss."""
        from . import _cabi
        r, nl, dev = self.rank, self.n_local, self.device
        Fn.peer_push(self.desc, stats, self.off_stats + r * nl * 4 * _cabi.STATS_STRIDE, partials,
                     self.off_partials + r * 8 * _cabi.N_PARTIALS, _cabi.PEER_FLAG_STATS, include_self=True)
        Fn.peer_wait(self.desc, _cabi.PEER_FLAG_STATS, dev)
        partials_global, loss = kernels.finalize_sets(prob, self.partial_sets)
        if want_grad:
            self.pending = True
        else:
            Fn.peer_end_step(self.desc, _cabi.PEER_FLAG_DONE, dev)
        return partials_global, loss

    def backward(self, partials_global, grad_out, prob, kernels, out_dtype):
        from . import _cabi
        if not self.pending:
            raise RuntimeError("ShardedSupConLoss (peer exchange): backward() without a pending forward (a second "
                               "backward through the same graph is not supported in this mode)")
        dz = kernels.backward_rows(self.z_all, self.labels_all, self.stats_all, partials_global, grad_out, prob,
                                   out_dtype)
        Fn.peer_end_step(self.desc, _cabi.PEER_FLAG_DONE, self.device)
        self.pending = False
        return dz


def gather_and_forward(z_local, labels_local, make_prob, group, kernels):
    """all-gather(z, labels) overlapped with the forward over this rank's own columns.

    The local block is copied into place first and the all-gather runs in place on a side stream, so the
    phase-1 kernels (which read only that block) race with nothing.  Returns (z_all, labels_all, prob,
    row_stats, partials)."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    n_local, d = z_local.shape
    dev = z_local.device
    prob = make_prob(n_local * world, d, rank * n_local, n_local)
    two_phase = dev.type == "cuda" and hasattr(kernels, "forward_rows_local")
    if not two_phase:
        z_all, labels_all = gather_inputs(z_local, labels_local, group)
        stats, partials = kernels.forward_rows(z_all, labels_all, prob)
        return z_all, labels_all, prob, stats, partials
    z_all = torch.empty((world * n_local, d), dtype=z_local.dtype, device=dev)
    y_all = torch.empty(world * n_local, dtype=labels_local.dtype, device=dev)
    zb, yb = z_all[rank * n_local:(rank + 1) * n_local], y_all[rank * n_local:(rank + 1) * n_local]
    zb.copy_(z_local)
    yb.copy_(labels_local)
    cur, comm = torch.cuda.current_stream(dev), _comm_stream(dev)
    comm.wait_stream(cur)
    with torch.cuda.stream(comm):
        with _coalesced(group, dev):
            dist.all_gather_into_tensor(z_all, zb, group=group)
            dist.all_gather_into_tensor(y_all, yb, group=group)
    z_all.record_stream(comm)
    y_all.record_stream(comm)
    ws = kernels.forward_rows_local(z_all, y_all, prob)      # runs while the all-gather is in flight
    cur.wait_stream(comm)
    stats, partials = kernels.forward_rows_remote(z_all, y_all, prob, ws)
    return z_all, y_all, prob, stats, partials


def _all_gather_rows(x: torch.Tensor, group) -> torch.Tensor:
    world = dist.get_world_size(group)
    out = torch.empty((world * x.size(0),) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, x.contiguous(), group=group)
    return out


def _coalesced(group, device):
    """One NCCL group launch for the collectives issued inside the block (falls back to
    plain sequential collectives on backends without coalescing support, e.g. gloo)."""
    import contextlib
    mgr = getattr(dist, "_coalescing_manager", None)
    if mgr is None or device.type != "cuda":
        return contextlib.nullcontext()
    return mgr(group=group, device=device, async_ops=False)


def gather_inputs(z_local: torch.Tensor, labels_local: torch.Tensor, group=None):
    """all-gather of embeddings and labels in ONE collective launch. Returns (z_all, labels_all)."""
    world = dist.get_world_size(group)
    z_all = torch.empty((world * z_local.size(0), z_local.size(1)), dtype=z_local.dtype, device=z_local.device)
    y_all = torch.empty(world * labels_local.size(0), dtype=labels_local.dtype, device=labels_local.device)
    with _coalesced(group, z_local.device):
        dist.all_gather_into_tensor(z_all, z_local.contiguous(), group=group)
        dist.all_gather_into_tensor(y_all, labels_local.contiguous(), group=group)
    return z_all, y_all


def exchange_stats(partials: torch.Tensor, stats: torch.Tensor, group=None):
    """Global partial sums + row statistics of every rank in ONE collective launch: the 8 fp64 partial
    sums travel as 16 fp32 words beside the statistics (two all-gathers of the same dtype coalesce; an
    all-reduce would not) and are summed on every rank in rank order, so the result is deterministic.
    ``partials`` is overwritten with the global sums; returns stats_all."""
    world = dist.get_world_size(group)
    stats_all = torch.empty((world * stats.size(0),) + tuple(stats.shape[1:]), dtype=stats.dtype, device=stats.device)
    if partials.dtype == torch.float64 and stats.dtype == torch.float32:
        p32 = partials.view(torch.float32)
        p_all = torch.empty(world * p32.numel(), dtype=torch.float32, device=partials.device)
        with _coalesced(group, stats.device):
            dist.all_gather_into_tensor(p_all, p32, group=group)
            dist.all_gather_into_tensor(stats_all, stats.contiguous(), group=group)
        sets = p_all.view(torch.float64).view(world, -1)
        summed = sets.sum(dim=0)
        summed[5:] = sets[0, 5:]        # global label-derived counts / fixed maximum: identical on every rank
        partials.copy_(summed)
    else:   # generic fallback (CPU stand-in kernels in the gloo tests)
        keep = partials[5:].clone()
        dist.all_reduce(partials, op=dist.ReduceOp.SUM, group=group)
        partials[5:] = keep
        dist.all_gather_into_tensor(stats_all, stats.contiguous(), group=group)
    return stats_all


def exchange_and_local_backward(z_all, labels_all, prob, stats, partials, group, kernels, want_grad=True):
    """The exchange after the forward, overlapped with the part of the backward that does not need it.

    Side stream: ONE coalesced NCCL launch {all-gather partial sums, all-gather row statistics}, then one kernel
    that sums the partials in rank order and writes the scalar loss.  Current stream, meanwhile (only when a
    gradient is wanted): the backward over the rank's OWN columns.  Returns (stats_all, partials_global, loss,
    workspace of the started backward or None)."""
    world = dist.get_world_size(group)
    dev = stats.device
    cur, comm = torch.cuda.current_stream(dev), _comm_stream(dev)
    stats_all = torch.empty((world * stats.size(0), stats.size(1)), dtype=stats.dtype, device=dev)
    p32 = partials.view(torch.float32)
    p_all = torch.empty(world * p32.numel(), dtype=torch.float32, device=dev)
    comm.wait_stream(cur)
    with torch.cuda.stream(comm):
        with _coalesced(group, dev):
            dist.all_gather_into_tensor(p_all, p32, group=group)
            if want_grad:
                dist.all_gather_into_tensor(stats_all, stats, group=group)
        partials_global, loss = kernels.finalize_sets(prob, p_all.view(torch.float64))
    for t in (stats_all, p_all, partials_global, loss, stats, partials):
        t.record_stream(comm)
    ws = kernels.backward_rows_local(z_all, labels_all, stats, partials, prob) if want_grad else None
    cur.wait_stream(comm)
    return stats_all, partials_global, loss, ws


_CHECKED_SHARDS = set()


def check_equal_shards(n_local: int, device, group=None):
    """Every rank must contribute the same number of rows (row_offset = rank * n_local; all_gather_into_tensor
    needs equal shards).  Verified once per distinct local size: a ragged last batch raises here instead of
    hanging or corrupting the collective."""
    key = (id(group), n_local)
    if key in _CHECKED_SHARDS:
        return
    t = torch.tensor([n_local, -n_local], device=device, dtype=torch.int64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    lo, hi = -int(t[1]), int(t[0])
    if lo != hi:
        raise ValueError(f"ShardedSupConLoss needs the same local batch size on every rank (got between {lo} and {hi} "
                         f"rows): use drop_last / the equal-step BalancedBatchSampler")
    _CHECKED_SHARDS.add(key)


class _ShardedSupCon(torch.autograd.Function):
    @staticmethod
    def forward(ctx, z_local, labels_local, cfg, group, kernels, peer=None):
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        zc = Fn.canonical_z(z_local.detach())
        check_equal_shards(zc.size(0), zc.device, group)

        def make_prob(n_total, d, row_offset, n_rows):
            return Fn.make_problem(n_total, d, Fn._dtype_id(zc), row_offset=row_offset, n_rows=n_rows, **cfg)

        ctx.peer = None
        if peer is not None:      # exchange through peer memory: this library's kernels only
            n_local = zc.size(0)
            prob = make_prob(n_local * world, zc.size(1), rank * n_local, n_local)
            want_grad = ctx.needs_input_grad[0]
            partials, loss = peer.forward(zc, labels_local, prob, kernels, want_grad)
            if want_grad:
                ctx.save_for_backward(partials)
                ctx.peer, ctx.prob, ctx.kernels, ctx.in_dtype, ctx.work_dtype = peer, prob, kernels, z_local.dtype, zc.dtype
            return Fn._loss_dtype(loss, z_local.dtype)

        z_all, labels_all, prob, stats, partials = gather_and_forward(zc, labels_local, make_prob, group, kernels)
        want_grad = ctx.needs_input_grad[0]
        overlap = zc.device.type == "cuda" and hasattr(kernels, "backward_rows_local")
        ws = None
        if overlap:
            stats_all, partials, loss, ws = exchange_and_local_backward(z_all, labels_all, prob, stats, partials,
                                                                        group, kernels, want_grad)
        else:
            if want_grad:
                stats_all = exchange_stats(partials, stats, group)
            else:
                keep = partials[5:].clone()
                dist.all_reduce(partials, op=dist.ReduceOp.SUM, group=group)
                partials[5:] = keep
            loss = kernels.finalize(prob, partials)
        if want_grad:
            ctx.save_for_backward(z_all, labels_all, stats_all, partials)
            ctx.prob, ctx.kernels, ctx.in_dtype, ctx.work_dtype = prob, kernels, z_local.dtype, zc.dtype
            ctx.ws = ws
        return Fn._loss_dtype(loss, z_local.dtype)

    @staticmethod
    def backward(ctx, grad_out):
        if ctx.peer is not None:
            (partials,) = ctx.saved_tensors
            dz = ctx.peer.backward(partials, grad_out, ctx.prob, ctx.kernels, ctx.work_dtype)
            return dz.to(ctx.in_dtype), None, None, None, None, None
        z_all, labels_all, stats_all, partials = ctx.saved_tensors
        if ctx.ws is not None:
            dz = ctx.kernels.backward_rows_remote(z_all, labels_all, stats_all, partials, grad_out, ctx.prob, ctx.ws,
                                                  out_dtype=ctx.work_dtype)
            ctx.ws = None
        else:
            dz = ctx.kernels.backward_rows(z_all, labels_all, stats_all, partials, grad_out, ctx.prob, ctx.work_dtype)
        return dz.to(ctx.in_dtype), None, None, None, None, None


class ShardedSupConLoss(torch.nn.Module):
    """SupConBinaryLoss over the global batch of all ranks (same constructor and
    call signature as reference loss.py:19-25,110-114, plus ``group``).

    Every rank must pass the same number of rows per call (equal shards; checked, a mismatch raises).
    When ``z`` requires a gradient, forward() already launches the part of the backward that needs no
    exchange (the rank's own columns) so that it overlaps the all-gather of the row statistics; a second
    backward() through the same graph (retain_graph) recomputes the whole backward."""

    def __init__(self, temperature: float = 0.2, similarity: str = "geodesic", uniformity_weight: float = 0.0,
                 uniformity_t: float = 2.0, group: Optional[dist.ProcessGroup] = None, kernels=None,
                 exchange: str = "nccl"):
        """``exchange``: "nccl" = all-gathers through torch.distributed (works on any group);
        "peer" = the library's own kernels write rows and row statistics straight into every peer's buffer over
        NVLink (symmetric memory; one node with peer access; forward and its backward must alternate);
        "auto" = "peer" when the symmetric buffer can be set up, else "nccl"."""
        super().__init__()
        self.tau = temperature
        self.similarity = similarity.lower()
        self.lambda_uni = float(uniformity_weight)
        self.uni_t = float(uniformity_t)
        Fn.similarity_id(similarity)
        self.group = group
        self.kernels = kernels if kernels is not None else _CudaKernels
        self.kernel_flags = 0
        self.assume_unit_rows = None   # see SupConBinaryLoss.assume_unit_rows
        if exchange not in ("nccl", "peer", "auto"):
            raise ValueError(f"Unknown exchange: {exchange}")
        self.exchange = exchange
        self._peers = {}               # (n_local, d, dtype) -> PeerExchange

    def forward(self, z: torch.Tensor, labels: torch.Tensor, topk_neg: int = 32, alpha: float = 0.0):
        if not (dist.is_available() and dist.is_initialized()):
            raise RuntimeError("ShardedSupConLoss needs an initialised torch.distributed process group")
        if self.kernels is _CudaKernels:
            Fn._require_cuda(z, "z")
        sim = Fn.similarity_id(self.similarity)
        cfg = dict(tau=self.tau, similarity=sim, lambda_uni=self.lambda_uni,
                   uni_t=self.uni_t, topk=topk_neg, alpha=alpha,
                   flags=self.kernel_flags | Fn.unit_rows_flag(z, sim, self.assume_unit_rows))
        lab = Fn.canonical_labels(labels, z.size(0))
        peer = None
        if self.exchange != "nccl" and self.kernels is _CudaKernels:
            peer = self._peer_for(z)
            if peer is not None:
                from . import _cabi
                cfg["flags"] |= _cabi.FLAG_PEER_EXCHANGE
        return _ShardedSupCon.apply(z, lab, cfg, self.group, self.kernels, peer)

    def _peer_for(self, z):
        work_dtype = z.dtype if z.dtype in (torch.float32, torch.bfloat16) else torch.float32
        key = (z.size(0), z.size(1), work_dtype)
        if key not in self._peers:
            check_equal_shards(z.size(0), z.device, self.group)
            try:
                self._peers[key] = PeerExchange(self.group, z.size(0), z.size(1), work_dtype, z.device)
            except Exception as exc:  # noqa: BLE001  (no peer access / symmetric memory unavailable)
                if self.exchange == "peer":
                    raise
                import warnings
                warnings.warn(f"ShardedSupConLoss: peer exchange unavailable ({type(exc).__name__}: {exc}); using NCCL")
                self._peers[key] = None
        return self._peers[key]
