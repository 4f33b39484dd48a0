"""fp64 torch-autograd reference of the SupCon loss with a cross-batch memory (wav2vec_contr_loss_b200/memory.py).

Anchors are the batch rows i < B; columns are the batch followed by the M memory rows, j != i.  lse, positives,
negatives and the top-K hard negatives (value desc, index asc) run over all B + M columns; |A_f|, |A_m| count
anchors; the uniformity term is over the batch's own pairs i < j < B.  The memory is a constant, so autograd's
gradient with respect to the batch is d loss / d z_batch.  With M = 0 this is the reference loss (oracle.closed_form).
"""
import math

import torch

INT_MAX = 2**31 - 1


def memory_loss(z_batch, y_batch, z_mem=None, y_mem=None, *, tau, similarity, lam=0.0, t=2.0, topk=32, alpha=0.0,
                want_grad=True):
    """Returns dict(loss float, dz [B, d] fp64 or None, lse, npos, nneg, thr_val, thr_idx, member [B, B+M] bool)."""
    zb = z_batch.detach().to("cpu", torch.float64).clone().requires_grad_(want_grad)
    yb = y_batch.detach().to("cpu").reshape(-1)
    b, d = zb.shape
    if z_mem is None or z_mem.numel() == 0:
        zm = torch.zeros(0, d, dtype=torch.float64)
        ym = yb[:0]
    else:
        zm = z_mem.detach().to("cpu", torch.float64)
        ym = y_mem.detach().to("cpu").reshape(-1)
    cols = torch.cat([zb, zm])
    yc = torch.cat([yb, ym])
    n = cols.size(0)
    c = zb @ cols.t()
    if similarity == "cosine":
        s = c
    else:
        hi = 1.0 - 1e-7
        s = 2.0 * (1.0 - torch.acos(c.clamp(-hi, hi)) / math.pi) - 1.0
    lg = s / tau
    self_m = torch.zeros(b, n, dtype=torch.bool)
    self_m[torch.arange(b), torch.arange(b)] = True
    pos = (yb.view(-1, 1) == yc.view(1, -1)) & ~self_m
    neg = ~pos & ~self_m
    lse = torch.logsumexp(lg.masked_fill(self_m, float("-inf")), dim=1)
    npos, nneg = pos.sum(1), neg.sum(1)
    pos_mean = (lg * pos).sum(1) / npos.clamp_min(1)
    # hard negatives: stable descending sort of the (detached) similarities = (value desc, index asc)
    order = torch.sort(s.detach().masked_fill(~neg, float("-inf")), dim=1, descending=True, stable=True).indices
    k_i = nneg.clamp_max(max(int(topk), 0))
    member = torch.zeros_like(neg)
    member.scatter_(1, order, torch.arange(n).view(1, -1) < k_i.view(-1, 1))
    member &= neg
    last = (k_i - 1).clamp_min(0).view(-1, 1)
    thr_idx = order.gather(1, last).view(-1)
    thr_val = s.detach().gather(1, thr_idx.view(-1, 1)).view(-1)
    all_sel = k_i >= nneg
    thr_val = torch.where(all_sel, torch.full_like(thr_val, float("-inf")), thr_val)
    thr_idx = torch.where(all_sel, torch.full_like(thr_idx, INT_MAX), thr_idx)

    in_f = npos > 0
    in_m = in_f & (nneg > 0) & (int(topk) >= 1)
    if bool(in_f.any()):
        full = (lse - pos_mean)[in_f].mean()
        if bool(in_m.any()):
            lse_m = torch.logsumexp(lg[in_m].masked_fill(~(pos | member)[in_m], float("-inf")), dim=1)
            mined = (lse_m - pos_mean[in_m]).mean()
        else:
            mined = full
        loss = (1.0 - alpha) * full + alpha * mined
    else:
        loss = zb.sum() * 0.0
    if lam > 0.0 and b > 1:
        nrm = (zb * zb).sum(1)
        g = zb @ zb.t()
        d2 = (nrm.view(-1, 1) + nrm.view(1, -1) - 2.0 * g).clamp_min(0.0)
        iu = torch.triu_indices(b, b, offset=1)
        loss = loss + lam * torch.log(torch.exp(-t * d2[iu[0], iu[1]]).mean() + 1e-8)
    dz = None
    if want_grad:
        (dz,) = torch.autograd.grad(loss, zb, allow_unused=True)
        if dz is None:
            dz = torch.zeros_like(zb)
    return dict(loss=float(loss.detach()), dz=dz, lse=lse.detach(), npos=npos, nneg=nneg, thr_val=thr_val,
                thr_idx=thr_idx, member=member)
