"""TEST INFRASTRUCTURE ONLY -- CPU oracle for the Stage-1 SupCon objective.

Two independent restatements of the reference algorithm:

``anchor_loop_loss``  a per-anchor loop that follows the reference's control
    flow (reference loss.py:110-153 for the binary class, :168-210 for the
    multi-class class) using autograd.  This is the *port* that ``bench.py``
    times as the CPU baseline on the GPU box, where /root/reference is absent.

``closed_form``  the vectorised closed form of SURVEY.md Appendix A (forward and
    analytic backward), evaluated in row blocks so it also runs at large N.  It
    is written in the same "row stats -> (G + G^T) z" shape the CUDA path uses
    (``rowblock_forward`` / ``rowblock_backward``), so the multi-rank host logic
    can be exercised on CPU against it.

Tie rule for hard-negative selection: (similarity descending, index ascending),
i.e. lowest index wins (north_star); the reference itself uses an unstable sort
whose tie order is unspecified (reference loss.py:67-68).

Parity pinning: see oracle/__init__.py -- pinned against the live reference in
tests/test_oracle_vs_reference.py (build container) and against the committed
fixtures in tests/golden/ everywhere.
"""
import math
from typing import Dict, Optional

import torch

COSINE, GEODESIC = 0, 1
_SIM_IDS = {"cosine": COSINE, "geodesic": GEODESIC}

# indices into the partial-sum vector exchanged between ranks
P_SUM_FULL, P_CNT_FULL, P_SUM_MINED, P_CNT_MINED, P_SUM_W = 0, 1, 2, 3, 4
N_PARTIALS = 8


def sim_id(similarity: str) -> int:
    s = similarity.lower()
    if s not in _SIM_IDS:
        raise ValueError(f"Unknown similarity: {similarity}")
    return _SIM_IDS[s]


# --------------------------------------------------------------------------
# 1. per-anchor loop port (timed CPU baseline; mirrors reference control flow)
# --------------------------------------------------------------------------
def _pair_sim(z: torch.Tensor, similarity: str) -> torch.Tensor:
    """reference loss.py:96-107."""
    gram = z @ z.t()
    if similarity == "cosine":
        return gram
    eps = 1e-7
    ang = torch.acos(gram.clamp(-1.0 + eps, 1.0 - eps))
    unit = 1.0 - ang / math.pi
    return 2.0 * unit - 1.0


def anchor_loop_loss(z, labels, *, temperature=0.2, similarity="geodesic",
                     uniformity_weight=0.0, uniformity_t=2.0, topk_neg=32, alpha=0.0):
    """Per-anchor port of SupConBinaryLoss.forward (reference loss.py:110-153).

    Same op sequence per anchor as the reference (boolean-index, logsumexp,
    full-row sort, cat) so its CPU cost is representative of the reference's.
    """
    similarity = similarity.lower()
    sim_id(similarity)
    n = z.size(0)
    dev = z.device
    diag = torch.eye(n, device=dev, dtype=torch.bool)
    sim = _pair_sim(z, similarity).masked_fill(diag, float("-inf"))
    col = labels.view(-1, 1)
    same = (col == col.t()) & ~diag
    diff = ~same & ~diag

    full_terms, mined_terms = [], []
    for a in range(n):
        row, pm, nm = sim[a], same[a], diff[a]
        # reference loss.py:36-49
        scaled = row / temperature
        has_pos = bool(pm.any())
        if has_pos:
            pl = scaled[pm]
            full_terms.append(-(pl - torch.logsumexp(scaled, dim=0)).mean())
        # reference loss.py:51-73
        if has_pos and bool(nm.any()):
            ps, ns = row[pm], row[nm]
            k = min(topk_neg, ns.numel())
            if k >= 1:
                hard, _ = torch.sort(ns, descending=True)
                lg = torch.cat([ps, hard[:k]], dim=0) / temperature
                lp = lg - torch.logsumexp(lg, dim=0)
                mined_terms.append(-lp[: ps.numel()].mean())

    if not full_terms:
        total = torch.tensor(0.0, device=dev, requires_grad=True)
    else:
        lf = torch.stack(full_terms).mean()
        lm = torch.stack(mined_terms).mean() if mined_terms else lf
        total = (1.0 - alpha) * lf + alpha * lm
    if uniformity_weight > 0.0 and n > 1:
        # reference loss.py:77-93
        d2 = torch.pdist(z, p=2).pow(2)
        total = total + uniformity_weight * torch.log(torch.exp(-uniformity_t * d2).mean() + 1e-8)
    return total


def anchor_loop_multiclass(z, labels, temperature=0.1):
    """Per-anchor port of SupConMultiClassLoss.forward (reference loss.py:168-210)."""
    assert labels.dim() == 1 and labels.size(0) == z.size(0), "labels must be shape (B,)"
    n = z.size(0)
    diag = torch.eye(n, dtype=torch.bool, device=z.device)
    lg = (z @ z.t() / temperature).masked_fill(diag, float("-inf"))
    col = labels.view(-1, 1)
    same = (col == col.t()) & ~diag
    terms = []
    for a in range(n):
        idx = torch.nonzero(same[a]).squeeze(-1)
        if idx.numel() == 0:
            continue
        terms.append(-(lg[a, idx] - torch.logsumexp(lg[a, ~diag[a]], dim=0)).mean())
    if not terms:
        return torch.tensor(0.0, device=z.device, requires_grad=True)
    return torch.stack(terms).mean()


# --------------------------------------------------------------------------
# 2. closed form (SURVEY.md Appendix A), row-blocked
# --------------------------------------------------------------------------
def _clamp_bounds(dtype):
    # the reference clamps an fp32 tensor with python floats: the bound that is
    # applied is fp32(1-1e-7) = 1-2^-23 (SURVEY Appendix C).  In fp64: 1-1e-7.
    if dtype == torch.float32:
        hi = float(torch.tensor(1.0 - 1e-7, dtype=torch.float32))
    else:
        hi = 1.0 - 1e-7
    return -hi, hi


def _sim_and_slope(c: torch.Tensor, similarity: int):
    """similarity s(c) and ds/dc (reference loss.py:96-107; Appendix A)."""
    if similarity == COSINE:
        return c, None
    lo, hi = _clamp_bounds(c.dtype)
    ch = c.clamp(lo, hi)
    s = 2.0 * (1.0 - torch.acos(ch) / math.pi) - 1.0
    slope = (2.0 / math.pi) / torch.sqrt(1.0 - ch * ch)
    slope = torch.where((c >= lo) & (c <= hi), slope, torch.zeros_like(slope))
    return s, slope


def rowblock_forward(z_all, labels_all, row_offset, n_rows, *, tau, similarity, topk,
                     lambda_uni=0.0, uni_t=2.0, block=1024, want_topk_idx=False):
    """Forward for the rows [row_offset, row_offset+n_rows) against all columns.

    Returns ``stats`` (dict of per-row tensors: lse, lse_m, npos, nneg, thr_val,
    thr_idx, wsum, pos_mean) and ``partials`` (float64 tensor [N_PARTIALS]: sum of
    per-anchor full losses, |A_f|, sum of mined losses, |A_m|, sum_{i,j!=i} w_ij).
    ``thr_val/thr_idx`` is the lowest-ranked selected hard negative under the
    (value desc, index asc) order; (-inf, INT_MAX) when every negative is selected.
    Everything is computed on ``z_all``'s device (``labels_all`` must live there too), so
    large batches can be evaluated in fp64 on a GPU; ``rowblock_backward`` likewise.
    """
    n = z_all.size(0)
    dt, dev = z_all.dtype, z_all.device
    lab = labels_all.view(-1)
    INT_MAX = 2**31 - 1
    out = {k: [] for k in ("lse", "lse_m", "npos", "nneg", "thr_val", "thr_idx", "wsum", "pos_mean")}
    topk_lists = []
    nrm_all = (z_all * z_all).sum(1)
    for r0 in range(row_offset, row_offset + n_rows, block):
        r1 = min(r0 + block, row_offset + n_rows)
        rows = torch.arange(r0, r1, device=dev)
        c = z_all[r0:r1] @ z_all.t()
        s, _ = _sim_and_slope(c, similarity)
        lg = s / tau
        self_m = torch.zeros_like(lg, dtype=torch.bool)
        self_m[torch.arange(r1 - r0, device=dev), rows] = True
        pos = (lab[r0:r1].view(-1, 1) == lab.view(1, -1)) & ~self_m
        neg = ~pos & ~self_m
        lgm = lg.masked_fill(self_m, float("-inf"))
        lse = torch.logsumexp(lgm, dim=1)
        npos = pos.sum(1)
        nneg = neg.sum(1)
        pos_mean = (lg * pos).sum(1) / npos.clamp_min(1)
        # hard negatives: stable descending sort => ties resolved to lowest index
        negval = s.masked_fill(~neg, float("-inf"))
        order = torch.sort(negval, dim=1, descending=True, stable=True).indices
        k_i = nneg.clamp_max(max(int(topk), 0))
        rank = torch.arange(n, device=dev).view(1, -1)
        sel_sorted = rank < k_i.view(-1, 1)
        member = torch.zeros_like(neg)
        member.scatter_(1, order, sel_sorted)
        member &= neg
        lse_m = torch.logsumexp(lg.masked_fill(~(pos | member), float("-inf")), dim=1)
        last = (k_i - 1).clamp_min(0).view(-1, 1)
        thr_idx = order.gather(1, last).view(-1)
        thr_val = s.gather(1, thr_idx.view(-1, 1)).view(-1)
        all_sel = (k_i >= nneg)
        thr_val = torch.where(all_sel, torch.full_like(thr_val, float("-inf")), thr_val)
        thr_idx = torch.where(all_sel, torch.full_like(thr_idx, INT_MAX), thr_idx)
        if lambda_uni > 0.0:
            d2 = (nrm_all[r0:r1].view(-1, 1) + nrm_all.view(1, -1) - 2.0 * c).clamp_min(0.0)
            w = torch.exp(-uni_t * d2).masked_fill(self_m, 0.0)
            wsum = w.sum(1)
        else:
            wsum = torch.zeros(r1 - r0, dtype=dt, device=dev)
        for k, v in (("lse", lse), ("lse_m", lse_m), ("npos", npos), ("nneg", nneg),
                     ("thr_val", thr_val), ("thr_idx", thr_idx), ("wsum", wsum), ("pos_mean", pos_mean)):
            out[k].append(v)
        if want_topk_idx:
            for i in range(r1 - r0):
                topk_lists.append(order[i, : int(k_i[i])].tolist())
    stats = {k: torch.cat(v) for k, v in out.items()}
    in_f = stats["npos"] > 0
    in_m = in_f & (stats["nneg"] > 0) & (int(topk) >= 1)
    l_full = stats["lse"] - stats["pos_mean"]
    l_mined = stats["lse_m"] - stats["pos_mean"]
    partials = torch.zeros(N_PARTIALS, dtype=torch.float64, device=dev)
    partials[P_SUM_FULL] = l_full[in_f].double().sum()
    partials[P_CNT_FULL] = in_f.sum()
    partials[P_SUM_MINED] = l_mined[in_m].double().sum()
    partials[P_CNT_MINED] = in_m.sum()
    partials[P_SUM_W] = stats["wsum"].double().sum()
    if want_topk_idx:
        stats["topk_idx"] = topk_lists
    return stats, partials


def loss_from_partials(partials, n_total, *, alpha, lambda_uni):
    """Scalar loss and the global coefficients the backward needs.

    reference loss.py:137-151 (alpha blend, empty-set fallbacks, uniformity)."""
    cnt_f = float(partials[P_CNT_FULL])
    cnt_m = float(partials[P_CNT_MINED])
    coef = {"w_full": 0.0, "w_mined": 0.0, "cnt_f": cnt_f, "cnt_m": cnt_m, "uni_scale": 0.0}
    if cnt_f == 0:
        main = 0.0
    else:
        full = float(partials[P_SUM_FULL]) / cnt_f
        if cnt_m == 0:
            mined = full
            coef["w_full"], coef["w_mined"] = 1.0, 0.0
        else:
            mined = float(partials[P_SUM_MINED]) / cnt_m
            coef["w_full"], coef["w_mined"] = 1.0 - alpha, alpha
        main = (1.0 - alpha) * full + alpha * mined
    if lambda_uni > 0.0 and n_total > 1:
        pairs2 = float(n_total) * float(n_total - 1)          # ordered pairs = 2M
        m = float(partials[P_SUM_W]) / pairs2
        main = main + lambda_uni * math.log(m + 1e-8)
        coef["uni_scale"] = lambda_uni / ((pairs2 / 2.0) * (m + 1e-8))   # lambda / (M (m+eps))
    return main, coef


def rowblock_backward(z_all, labels_all, row_offset, n_rows, stats_all, coef, *, tau, similarity,
                      topk, lambda_uni=0.0, uni_t=2.0, block=1024):
    """dz for the owned rows using only column *stats* of the other rows:
    dz_i = sum_j (G_ij + G_ji) z_j (+ uniformity), Appendix A with H = G + G^T."""
    n = z_all.size(0)
    dt, dev = z_all.dtype, z_all.device
    lab = labels_all.view(-1)
    npos_all = stats_all["npos"].to(dt)
    in_f = stats_all["npos"] > 0
    in_m = in_f & (stats_all["nneg"] > 0) & (int(topk) >= 1)
    a_f = in_f.to(dt) * (coef["w_full"] / max(coef["cnt_f"], 1.0) / tau)
    a_m = in_m.to(dt) * (coef["w_mined"] / max(coef["cnt_m"], 1.0) / tau)
    inv_p = torch.where(in_f, 1.0 / npos_all.clamp_min(1), torch.zeros_like(npos_all))
    nrm_all = (z_all * z_all).sum(1)
    idx_all = torch.arange(n, device=dev)
    dz = torch.zeros(n_rows, z_all.size(1), dtype=dt, device=dev)
    for r0 in range(row_offset, row_offset + n_rows, block):
        r1 = min(r0 + block, row_offset + n_rows)
        R = slice(r0, r1)
        rows = torch.arange(r0, r1, device=dev)
        c = z_all[R] @ z_all.t()
        s, slope = _sim_and_slope(c, similarity)
        lg = s / tau
        self_m = torch.zeros_like(lg, dtype=torch.bool)
        self_m[torch.arange(r1 - r0, device=dev), rows] = True
        pos = (lab[R].view(-1, 1) == lab.view(1, -1)) & ~self_m
        neg = ~pos & ~self_m
        # row-side membership: j in top_i ; column-side: i in top_j
        mem_row = pos | (neg & ((s > stats_all["thr_val"][R].view(-1, 1)) |
                                ((s == stats_all["thr_val"][R].view(-1, 1)) &
                                 (idx_all.view(1, -1) <= stats_all["thr_idx"][R].view(-1, 1)))))
        mem_col = pos | (neg & ((s > stats_all["thr_val"].view(1, -1)) |
                                ((s == stats_all["thr_val"].view(1, -1)) &
                                 (rows.view(-1, 1) <= stats_all["thr_idx"].view(1, -1)))))
        e_row = torch.exp(lg - stats_all["lse"][R].view(-1, 1))
        e_col = torch.exp(lg - stats_all["lse"].view(1, -1))
        em_row = torch.exp(lg - stats_all["lse_m"][R].view(-1, 1)) * mem_row
        em_col = torch.exp(lg - stats_all["lse_m"].view(1, -1)) * mem_col
        posf = pos.to(dt)
        g_row = a_f[R].view(-1, 1) * (e_row - posf * inv_p[R].view(-1, 1)) + \
                a_m[R].view(-1, 1) * (em_row - posf * inv_p[R].view(-1, 1))
        g_col = a_f.view(1, -1) * (e_col - posf * inv_p.view(1, -1)) + \
                a_m.view(1, -1) * (em_col - posf * inv_p.view(1, -1))
        h = g_row + g_col
        if slope is not None:
            h = h * slope
        h = h.masked_fill(self_m, 0.0)
        blk = h @ z_all
        if coef["uni_scale"] != 0.0:
            d2 = (nrm_all[R].view(-1, 1) + nrm_all.view(1, -1) - 2.0 * c).clamp_min(0.0)
            w = torch.exp(-uni_t * d2).masked_fill(self_m, 0.0)
            cu = coef["uni_scale"] * (-2.0 * uni_t)
            blk = blk + cu * (w.sum(1, keepdim=True) * z_all[R] - w @ z_all)
        dz[r0 - row_offset: r1 - row_offset] = blk
    return dz


def closed_form(z, labels, *, temperature=0.2, similarity="geodesic", uniformity_weight=0.0,
                uniformity_t=2.0, topk_neg=32, alpha=0.0, dtype=torch.float64, block=1024,
                want_grad=True, want_topk_idx=False) -> Dict[str, object]:
    """Loss (python float), dz (tensor, ``dtype``) and row stats for the whole batch."""
    sid = sim_id(similarity)
    zz = z.detach().to("cpu").to(dtype)
    lab = _canon_labels(labels)
    n = zz.size(0)
    stats, partials = rowblock_forward(zz, lab, 0, n, tau=temperature, similarity=sid, topk=topk_neg,
                                       lambda_uni=uniformity_weight, uni_t=uniformity_t, block=block,
                                       want_topk_idx=want_topk_idx)
    loss, coef = loss_from_partials(partials, n, alpha=alpha, lambda_uni=uniformity_weight)
    res = {"loss": loss, "stats": stats, "partials": partials, "coef": coef}
    if want_grad:
        res["dz"] = rowblock_backward(zz, lab, 0, n, stats, coef, tau=temperature, similarity=sid,
                                      topk=topk_neg, lambda_uni=uniformity_weight, uni_t=uniformity_t,
                                      block=block)
    return res


def _canon_labels(labels: torch.Tensor) -> torch.Tensor:
    lab = labels.detach().to("cpu").view(-1)
    if lab.is_floating_point():
        lab = torch.unique(lab, return_inverse=True)[1]
    return lab.to(torch.int64)


# --------------------------------------------------------------------------
# 3. normalisation either side of the loss (reference stage1_utils.py:123,149)
# --------------------------------------------------------------------------
def normalize_fwd(x: torch.Tensor, eps: float = 1e-12):
    nrm = x.norm(dim=1, keepdim=True).clamp_min(eps)
    return x / nrm, nrm


def normalize_bwd(z: torch.Tensor, nrm: torch.Tensor, dz: torch.Tensor):
    return (dz - z * (z * dz).sum(1, keepdim=True)) / nrm


# --------------------------------------------------------------------------
# 4. synthetic inputs (SURVEY.md section 8d) -- shared by tests and bench
# --------------------------------------------------------------------------
def make_inputs(n: int, d: int = 256, kind: str = "iso", seed: int = 1337, classes: int = 2,
                sigma: float = 1.0):
    """x (n,d) fp32 un-normalised and balanced labels (int64)."""
    g = torch.Generator().manual_seed(seed)
    if classes == 2:
        y = torch.zeros(n, dtype=torch.int64)
        y[torch.randperm(n, generator=g)[: n // 2]] = 1
    else:
        y = torch.randint(0, classes, (n,), generator=g, dtype=torch.int64)
    if kind == "iso":
        x = torch.randn(n, d, generator=g)
    elif kind == "clustered":
        mu = torch.nn.functional.normalize(torch.randn(classes, d, generator=g), dim=1)
        x = mu[y] + sigma * torch.randn(n, d, generator=g) / math.sqrt(d)
    elif kind == "ties":
        x = torch.randn(n, d, generator=g)
        pairs = torch.randperm(n // 2, generator=g)[: max(1, n // 40)]
        x[2 * pairs + 1] = x[2 * pairs]
    else:
        raise ValueError(kind)
    return x, y


def appendix_b_inputs(b: int, d: int):
    """RNG-free inputs of SURVEY.md Appendix B (float64)."""
    i = torch.arange(b, dtype=torch.float64).view(-1, 1)
    j = torch.arange(d, dtype=torch.float64).view(1, -1)
    x = torch.sin(0.37 * i + 0.11 * j + 0.05 * i * j) + 0.25 * torch.cos(1.3 * i - 0.7 * j)
    y = ((7 * torch.arange(b)) % 5 < 2).to(torch.int64)
    return x, y
