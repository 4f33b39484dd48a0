"""GPU parity, round-2 additions (VERDICT r01 "next round" items 3 and 4):
  * the tensor path on rows that are NOT L2-normalised (z taken as given, loss.py:110-121);
  * hard-negative index sets through the TENSOR path held to equality on exact-arithmetic inputs;
  * the headline size N = 65536: every row's statistics and the loss against a plain fp64 evaluation,
    sampled rows (statistics, top-K sets, dz) against the oracle's brute force;
  * two-phase backward (own columns first) == single-phase backward == oracle;
  * rank-ordered partial-sum kernel (supcon_finalize_sets);
  * duplicate rows + uniformity term on all three kernel families.
Tolerances (north_star): 1e-5 relative fp32 path, 2e-3 bf16-input path, index sets exact."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import supcon_oracle as O
import gpu_util as G
from wav2vec_contr_loss_b200 import _cabi
from wav2vec_contr_loss_b200 import functional as Fn

pytestmark = pytest.mark.gpu

TOL_F32 = 1e-5
TOL_BF16 = 2e-3


def _tc_problem(n, *, tau=0.07, sim="cosine", lam=0.0, topk=15, alpha=0.0, row_offset=0, n_rows=None, flags=2):
    return Fn.make_problem(n, 256, _cabi.BF16, tau=tau, similarity=Fn.similarity_id(sim), lambda_uni=lam, uni_t=2.0,
                           topk=topk, alpha=alpha, flags=flags, row_offset=row_offset, n_rows=n_rows)


# ---------------------------------------------------------------------------------------------------------
# un-normalised rows on the tensor path (ADVICE r01 medium / VERDICT weak #1)
# ---------------------------------------------------------------------------------------------------------
def _scaled_rows(n, scale, seed=11):
    x, y = O.make_inputs(n, 256, "iso", seed=seed)
    z = F.normalize(x, dim=1)
    if scale == "3x":
        z = 3.0 * z                               # the VERDICT's case: cosine logits reach 9 / tau
    elif scale == "ragged":
        z = z * (1.0 + 0.5 * torch.rand(n, 1, generator=torch.Generator().manual_seed(3)))   # |z| in [1, 1.5]
    return z.to(torch.bfloat16), y


@pytest.mark.parametrize("tau", [0.07, 0.03])
@pytest.mark.parametrize("sim", ["cosine", "geodesic"])
@pytest.mark.parametrize("scale", ["3x", "ragged"])
def test_bf16_unnormalised_rows_through_the_module(cuda_device, tau, sim, scale):
    """z is taken as given (loss.py:110-121).  bf16, d = 256, N >= 256 with rows that are NOT unit norm and no
    promise: cosine takes the exact path (online maximum), geodesic the tensor path (its similarities are in
    [-1, 1] whatever the norms).  Either way: finite, within the bf16 tolerance of the oracle."""
    zb, y = _scaled_rows(512, scale)
    kw = dict(tau=tau, similarity=sim, lam=0.0, t=2.0, topk=15, alpha=0.5)
    ref = G.oracle_for(zb.float(), y, **kw)
    loss, dz = G.kernel_loss_and_grad(zb, y, dtype=torch.bfloat16, **kw)
    assert math.isfinite(loss) and bool(torch.isfinite(dz).all())
    assert loss == pytest.approx(ref["loss"], rel=TOL_BF16)
    assert G.rel_err(dz, ref["dz"]) < 3 * TOL_BF16      # dz additionally rounded to bf16 by autograd


def test_tensor_path_follows_the_row_norms_it_can_and_poisons_the_rest(cuda_device):
    """Under the unit-rows promise the fixed maximum is max(1, max |z|^2) found on the device.  Norms up to
    sqrt(tau / 0.025) are evaluated correctly (nothing can underflow); beyond that the promise is broken in a way
    a fixed maximum cannot absorb and the result is NaN -- loud, not silently wrong (VERDICT r01 weak #1)."""
    n = 512
    zb, y = _scaled_rows(n, "ragged")                  # max |z|^2 ~ 2.25 <= 0.07 / 0.025 = 2.8
    zz = Fn.canonical_z(zb.to(cuda_device))
    yy = Fn.canonical_labels(y.to(cuda_device), n)
    kw = dict(tau=0.07, similarity="cosine", lam=0.0, t=2.0, topk=15, alpha=0.5)
    ref = G.oracle_for(zb.float(), y, **kw)
    prob = _tc_problem(n, tau=0.07, topk=15, alpha=0.5, flags=_cabi.FLAG_UNIT_ROWS | _cabi.FLAG_FORCE_TENSOR)
    stats, partials, loss = Fn.forward_rows(zz, yy, prob, want_loss=True)
    assert float(partials[_cabi.P_FIXMAX]) == pytest.approx(float((zb.float() ** 2).sum(1).max()), rel=1e-5)
    assert float(loss) == pytest.approx(ref["loss"], rel=TOL_BF16)
    assert float((stats[:, 0].double().cpu() - ref["stats"]["lse"]).abs().max()) < 2e-3
    dz = Fn.backward_rows(zz, yy, stats, partials, None, prob, out_dtype=torch.float32)
    assert G.rel_err(dz.cpu(), ref["dz"]) < TOL_BF16
    # tau = 0.03: the same rows exceed tau / 0.025 = 1.2 -> poisoned; 3x rows likewise at any tau of this path
    for zbad, tau in ((zb, 0.03), (_scaled_rows(n, "3x")[0], 0.07)):
        zz = Fn.canonical_z(zbad.to(cuda_device))
        prob = _tc_problem(n, tau=tau, topk=15, alpha=0.0, flags=_cabi.FLAG_UNIT_ROWS | _cabi.FLAG_FORCE_TENSOR)
        stats, partials, loss = Fn.forward_rows(zz, yy, prob, want_loss=True)
        assert math.isnan(float(loss)) and math.isnan(float(partials[_cabi.P_FIXMAX]))
        dz = Fn.backward_rows(zz, yy, stats, partials, None, prob, out_dtype=torch.float32)
        assert bool(torch.isnan(dz).all())
    # the promise through the module: assume_unit_rows = True on un-normalised rows is the caller's error -> NaN
    loss, _ = G.kernel_loss_and_grad(_scaled_rows(n, "3x")[0], y, dtype=torch.bfloat16, unit_rows=True, **kw)
    assert math.isnan(loss)


def test_unit_rows_keep_the_fixed_maximum_at_exactly_one(cuda_device):
    """bf16 rounding moves |z|^2 off 1 by up to ~0.4 %: the maximum snaps to 1 so that unit rows are
    evaluated exactly as before (and identically on every rank / phase)."""
    x, y = O.make_inputs(1024, 256, "iso")
    zb = F.normalize(x, dim=1).to(torch.bfloat16)
    out = G.kernel_stats(zb, y, dtype=torch.bfloat16, flags=_cabi.FLAG_UNIT_ROWS, tau=0.07, similarity="cosine",
                         topk=15, alpha=0.0)
    assert float(out["partials"][_cabi.P_FIXMAX]) == 1.0
    # label-derived global anchor counts ride along in the partials
    assert float(out["partials"][_cabi.P_GCNT_FULL]) == 1024.0
    assert float(out["partials"][_cabi.P_GCNT_MINED]) == 1024.0


# ---------------------------------------------------------------------------------------------------------
# hard-negative sets on the tensor path: equality, exact-arithmetic inputs (VERDICT weak #2)
# ---------------------------------------------------------------------------------------------------------
def _exact_arith_inputs_d256(n, seed, classes=3):
    """Entries in {0, +-1/16, +-1/32}: exactly representable in bf16, every dot product is a multiple of 2^-10
    below 1 in magnitude -> exact in fp32 (any summation order) and in fp64.  |z|^2 ~ 0.5 <= 1.  The few
    hundred distinct similarity values among thousands of columns give MANY exact ties."""
    g = torch.Generator().manual_seed(seed)
    vals = torch.tensor([0.0, 0.0625, -0.0625, 0.03125, -0.03125])
    z = vals[torch.randint(0, 5, (n, 256), generator=g)]
    y = torch.randint(0, classes, (n,), generator=g)
    return z, y


@pytest.mark.parametrize("n,k", [(1024, 15), (1024, 32), (2304, 15), (2304, 32), (4096, 7)])
def test_tensor_path_hard_negative_sets_bit_exact(cuda_device, n, k):
    z, y = _exact_arith_inputs_d256(n, seed=n + k)
    zb = z.to(torch.bfloat16)
    assert torch.equal(zb.float(), z)
    kw = dict(tau=0.07, similarity="cosine", lam=0.0, t=2.0, topk=k, alpha=1.0)
    ref = G.oracle_for(z, y, want_topk_idx=False, **kw)
    zz = Fn.canonical_z(zb.to(cuda_device))
    yy = Fn.canonical_labels(y.to(cuda_device), n)
    prob = _tc_problem(n, topk=k, alpha=1.0)
    stats, partials, loss = Fn.forward_rows(zz, yy, prob, want_loss=True)
    st = stats.cpu()
    # the threshold (value, index) of every row == the stable-sort oracle's: with the values exact this pins the
    # whole selected set {s > thr} U {s == thr, j <= idx}
    assert torch.equal(st.view(torch.int32)[:, _cabi.ST_THR_IDX].long(), ref["stats"]["thr_idx"])
    assert torch.equal(st[:, _cabi.ST_THR_VAL].double(), ref["stats"]["thr_val"])
    n_tied = int((ref["stats"]["thr_val"].view(-1, 1) == (z.double() @ z.double().t())).sum(1).gt(1).sum())
    assert n_tied > n // 4            # the inputs do put ties at the K-th boundary of many rows
    assert float(loss) == pytest.approx(ref["loss"], rel=1e-5)
    dz = Fn.backward_rows(zz, yy, stats, partials, None, prob, out_dtype=torch.float32)
    assert G.rel_err(dz.cpu(), ref["dz"]) < TOL_BF16          # H is rounded to bf16 before the second GEMM


def test_tensor_path_ties_layout_sets_exact(cuda_device):
    """SURVEY 8d 'ties' layout (duplicated rows) on the tensor path: exact duplicates produce exactly equal
    similarities (the tcgen05 Gram is bit-symmetric), so lowest-index-wins is decidable and must hold."""
    n = 2048
    x, y = O.make_inputs(n, 256, "ties")
    zb = F.normalize(x, dim=1).to(torch.bfloat16)
    kw = dict(tau=0.07, similarity="cosine", lam=0.0, t=2.0, topk=15, alpha=1.0)
    ref = G.oracle_for(zb.float(), y, **kw)
    out = G.kernel_stats(zb, y, dtype=torch.bfloat16, flags=2, **kw)
    got = out["stats"].cpu().view(torch.int32)[:, _cabi.ST_THR_IDX].long()
    # rows whose K-th boundary is an exact tie in fp64 as well: decided by index, must agree
    sims = zb.double() @ zb.double().t()
    sims.fill_diagonal_(-9.0)
    neg = y.view(-1, 1) != y.view(1, -1)
    tied = ((sims == ref["stats"]["thr_val"].view(-1, 1)) & neg).sum(1) > 1
    assert int(tied.sum()) > 0
    assert torch.equal(got[tied], ref["stats"]["thr_idx"][tied])
    assert float((got == ref["stats"]["thr_idx"]).float().mean()) >= 0.999   # fp32- vs fp64-rounded near-ties elsewhere


# ---------------------------------------------------------------------------------------------------------
# N = 65536 (BASELINE configs[3], the headline size)
# ---------------------------------------------------------------------------------------------------------
def _plain_fp64_row_stats(zz, yy, tau, block=2048):
    """lse_i, mean positive logit and |pos_i| of EVERY row by direct evaluation in fp64 on the device (plain
    torch: a Gram block, a masked logsumexp) -- the same quantities oracle.rowblock_forward returns, without the
    full-row sort that makes the oracle itself impractical for all 65536 rows."""
    n = zz.size(0)
    z64 = zz.double()
    lse, pmean, npos = [], [], []
    for r0 in range(0, n, block):
        lg = (z64[r0:r0 + block] @ z64.t()) / tau
        idx = torch.arange(r0, min(r0 + block, n), device=zz.device)
        same = yy[r0:r0 + block].view(-1, 1) == yy.view(1, -1)
        same[torch.arange(idx.numel(), device=zz.device), idx] = False
        pmean.append((lg * same).sum(1) / same.sum(1).clamp_min(1))
        npos.append(same.sum(1))
        lg[torch.arange(idx.numel(), device=zz.device), idx] = float("-inf")
        lse.append(torch.logsumexp(lg, dim=1))
    return torch.cat(lse), torch.cat(pmean), torch.cat(npos)


def test_headline_size_n65536_bf16(cuda_device):
    n, tau, k = 65536, 0.07, 15
    x, y = O.make_inputs(n, 256, "iso")
    zb = F.normalize(x, dim=1).to(torch.bfloat16)
    zz = Fn.canonical_z(zb.to(cuda_device))
    yy = Fn.canonical_labels(y.to(cuda_device), n)

    # --- alpha = 0 (the bench configuration): every row + the loss against the plain fp64 evaluation
    prob = _tc_problem(n, tau=tau, topk=k, alpha=0.0)
    stats, partials, loss = Fn.forward_rows(zz, yy, prob, want_loss=True)
    lse64, pmean64, npos64 = _plain_fp64_row_stats(zz, yy, tau)
    assert torch.equal(stats.view(torch.int32)[:, _cabi.ST_NPOS].long(), npos64)
    assert float((stats[:, _cabi.ST_LSE].double() - lse64).abs().max()) < 1e-4
    assert float((stats[:, _cabi.ST_POS_MEAN].double() - pmean64).abs().max()) < 1e-4
    loss64 = float((lse64 - pmean64)[npos64 > 0].mean())
    assert float(loss) == pytest.approx(loss64, rel=1e-5)
    assert loss64 == pytest.approx(math.log(n - 1) + 0.5 * (1.0 / (256 * tau * tau)), rel=2e-3)   # iso: ln(N-1) + var/2
    dz = Fn.backward_rows(zz, yy, stats, partials, None, prob, out_dtype=torch.float32)

    # --- sampled rows against the oracle's brute force (4 windows x 16 rows): statistics and dz rows.
    # dz_i needs the statistics of ALL columns: the fp64 evaluation above (validated row by row) supplies them.
    z64c, yc = zb.double(), y
    stats_all = dict(lse=lse64.cpu(), lse_m=lse64.cpu(), npos=npos64.cpu(), nneg=(n - 1 - npos64).cpu(),
                     thr_val=torch.full((n,), float("inf"), dtype=torch.float64),
                     thr_idx=torch.full((n,), -1, dtype=torch.int64), wsum=torch.zeros(n, dtype=torch.float64),
                     pos_mean=pmean64.cpu())
    part = torch.zeros(O.N_PARTIALS, dtype=torch.float64)
    part[O.P_SUM_FULL], part[O.P_CNT_FULL] = float((lse64 - pmean64)[npos64 > 0].sum()), float((npos64 > 0).sum())
    _, coef = O.loss_from_partials(part, n, alpha=0.0, lambda_uni=0.0)
    g = torch.Generator().manual_seed(65536)
    windows = [int(v) for v in torch.randint(0, n - 16, (4,), generator=g)] + [0, n - 16]
    for r0 in windows:
        st, _ = O.rowblock_forward(z64c, yc, r0, 16, tau=tau, similarity=O.COSINE, topk=k)
        got = stats[r0:r0 + 16].cpu()
        assert float((got[:, _cabi.ST_LSE].double() - st["lse"]).abs().max()) < 1e-4
        assert torch.equal(got.view(torch.int32)[:, _cabi.ST_NPOS].long(), st["npos"])
        want = O.rowblock_backward(z64c, yc, r0, 16, stats_all, coef, tau=tau, similarity=O.COSINE, topk=k)
        assert G.rel_err(dz[r0:r0 + 16].cpu(), want) < TOL_BF16, f"dz rows {r0}..{r0 + 15}"

    # --- alpha = 0.5, top-15 mining at N = 65536: threshold (value, index) of the sampled rows == brute force
    prob_m = _tc_problem(n, tau=tau, topk=k, alpha=0.5)
    stats_m, partials_m, loss_m = Fn.forward_rows(zz, yy, prob_m, want_loss=True)
    assert math.isfinite(float(loss_m))
    for r0 in windows:
        st, _ = O.rowblock_forward(z64c, yc, r0, 16, tau=tau, similarity=O.COSINE, topk=k)
        got = stats_m[r0:r0 + 16].cpu()
        assert torch.equal(got.view(torch.int32)[:, _cabi.ST_THR_IDX].long(), st["thr_idx"]), f"rows {r0}.."
        assert float((got[:, _cabi.ST_THR_VAL].double() - st["thr_val"]).abs().max()) < 1e-6
        assert float((got[:, _cabi.ST_LSE_M].double() - st["lse_m"]).abs().max()) < 1e-4


# ---------------------------------------------------------------------------------------------------------
# two-phase backward, partial-sum kernel
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sim,lam,alpha,k", [("cosine", 0.0, 0.0, 15), ("cosine", 0.0, 0.5, 15),
                                             ("geodesic", 0.0, 1.0, 7), ("cosine", 0.05, 0.0, 15)])
def test_two_phase_backward_equals_single_phase(cuda_device, sim, lam, alpha, k):
    """supcon_backward_rows_local (own columns, own statistics, label-derived global counts, no grad_out yet)
    + _remote (the rest, everyone's statistics, global sums, grad_out) == supcon_backward_rows == oracle.
    With the uniformity term the local call must decline (its coefficient needs the global sum)."""
    n = 2048
    # exact duplicates ("ties") only with cosine: under geodesic similarity d acos(c) at c ~ 1 makes the gradient
    # through a duplicated pair ill-conditioned (SURVEY H7) and no fixed tolerance against fp64 is meaningful
    x, y = O.make_inputs(n, 256, "ties" if sim == "cosine" else "iso", classes=3)
    zb = F.normalize(x, dim=1).to(torch.bfloat16)
    zz = Fn.canonical_z(zb.to(cuda_device))
    yy = Fn.canonical_labels(y.to(cuda_device), n)
    kw = dict(tau=0.07, sim=sim, lam=lam, topk=k, alpha=alpha)
    whole = _tc_problem(n, **kw)
    stats_all, partials_all, _ = Fn.forward_rows(zz, yy, whole, want_loss=True)
    ref = G.oracle_for(zb.float(), y, tau=0.07, similarity=sim, lam=lam, t=2.0, topk=k, alpha=alpha)
    g = torch.tensor(1.7, device=cuda_device)
    for row_offset, n_rows in ((512, 768), (0, 256), (1792, 256)):
        prob = _tc_problem(n, row_offset=row_offset, n_rows=n_rows, **kw)
        s_loc, p_loc, _ = Fn.forward_rows(zz, yy, prob, want_loss=False)
        assert float(p_loc[_cabi.P_GCNT_FULL]) == float(partials_all[_cabi.P_CNT_FULL])     # counts from the labels
        assert float(p_loc[_cabi.P_GCNT_MINED]) == float(partials_all[_cabi.P_CNT_MINED])
        dz1 = Fn.backward_rows(zz, yy, stats_all, partials_all, g, prob, out_dtype=torch.float32)
        ws = Fn.backward_rows_local(zz, yy, s_loc, p_loc, prob)
        dz2 = Fn.backward_rows_remote(zz, yy, stats_all, partials_all, g, prob, ws, out_dtype=torch.float32)
        assert G.rel_err(dz2.cpu(), dz1.cpu()) < 1e-5                 # same tiles, different summation split
        assert G.rel_err(dz2.cpu() / 1.7, ref["dz"][row_offset:row_offset + n_rows]) < TOL_BF16


def test_finalize_sets_sums_in_rank_order(cuda_device):
    g = torch.Generator().manual_seed(0)
    sets = torch.rand(5, 8, generator=g, dtype=torch.float64)
    sets[:, 1] = torch.tensor([100., 90., 110., 95., 105.])      # |A_f| per rank
    sets[:, 3] = sets[:, 1]
    sets[:, 0] *= 400.0; sets[:, 2] *= 380.0
    sets[:, 5:] = torch.tensor([500.0, 500.0, 1.0])               # global quantities, identical on every rank
    prob = Fn.make_problem(500, 256, _cabi.BF16, tau=0.07, similarity=_cabi.COSINE, lambda_uni=0.1, topk=15, alpha=0.3)
    partials, loss = Fn.finalize_sets(prob, sets.to(cuda_device))
    want = sets[0].clone()
    for r in range(1, 5):
        want[:5] += sets[r, :5]                                   # rank order, fp64
    assert torch.equal(partials.cpu(), want)
    assert float(loss) == pytest.approx(float(Fn.finalize(prob, want.to(cuda_device))), rel=0, abs=0)
    ref, _ = O.loss_from_partials(want, 500, alpha=0.3, lambda_uni=0.1)
    assert float(loss) == pytest.approx(ref, rel=1e-6)


# ---------------------------------------------------------------------------------------------------------
# duplicate rows + uniformity on every kernel family (DESIGN r01 plan item 7)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family", ["small", "ffma", "tensor"])
@pytest.mark.parametrize("sim", ["cosine", "geodesic"])
def test_duplicate_rows_with_uniformity(cuda_device, family, sim):
    """Exact duplicates: zero distance (w = 1, gradient of the uniformity term through that pair is 0, as
    torch.pdist's backward gives).  Cosine: loss and dz against the oracle.  Geodesic: the loss only -- the
    slope (2/pi)/sqrt(1 - c^2) of a duplicated pair (c within an ulp of the clamp at 1 - 2^-23) is ~1e3 and flips
    with the last bit of c, so fp32 (kernel, reference) and fp64 (oracle) gradients differ by O(1) there
    (SURVEY H7 / Appendix C); dz must still be finite."""
    n = {"small": 96, "ffma": 384, "tensor": 512}[family]
    dtype = torch.bfloat16 if family == "tensor" else torch.float32
    flags = {"small": 0, "ffma": 4 | 1, "tensor": 2}[family]
    x, y = O.make_inputs(n, 256, "ties", classes=2, seed=21)
    x[5] = x[4]; x[6] = x[4]; y[5] = y[4]; y[6] = 1 - y[4]          # a triple: positive and negative duplicates
    z = F.normalize(x, dim=1).to(dtype)
    kw = dict(tau=0.1, similarity=sim, lam=0.2, t=2.0, topk=7, alpha=0.4)
    ref = G.oracle_for(z.float(), y, **kw)
    loss, dz = G.kernel_loss_and_grad(z, y, dtype=dtype, flags=flags, **kw)
    tol = TOL_F32 if dtype == torch.float32 else TOL_BF16
    assert loss == pytest.approx(ref["loss"], rel=tol)
    assert bool(torch.isfinite(dz).all())
    if sim == "cosine":
        assert G.rel_err(dz, ref["dz"]) < (tol if dtype == torch.float32 else 3 * tol)
    else:   # rows not involved in a duplicated pair are well-conditioned: compare those
        keep = torch.ones(n, dtype=torch.bool)
        dup = (z.float() @ z.float().t()).fill_diagonal_(0).gt(0.999).any(1)
        keep &= ~dup
        assert int(keep.sum()) > n // 2
        assert G.rel_err(dz[keep], ref["dz"][keep]) < (50 * tol if dtype == torch.float32 else 3 * tol)


# ---------------------------------------------------------------------------------------------------------
# single-launch kernel for mid-size batches, 160 < N <= 320 (supcon_mid.cu): the reference's default batch (256)
# ---------------------------------------------------------------------------------------------------------
MID_CASES = [
    # n, d, kind, classes, sim, tau, lam, K, alpha
    (256, 256, "iso", 2, "cosine", 0.07, 0.0, 15, 0.0),          # stage1_config.py defaults: batch 256, hidden 256
    (256, 256, "iso", 2, "geodesic", 0.2, 0.2, 15, 0.5),
    (161, 256, "clustered", 3, "cosine", 0.07, 0.05, 15, 1.0),
    (300, 64, "iso", 5, "geodesic", 0.1, 0.0, 32, 0.37),
    (320, 256, "ties", 2, "cosine", 0.07, 0.0, 15, 0.5),
    (320, 256, "iso", 2, "cosine", 0.07, 0.1, 600, 1.0),         # K >= all negatives
    (288, 128, "iso", 7, "cosine", 0.5, 0.0, 0, 0.0),            # multi-class class: K = 0
]


@pytest.mark.parametrize("n,d,kind,classes,sim,tau,lam,k,alpha", MID_CASES)
def test_mid_size_single_launch_kernel_fp32(cuda_device, n, d, kind, classes, sim, tau, lam, k, alpha):
    """fp32, whole batch on one GPU, 160 < N <= 320: loss and dz from ONE cluster launch (default flags) agree with
    the oracle at 1e-5 and with the tiled exact kernels (flags = 4) -- same formulas, same fixed k-order."""
    x, y = O.make_inputs(n, d, kind, classes=classes)
    z = F.normalize(x, dim=1)
    kw = dict(tau=tau, similarity=sim, lam=lam, t=2.0, topk=k, alpha=alpha)
    ref = G.oracle_for(z, y, **kw)
    loss, dz = G.kernel_loss_and_grad(z, y, **kw)
    assert loss == pytest.approx(ref["loss"], rel=TOL_F32, abs=1e-6)
    assert G.rel_err(dz, ref["dz"]) < TOL_F32
    loss_t, dz_t = G.kernel_loss_and_grad(z, y, flags=4, **kw)
    assert loss_t == pytest.approx(loss, rel=1e-6)
    assert G.rel_err(dz, dz_t) < 1e-5
    if k >= 1 and alpha != 0.0:       # hard-negative thresholds: identical (value, index) in both kernel families
        a = G.kernel_stats(z, y, flags=0, **{**kw, "alpha": alpha})
        b = G.kernel_stats(z, y, flags=4, **{**kw, "alpha": alpha})
        assert torch.equal(a["stats"].view(torch.int32)[:, _cabi.ST_THR_IDX], b["stats"].view(torch.int32)[:, _cabi.ST_THR_IDX])
        assert torch.equal(a["stats"][:, _cabi.ST_THR_VAL], b["stats"][:, _cabi.ST_THR_VAL])


# ---------------------------------------------------------------------------------------------------------
# backward beyond L2: the work list ordered by column panels (z > 48 MB)
# ---------------------------------------------------------------------------------------------------------
def test_backward_column_panels_beyond_l2(cuda_device):
    """N = 131072 (z = 64 MB -> the backward's list is cut into 3 column panels): dz of a rank's 8192 rows, sampled
    windows against the oracle's brute force (which is given every row's statistics from the forward, themselves
    checked on the sampled rows), and the whole block against a second evaluation that shifts the panel boundaries
    (another row offset -> other CTA ranges): the partial records of the panels must add up identically."""
    n, nl, tau = 131072, 8192, 0.07
    x, y = O.make_inputs(n, 256, "iso")
    zb = F.normalize(x, dim=1).to(torch.bfloat16)
    zz = Fn.canonical_z(zb.to(cuda_device))
    yy = Fn.canonical_labels(y.to(cuda_device), n)
    whole = _tc_problem(n, tau=tau, topk=15, alpha=0.0)
    stats_all, partials, loss = Fn.forward_rows(zz, yy, whole, want_loss=True)
    assert float(loss) == pytest.approx(math.log(n - 1) + 0.5 / (256 * tau * tau), rel=2e-3)
    r0 = 5 * nl
    prob = _tc_problem(n, tau=tau, topk=15, alpha=0.0, row_offset=r0, n_rows=nl)
    dz = Fn.backward_rows(zz, yy, stats_all, partials, None, prob, out_dtype=torch.float32)
    st = stats_all.cpu()
    stats_dict = dict(lse=st[:, _cabi.ST_LSE].double(), lse_m=st[:, _cabi.ST_LSE].double(),
                      npos=st.view(torch.int32)[:, _cabi.ST_NPOS].long(), nneg=st.view(torch.int32)[:, _cabi.ST_NNEG].long(),
                      thr_val=torch.full((n,), float("inf"), dtype=torch.float64),
                      thr_idx=torch.full((n,), -1, dtype=torch.int64), wsum=torch.zeros(n, dtype=torch.float64),
                      pos_mean=st[:, _cabi.ST_POS_MEAN].double())
    _, coef = O.loss_from_partials(partials.cpu(), n, alpha=0.0, lambda_uni=0.0)
    z64 = zb.double()
    for w0 in (r0, r0 + 4093, r0 + nl - 16):
        fw, _ = O.rowblock_forward(z64, y, w0, 16, tau=tau, similarity=O.COSINE, topk=15)
        assert float((st[w0:w0 + 16, _cabi.ST_LSE].double() - fw["lse"]).abs().max()) < 1e-4
        want = O.rowblock_backward(z64, y, w0, 16, stats_dict, coef, tau=tau, similarity=O.COSINE, topk=15)
        assert G.rel_err(dz[w0 - r0:w0 - r0 + 16].cpu(), want) < TOL_BF16, f"rows {w0}.."
    # the same rows as part of a differently placed block: other CTA ranges / panel cuts, same sums
    prob2 = _tc_problem(n, tau=tau, topk=15, alpha=0.0, row_offset=r0 - 2048, n_rows=nl)
    dz2 = Fn.backward_rows(zz, yy, stats_all, partials, None, prob2, out_dtype=torch.float32)
    assert G.rel_err(dz2[2048:].cpu(), dz[:nl - 2048].cpu()) < 1e-5


# ---------------------------------------------------------------------------------------------------------
# positives by linearity (round 2): sum over positives from class sums for <= 32 classes, per pair beyond
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("classes", [1, 2, 5, 32, 33, 100])
@pytest.mark.parametrize("lam", [0.0, 0.05])
def test_tensor_path_positive_sums_for_any_class_count(cuda_device, classes, lam):
    """cosine, no mining, whole forward on the tensor path: loss, row statistics (pos_mean) and dz against the
    oracle whether the positives' sum comes from the class sums (<= TC_CMAX = 32 classes) or from the sweep."""
    n, tau = 1000, 0.07                     # ragged: 8 row blocks, the last one partial
    x, _ = O.make_inputs(n, 256, "iso", seed=5)
    g = torch.Generator().manual_seed(classes)
    y = torch.randint(0, classes, (n,), generator=g) * 7 - 3           # arbitrary label values
    zb = F.normalize(x, dim=1).to(torch.bfloat16)
    want = G.oracle_for(zb.double(), y, tau=tau, similarity="cosine", lam=lam, topk=15, alpha=0.0)
    loss, dz = G.kernel_loss_and_grad(zb, y, tau=tau, similarity="cosine", lam=lam, topk=15, alpha=0.0,
                                      dtype=torch.bfloat16, device=cuda_device, unit_rows=True)
    assert loss == pytest.approx(want["loss"], rel=TOL_BF16)
    assert G.rel_err(dz, want["dz"]) < 2 * TOL_BF16 or float(want["dz"].norm()) < 1e-9   # dz rounded to bf16 by autograd
    # row statistics straight from the C-ABI: mean positive logit of every row
    zz = Fn.canonical_z(zb.to(cuda_device))
    yy = Fn.canonical_labels(y.to(cuda_device), n)
    prob = _tc_problem(n, tau=tau, topk=15, alpha=0.0, lam=lam)
    stats, _, _ = Fn.forward_rows(zz, yy, prob, want_loss=True)
    s64 = zb.double() @ zb.double().T
    same = (y[:, None] == y[None, :]) & ~torch.eye(n, dtype=torch.bool)
    npos = same.sum(1)
    pmean = torch.where(npos > 0, (s64 * same).sum(1) / tau / npos.clamp(min=1), torch.zeros(n, dtype=torch.float64))
    assert torch.equal(stats.view(torch.int32)[:, _cabi.ST_NPOS].long().cpu(), npos)
    assert float((stats[:, _cabi.ST_POS_MEAN].double().cpu() - pmean).abs().max()) < 2e-4
    # the class-sum route and the per-pair route, pinned by flag, forward and backward, against each other and
    # against the oracle (the per-pair backward rounds the positives' term to bf16 inside H, the class-sum one
    # adds it in fp32: the class-sum gradient is the closer one)
    outs = {}
    for name, fl in (("class_sums", _cabi.FLAG_CLASS_SUMS), ("per_pair", _cabi.FLAG_NO_CLASS_SUMS)):
        pr = _tc_problem(n, tau=tau, topk=15, alpha=0.0, lam=lam, flags=_cabi.FLAG_FORCE_TENSOR | fl)
        st, pa, ls = Fn.forward_rows(zz, yy, pr, want_loss=True)
        gz = Fn.backward_rows(zz, yy, st, pa, None, pr, out_dtype=torch.float32)
        outs[name] = (float(ls), st.cpu(), gz.double().cpu())
        assert float(ls) == pytest.approx(want["loss"], rel=TOL_BF16)
        assert G.rel_err(gz.double().cpu(), want["dz"]) < TOL_BF16 or float(want["dz"].norm()) < 1e-9
    assert outs["class_sums"][0] == pytest.approx(outs["per_pair"][0], rel=1e-6)
    assert float((outs["class_sums"][1][:, _cabi.ST_POS_MEAN] - outs["per_pair"][1][:, _cabi.ST_POS_MEAN]).abs().max()) < 1e-4
    assert torch.equal(outs["class_sums"][1][:, _cabi.ST_LSE], outs["per_pair"][1][:, _cabi.ST_LSE])
    if float(want["dz"].norm()) > 1e-9:
        assert G.rel_err(outs["class_sums"][2], outs["per_pair"][2]) < TOL_BF16
    # through the module with the class-sum route pinned: the backward takes the label table and the class sums
    # out of the workspace the forward left (SUPCON_FLAG_WS_FROM_FORWARD) instead of rebuilding them
    loss_m, dz_m = G.kernel_loss_and_grad(zb, y, tau=tau, similarity="cosine", lam=lam, topk=15, alpha=0.0,
                                          dtype=torch.bfloat16, device=cuda_device, unit_rows=True,
                                          flags=_cabi.FLAG_CLASS_SUMS)
    assert loss_m == pytest.approx(outs["class_sums"][0], rel=1e-6)
    if float(want["dz"].norm()) > 1e-9:
        assert G.rel_err(dz_m, want["dz"]) < 2 * TOL_BF16                  # dz rounded to bf16 by autograd
        assert G.rel_err(dz_m, outs["class_sums"][2]) < 4e-3               # = the bf16 rounding of the same gradient
