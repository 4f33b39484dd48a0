"""GPU: hard-negative mining with more than 32 negatives per row against the fp64 oracle.

With alpha > 0 and K > 32 only the exact fp32 kernels (csrc/supcon_ffma.cu) run: the tensor path keeps at most 32
list entries per row, and the single-launch small / mid kernels take K > 32 only when it selects every negative.
Those kernels select the K hardest negatives of a row by one of three mechanisms:
  * one in-sweep list of up to 128 entries per row, when the forward sweeps all columns in one CTA;
  * one list per column split, merged by ffma_fwd_merge_kernel (K <= 128, mid-size N);
  * rounds of at most 128 entries for K > 128 over one sweep: round r admits only negatives ranked after the last
    entry of round r - 1.
An off-by-one-tie in any of them moves one exp term among hundreds of the loss and one column of the gradient,
so most cases use inputs whose dot products are exact (entries in {0, +-1/2, +-1/4}): exact ties then sit across
rank K and the round boundaries of most rows, and thresholds, counts and index sets must equal the oracle's.
Tolerances as in the rest of the suite: loss and dz 1e-5 relative on the fp32 path."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

import debug_lib as D
import gpu_util as G
from memory_ref import memory_loss
from oracle import supcon_oracle as O
from test_gpu_parity import _exact_arith_inputs
from test_gpu_parity_r02 import _exact_arith_inputs_d256
from test_memory_gpu import EXACT_PATH_MEMORY, EXACT_PATH_TOPK
from test_memory_gpu import _index_sets
from test_memory_gpu import _inputs as _memory_inputs
from test_memory_gpu import _kernel as _memory_kernel
from wav2vec_contr_loss_b200 import _cabi
from wav2vec_contr_loss_b200 import functional as Fn

pytestmark = pytest.mark.gpu

TOL_F32 = 1e-5
TOL_BF16 = 2e-3
LIST_CAP = 128              # entries of one selection round (ffma_kcap)
NEAR_TIE = 1e-6             # fp64 gap below which fp32 rounding may order two random similarities either way

# N, K of the exact-arithmetic sweep: every row has more than K negatives (3 classes: about 2N/3 each)
SWEEP_K = (33, 64, 127, 128, 129, 200, 255, 256, 257, 400)
SWEEP_CASES = [(n, k) for n in (448, 1024, 2048) for k in SWEEP_K if k < {448: 285, 1024: 672, 2048: 1336}[n]]
# classes of 600 / 300 / 100 / 24 rows at N = 1024 have 424 / 724 / 924 / 1000 negatives per row
IMBALANCED_SIZES = (600, 300, 100, 24)
IMBALANCED_K = (423, 424, 500, 723, 724, 999)
# B = 64 anchors against an exact-arithmetic memory of M rows, K below every anchor's negative count
MEMORY_CASES = [(300, 64), (300, 128), (300, 129), (1000, 64), (1000, 128), (1000, 129), (1000, 300),
                (4096, 64), (4096, 128), (4096, 129), (4096, 300)]


def _ffma_plan(n_total, k, *, d=16, n_rows=None, flags=0):
    """{fwd_splits, bwd_splits, kcap, rounds} of the exact path for a mined fp32 problem"""
    prob = Fn.make_problem(n_total, d, _cabi.F32, tau=0.5, similarity=_cabi.COSINE, topk=k, alpha=1.0, n_rows=n_rows,
                           flags=flags)
    out = (ctypes.c_int32 * 4)()
    D.check(D.load().supcon_debug_ffma_plan(ctypes.byref(prob), out, 4), "supcon_debug_ffma_plan")
    return dict(zip(("fwd_splits", "bwd_splits", "kcap", "rounds"), out))


def _mechanism(plan):
    if plan["rounds"] > 1:
        return "rounds"
    return "merge" if plan["fwd_splits"] > 1 else "one list"


def test_cases_cover_every_selection_mechanism(cuda_device):
    """the matrices below reach each selection mechanism on this device, with a memory too, so that a change to
    the plan cannot move them all onto one path unnoticed"""
    sweep = [(k, _ffma_plan(n, k)) for n, k in SWEEP_CASES]
    sweep += [(k, _ffma_plan(sum(IMBALANCED_SIZES), k)) for k in IMBALANCED_K]
    memory = {_mechanism(_ffma_plan(64 + m, k, n_rows=64, flags=_cabi.FLAG_MEMORY_COLUMNS)) for m, k in MEMORY_CASES}
    random_memory = set()      # test_memory_gpu.test_exact_path_fp32 where its anchors have more than K negatives
    for m in EXACT_PATH_MEMORY:
        for k in EXACT_PATH_TOPK:
            _, yb, _, ym = _memory_inputs(64, m, seed=m + k)
            if k > 32 and int((yb.view(-1, 1) != torch.cat([yb, ym]).view(1, -1)).sum(1).min()) > k:
                random_memory.add(_mechanism(_ffma_plan(64 + m, k, d=256, n_rows=64, flags=_cabi.FLAG_MEMORY_COLUMNS)))
    assert all(p["kcap"] == min(k, LIST_CAP) for k, p in sweep)
    assert any(_mechanism(p) == "one list" and 32 < k <= LIST_CAP for k, p in sweep)
    assert any(_mechanism(p) == "merge" and k == LIST_CAP for k, p in sweep)     # the merge's array full
    assert any(p["rounds"] == 2 for _, p in sweep) and any(p["rounds"] >= 3 for _, p in sweep)
    assert all(p["fwd_splits"] == 1 for _, p in sweep if p["rounds"] > 1)
    assert memory == {"one list", "merge", "rounds"}
    assert random_memory == {"merge", "rounds"}


def _sorted_negatives(z, y, similarity="cosine"):
    """fp64 similarities of each row's negatives in descending order (-inf padded), as the oracle ranks them"""
    c = z.double() @ z.double().t()
    s, _ = O._sim_and_slope(c, O.sim_id(similarity))
    neg = y.view(-1, 1) != y.view(1, -1)
    return torch.sort(s.masked_fill(~neg, float("-inf")), dim=1, descending=True).values


def _check_exact_selection(z, y, k):
    """statistics, thresholds and index sets of the exact path equal the oracle's on exact-arithmetic inputs"""
    kw = dict(tau=0.5, similarity="cosine", lam=0.0, t=2.0, topk=k, alpha=1.0)
    out = G.kernel_stats(z, y, flags=_cabi.FLAG_NO_SMALL, **kw)
    ref = G.oracle_for(z, y, want_topk_idx=True, **kw)
    rs = ref["stats"]
    st = out["stats"].cpu()
    si = st.view(torch.int32)
    assert torch.equal(si[:, _cabi.ST_NPOS].long(), rs["npos"])
    assert torch.equal(si[:, _cabi.ST_NNEG].long(), rs["nneg"])
    assert torch.equal(si[:, _cabi.ST_THR_IDX].long(), rs["thr_idx"])
    assert torch.equal(st[:, _cabi.ST_THR_VAL].double(), rs["thr_val"])
    assert torch.allclose(st[:, _cabi.ST_LSE_M].double(), rs["lse_m"], rtol=TOL_F32, atol=TOL_F32)
    want = torch.full((z.size(0), k), -1, dtype=torch.int64)
    for i, cols in enumerate(rs["topk_idx"]):
        want[i, :len(cols)] = torch.tensor(sorted(cols), dtype=torch.int64)
    assert torch.equal(out["idx"].cpu().long(), want)
    assert float(out["loss"]) == pytest.approx(ref["loss"], rel=TOL_F32)
    dz = Fn.backward_rows(out["z"], out["y"], out["stats"], out["partials"], None, out["prob"],
                          out_dtype=torch.float32)
    assert G.rel_err(dz.cpu(), ref["dz"]) < TOL_F32
    return rs


@pytest.mark.parametrize("n,k", SWEEP_CASES)
def test_exact_sets_across_round_and_split_boundaries(cuda_device, n, k):
    """cosine, tau 0.5, alpha 1: every row mines; exact ties straddle rank K and the round boundaries"""
    z, y = _exact_arith_inputs(n, 16, seed=n)
    rs = _check_exact_selection(z, y, k)
    assert bool((rs["nneg"] > k).all())
    sv = _sorted_negatives(z, y)
    for rank in [k] + [r for r in (LIST_CAP, 2 * LIST_CAP) if k > r]:
        tied = (sv[:, rank - 1] == sv[:, rank]).double().mean()
        assert float(tied) > 0.5, f"ties across rank {rank} in only {float(tied):.0%} of rows"


@pytest.mark.parametrize("k", IMBALANCED_K)
def test_rows_of_one_block_need_different_round_counts(cuda_device, k):
    """imbalanced classes, shuffled so that each 64-row block mixes them: in one CTA some rows select every
    negative (threshold (-inf, INT_MAX)) while others mine in ceil(K / 128) rounds; K = 424 and 724 equal a
    class's negative count exactly, K = 423 and 723 (and 999) leave that class one negative out"""
    n = sum(IMBALANCED_SIZES)
    z, _ = _exact_arith_inputs(n, 16, seed=k)
    sizes = torch.tensor(IMBALANCED_SIZES)
    y = torch.repeat_interleave(torch.arange(len(sizes)), sizes)
    y = y[torch.randperm(n, generator=torch.Generator().manual_seed(k))]
    rs = _check_exact_selection(z, y, k)
    mines = rs["nneg"] > k
    assert bool(mines.any())
    if bool((n - sizes <= k).any()):
        blocks = mines.view(-1, 64)
        assert bool((blocks.any(1) & ~blocks.all(1)).any())        # a 64-row block holding both kinds of row
        assert bool((rs["thr_idx"][~mines] == 2**31 - 1).all())
    assert bool((rs["nneg"] == k + 1).any()) == (k in (423, 723, 999))


@pytest.mark.parametrize("n", [1024, 2048])
@pytest.mark.parametrize("k", [64, 200])
@pytest.mark.parametrize("sim", ["cosine", "geodesic"])
@pytest.mark.parametrize("lam", [0.0, 0.2])
@pytest.mark.parametrize("alpha", [0.5, 1.0])
def test_random_unit_rows_fp32(cuda_device, n, k, sim, lam, alpha):
    """random unit rows, d = 256, tau 0.07.  fp64 gaps between the K-th and (K+1)-th negative reach 1e-9 here,
    below fp32 rounding of a 256-term dot product (and of acosf), so a row may rank such a pair either way: every
    row with a wider gap must select exactly the oracle's set, and at least 99.9 % of all rows must"""
    x, y = O.make_inputs(n, 256, "iso", seed=n + k)
    z = F.normalize(x, dim=1)
    kw = dict(tau=0.07, similarity=sim, lam=lam, t=2.0, topk=k, alpha=alpha)
    out = G.kernel_stats(z, y, flags=_cabi.FLAG_NO_SMALL, **kw)
    ref = G.oracle_for(z, y, want_topk_idx=True, **kw)
    assert float(out["loss"]) == pytest.approx(ref["loss"], rel=TOL_F32)
    dz = Fn.backward_rows(out["z"], out["y"], out["stats"], out["partials"], None, out["prob"],
                          out_dtype=torch.float32)
    assert G.rel_err(dz.cpu(), ref["dz"]) < TOL_F32
    sv = _sorted_negatives(z, y, sim)
    decided = (sv[:, k - 1] - sv[:, k]) >= NEAR_TIE
    same_thr = out["stats"].cpu().view(torch.int32)[:, _cabi.ST_THR_IDX].long() == ref["stats"]["thr_idx"]
    assert bool(same_thr[decided].all())
    assert float(same_thr.double().mean()) >= 0.999
    idx = out["idx"].cpu().long()
    for i in torch.nonzero(decided).view(-1).tolist():
        assert idx[i].tolist() == sorted(ref["stats"]["topk_idx"][i]), f"row {i}"


def test_tensor_and_exact_paths_meet_at_k32_bf16(cuda_device):
    """bf16, d = 256, unit-rows promise, exact inputs: K = 32 takes the tensor path, K = 33 the exact path on
    bf16 loads; both give the oracle's thresholds bit for bit"""
    n = 1024
    z, y = _exact_arith_inputs_d256(n, seed=33)
    zb = z.to(torch.bfloat16)
    assert torch.equal(zb.float(), z)
    for k in (32, 33):
        kw = dict(tau=0.07, similarity="cosine", lam=0.0, t=2.0, topk=k, alpha=1.0)
        ref = G.oracle_for(z, y, **kw)
        prob = Fn.make_problem(n, 256, _cabi.BF16, tau=0.07, similarity=_cabi.COSINE, topk=k, alpha=1.0,
                               flags=_cabi.FLAG_UNIT_ROWS)
        tc_out = (ctypes.c_int32 * 16)()
        rc = D.load().supcon_debug_plan(ctypes.byref(prob), tc_out, 16)
        forced = dict(kw, dtype=torch.bfloat16, flags=_cabi.FLAG_UNIT_ROWS | _cabi.FLAG_FORCE_TENSOR)
        if k == 32:
            D.check(rc, "supcon_debug_plan")
            tc = G.kernel_stats(zb, y, **forced)
        else:
            assert rc == -2                                       # SUPCON_E_UNSUPPORTED
            with pytest.raises(RuntimeError):
                G.kernel_stats(zb, y, **forced)
        out = G.kernel_stats(zb, y, dtype=torch.bfloat16, flags=_cabi.FLAG_UNIT_ROWS, **kw)
        st = out["stats"].cpu()
        si = st.view(torch.int32)
        assert torch.equal(si[:, _cabi.ST_THR_IDX].long(), ref["stats"]["thr_idx"])
        assert torch.equal(st[:, _cabi.ST_THR_VAL].double(), ref["stats"]["thr_val"])
        assert bool((ref["stats"]["nneg"] > k).all())
        assert float(out["loss"]) == pytest.approx(ref["loss"], rel=TOL_F32)
        dz = Fn.backward_rows(out["z"], out["y"], out["stats"], out["partials"], None, out["prob"],
                              out_dtype=torch.float32)
        if k == 32:
            assert torch.equal(si[:, [2, 3, 5]], tc["stats"].cpu().view(torch.int32)[:, [2, 3, 5]])
            assert G.rel_err(dz.cpu(), ref["dz"]) < TOL_BF16      # H is rounded to bf16 before the second GEMM
        else:
            assert G.rel_err(dz.cpu(), ref["dz"]) < TOL_F32       # fp32 math on the exact bf16 values
    kw = dict(tau=0.07, similarity="cosine", topk=64, alpha=0.5)
    loss, dz = G.kernel_loss_and_grad(zb, y, dtype=torch.bfloat16, unit_rows=True, **kw)
    ref = G.oracle_for(z, y, **kw)
    assert loss == pytest.approx(ref["loss"], rel=TOL_F32)
    assert G.rel_err(dz, ref["dz"]) < 2 * TOL_BF16                # dz rounded to bf16 on return


@pytest.mark.parametrize("n,k", [(100, 40), (100, 33), (100, 99), (300, 40), (300, 100), (300, 299)])
def test_single_launch_kernels_decline_mining_beyond_32(cuda_device, n, k):
    """through the module: 32 < K < N - 1 runs on the tiled kernels (bit-identical to a call that excludes the
    single-launch kernels); K = N - 1 selects every negative and stays on the single-launch kernels"""
    x, y = O.make_inputs(n, 64, "iso", classes=3, seed=n)
    z = F.normalize(x, dim=1)
    kw = dict(tau=0.1, similarity="cosine", lam=0.1, t=2.0, topk=k, alpha=0.5)
    loss, dz = G.kernel_loss_and_grad(z, y, **kw)
    ref = G.oracle_for(z, y, **kw)
    assert loss == pytest.approx(ref["loss"], rel=TOL_F32)
    assert G.rel_err(dz, ref["dz"]) < TOL_F32
    if k < n - 1:
        assert bool((ref["stats"]["nneg"] > k).any())
        tiled_loss, tiled_dz = G.kernel_loss_and_grad(z, y, flags=_cabi.FLAG_NO_SMALL, **kw)
        assert loss == tiled_loss and torch.equal(dz, tiled_dz)


@pytest.mark.parametrize("m,k", MEMORY_CASES)
@pytest.mark.parametrize("sim", ["cosine", "geodesic"])
def test_memory_columns_exact_sets(cuda_device, m, k, sim):
    """64 anchors against an exact-arithmetic memory in each selection mechanism: loss, dz, thresholds and
    index sets (memory indices included) against the fp64 reference with a memory"""
    z, y = _exact_arith_inputs(64 + m, 16, seed=m + k)
    zb, yb, zm, ym = z[:64], y[:64], z[64:], y[64:]
    kw = dict(tau=0.5, sim=sim, lam=0.2, k=k, alpha=0.5)
    out = _memory_kernel(zb, yb, zm, ym, dtype=torch.float32, flags=0, want_idx=True, **kw)
    ref = memory_loss(zb, yb, zm, ym, tau=0.5, similarity=sim, lam=0.2, t=2.0, topk=k, alpha=0.5)
    assert bool((ref["nneg"] > k).all())
    assert out["loss"] == pytest.approx(ref["loss"], rel=TOL_F32)
    assert G.rel_err(out["dz"], ref["dz"]) < TOL_F32
    si = out["stats"].view(torch.int32)
    assert torch.equal(si[:, _cabi.ST_NPOS].long(), ref["npos"]) and torch.equal(si[:, _cabi.ST_NNEG].long(), ref["nneg"])
    assert torch.equal(si[:, _cabi.ST_THR_IDX].long(), ref["thr_idx"])
    if sim == "cosine":
        assert torch.equal(out["stats"][:, _cabi.ST_THR_VAL].double(), ref["thr_val"])
    assert torch.equal(out["idx"].long(), _index_sets(ref["member"], k))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_memory_module_three_steps_k200(cuda_device, dtype):
    """MemorySupConLoss at topk_neg = 200 over a memory of about 1000 rows: two selection rounds over batch +
    memory (bf16 under the unit-rows promise too, since K > 32); each step equals the reference on the memory as
    it stood before the call"""
    from wav2vec_contr_loss_b200.memory import MemorySupConLoss
    dev = torch.device("cuda:0")
    mod = MemorySupConLoss(0.07, "cosine", 0.2, 2.0, memory_size=1150)
    mod.assume_unit_rows = dtype == torch.bfloat16
    z0, y0, _, _ = _memory_inputs(1000, 0, seed=98)
    mod.memory.enqueue(z0.to(dev, dtype), y0.to(dev), unit_rows=True)
    for step in range(3):
        zb, yb, _, _ = _memory_inputs(64, 0, seed=20 + step)
        snap_z = mod.memory.embeddings.float().cpu().clone()
        snap_y = mod.memory.keys.long().cpu().clone()
        z = zb.to(dev, dtype).requires_grad_(True)
        loss = mod(z, yb.to(dev), topk_neg=200, alpha=0.5)
        loss.backward()
        ref = memory_loss(z.detach().float().cpu(), yb, snap_z, snap_y, tau=0.07, similarity="cosine", lam=0.2,
                          t=2.0, topk=200, alpha=0.5)
        assert bool((ref["nneg"] > 200).all())
        assert float(loss) == pytest.approx(ref["loss"], rel=TOL_F32)
        assert G.rel_err(z.grad.double().cpu(), ref["dz"]) < (TOL_F32 if dtype == torch.float32 else 2 * TOL_BF16)
