"""GPU: every rank's share of a row-sharded step, emulated on one GPU and checked row by row.

ShardedSupConLoss (distributed.py) has rank r own rows [r n, (r + 1) n) of the N x N problem and issue, in this
order: supcon_forward_rows_local + _remote, supcon_finalize_sets over every rank's partial sums in rank order,
supcon_backward_rows_local (own statistics) + _remote (everyone's statistics, global sums, grad_out).
emulate_step() issues exactly those calls for every rank of a batch on one device; the collectives become
torch.cat / torch.stack, which copy exactly, so only the transport is left out.

Every rank's rows are then held to:
  * the fp64 oracle, row by row (oracle.rowblock_forward / rowblock_backward, evaluated on the device): counts
    exactly, lse / lse_m / pos_mean within 1e-4 absolute on the tensor path and 1e-5 max(1, |ref|) on the exact
    path, each row's dz within 4e-3 / 1e-5 of its reference row (floored at the block's RMS row norm, so that a
    row whose gradient nearly cancels does not decide the test).  A norm over a whole block would hide a mistake
    confined to a few rows: 128 rows of a 16384-row batch losing one column tile move the loss by ~6e-6;
  * the whole-batch call of the same kernels: counts, thresholds, the label-derived global counts and the fixed
    maximum bit for bit (the Gram is computed in the same order whatever the row blocking), and each rank's
    backward fed the whole batch's statistics within 1e-5 of the whole batch's dz rows (only the grouping of the
    fp32 partial records differs).

The shapes are those of a Stage-1 run at 64 rows per GPU (64-row tensor-path shards at offsets that are not a
multiple of 128, which take the single-phase calls), 128-row aligned shards (the two-phase calls, with and without
SUPCON_FLAG_PEER_EXCHANGE), ranks whose own rows have a smaller maximum |z|^2 than the batch (the merge rescales
their own-column records), ragged fp32 shards whose 64-row blocks straddle ranks, and exact ties."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

import debug_lib as D
from oracle import supcon_oracle as O
from test_gpu_parity_r02 import _exact_arith_inputs_d256
from wav2vec_contr_loss_b200 import _cabi
from wav2vec_contr_loss_b200 import functional as Fn

pytestmark = pytest.mark.gpu

GRAD_OUT = 1.7
TOL_LOSS = {True: 2e-3, False: 1e-5}          # keyed by "tensor path"
TOL_DZ_ROW = {True: 4e-3, False: 1e-5}        # tensor path: H is rounded to bf16 before the second GEMM
TOL_WSUM = {True: 1e-4, False: 1e-5}          # relative
TOL_STAT_TC = 1e-4                            # lse, lse_m, pos_mean absolute (the N = 65536 test's bar)
TOL_STAT_EXACT = 1e-5                         # times max(1, |ref|)
TOL_SAME_TILES = 1e-5                         # same similarity tiles and statistics, other fp32 summation order
UNIT = _cabi.FLAG_UNIT_ROWS
PEER = _cabi.FLAG_PEER_EXCHANGE

# largest per-row dz metric against the oracle seen per case group (read out when reporting the margins)
DZ_METRIC_MAX = {}


def _cfg(tau=0.07, sim="cosine", lam=0.0, topk=15, alpha=0.0):
    return dict(tau=tau, similarity=O.sim_id(sim), lambda_uni=lam, uni_t=2.0, topk=topk, alpha=alpha)


# (dtype, R, cfg) -- 64 rows per rank
STAGE1_CASES = [(dt, r, _cfg(lam=lam, alpha=alpha)) for dt in ("bf16", "f32") for r in (2, 4, 8)
                for alpha in (0.0, 0.5) for lam in (0.0, 0.05)]
STAGE1_CASES += [("bf16", 4, _cfg(tau=0.1, sim="geodesic", lam=0.05, alpha=0.5)),
                 ("f32", 8, _cfg(tau=0.1, sim="geodesic", lam=0.05, alpha=0.5))]
ALIGNED_SHAPES = [(1024, 8), (2048, 2), (2048, 4), (16384, 8)]          # (N, R): 128 .. 2048 rows per rank
RAGGED_NORM_N, RAGGED_NORM_R = 2048, 4
RAGGED_F32_SHAPES = [(1000, 8), (1000, 5)]                              # 125 / 200 rows per rank, d = 200
RAGGED_F32_CFG = _cfg(tau=0.1, sim="geodesic", lam=0.1, topk=15, alpha=0.37)
TIE_SHAPES = [(512, 8), (2048, 8)]                                      # 64 / 256 rows per rank


def _id(case):
    dt, r, cfg = case
    return f"{dt}-R{r}-{'geo' if cfg['similarity'] else 'cos'}-a{cfg['alpha']}-l{cfg['lambda_uni']}"


# ---------------------------------------------------------------------------------------------------------
# the emulated step
# ---------------------------------------------------------------------------------------------------------
def _rank_problems(z, R, cfg, flags):
    n_total, d = z.shape
    assert n_total % R == 0
    n = n_total // R
    return [Fn.make_problem(n_total, d, Fn._dtype_id(z), row_offset=r * n, n_rows=n, flags=flags, **cfg)
            for r in range(R)]


def _rank_backwards(z, y, probs, own_stats, own_partials, stats_all, partials_global):
    """every rank's backward_rows_local (own statistics and partials) + backward_rows_remote; grad_out = 1.7"""
    g = torch.tensor(GRAD_OUT, device=z.device)
    dz = []
    for prob, st, pt in zip(probs, own_stats, own_partials):
        ws = Fn.backward_rows_local(z, y, st, pt, prob)
        dz.append(Fn.backward_rows_remote(z, y, stats_all, partials_global, g, prob, ws, out_dtype=torch.float32))
    return dz


def emulate_step(z, y, R, cfg, flags):
    """What _ShardedSupCon issues on ranks 0..R-1 of one step, on one device.  z: [N, d] fp32 / bf16 on the
    device, y: int32 class keys.  Returns per-rank statistics and partial sums, every rank's (global partials,
    loss) from finalize_sets, and per-rank dz (grad_out-scaled, fp32)."""
    probs = _rank_problems(z, R, cfg, flags)
    stats, partials = [], []
    for prob in probs:
        ws = Fn.forward_rows_local(z, y, prob)
        st, pt = Fn.forward_rows_remote(z, y, prob, ws)
        stats.append(st)
        partials.append(pt)
    sets = torch.stack(partials)                                   # the all-gather of the partial sums
    finals = [Fn.finalize_sets(prob, sets) for prob in probs]     # every rank sums them itself
    partials_global, loss = finals[0]
    dz = _rank_backwards(z, y, probs, stats, partials, torch.cat(stats), partials_global)
    return dict(R=R, n=z.size(0) // R, probs=probs, stats=stats, partials=partials, finals=finals,
                partials_global=partials_global, loss=loss, dz=dz)


def _whole_batch(z, y, cfg, flags):
    """the same problem as one call over all rows, on the tiled kernels (the single-launch small / mid kernels
    evaluate in another order)"""
    prob = Fn.make_problem(z.size(0), z.size(1), Fn._dtype_id(z), flags=flags | _cabi.FLAG_NO_SMALL, **cfg)
    stats, partials, loss = Fn.forward_rows(z, y, prob, want_loss=True)
    dz = Fn.backward_rows(z, y, stats, partials, torch.tensor(GRAD_OUT, device=z.device), prob,
                          out_dtype=torch.float32)
    return dict(stats=stats, partials=partials, loss=loss, dz=dz)


_ORACLE = {}


def _oracle(key, z, y64, cfg):
    """fp64 statistics, loss and dz of every row of the batch, on the device, of the values the kernels read.
    ``key`` names the inputs so that cases differing only in flags share one evaluation; None = not kept."""
    k = (key, tuple(sorted(cfg.items())))
    if key is None or k not in _ORACLE:
        z64 = z.double()
        kw = dict(tau=cfg["tau"], similarity=cfg["similarity"], topk=cfg["topk"], lambda_uni=cfg["lambda_uni"],
                  uni_t=cfg["uni_t"])
        stats, partials = O.rowblock_forward(z64, y64, 0, z.size(0), **kw)
        loss, coef = O.loss_from_partials(partials, z.size(0), alpha=cfg["alpha"], lambda_uni=cfg["lambda_uni"])
        dz = O.rowblock_backward(z64, y64, 0, z.size(0), stats, coef, **kw)
        ref = dict(stats=stats, loss=loss, dz=dz)
        if key is None:
            return ref
        _ORACLE[k] = ref
    return _ORACLE[k]


# ---------------------------------------------------------------------------------------------------------
# checks
# ---------------------------------------------------------------------------------------------------------
def _dz_metric(dz, ref):
    """per row: |dz_i - ref_i| / max(|ref_i|, RMS row norm of the block)"""
    dz, ref = dz.double(), ref.double()
    rn = ref.norm(dim=1)
    floor = float(rn.pow(2).mean().sqrt())
    return (dz - ref).norm(dim=1) / rn.clamp_min(max(floor, 1e-30))


def _assert_rows(ok, what, err=None):
    if not bool(ok.all()):
        bad = torch.nonzero(~ok).view(-1)
        detail = f"; worst {float(err.max()):.3e}" if err is not None else ""
        raise AssertionError(f"{what}: {bad.numel()} rows fail, first {bad[:8].tolist()}{detail}")


def _check_against_oracle(group, out, ref, cfg, tc, ties=False):
    R, n = out["R"], out["n"]
    rs = ref["stats"]
    mining = cfg["alpha"] != 0.0 and cfg["topk"] >= 1
    for r in range(R):
        blk = slice(r * n, (r + 1) * n)
        st = out["stats"][r]
        si = st.view(torch.int32)
        where = f"{group} rank {r}"
        _assert_rows(si[:, _cabi.ST_NPOS].long() == rs["npos"][blk], f"{where} npos")
        _assert_rows(si[:, _cabi.ST_NNEG].long() == rs["nneg"][blk], f"{where} nneg")
        if ties:
            _assert_rows(si[:, _cabi.ST_THR_IDX].long() == rs["thr_idx"][blk], f"{where} thr_idx")
            _assert_rows(st[:, _cabi.ST_THR_VAL].double() == rs["thr_val"][blk], f"{where} thr_val")
        cols = [(_cabi.ST_LSE, "lse"), (_cabi.ST_POS_MEAN, "pos_mean")] + ([(_cabi.ST_LSE_M, "lse_m")] if mining else [])
        for c, key in cols:
            want = rs[key][blk]
            err = (st[:, c].double() - want).abs()
            bound = TOL_STAT_TC if tc else TOL_STAT_EXACT * want.abs().clamp_min(1.0)
            _assert_rows(err <= bound, f"{where} {key}", err)
        if cfg["lambda_uni"] > 0.0:
            want = rs["wsum"][blk]
            err = (st[:, _cabi.ST_WSUM].double() - want).abs() / want.abs()
            _assert_rows(err <= TOL_WSUM[tc], f"{where} wsum", err)
        in_f = rs["npos"][blk] > 0
        in_m = in_f & (rs["nneg"][blk] > 0) & (cfg["topk"] >= 1)
        assert float(out["partials"][r][_cabi.P_CNT_FULL]) == int(in_f.sum()), where
        assert float(out["partials"][r][_cabi.P_CNT_MINED]) == int(in_m.sum()), where
    for pg, loss in out["finals"]:                     # every rank derives the same global sums and loss
        assert torch.equal(pg, out["partials_global"]) and torch.equal(loss, out["loss"])
    assert float(out["loss"]) == pytest.approx(ref["loss"], rel=TOL_LOSS[tc])
    worst = 0.0
    for r in range(R):
        m = _dz_metric(out["dz"][r] / GRAD_OUT, ref["dz"][r * n:(r + 1) * n])
        _assert_rows(m <= TOL_DZ_ROW[tc], f"{group} rank {r} dz", m)
        worst = max(worst, float(m.max()))
    DZ_METRIC_MAX[group] = max(DZ_METRIC_MAX.get(group, 0.0), worst)


def _check_against_whole(group, z, y, out, whole):
    R, n = out["R"], out["n"]
    exact_cols = [_cabi.ST_NPOS, _cabi.ST_NNEG, _cabi.ST_THR_VAL, _cabi.ST_THR_IDX]
    wi = whole["stats"].view(torch.int32)[:, exact_cols]
    for r in range(R):
        blk = slice(r * n, (r + 1) * n)
        same = out["stats"][r].view(torch.int32)[:, exact_cols] == wi[blk]
        _assert_rows(same.all(1), f"{group} rank {r}: counts / thresholds differ from the whole-batch call")
        # label-derived |A_f|, |A_m| and the fixed maximum: global quantities, bit-identical on every rank
        assert torch.equal(out["partials"][r][_cabi.P_GCNT_FULL:], whole["partials"][_cabi.P_GCNT_FULL:]), \
            f"{group} rank {r}"
    # backward in isolation: every rank fed the whole batch's statistics and sums
    probs = out["probs"]
    own = [whole["stats"][r * n:(r + 1) * n] for r in range(R)]
    dz = _rank_backwards(z, y, probs, own, [whole["partials"]] * R, whole["stats"], whole["partials"])
    for r in range(R):
        m = _dz_metric(dz[r], whole["dz"][r * n:(r + 1) * n])
        _assert_rows(m <= TOL_SAME_TILES, f"{group} rank {r}: backward on the whole batch's statistics", m)


def _run(group, key, z_cpu, y_cpu, R, cfg, flags, tc, ties=False):
    dev = torch.device("cuda:0")
    z = Fn.canonical_z(z_cpu.to(dev))
    y = Fn.canonical_labels(y_cpu.to(dev), z.size(0))
    out = emulate_step(z, y, R, cfg, flags)
    ref = _oracle(key, z, y_cpu.to(dev), cfg)
    _check_against_oracle(group, out, ref, cfg, tc, ties)
    _check_against_whole(group, z, y, out, _whole_batch(z, y, cfg, flags))
    return out, ref


def _unit_rows(n, d, dtype, seed, classes=2):
    x, y = O.make_inputs(n, d, "iso", seed=seed, classes=classes)
    return F.normalize(x, dim=1).to(dtype), y


_DT = {"bf16": torch.bfloat16, "f32": torch.float32}


def _ragged_norm_inputs():
    """rank 0's rows unit, the other ranks' rows scaled to |z|^2 in [1, 2.25] (the promise allows tau / 0.025)"""
    n = RAGGED_NORM_N
    x, y = O.make_inputs(n, 256, "iso", seed=77, classes=3)
    s = 1.0 + 0.5 * torch.rand(n, 1, generator=torch.Generator().manual_seed(78))
    s[: n // RAGGED_NORM_R] = 1.0
    return (F.normalize(x, dim=1) * s).to(torch.bfloat16), y


# ---------------------------------------------------------------------------------------------------------
# routes
# ---------------------------------------------------------------------------------------------------------
def _tc_plan(prob):
    """tensor-path plan {two_phase, fwd_local_ctas} or None when the problem takes the exact path"""
    out = (ctypes.c_int32 * 16)()
    rc = D.load().supcon_debug_plan(ctypes.byref(prob), out, 16)
    if rc == -2:                                                  # SUPCON_E_UNSUPPORTED
        return None
    D.check(rc, "supcon_debug_plan")
    return dict(two_phase=out[6], fwd_local_ctas=out[7])


def _shard_probs(n_total, d, dtype, R, cfg, flags):
    z = torch.empty((n_total, d), dtype=dtype, device="meta")
    return _rank_problems(z, R, cfg, flags)


def test_cases_reach_the_routes_they_are_meant_for(cuda_device):
    """so that a later change to the plan cannot quietly move every case onto one path"""
    for dt, R, cfg in STAGE1_CASES:
        for prob in _shard_probs(64 * R, 256, _DT[dt], R, cfg, UNIT):
            plan = _tc_plan(prob)
            if dt == "f32" or R == 2:
                assert plan is None                               # exact path (N = 128: below the tensor path)
            else:
                assert plan is not None and plan["two_phase"] == 0, (dt, R, prob.row_offset)
        assert R == 2 or any(p.row_offset % 128 == 64 for p in _shard_probs(64 * R, 256, _DT[dt], R, cfg, UNIT))
    for n, R in ALIGNED_SHAPES + [(RAGGED_NORM_N, RAGGED_NORM_R)]:
        for flags in (UNIT, UNIT | PEER):
            for prob in _shard_probs(n, 256, torch.bfloat16, R, _cfg(alpha=0.5), flags):
                assert _tc_plan(prob)["two_phase"] == 1, (n, R, flags)
        shared = _tc_plan(_shard_probs(n, 256, torch.bfloat16, R, _cfg(), UNIT)[1])["fwd_local_ctas"]
        peer = _tc_plan(_shard_probs(n, 256, torch.bfloat16, R, _cfg(), UNIT | PEER)[1])["fwd_local_ctas"]
        assert shared <= peer
        if n == 16384:       # a rank owning 1/8 of the columns leaves SMs to the all-gather unless peers exchange
            assert shared < peer, (shared, peer)
    for n, R in TIE_SHAPES:
        for prob in _shard_probs(n, 256, torch.bfloat16, R, _cfg(topk=32, alpha=1.0), UNIT):
            assert _tc_plan(prob)["two_phase"] == (1 if n // R % 128 == 0 else 0)
    for n, R in RAGGED_F32_SHAPES:
        for prob in _shard_probs(n, 200, torch.float32, R, RAGGED_F32_CFG, UNIT):
            assert _tc_plan(prob) is None
            out = (ctypes.c_int32 * 4)()
            D.check(D.load().supcon_debug_ffma_plan(ctypes.byref(prob), out, 4), "supcon_debug_ffma_plan")
            assert out[0] > 1 and out[1] > 1, (n, R, list(out))      # column splits merged / reduced


# ---------------------------------------------------------------------------------------------------------
# case groups
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", STAGE1_CASES, ids=[_id(c) for c in STAGE1_CASES])
def test_stage1_shards_of_64_rows(cuda_device, case):
    """the Stage-1 batch of 64 rows per GPU on 2, 4 and 8 ranks: bf16 at N = 256 / 512 on the tensor path with
    row offsets 64 mod 128 (single phase: the 128-row A tile holds the next rank's rows, or runs past N on the
    last rank), bf16 at N = 128 and fp32 on the exact path"""
    dt, R, cfg = case
    n = 64 * R
    z, y = _unit_rows(n, 256, _DT[dt], seed=n + R)
    tc = dt == "bf16" and n >= 256
    _run(f"stage1-{dt}-{'tensor' if tc else 'exact'}", None, z, y, R, cfg, UNIT, tc)


@pytest.mark.parametrize("peer", [False, True], ids=["nccl", "peer"])
@pytest.mark.parametrize("lam", [0.0, 0.05])
@pytest.mark.parametrize("alpha", [0.0, 0.5])
@pytest.mark.parametrize("n,R", ALIGNED_SHAPES)
def test_aligned_two_phase_shards(cuda_device, n, R, alpha, lam, peer):
    """128-row aligned shards take the two-phase calls; lambda > 0 makes the own-column backward decline (its
    coefficient needs the global sum of W) and the remote call do the whole backward"""
    z, y = _unit_rows(n, 256, torch.bfloat16, seed=n, classes=3)
    cfg = _cfg(lam=lam, alpha=alpha)
    _run("aligned", ("aligned", n), z, y, R, cfg, UNIT | (PEER if peer else 0), tc=True)


@pytest.mark.parametrize("alpha", [0.0, 0.5])
def test_own_columns_with_a_smaller_fixed_maximum(cuda_device, alpha):
    """rank 0's rows are unit, the others' reach |z|^2 = 2.25: the own-column phase of rank 0 evaluates its
    records against max |z|^2 = 1, and the merge must rescale them to the batch's maximum"""
    z, y = _ragged_norm_inputs()
    n = RAGGED_NORM_N // RAGGED_NORM_R
    nrm2 = (z.float() ** 2).sum(1)
    own_max = [float(nrm2[r * n:(r + 1) * n].max()) for r in range(RAGGED_NORM_R)]
    assert own_max[0] < 1.01 < 2.2 < max(own_max)
    out, _ = _run("ragged-norms", None, z, y, RAGGED_NORM_R, _cfg(alpha=alpha), UNIT, tc=True)
    assert float(out["partials"][0][_cabi.P_FIXMAX]) == pytest.approx(max(own_max), rel=1e-5)


@pytest.mark.parametrize("n,R", RAGGED_F32_SHAPES)
def test_ragged_fp32_shards(cuda_device, n, R):
    """125 / 200 rows per rank: the exact path's 64-row blocks straddle rank boundaries"""
    z, y = _unit_rows(n, 200, torch.float32, seed=n + R, classes=3)
    _run("ragged-f32", None, z, y, R, RAGGED_F32_CFG, UNIT, tc=False)


@pytest.mark.parametrize("k", [15, 32])
@pytest.mark.parametrize("n,R", TIE_SHAPES)
def test_exact_ties_on_every_rank(cuda_device, n, R, k):
    """entries in {0, +-1/16, +-1/32}: every similarity is exact, many rows have exact ties at rank K, and each
    rank's thresholds must equal the oracle's bit for bit"""
    z, y = _exact_arith_inputs_d256(n, seed=n + k)
    zb = z.to(torch.bfloat16)
    assert torch.equal(zb.float(), z)
    cfg = _cfg(topk=k, alpha=1.0)
    _, ref = _run("ties", None, zb, y, R, cfg, UNIT, tc=True, ties=True)
    zz = zb.to(cuda_device).double()
    tied = ((zz @ zz.t()) == ref["stats"]["thr_val"].view(-1, 1)).sum(1) > 1
    assert int(tied.sum()) > n // 4


@pytest.mark.parametrize("dtype", ["bf16", "f32"])
def test_rank_counts_agree_row_by_row(cuda_device, dtype):
    """the concatenated dz of R = 2, 4 and 8 ranks of one batch agree row by row.  fp32: whole emulated steps.
    bf16: each rank count's backward on the same (whole-batch) statistics -- statistics summed over other column
    splits differ in the last fp32 bits, which can move an entry of H across a bf16 rounding boundary"""
    dev = torch.device("cuda:0")
    n = 2048 if dtype == "bf16" else 512
    zc, yc = _unit_rows(n, 256, _DT[dtype], seed=5 * n)
    z = Fn.canonical_z(zc.to(dev))
    y = Fn.canonical_labels(yc.to(dev), n)
    cfg = _cfg(lam=0.0 if dtype == "bf16" else 0.05, alpha=0.5)
    whole = _whole_batch(z, y, cfg, UNIT)
    dz = {}
    for R in (2, 4, 8):
        if dtype == "bf16":
            k = n // R
            own = [whole["stats"][r * k:(r + 1) * k] for r in range(R)]
            dz[R] = torch.cat(_rank_backwards(z, y, _rank_problems(z, R, cfg, UNIT), own, [whole["partials"]] * R,
                                              whole["stats"], whole["partials"]))
        else:
            dz[R] = torch.cat(emulate_step(z, y, R, cfg, UNIT)["dz"])
    for R in (4, 8):
        m = _dz_metric(dz[R], dz[2])
        _assert_rows(m <= TOL_SAME_TILES, f"R = {R} against R = 2", m)
