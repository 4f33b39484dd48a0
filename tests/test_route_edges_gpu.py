"""GPU: every single-GPU route at its edges, through both whole-batch entries, row by row against the fp64 oracle.

Each case first asserts, through the test library's route report (supcon_debug_route), which kernel family its
problem takes -- the map itself is pinned by tests/test_route_map.py -- and then runs the same inputs through
  * supcon_loss_and_grad (what the module calls up to N = 320), and
  * supcon_forward_rows + supcon_backward_rows with grad_out = 1.7 (the module above N = 320; the memory and
    cached-batch steps at every size),
each twice, with fp32 and with bf16 dz.  Per case and entry:
  * row statistics against the fp64 oracle (oracle.rowblock_forward, on the device, of the values the kernels read):
    npos / nneg exactly, lse / pos_mean / lse_m within 1e-5 max(1, |ref|) on the exact routes and 1e-4 absolute on
    the tensor path, wsum within 1e-5 / 1e-4 relative; on the exact-arithmetic grids the hard-negative threshold
    (value, index) bit for bit;
  * the loss within 1e-5 / 2e-3 relative, and dz row by row within 1e-5 / 4e-3 of the oracle's row (floored at the
    RMS row norm), naming the failing rows.  A matrix norm would hide a mistake confined to a few rows (a ragged
    last CTA, a tail tile, one dropped column);
  * the bf16 dz equal, bit for bit, to the fp32 dz of the same call rounded to nearest even: every route stores
    __float2bfloat16 of the fp32 value it would have stored;
  * the second call bit-identical to the first (statistics, partial sums, loss, dz): every route sums in a fixed
    order;
  * the neighbour across the edge: single-launch kernels against the tiled ones (SUPCON_FLAG_NO_SMALL) within 1e-5
    per row, with the mid kernel's thresholds bit-identical to the tiled kernels'; the tensor path against the exact
    one (SUPCON_FLAG_FORCE_EXACT) within the tensor path's 4e-3 per row, since only it rounds H to bf16.

Hard-negative mining is decided by a comparison, so inputs are chosen where fp32 and fp64 rank the negatives
alike: cosine mining runs on exact-arithmetic grids (every dot product exact, ties exact and broken by lowest index
on every route), and every random mining case asserts, before comparing, that each row's fp64 gap between its K-th
and (K+1)-th negative exceeds 2e-5 (the seeds were chosen so; the assertion keeps a change to the generator from
weakening a case silently).  Geodesic cases hold no duplicate rows (the slope is ill-conditioned at c = 1)."""
import math

import pytest
import torch
import torch.nn.functional as F

import debug_lib as D
from oracle import supcon_oracle as O
from test_rank_shards_gpu import _assert_rows, _dz_metric
from test_route_map import small_d_max
from wav2vec_contr_loss_b200 import _cabi
from wav2vec_contr_loss_b200 import functional as Fn

pytestmark = pytest.mark.gpu

GRAD_OUT = 1.7
TOL_LOSS = {True: 2e-3, False: 1e-5}          # keyed by "tensor path"
TOL_DZ_ROW = {True: 4e-3, False: 1e-5}        # tensor path: H is rounded to bf16 before the second GEMM
TOL_WSUM = {True: 1e-4, False: 1e-5}          # relative
TOL_STAT_TC = 1e-4                            # lse, lse_m, pos_mean absolute
TOL_STAT_EXACT = 1e-5                         # times max(1, |ref|)
TOL_NEIGHBOUR = 1e-5                          # single-launch against tiled: same formulas, other summation order
MIN_GAP = 2e-5                                # fp64 gap between the K-th and (K+1)-th negative, random mining cases
UNIT = _cabi.FLAG_UNIT_ROWS
NO_SMALL, FORCE_EXACT = _cabi.FLAG_NO_SMALL, _cabi.FLAG_FORCE_EXACT
SMALL, MID, TENSOR, TILED = D.SMALL, D.MID, D.TENSOR, D.TILED

# largest per-row dz metric against the oracle seen per route (printed at the end of the session)
DZ_METRIC_MAX = {}


# ---------------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------------
def _cfg(tau=0.1, sim="cosine", lam=0.05, topk=15, alpha=0.5):
    return dict(tau=tau, similarity=O.sim_id(sim), lambda_uni=lam, uni_t=2.0, topk=topk, alpha=alpha)


def _unit(n, d, seed, classes=2):
    """random unit rows (fp32) and labels"""
    x, y = O.make_inputs(n, d, "iso", seed=seed, classes=classes)
    return F.normalize(x, dim=1), y


def _grid(n, d, seed, classes=3):
    """entries in {0, +-a, +-a/2} with a = 2^-ceil(log2(d) / 2): exact in bf16, every dot product a multiple of
    a^2 / 4 below 2 in magnitude -> exact in fp32 (any summation order) and fp64; |z|^2 ~ 0.5; many exact ties"""
    g = torch.Generator().manual_seed(seed)
    a = 2.0 ** -math.ceil(math.log2(d) / 2)
    vals = torch.tensor([0.0, a, -a, a / 2, -a / 2])
    return vals[torch.randint(0, 5, (n, d), generator=g)], torch.randint(0, classes, (n,), generator=g)


def mining_gaps(z, y, sim, k):
    """per row with more than k negatives: fp64 similarity gap between its k-th and (k+1)-th negative"""
    z64 = z.double()
    if k < 1 or k >= z64.size(0) - 1:
        return z64.new_zeros(0)
    s, _ = O._sim_and_slope(z64 @ z64.t(), sim)
    neg = y.view(-1, 1) != y.view(1, -1)
    v = s.masked_fill(~neg, float("-inf")).sort(dim=1, descending=True).values
    rows = neg.sum(1) > k
    return v[rows, k - 1] - v[rows, k]


# ---------------------------------------------------------------------------------------------------------
# the two entries
# ---------------------------------------------------------------------------------------------------------
def _bits(t):
    return t.contiguous().view(torch.int32 if t.element_size() == 4 else
                               torch.int64 if t.element_size() == 8 else torch.int16)


def _assert_same_bits(a, b, what):
    for k in a:
        assert torch.equal(_bits(a[k]), _bits(b[k])), f"{what}: {k} differs between two identical calls"


def _assert_bf16_is_rounded_fp32(dzb, dz32, what):
    want = dz32.to(torch.bfloat16)
    same = (_bits(dzb) == _bits(want)).all(1)
    _assert_rows(same, f"{what}: bf16 dz is not the fp32 dz rounded to nearest even")


def _loss_and_grad(z, y, prob):
    out = []
    for _ in range(2):
        loss, dz, st, pt = Fn.loss_and_grad(z, y, prob, out_dtype=torch.float32)
        out.append(dict(stats=st.clone(), partials=pt.clone(), loss=loss.clone(), dz=dz))
    _, dzb, _, _ = Fn.loss_and_grad(z, y, prob, out_dtype=torch.bfloat16)
    return out, dzb, 1.0


def _rows(z, y, prob):
    g = torch.tensor(GRAD_OUT, device=z.device)
    out = []
    for _ in range(2):
        st, pt, loss = Fn.forward_rows(z, y, prob, want_loss=True)
        dz = Fn.backward_rows(z, y, st, pt, g, prob, out_dtype=torch.float32)
        out.append(dict(stats=st.clone(), partials=pt.clone(), loss=loss.clone(), dz=dz))
    dzb = Fn.backward_rows(z, y, out[0]["stats"], out[0]["partials"], g, prob, out_dtype=torch.bfloat16)
    return out, dzb, GRAD_OUT


ENTRIES = {"loss_and_grad": _loss_and_grad, "forward_rows+backward_rows": _rows}

_ORACLE = {}


def _oracle(key, z, y64, cfg):
    """fp64 statistics, loss and dz of every row, on the device, of the values the kernels read (bf16 rows: their
    bf16 values); cached per input"""
    k = (key, tuple(sorted(cfg.items())))
    if k not in _ORACLE:
        z64 = z.double()
        kw = dict(tau=cfg["tau"], similarity=cfg["similarity"], topk=cfg["topk"], lambda_uni=cfg["lambda_uni"],
                  uni_t=cfg["uni_t"])
        stats, partials = O.rowblock_forward(z64, y64, 0, z.size(0), **kw)
        loss, coef = O.loss_from_partials(partials, z.size(0), alpha=cfg["alpha"], lambda_uni=cfg["lambda_uni"])
        dz = O.rowblock_backward(z64, y64, 0, z.size(0), stats, coef, **kw)
        _ORACLE[k] = dict(stats=stats, partials=partials, loss=loss, dz=dz)
    return _ORACLE[k]


def _check_oracle(where, run, scale, ref, cfg, tc, exact_grid):
    st, rs = run["stats"], ref["stats"]
    si = st.view(torch.int32)
    mining = cfg["alpha"] != 0.0 and cfg["topk"] >= 1
    _assert_rows(si[:, _cabi.ST_NPOS].long() == rs["npos"], f"{where} npos")
    _assert_rows(si[:, _cabi.ST_NNEG].long() == rs["nneg"], f"{where} nneg")
    if exact_grid and mining and cfg["similarity"] == _cabi.COSINE:
        _assert_rows(si[:, _cabi.ST_THR_IDX].long() == rs["thr_idx"], f"{where} thr_idx")
        _assert_rows(st[:, _cabi.ST_THR_VAL].double() == rs["thr_val"], f"{where} thr_val")
    cols = [(_cabi.ST_LSE, "lse"), (_cabi.ST_POS_MEAN, "pos_mean")] + ([(_cabi.ST_LSE_M, "lse_m")] if mining else [])
    for c, key in cols:
        want = rs[key]
        err = (st[:, c].double() - want).abs()
        bound = TOL_STAT_TC if tc else TOL_STAT_EXACT * want.abs().clamp_min(1.0)
        _assert_rows(err <= bound, f"{where} {key}", err)
    if cfg["lambda_uni"] > 0.0:
        want = rs["wsum"]
        err = (st[:, _cabi.ST_WSUM].double() - want).abs() / want.abs()
        _assert_rows(err <= TOL_WSUM[tc], f"{where} wsum", err)
    for slot in (_cabi.P_CNT_FULL, _cabi.P_CNT_MINED):
        assert float(run["partials"][slot]) == float(ref["partials"][slot]), f"{where} partial {slot}"
    assert float(run["loss"]) == pytest.approx(ref["loss"], rel=TOL_LOSS[tc], abs=1e-7), where
    m = _dz_metric(run["dz"], ref["dz"] * scale)
    _assert_rows(m <= TOL_DZ_ROW[tc], f"{where} dz", m)
    return float(m.max()) if m.numel() else 0.0


def _route_of(prob, z):
    r = D.route(prob, z)
    return r["loss_and_grad"], r["backward_rows"]


def run_case(name, z_cpu, y_cpu, cfg, flags, route, *, exact_grid=False, misalign=False, key=None):
    """route: the expected (supcon_loss_and_grad, supcon_backward_rows) routes"""
    dev = torch.device("cuda:0")
    if misalign:                          # rows start one element past a 16-byte boundary
        buf = torch.empty(z_cpu.numel() + 1, dtype=z_cpu.dtype, device=dev)
        z = buf[1:].view(z_cpu.shape)
        z.copy_(z_cpu.to(dev))
        assert z.data_ptr() % 16 != 0
    else:
        z = Fn.canonical_z(z_cpu.to(dev))
    y = Fn.canonical_labels(y_cpu.to(dev), z.size(0))
    n, d = z.shape
    prob = Fn.make_problem(n, d, Fn._dtype_id(z), flags=flags, **cfg)
    assert _route_of(prob, z) == route, f"{name}: takes {_route_of(prob, z)}, meant for {route}"
    tc = route[0] == TENSOR
    assert route[1] == (TENSOR if tc else TILED)
    ref = _oracle(key if key is not None else (name, n, d), z, y_cpu.to(dev), cfg)
    results = {}
    for entry, fn in ENTRIES.items():
        where = f"{name} [{entry}]"
        runs, dzb, scale = fn(z, y, prob)
        _assert_same_bits(runs[0], runs[1], where)
        _assert_bf16_is_rounded_fp32(dzb, runs[0]["dz"], where)
        worst = _check_oracle(where, runs[0], scale, ref, cfg, tc, exact_grid)
        fwd = D.route(prob, z)["loss_and_grad" if entry == "loss_and_grad" else "forward_rows"]
        rname = D.ROUTE_NAMES[fwd]
        if entry != "loss_and_grad" and fwd != route[1]:
            rname += f" forward + {D.ROUTE_NAMES[route[1]]} backward"
        DZ_METRIC_MAX[rname] = max(DZ_METRIC_MAX.get(rname, 0.0), worst)
        results[entry] = runs[0]
    # the neighbour across the edge
    if route[0] in (SMALL, MID):
        nb = Fn.make_problem(n, d, Fn._dtype_id(z), flags=flags | NO_SMALL, **cfg)
        assert _route_of(nb, z) == (TILED, TILED)
        runs, _, _ = _loss_and_grad(z, y, nb)
        mine = results["loss_and_grad"]
        m = _dz_metric(mine["dz"], runs[0]["dz"])
        _assert_rows(m <= TOL_NEIGHBOUR, f"{name}: {D.ROUTE_NAMES[route[0]]} against tiled dz", m)
        cols = [_cabi.ST_NPOS, _cabi.ST_NNEG] + ([_cabi.ST_THR_VAL, _cabi.ST_THR_IDX] if route[0] == MID else [])
        same = mine["stats"].view(torch.int32)[:, cols] == runs[0]["stats"].view(torch.int32)[:, cols]
        _assert_rows(same.all(1), f"{name}: {D.ROUTE_NAMES[route[0]]} against tiled counts / thresholds")
    if tc:
        nb = Fn.make_problem(n, d, Fn._dtype_id(z), flags=flags | FORCE_EXACT, **cfg)
        assert _route_of(nb, z)[1] == TILED
        runs, _, _ = _loss_and_grad(z, y, nb)
        m = _dz_metric(results["loss_and_grad"]["dz"], runs[0]["dz"])
        _assert_rows(m <= TOL_DZ_ROW[True], f"{name}: tensor against exact dz", m)
    return results


def _assert_gaps(z, y, cfg):
    if cfg["alpha"] == 0.0 or cfg["topk"] < 1:
        return
    gaps = mining_gaps(z.double(), y, cfg["similarity"], cfg["topk"])
    assert gaps.numel() == 0 or float(gaps.min()) > MIN_GAP, \
        f"inputs have a near-tie at rank K (gap {float(gaps.min()):.2e}): choose another seed"


@pytest.fixture(scope="module", autouse=True)
def _report_margins():
    yield
    for r, v in sorted(DZ_METRIC_MAX.items()):
        print(f"\nDZ_METRIC_MAX {r}: {v:.3e}", end="")
    print()


# ---------------------------------------------------------------------------------------------------------
# N across small / mid / tiled, fp32, d = 256
# ---------------------------------------------------------------------------------------------------------
N_EDGES = [2, 3, 8, 9, 31, 32, 33, 159, 160, 161, 255, 256, 257, 319, 320, 321]
GEO_N = sorted(N_EDGES + [64, 100])
# seeds whose random unit rows put no near-tie at rank K = 5 (geodesic), chosen on the CPU with mining_gaps
GEO_SEEDS = {159: 164, 160: 166, 255: 260, 256: 284, 257: 265, 319: 321, 320: 324, 321: 346}


def _n_route(n):
    r = SMALL if n <= 160 else MID if n <= 320 else TILED
    return (r, TILED)


@pytest.mark.parametrize("n", N_EDGES)
def test_n_edges_exact_grid_cosine_mining(cuda_device, n):
    """cosine, K = 15, alpha = 0.5, uniformity; exact arithmetic: thresholds bit for bit on every route"""
    z, y = _grid(n, 256, seed=1000 + n)
    run_case(f"N={n} grid", z, y, _cfg(), 0, _n_route(n), exact_grid=True)


@pytest.mark.parametrize("n", GEO_N)
def test_n_edges_random_geodesic_mining(cuda_device, n):
    """random unit rows, geodesic, K = 5, alpha = 0.5, uniformity.  Below 129 rows the small kernel splits each
    dot product over k (2 or 4 partial sums), so its Gram differs in the last bits from the tiled kernels' single
    fma chain: supcon_forward_rows + supcon_backward_rows must still select the same hard negatives"""
    z, y = _unit(n, 256, seed=GEO_SEEDS.get(n, n))
    cfg = _cfg(sim="geodesic", topk=5)
    _assert_gaps(z, y, cfg)
    run_case(f"N={n} geodesic", z, y, cfg, 0, _n_route(n))


@pytest.mark.parametrize("n", [31, 64, 100])
def test_mining_forward_rows_thresholds_are_the_tiled_backwards(cuda_device, n):
    """supcon_forward_rows hands its thresholds to a tiled supcon_backward_rows, which recomputes each similarity as
    one fma chain over k and selects {s > thr} U {s == thr, j <= thr_idx}.  The small kernel sums each dot product
    from k-slices below 129 rows, so its thresholds could differ from the tiled s in the last bit, and the backward
    dropped the K-th negative of those rows (dz rows off by up to 9e-2).  With mining the forward now runs on the
    tiled kernels: its thresholds are theirs bit for bit"""
    dev = cuda_device
    z0, y0 = _unit(n, 256, seed=GEO_SEEDS.get(n, n))
    z = Fn.canonical_z(z0.to(dev))
    y = Fn.canonical_labels(y0.to(dev), n)
    cfg = _cfg(sim="geodesic", topk=5)
    prob = Fn.make_problem(n, 256, _cabi.F32, **cfg)
    r = D.route(prob, z)
    assert (r["loss_and_grad"], r["forward_rows"], r["backward_rows"]) == (SMALL, TILED, TILED)
    st, _, _ = Fn.forward_rows(z, y, prob, want_loss=True)
    tiled, _, _ = Fn.forward_rows(z, y, Fn.make_problem(n, 256, _cabi.F32, flags=NO_SMALL, **cfg), want_loss=True)
    cols = [_cabi.ST_THR_VAL, _cabi.ST_THR_IDX]
    _assert_rows((st.view(torch.int32)[:, cols] == tiled.view(torch.int32)[:, cols]).all(1), "thresholds")


# ---------------------------------------------------------------------------------------------------------
# d across the capacity edges (recomputed from the layouts)
# ---------------------------------------------------------------------------------------------------------
def _d_edges():
    cases = []
    for n in (64, 128, 160):
        dmax = small_d_max(n)
        cases += [(n, dmax, SMALL), (n, dmax + 4, MID)]
    cases += [(32, small_d_max(32), SMALL), (320, 1024, MID), (161, 1024, MID), (64, 1028, TILED), (320, 1028, TILED)]
    return cases


@pytest.mark.parametrize("n,d,route", _d_edges())
def test_d_capacity_edges(cuda_device, n, d, route):
    z, y = _grid(n, d, seed=n * 7 + d)
    run_case(f"N={n} d={d}", z, y, _cfg(), 0, (route, TILED), exact_grid=True)


# ---------------------------------------------------------------------------------------------------------
# vector / scalar loads
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [100, 300])
@pytest.mark.parametrize("d", [19, 255, 257])
def test_odd_d_scalar_loads(cuda_device, n, d):
    z, y = _grid(n, d, seed=n + d)
    assert D.route(Fn.make_problem(n, d, _cabi.F32, **_cfg()), 1 << 20)["vec"] == 0
    run_case(f"N={n} d={d}", z, y, _cfg(), 0, (TILED, TILED), exact_grid=True)


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("n", [100, 300])
def test_misaligned_rows_scalar_loads(cuda_device, n, dtype):
    """z = buf[1:] of a flat buffer: the single-launch kernels decline it, the tiled kernels load element-wise"""
    z, y = _grid(n, 252, seed=3 * n)
    z = z.to(torch.bfloat16 if dtype == "bf16" else torch.float32)
    run_case(f"N={n} misaligned {dtype}", z, y, _cfg(), 0, (TILED, TILED), exact_grid=True, misalign=True,
             key=("misaligned", n, dtype))


def test_misaligned_bf16_at_a_tensor_shape_fails_cleanly(cuda_device):
    """the tensor map is encoded before any launch: a clean SUPCON_E_INVALID naming the alignment, no kernel runs"""
    dev = cuda_device
    z0, y0 = _unit(300, 256, seed=5)
    buf = torch.empty(300 * 256 + 1, dtype=torch.bfloat16, device=dev)
    z = buf[1:].view(300, 256)
    z.copy_(z0.to(dev))
    y = Fn.canonical_labels(y0.to(dev), 300)
    prob = Fn.make_problem(300, 256, _cabi.BF16, flags=UNIT, **_cfg())
    assert _route_of(prob, z) == (TENSOR, TENSOR)
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        Fn.loss_and_grad(z, y, prob)
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        Fn.forward_rows(z, y, prob, want_loss=True)
    stats = torch.zeros(300, _cabi.STATS_STRIDE, device=dev)
    partials = torch.zeros(_cabi.N_PARTIALS, dtype=torch.float64, device=dev)
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        Fn.backward_rows(z, y, stats, partials, None, prob)
    torch.cuda.synchronize()
    # the device is fine: the same rows, aligned, run
    zz = z.clone()
    loss, dz, _, _ = Fn.loss_and_grad(zz, y, prob)
    assert math.isfinite(float(loss)) and bool(dz.isfinite().all())


# ---------------------------------------------------------------------------------------------------------
# mining depth
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [150, 300])
@pytest.mark.parametrize("which", ["32", "33", "N-2", "N-1"])
def test_mining_depth(cuda_device, n, which):
    """K = 32 and K = N - 1 (every negative) stay on the single-launch kernels; K = 33 and N - 2 leave them"""
    k = {"32": 32, "33": 33, "N-2": n - 2, "N-1": n - 1}[which]
    single = SMALL if n <= 160 else MID
    route = single if which in ("32", "N-1") else TILED
    z, y = _grid(n, 256, seed=17 * n)
    run_case(f"N={n} K={k}", z, y, _cfg(topk=k), 0, (route, TILED), exact_grid=True, key=("depth", n))


@pytest.mark.parametrize("n", [150, 300])
def test_mining_off(cuda_device, n):
    """K = 0 (no hard-negative term at all), and alpha = 0 with K = 15 (the term has no weight)"""
    single = SMALL if n <= 160 else MID
    z, y = _grid(n, 256, seed=17 * n)
    run_case(f"N={n} K=0", z, y, _cfg(topk=0), 0, (single, TILED), exact_grid=True, key=("depth", n))
    run_case(f"N={n} alpha=0", z, y, _cfg(alpha=0.0), 0, (single, TILED), exact_grid=True, key=("depth", n))


def test_rows_with_fewer_negatives_than_k(cuda_device):
    """labels 140 : 10 at N = 150: the 140 rows of the large class have 10 negatives, fewer than K = 15"""
    z, _ = _grid(150, 256, seed=140)
    y = torch.zeros(150, dtype=torch.int64)
    y[torch.randperm(150, generator=torch.Generator().manual_seed(10))[:10]] = 1
    for flags, route in ((0, SMALL), (NO_SMALL, TILED)):
        run_case(f"140:10 flags={flags}", z, y, _cfg(), flags, (route, TILED), exact_grid=True, key="140:10")


# ---------------------------------------------------------------------------------------------------------
# labels on each route
# ---------------------------------------------------------------------------------------------------------
LABEL_ROUTES = [(64, "f32", SMALL), (200, "f32", MID), (400, "f32", TILED), (512, "bf16", TENSOR)]


@pytest.mark.parametrize("labels", ["one-class", "all-distinct", "singleton"])
@pytest.mark.parametrize("n,dtype,route", LABEL_ROUTES)
def test_label_layouts_on_each_route(cuda_device, n, dtype, route, labels):
    z, y = _grid(n, 256, seed=n + 11)
    if labels == "one-class":            # no negatives: mining has nothing to select
        y = torch.zeros(n, dtype=torch.int64)
    elif labels == "all-distinct":       # no positives: only the uniformity term has a gradient
        y = torch.arange(n)
    else:                                # one row alone in its class
        y = (torch.arange(n) % 2) + 1
        y[n // 3] = 0
    z = z.to(torch.bfloat16 if dtype == "bf16" else torch.float32)
    flags = UNIT if dtype == "bf16" else 0
    run_case(f"N={n} {labels}", z, y, _cfg(), flags, (route, route if route == TENSOR else TILED), exact_grid=True)


# ---------------------------------------------------------------------------------------------------------
# the tensor path, bf16, d = 256
# ---------------------------------------------------------------------------------------------------------
TC_N = [255, 256, 257, 383, 384, 385, 511, 512, 513]
# seeds without a near-tie at rank K = 5 (cosine, bf16 rows), chosen like GEO_SEEDS
TC_SEEDS = {255: 768, 256: 772, 257: 773, 383: 1157, 384: 1159, 385: 1156, 511: 1570, 512: 1540, 513: 1547}


@pytest.mark.parametrize("n", TC_N)
def test_tensor_path_row_blocks(cuda_device, n):
    """the last 256-row forward block or 128-row backward block holds one row at 257, 385, 513; 255 is mid"""
    z, y = _unit(n, 256, seed=TC_SEEDS[n])
    z = z.to(torch.bfloat16)
    cfg = _cfg(topk=5)
    _assert_gaps(z, y, cfg)
    route = (MID, TILED) if n < 256 else (TENSOR, TENSOR)
    run_case(f"N={n} bf16", z, y, cfg, UNIT, route)


@pytest.mark.parametrize("tau,route", [(0.025, TENSOR), (0.0249, MID)])
def test_tensor_path_temperature_edge(cuda_device, tau, route):
    z, y = _unit(300, 256, seed=25)
    run_case(f"tau={tau}", z.to(torch.bfloat16), y, _cfg(tau=tau, alpha=0.0), UNIT,
             (route, TENSOR if route == TENSOR else TILED))


@pytest.mark.parametrize("sim,route", [("geodesic", TENSOR), ("cosine", MID)])
def test_tensor_path_without_the_unit_rows_promise(cuda_device, sim, route):
    """geodesic needs no promise; cosine without it is exact"""
    z, y = _unit(300, 256, seed=31)
    run_case(f"{sim} no promise", z.to(torch.bfloat16), y, _cfg(sim=sim, alpha=0.0), 0,
             (route, TENSOR if route == TENSOR else TILED), key=("no-promise", 300))


@pytest.mark.parametrize("k,route", [(32, TENSOR), (33, TILED)])
def test_tensor_path_mining_depth(cuda_device, k, route):
    z, y = _grid(300, 256, seed=332)
    run_case(f"bf16 K={k}", z.to(torch.bfloat16), y, _cfg(topk=k), UNIT, (route, route), exact_grid=True,
             key=("bf16-depth", 300))


@pytest.mark.parametrize("classes", [3, 33])
@pytest.mark.parametrize("n,sums", [(32767, 0), (32768, 1)])
def test_class_sums_switch(cuda_device, n, sums, classes):
    """cosine, unmined: class sums from 2^30 pairs; with 33 classes the device falls back to per-pair sums"""
    z, y = _unit(32768, 256, seed=classes, classes=classes)
    z, y = z[:n].to(torch.bfloat16), y[:n]
    prob = Fn.make_problem(n, 256, _cabi.BF16, flags=UNIT, **_cfg(alpha=0.0, lam=0.0))
    r = D.route(prob, 1 << 20)
    assert r["fwd_class_sums"] == r["bwd_class_sums"] == sums
    run_case(f"N={n} {classes} classes", z, y, _cfg(alpha=0.0, lam=0.0), UNIT, (TENSOR, TENSOR))
