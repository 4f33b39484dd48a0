"""The single-GPU route map, read from the dispatcher's own predicates (supcon_debug_route; no device needed).

supcon_api.cu sends every whole-batch call to one of four kernel families:

  small   supcon_small.cu  N <= 160, d % 4 == 0, d <= 1024, z 16-byte aligned, small_layout <= 224 KiB,
                           mining K <= 32 or K >= N - 1; not NO_SMALL / FORCE_TENSOR / MEMORY_COLUMNS.
                           supcon_forward_rows with mining: tiled instead (its backward, always tiled, must
                           recompute the forward's Gram bit for bit to find the same hard negatives)
  mid     supcon_mid.cu    not small, N <= 320, the same d / alignment / K rules, mid_layout(N, d, 32) <= 224 KiB,
                           the tensor path not eligible, and a cluster of 16 CTAs (8 when N <= 256) co-schedules
  tensor  supcon_tc.cu     bf16, d == 256, N >= 256, tau >= 0.025, K <= 32 when mining, cosine only with the
                           unit-rows promise (or FORCE_TENSOR); not FORCE_EXACT.  Class sums from N_rows N >= 2^30
                           (or CLASS_SUMS), cosine, unmined, not NO_CLASS_SUMS, never in a memory backward
  tiled   supcon_ffma.cu   everything else; vector loads only when d % 4 == 0 and z is 16-byte (fp32) / 8-byte
                           (bf16) aligned

`expected()` below is that table.  A change to a predicate in the dispatcher changes what these tests expect, so it
has to change this file too, where a reviewer reads it; tests/test_route_edges_gpu.py runs every edge named here on
the device."""
import ctypes

import pytest

import debug_lib as D
from wav2vec_contr_loss_b200 import _cabi
from wav2vec_contr_loss_b200 import functional as Fn

SMALL, MID, TENSOR, TILED = D.SMALL, D.MID, D.TENSOR, D.TILED
F32, BF16 = _cabi.F32, _cabi.BF16
COS, GEO = _cabi.COSINE, _cabi.GEODESIC
UNIT = _cabi.FLAG_UNIT_ROWS
KIB224 = 224 * 1024
ALIGNED = 1 << 20              # a 256-byte aligned address: only the alignment of z enters the route
E_INVALID = -1                 # SUPCON_E_INVALID


# ---------------------------------------------------------------------------------------------------------
# shared-memory layouts of the single-launch kernels (supcon_small.cu small_layout, supcon_mid.cu mid_layout)
# ---------------------------------------------------------------------------------------------------------
def _tail(o, np_, rows):
    """norms, labels, local and gathered statistics, 8-byte alignment, partial sums"""
    o += 2 * np_ * 4 + rows * _cabi.STATS_STRIDE * 4 + np_ * _cabi.STATS_STRIDE * 4
    return ((o + 7) & ~7) + _cabi.N_PARTIALS * 8


def small_layout_bytes(n, d):
    rows, np_, ld = (n + 7) // 8, (n + 31) // 32 * 32, d + 4
    groups = min(4, max(1, 256 // np_))
    return _tail(n * ld * 4 + 2 * rows * np_ * 4 + groups * rows * np_ * 4, np_, rows)


def mid_layout_bytes(n, d, rows=32):
    np_, ld = (n + 31) // 32 * 32, d + 4
    return _tail(rows * ld * 4 + 2 * rows * np_ * 4, np_, rows)


def small_d_max(n):
    """largest d (a multiple of 4, at most 1024) whose small-kernel layout fits 224 KiB"""
    return max(d for d in range(4, 1025, 4) if small_layout_bytes(n, d) <= KIB224)


def mid_d_max(n):
    return max(d for d in range(4, 1025, 4) if mid_layout_bytes(n, d) <= KIB224)


# ---------------------------------------------------------------------------------------------------------
# the table
# ---------------------------------------------------------------------------------------------------------
def problem(n, d, dtype=F32, *, sim=COS, tau=0.07, topk=15, alpha=0.0, flags=0, n_rows=None):
    return Fn.make_problem(n, d, dtype, tau=tau, similarity=sim, topk=topk, alpha=alpha, flags=flags, n_rows=n_rows)


def expected(p, addr=ALIGNED, cluster=16):
    """the route map of the module docstring, written out independently of the C++"""
    f = p.flags
    whole = p.row_offset == 0 and p.n_rows == p.n_total
    mine = p.alpha != 0.0 and p.topk >= 1
    k_ok = not mine or p.topk <= 32 or p.topk >= p.n_total - 1
    single = not (f & (_cabi.FLAG_NO_SMALL | _cabi.FLAG_FORCE_TENSOR | _cabi.FLAG_MEMORY_COLUMNS))
    shape_ok = whole and p.d % 4 == 0 and p.d <= 1024 and addr % 16 == 0 and k_ok
    small_ok = shape_ok and p.n_total <= 160 and small_layout_bytes(p.n_total, p.d) <= KIB224
    tc = (not f & _cabi.FLAG_FORCE_EXACT and p.z_dtype == BF16 and p.d == 256 and p.tau >= 0.025
          and (p.similarity == GEO or f & (UNIT | _cabi.FLAG_FORCE_TENSOR))
          and not (p.alpha != 0.0 and p.topk > 32) and p.n_total >= 256)
    mid_ok = (shape_ok and not small_ok and p.n_total <= 320 and mid_layout_bytes(p.n_total, p.d) <= KIB224
              and not tc)
    if single and small_ok:
        fwd = SMALL
    elif single and mid_ok and cluster != 0:
        fwd = MID
    else:
        fwd = TENSOR if tc else TILED
    sums = bool(tc and p.similarity == COS and not mine and not f & _cabi.FLAG_NO_CLASS_SUMS
                and (p.n_rows * p.n_total >= 2**30 or f & _cabi.FLAG_CLASS_SUMS))
    return dict(loss_and_grad=fwd, forward_rows=TILED if fwd == SMALL and mine else fwd,
                backward_rows=TENSOR if tc else TILED,
                vec=int(p.d % 4 == 0 and addr % (8 if p.z_dtype == BF16 else 16) == 0),
                fwd_class_sums=int(sums), bwd_class_sums=int(sums and not f & _cabi.FLAG_MEMORY_COLUMNS))


def _check(p, addr=ALIGNED, **want):
    got = D.route(p, addr)
    exp = expected(p, addr, cluster=got["cluster"])
    exp.update(want)
    got.pop("cluster")
    assert got == exp, (p.n_total, p.d, p.z_dtype, p.flags, p.topk, p.alpha, addr)


def _routes(p, addr=ALIGNED):
    r = D.route(p, addr)
    return r["loss_and_grad"], r["backward_rows"]


# ---------------------------------------------------------------------------------------------------------
# the capacity edges, recomputed from the layouts
# ---------------------------------------------------------------------------------------------------------
def test_layout_edges_are_where_the_suite_puts_them():
    """tests/test_route_edges_gpu.py names these d edges; the layouts must still put them there"""
    assert [small_d_max(n) for n in (64, 128, 160, 32)] == [832, 368, 280, 1024]
    assert mid_d_max(320) == 1024
    assert small_layout_bytes(64, 836) > KIB224 >= mid_layout_bytes(64, 836)


@pytest.mark.parametrize("n", [2, 3, 8, 9, 31, 32, 33, 64, 100, 128, 159, 160])
def test_small_capacity_edge_in_d(n):
    dmax = small_d_max(n)
    assert _routes(problem(n, dmax)) == (SMALL, TILED)
    nxt = problem(n, dmax + 4)
    want = (MID if dmax + 4 <= 1024 else TILED, TILED)
    assert _routes(nxt) == want or D.route(nxt, ALIGNED)["cluster"] == 0
    _check(nxt)


@pytest.mark.parametrize("n,d,route", [
    (64, 832, SMALL), (64, 836, MID), (128, 368, SMALL), (128, 372, MID), (160, 280, SMALL), (160, 284, MID),
    (32, 1024, SMALL), (320, 1024, MID), (64, 1028, TILED), (320, 1028, TILED), (161, 1024, MID)])
def test_named_d_edges(n, d, route):
    p = problem(n, d)
    r = D.route(p, ALIGNED)
    if route == MID and r["cluster"] == 0:
        route = TILED
    assert (r["loss_and_grad"], r["forward_rows"], r["backward_rows"]) == (route, route, TILED)
    _check(p)


@pytest.mark.parametrize("n", [2, 3, 8, 9, 31, 32, 33, 159, 160, 161, 255, 256, 257, 319, 320, 321])
def test_n_edges_fp32_d256(n):
    want = SMALL if n <= 160 else MID if n <= 320 else TILED
    r = D.route(problem(n, 256), ALIGNED)
    if want == MID and r["cluster"] == 0:
        want = TILED
    assert r["loss_and_grad"] == want and r["backward_rows"] == TILED
    assert _routes(problem(n, 256, flags=_cabi.FLAG_NO_SMALL)) == (TILED, TILED)
    _check(problem(n, 256))


# ---------------------------------------------------------------------------------------------------------
# loads, alignment, mining depth
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [100, 300])
@pytest.mark.parametrize("d", [19, 255, 257])
def test_odd_d_takes_the_scalar_tiled_path(n, d):
    for dt in (F32, BF16):
        p = problem(n, d, dt)
        assert _routes(p) == (TILED, TILED)
        assert D.route(p, ALIGNED)["vec"] == 0
        _check(p)


@pytest.mark.parametrize("n", [100, 300])
def test_misaligned_z_takes_the_scalar_tiled_path(n):
    """z one element past a 16-byte boundary (a view buf[1:] of a flat buffer)"""
    for dt, elem in ((F32, 4), (BF16, 2)):
        p = problem(n, 252, dt)
        assert _routes(p, ALIGNED + elem) == (TILED, TILED)
        assert D.route(p, ALIGNED + elem)["vec"] == 0
        assert D.route(p, ALIGNED)["vec"] == 1
        _check(p, ALIGNED + elem)
    # bf16 rows need 8-byte alignment for vector loads, the single-launch kernels 16
    p = problem(100, 252, BF16)
    assert D.route(p, ALIGNED + 8)["vec"] == 1 and _routes(p, ALIGNED + 8) == (TILED, TILED)


def test_misaligned_bf16_at_a_tensor_shape_stays_on_the_tensor_path():
    """the tensor path's TMA descriptor rejects it: the call fails cleanly (tested on the device)"""
    p = problem(300, 256, BF16, flags=UNIT)
    assert _routes(p, ALIGNED + 2) == (TENSOR, TENSOR)


@pytest.mark.parametrize("n", [150, 300])
def test_mining_depth_moves_problems_off_and_back_onto_the_single_launch_kernels(n):
    single = SMALL if n <= 160 else MID
    for k, want in ((32, single), (33, TILED), (n - 2, TILED), (n - 1, single), (n + 5, single)):
        r = D.route(problem(n, 256, topk=k, alpha=0.5), ALIGNED)
        w = TILED if (want == MID and r["cluster"] == 0) else want
        assert r["loss_and_grad"] == w, (n, k)
        _check(problem(n, 256, topk=k, alpha=0.5))
    # without mining the list length does not matter
    assert D.route(problem(n, 256, topk=33, alpha=0.0), ALIGNED)["loss_and_grad"] in (single, TILED)
    _check(problem(n, 256, topk=33, alpha=0.0))


# ---------------------------------------------------------------------------------------------------------
# the tensor path
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [255, 256, 257, 383, 384, 385, 511, 512, 513])
def test_tensor_path_from_256_rows(n):
    p = problem(n, 256, BF16, flags=UNIT)
    want = (TENSOR, TENSOR) if n >= 256 else (MID, TILED)
    r = _routes(p)
    assert r == want or (n == 255 and r == (TILED, TILED) and D.route(p, ALIGNED)["cluster"] == 0)
    _check(p)
    assert _routes(problem(n, 256, F32, flags=UNIT))[1] == TILED


def test_tensor_path_eligibility_edges():
    def fb(**kw):
        return _routes(problem(300, 256, BF16, **kw))
    assert fb(tau=0.025, flags=UNIT) == (TENSOR, TENSOR)
    assert fb(tau=0.0249, flags=UNIT) == (MID, TILED) or fb(tau=0.0249, flags=UNIT) == (TILED, TILED)
    assert fb(sim=GEO) == (TENSOR, TENSOR)                           # geodesic needs no promise
    assert fb(sim=COS)[1] == TILED                                   # cosine without it: exact
    assert fb(sim=COS, flags=_cabi.FLAG_FORCE_TENSOR) == (TENSOR, TENSOR)
    assert fb(topk=32, alpha=0.5, flags=UNIT) == (TENSOR, TENSOR)
    assert fb(topk=33, alpha=0.5, flags=UNIT) == (TILED, TILED)       # K = 33 also leaves the mid kernel
    assert fb(topk=33, alpha=0.0, flags=UNIT) == (TENSOR, TENSOR)     # unmined: K is not used
    assert fb(flags=UNIT | _cabi.FLAG_FORCE_EXACT)[1] == TILED
    assert _routes(problem(300, 255, BF16, flags=UNIT)) == (TILED, TILED)
    for kw in (dict(tau=0.025, flags=UNIT), dict(tau=0.0249, flags=UNIT), dict(sim=GEO), dict(sim=COS),
               dict(topk=32, alpha=0.5, flags=UNIT), dict(topk=33, alpha=0.5, flags=UNIT),
               dict(flags=UNIT | _cabi.FLAG_FORCE_EXACT), dict(sim=COS, flags=_cabi.FLAG_FORCE_TENSOR)):
        _check(problem(300, 256, BF16, **kw))


@pytest.mark.parametrize("n,sums", [(32767, 0), (32768, 1), (65536, 1)])
def test_class_sums_switch_on_at_2_to_the_30_pairs(n, sums):
    r = D.route(problem(n, 256, BF16, flags=UNIT), ALIGNED)
    assert (r["loss_and_grad"], r["backward_rows"]) == (TENSOR, TENSOR)
    assert r["fwd_class_sums"] == r["bwd_class_sums"] == sums
    _check(problem(n, 256, BF16, flags=UNIT))


def test_class_sum_flags_and_their_exclusions():
    def sums(n=1024, **kw):
        r = D.route(problem(n, 256, BF16, **kw), ALIGNED)
        return r["fwd_class_sums"], r["bwd_class_sums"]
    assert sums(flags=UNIT) == (0, 0)
    assert sums(flags=UNIT | _cabi.FLAG_CLASS_SUMS) == (1, 1)
    assert sums(n=65536, flags=UNIT | _cabi.FLAG_NO_CLASS_SUMS) == (0, 0)
    assert sums(n=65536, flags=UNIT, topk=15, alpha=0.5) == (0, 0)     # mined
    assert sums(n=65536, flags=UNIT, topk=15, alpha=0.0) == (1, 1)     # K without mining
    assert sums(n=65536, sim=GEO) == (0, 0)                            # geodesic
    assert sums(n=65536, flags=UNIT | _cabi.FLAG_FORCE_EXACT) == (0, 0)
    # a memory backward never sums by class: memory columns carry no coefficient
    assert sums(n=65536, flags=UNIT | _cabi.FLAG_MEMORY_COLUMNS, n_rows=32768) == (1, 0)
    for kw in (dict(flags=UNIT), dict(flags=UNIT | _cabi.FLAG_CLASS_SUMS),
               dict(n=65536, flags=UNIT | _cabi.FLAG_NO_CLASS_SUMS), dict(n=65536, flags=UNIT, alpha=0.5),
               dict(n=65536, sim=GEO), dict(n=65536, flags=UNIT | _cabi.FLAG_MEMORY_COLUMNS, n_rows=32768)):
        n = kw.pop("n", 1024)
        _check(problem(n, 256, BF16, **kw))


# ---------------------------------------------------------------------------------------------------------
# flags
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [64, 160, 200, 320])
def test_flags_that_leave_the_single_launch_kernels(n):
    assert _routes(problem(n, 256, flags=_cabi.FLAG_NO_SMALL)) == (TILED, TILED)
    assert _routes(problem(n, 256, flags=_cabi.FLAG_FORCE_TENSOR)) == (TILED, TILED)   # fp32: the call fails
    assert _routes(problem(n, 256, flags=_cabi.FLAG_FORCE_EXACT))[0] in (SMALL, MID, TILED)
    # a memory problem never takes them, not even with an empty memory (n_rows == n_total)
    assert _routes(problem(n, 256, flags=_cabi.FLAG_MEMORY_COLUMNS)) == (TILED, TILED)
    assert _routes(problem(n, 256, flags=_cabi.FLAG_MEMORY_COLUMNS, n_rows=n // 2)) == (TILED, TILED)
    for f in (_cabi.FLAG_NO_SMALL, _cabi.FLAG_FORCE_TENSOR, _cabi.FLAG_FORCE_EXACT, _cabi.FLAG_MEMORY_COLUMNS, UNIT):
        _check(problem(n, 256, flags=f))
        _check(problem(n, 256, BF16, flags=f))


def test_memory_columns_on_the_tensor_path():
    p = problem(4096, 256, BF16, flags=UNIT | _cabi.FLAG_MEMORY_COLUMNS, n_rows=512)
    assert _routes(p) == (TENSOR, TENSOR)
    _check(p)


def test_unit_rows_small_bf16_batches_stay_exact():
    """the promise alone does not move a batch below 256 rows onto the tensor path"""
    for n in (64, 160, 255):
        assert _routes(problem(n, 256, BF16, flags=UNIT))[1] == TILED


def test_rows_of_a_shard_never_take_the_single_launch_kernels():
    p = Fn.make_problem(128, 256, F32, tau=0.07, similarity=COS, row_offset=64, n_rows=64)
    assert _routes(p) == (TILED, TILED)


@pytest.mark.parametrize("n", [2, 33, 64, 100, 128, 129, 160])
def test_mining_forward_rows_leaves_the_small_kernel(n):
    """supcon_loss_and_grad keeps the small kernel (its backward reuses the kernel's own Gram); a separate
    supcon_forward_rows with mining takes the tiled kernels, whose fma chain the tiled backward recomputes"""
    r = D.route(problem(n, 256, topk=5, alpha=0.5), ALIGNED)
    assert (r["loss_and_grad"], r["forward_rows"], r["backward_rows"]) == (SMALL, TILED, TILED)
    for kw in (dict(topk=5, alpha=0.0), dict(topk=0, alpha=0.5)):         # unmined: the small kernel
        r = D.route(problem(n, 256, **kw), ALIGNED)
        assert (r["loss_and_grad"], r["forward_rows"]) == (SMALL, SMALL)
    r = D.route(problem(200, 256, topk=5, alpha=0.5), ALIGNED)         # the mid kernel shares the tiled chain
    assert r["forward_rows"] == r["loss_and_grad"]


def test_cluster_slot_without_a_device():
    """-1 without a device; on one, 16 or 8 for a mid problem and 0 for any other"""
    import torch
    r = D.route(problem(200, 256), ALIGNED)["cluster"]
    if not torch.cuda.is_available():
        assert r == -1
    else:
        assert r in (16, 8)
        assert D.route(problem(64, 256), ALIGNED)["cluster"] == 0


def test_sweep_agrees_with_the_table():
    """a grid over every input of the table"""
    for n in (2, 33, 64, 128, 160, 161, 256, 300, 320, 321, 1024):
        for d in (19, 252, 256, 368, 372, 1024, 1028):
            for dt in (F32, BF16):
                for sim, flags in ((COS, 0), (COS, UNIT), (GEO, 0)):
                    for tau in (0.07, 0.0249):
                        for topk, alpha in ((15, 0.0), (32, 0.5), (33, 0.5), (n - 1, 0.5)):
                            for addr in (ALIGNED, ALIGNED + 4):
                                _check(problem(n, d, dt, sim=sim, tau=tau, topk=topk, alpha=alpha, flags=flags),
                                       addr)


def test_report_rejects_bad_arguments():
    out = (ctypes.c_int32 * 7)()
    p = problem(64, 256)
    assert D.load().supcon_debug_route(ctypes.byref(p), ctypes.c_void_p(ALIGNED), out, 6) == E_INVALID
    bad = problem(64, 256, n_rows=65)
    assert D.load().supcon_debug_route(ctypes.byref(bad), ctypes.c_void_p(ALIGNED), out, 7) == E_INVALID
