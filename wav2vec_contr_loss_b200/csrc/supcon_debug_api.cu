// TEST-ONLY entry points (libsupcon_b200_test.so; declared in csrc/supcon_debug.h, not in the public header):
// the tcgen05/TMA building-block diagnostic, host-side introspection of the tensor path's work distribution, of
// the exact path's column splits and top-K selection rounds, and of the route the dispatcher picks.
// The product library libsupcon_b200.so does not contain this file.
#include <string>

#include "supcon_debug.h"
#include "supcon_internal.h"

using namespace supcon;

namespace {
thread_local std::string g_dbg_err;
int dbg_fail(int code, const char* msg) {
  g_dbg_err = msg;
  return code;
}
int dbg_validate(const supcon_problem_t* p) {
  if (!p || p->n_total < 2 || p->d < 1 || p->n_rows < 1 || p->row_offset < 0 ||
      p->row_offset + p->n_rows > p->n_total || !(p->tau > 0.f))
    return dbg_fail(SUPCON_E_INVALID, "bad problem");
  return 0;
}
}  // namespace

extern "C" {

const char* supcon_debug_last_error(void) { return g_dbg_err.c_str(); }

int supcon_debug_tc_tile(const void* z_bf16, int32_t n, int32_t d, int32_t row_i, int32_t row_j, float* s_out,
                         float* o_out, void* stream) {
  if (!z_bf16 || !s_out || !o_out) return dbg_fail(SUPCON_E_INVALID, "NULL buffer passed to supcon_debug_tc_tile");
  const char* err = "";
  int rc = tc_debug_tile(z_bf16, n, d, row_i, row_j, s_out, o_out, reinterpret_cast<cudaStream_t>(stream), &err);
  if (rc) return dbg_fail(rc, err);
  return 0;
}

int supcon_debug_plan(const supcon_problem_t* p, int32_t* out, int32_t n_out) {
  if (int rc = dbg_validate(p)) return rc;
  if (!out || n_out < 1) return dbg_fail(SUPCON_E_INVALID, "bad arguments to supcon_debug_plan");
  if (!tc_supported(p)) return dbg_fail(SUPCON_E_UNSUPPORTED, "problem does not take the tensor path");
  return tc_debug_plan(p, out, n_out);
}

int supcon_debug_ffma_plan(const supcon_problem_t* p, int32_t* out, int32_t n_out) {
  if (int rc = dbg_validate(p)) return rc;
  if (!out || n_out < 4) return dbg_fail(SUPCON_E_INVALID, "bad arguments to supcon_debug_ffma_plan");
  const FfmaPlan pl = ffma_plan(p);
  const bool mine = p->alpha != 0.f && p->topk >= 1;
  out[0] = pl.fwd_splits;
  out[1] = pl.bwd_splits;
  out[2] = pl.kcap;
  out[3] = mine ? (p->topk + pl.kcap - 1) / pl.kcap : 0;
  return 0;
}

int supcon_debug_route(const supcon_problem_t* p, const void* z, int32_t* out, int32_t n_out) {
  if (int rc = dbg_validate(p)) return rc;
  if (!out || n_out < 7) return dbg_fail(SUPCON_E_INVALID, "bad arguments to supcon_debug_route");
  enum { SMALL = 0, MID = 1, TENSOR = 2, TILED = 3 };
  int devices = 0;
  if (cudaGetDeviceCount(&devices) != cudaSuccess) { cudaGetLastError(); devices = 0; }
  const bool mid = use_mid(p, z);
  int cluster = -1;
  if (devices > 0) {
    cluster = 0;
    if (mid) {   // the occupancy query of pick_cluster, for a problem the mid kernel can hold
      SmallArgs s{};
      s.n = p->n_total; s.d = p->d; s.z_dtype = p->z_dtype; s.dz_dtype = SUPCON_F32;
      cluster = mid_cluster_ctas(s);
    }
  }
  // forward of supcon_loss_and_grad and supcon_forward_rows (the single-launch kernels also do the former's backward)
  const int after_small = mid && cluster != 0 ? MID : use_tc(p, false) ? TENSOR : TILED;
  out[0] = use_small(p, z) ? SMALL : after_small;
  out[1] = use_small_forward_rows(p, z) ? SMALL : after_small;
  out[2] = use_tc(p, true) ? TENSOR : TILED;
  out[3] = cluster;
  out[4] = vec_ok(z, p) ? 1 : 0;
  out[5] = use_tc(p, false) && tc_class_sums(p, false, 0) ? 1 : 0;
  out[6] = use_tc(p, true) && tc_class_sums(p, true, 0) ? 1 : 0;
  return 0;
}

int supcon_debug_sched(int32_t col_tiles, int32_t ctas, int64_t units, int32_t cta, int32_t row_block,
                       int64_t* range_begin, int64_t* range_end, int32_t* first_cta, int32_t* last_cta) {
  if (col_tiles < 1 || ctas < 1 || units < ctas || cta < 0 || cta >= ctas || !range_begin || !range_end ||
      !first_cta || !last_cta)
    return dbg_fail(SUPCON_E_INVALID, "bad arguments to supcon_debug_sched");
  long long b = 0, e = 0;
  int f = 0, l = 0;
  tc_debug_sched(col_tiles, ctas, units, cta, row_block, &b, &e, &f, &l);
  *range_begin = b; *range_end = e; *first_cta = f; *last_cta = l;
  return 0;
}

}  // extern "C"
