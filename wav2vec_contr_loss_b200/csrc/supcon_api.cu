// C-ABI dispatcher of libsupcon_b200.so (see include/supcon_b200.h).
//
// Routes each call to one of the kernel families:
//   small  single-launch cluster kernel for small batches   (supcon_small.cu)
//   tc     bf16 tcgen05/TMEM/TMA flash-style kernels         (supcon_tc.cu)
//   ffma   exact fp32 CUDA-core kernels, any shape           (supcon_ffma.cu)
// plus the producer of z (supcon_head.cu) and the row normalisation either side of the loss.
// There is no CPU path: if no CUDA kernel can take the problem the call fails.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <type_traits>

#include "supcon_common.cuh"
#include "supcon_internal.h"

namespace supcon {
namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  g_err = std::string(what) + ": " + cudaGetErrorString(e);
  return (int)e;
}

int validate(const supcon_problem_t* p) {
  if (!p) return fail(SUPCON_E_INVALID, "problem is NULL");
  if (p->n_total < 2) return fail(SUPCON_E_INVALID, "n_total must be >= 2 (got %d)", p->n_total);
  if (p->d < 1) return fail(SUPCON_E_INVALID, "d must be >= 1 (got %d)", p->d);
  if (p->n_rows < 1 || p->row_offset < 0 || p->row_offset + p->n_rows > p->n_total)
    return fail(SUPCON_E_INVALID, "row block [%d, %d) outside [0, %d)", p->row_offset,
                p->row_offset + p->n_rows, p->n_total);
  if (p->z_dtype != SUPCON_F32 && p->z_dtype != SUPCON_BF16)
    return fail(SUPCON_E_INVALID, "unknown z_dtype %d", p->z_dtype);
  if (p->similarity != SUPCON_COSINE && p->similarity != SUPCON_GEODESIC)
    return fail(SUPCON_E_INVALID, "Unknown similarity: %d", p->similarity);
  if (!(p->tau > 0.f)) return fail(SUPCON_E_INVALID, "tau must be > 0");
  if (p->flags & SUPCON_FLAG_MEMORY_COLUMNS) {
    if (p->row_offset != 0)
      return fail(SUPCON_E_INVALID, "SUPCON_FLAG_MEMORY_COLUMNS needs row_offset == 0 (got %d)", p->row_offset);
    // the tensor path masks memory columns out of the uniformity sums through exp(-t * inf) == 0
    if (p->lambda_uni > 0.f && !(p->uni_t > 0.f))
      return fail(SUPCON_E_INVALID, "SUPCON_FLAG_MEMORY_COLUMNS with lambda_uni > 0 needs uni_t > 0");
  }
  return 0;
}

// the rank owns every anchor: a whole batch, or a batch contrasted against a memory of earlier batches
bool owns_all_anchors(const supcon_problem_t* p) {
  return p->row_offset == 0 && (p->n_rows == p->n_total || (p->flags & SUPCON_FLAG_MEMORY_COLUMNS));
}

constexpr uint32_t FLAG_TC_FWD_ONLY = SUPCON_FLAG_DEBUG_TC_FWD_ONLY, FLAG_TC_BWD_ONLY = SUPCON_FLAG_DEBUG_TC_BWD_ONLY;

size_t workspace_need(const supcon_problem_t* p) {
  size_t need = ffma_workspace_bytes(p);
  if (!(p->flags & SUPCON_FLAG_FORCE_EXACT) && tc_supported(p)) {
    size_t t = tc_plan(p).total_bytes;
    if (t > need) need = t;
  }
  return need;
}

bool needs_mining(const supcon_problem_t* p) { return p->alpha != 0.f && p->topk >= 1; }

// A memory problem (SUPCON_FLAG_MEMORY_COLUMNS) never takes the single-launch kernels, not even with an empty memory
// (n_rows == n_total): its forward and backward are separate calls, and the backward's hard-negative membership test
// (s == thr) needs the forward's Gram arithmetic, which the small / mid kernels do not share with the tiled ones.
constexpr uint32_t NOT_SINGLE_LAUNCH = SUPCON_FLAG_NO_SMALL | SUPCON_FLAG_FORCE_TENSOR | SUPCON_FLAG_MEMORY_COLUMNS;

SmallArgs make_small(const supcon_problem_t* p, const void* z, const int32_t* labels) {
  SmallArgs s;
  memset(&s, 0, sizeof(s));
  s.z = z; s.labels = labels;
  s.n = p->n_total; s.d = p->d; s.z_dtype = p->z_dtype; s.dz_dtype = SUPCON_F32; s.similarity = p->similarity;
  s.topk = p->topk < 0 ? 0 : p->topk; s.mine = needs_mining(p) ? 1 : 0;
  s.tau = p->tau; s.alpha = p->alpha; s.lambda_uni = p->lambda_uni; s.uni_t = p->uni_t;
  return s;
}

FfmaArgs make_ffma(const supcon_problem_t* p, const void* z, const int32_t* labels, void* ws, bool backward = false,
                   bool use_plan = true) {
  FfmaArgs a;
  memset(&a, 0, sizeof(a));
  a.z = z; a.labels = labels;
  a.splits = 1; a.col_tiles = (p->n_total + 63) / 64; a.rows_pad = (p->n_rows + 63) / 64 * 64;
  if (use_plan && ws) ffma_bind_plan(a, ffma_plan(p), ws, backward);
  a.n_total = p->n_total; a.row_offset = p->row_offset; a.n_rows = p->n_rows; a.d = p->d;
  a.n_batch = batch_columns(p);
  a.z_dtype = p->z_dtype; a.similarity = p->similarity; a.topk = p->topk < 0 ? 0 : p->topk;
  a.mine = needs_mining(p) ? 1 : 0;
  int cap = ffma_kcap();
  a.kcap = a.mine ? (a.topk < cap ? a.topk : cap) : 0;
  a.vec_ok = vec_ok(z, p) ? 1 : 0;
  a.tau = p->tau; a.alpha = p->alpha; a.lambda_uni = p->lambda_uni; a.uni_t = p->uni_t;
  return a;
}

__global__ void finalize_kernel(const double* pg, float* loss_out, int n_batch, float tau, float alpha,
                                float lambda_uni, float uni_t) {
  if (threadIdx.x == 0 && blockIdx.x == 0)
    *loss_out = global_coef(pg, n_batch, tau, alpha, lambda_uni, uni_t).loss;
}

// sums the per-rank partial sums in rank order (deterministic, identical on every rank) and writes the loss.
// Slots SUPCON_P_GCNT_* / SUPCON_P_FIXMAX are global quantities every rank derived identically: copied, not summed.
__global__ void finalize_sets_kernel(const double* sets, int n_sets, double* partials_out, float* loss_out,
                                     int n_batch, float tau, float alpha, float lambda_uni, float uni_t) {
  __shared__ double pg[SUPCON_N_PARTIALS];
  const int k = threadIdx.x;
  if (k < SUPCON_N_PARTIALS) {
    double s = sets[k];
    if (k <= SUPCON_P_SUM_W)
      for (int r = 1; r < n_sets; ++r) s += sets[(int64_t)r * SUPCON_N_PARTIALS + k];
    pg[k] = s;
    partials_out[k] = s;
  }
  __syncthreads();
  if (k == 0 && loss_out) *loss_out = global_coef(pg, n_batch, tau, alpha, lambda_uni, uni_t).loss;
}

// ---- labels of any width -> int32 class keys: equal labels <-> equal keys (loss.py:123 compares with ==) ----
// int64 values outside int32 and float64 values that float32 cannot hold exactly cannot be keyed losslessly in 32
// bits: the kernel reports the row and traps (a loud device-side fault) instead of silently merging two classes.
// NaN never equals anything in the reference: every NaN row gets a key of its own.
template <typename T>
__global__ void label_keys_kernel(const T* __restrict__ in, int n, int32_t* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const T v = in[i];
  if constexpr (sizeof(T) == 8 && !std::is_floating_point<T>::value) {          // int64
    if (v != (T)(int32_t)v) {
      printf("supcon: integer label %lld (row %d) does not fit 32 bits; relabel the classes densely\n", (long long)v, i);
      __trap();
    }
    out[i] = (int32_t)v;
  } else {                                                                        // float32 / float64
    float f = (float)v;
    if constexpr (sizeof(T) == 8) {
      if (v == v && (double)f != (double)v) {
        printf("supcon: float64 label %.17g (row %d) is not exactly a float32; relabel the classes\n", (double)v, i);
        __trap();
      }
    }
    if (f != f) out[i] = 0x7fc00000 | (i & 0x3fffff);     // NaN: matches no other row
    else out[i] = __float_as_int(f + 0.0f);               // -0.0 == +0.0
  }
}

// ---- row L2 normalisation (stage1_utils.py:123,149): one warp per row ----
template <typename TO>
__global__ void normalize_fwd_kernel(const float* __restrict__ x, int n, int d, TO* __restrict__ z,
                                     float* __restrict__ norms) {
  int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (row >= n) return;
  const float* xr = x + (int64_t)row * d;
  float s = 0.f;
  for (int k = lane; k < d; k += 32) { float v = __ldg(xr + k); s = fmaf(v, v, s); }
  s = warp_sum(s);
  float nrm = fmaxf(sqrtf(s), 1e-12f);
  if (lane == 0 && norms) norms[row] = nrm;
  for (int k = lane; k < d; k += 32) {
    float v = __fdiv_rn(__ldg(xr + k), nrm);
    if constexpr (sizeof(TO) == 4) z[(int64_t)row * d + k] = v;
    else z[(int64_t)row * d + k] = __float2bfloat16(v);
  }
}

template <typename TZ, typename TG>
__global__ void normalize_bwd_kernel(const TZ* __restrict__ z, const float* __restrict__ norms,
                                     const TG* __restrict__ dz, int n, int d, float* __restrict__ dx) {
  int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  int lane = threadIdx.x & 31;
  if (row >= n) return;
  const TZ* zr = z + (int64_t)row * d;
  const TG* gr = dz + (int64_t)row * d;
  float s = 0.f;
  for (int k = lane; k < d; k += 32) s = fmaf(ld_elem<TZ>(zr + k), ld_elem<TG>(gr + k), s);
  s = warp_sum(s);
  float inv = __fdiv_rn(1.0f, norms[row]);
  for (int k = lane; k < d; k += 32)
    dx[(int64_t)row * d + k] = (ld_elem<TG>(gr + k) - ld_elem<TZ>(zr + k) * s) * inv;
}

}  // namespace

// ---- route predicates (declared in supcon_internal.h: the test library's route report calls these same ones) ----
bool use_tc(const supcon_problem_t* p, bool backward) {
  if (p->flags & SUPCON_FLAG_FORCE_EXACT) return false;
  if (!tc_supported(p)) return false;
  if (backward && (p->flags & FLAG_TC_FWD_ONLY)) return false;
  if (!backward && (p->flags & FLAG_TC_BWD_ONLY)) return false;
  return true;
}

bool vec_ok(const void* z, const supcon_problem_t* p) {
  size_t al = p->z_dtype == SUPCON_BF16 ? 8 : 16;
  return (p->d % 4 == 0) && ((reinterpret_cast<uintptr_t>(z) % al) == 0);
}

bool use_small(const supcon_problem_t* p, const void* z) {
  if (p->flags & NOT_SINGLE_LAUNCH) return false;
  return small_supported(p, z);
}
// supcon_forward_rows' statistics feed a supcon_backward_rows on the tiled kernels, whose hard-negative membership test
// (s > thr || s == thr && j <= thr_idx) recomputes s as one fma chain over k.  Below 129 rows the small kernel sums
// each dot product from 2 or 4 k-slices, so its threshold can differ from the tiled s in the last bit and drop the K-th
// negative from the backward's set: a mining forward there runs on the tiled kernels.  (The mid kernel's chain is the
// tiled kernels' own; supcon_loss_and_grad's small-kernel backward reuses its own Gram.)
bool use_small_forward_rows(const supcon_problem_t* p, const void* z) {
  return use_small(p, z) && !needs_mining(p);
}
// mid-size single-launch kernel: exact fp32 math, so it yields to the tensor path where that one is eligible
bool use_mid(const supcon_problem_t* p, const void* z) {
  if (p->flags & NOT_SINGLE_LAUNCH) return false;
  if (use_tc(p, false) || use_tc(p, true)) return false;
  return !small_supported(p, z) && mid_supported(p, z);
}

}  // namespace supcon

using namespace supcon;

extern "C" {

int supcon_abi_version(void) { return SUPCON_ABI_VERSION; }
const char* supcon_last_error(void) { return g_err.c_str(); }

int supcon_workspace_bytes(const supcon_problem_t* p, size_t* bytes_out) {
  if (int rc = validate(p)) return rc;
  if (!bytes_out) return fail(SUPCON_E_INVALID, "bytes_out is NULL");
  *bytes_out = workspace_need(p);
  return 0;
}

}  // extern "C"

namespace {
// supcon_forward_rows (mem_filled == NULL) and supcon_forward_rows_memory: the plan, the workspace and the route
// depend on the problem alone, never on the device fill level, so one captured graph serves every fill level
int forward_rows(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all, const int32_t* mem_filled,
                 float* row_stats, double* partials, float* loss_out, void* workspace, size_t workspace_bytes,
                 void* stream, const char* who) {
  if (!z_all || !labels_all || !row_stats || !partials || !workspace)
    return fail(SUPCON_E_INVALID, "NULL buffer passed to %s", who);
  if (workspace_bytes < workspace_need(p))
    return fail(SUPCON_E_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, workspace_need(p));
  if ((p->flags & SUPCON_FLAG_FORCE_TENSOR) && !tc_supported(p))
    return fail(SUPCON_E_UNSUPPORTED, "tensor-core path needs bf16 z, d == 256, tau >= 0.025, N >= 256, top-K <= 32");
  if (loss_out && !owns_all_anchors(p))
    return fail(SUPCON_E_INVALID, "loss_out needs a rank that owns every row; use supcon_finalize");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (use_small_forward_rows(p, z_all)) {   // whole batch on this rank, small N: one launch, statistics + loss only
    SmallArgs s = make_small(p, z_all, labels_all);
    s.row_stats = row_stats; s.partials = partials; s.loss_out = loss_out;
    cudaError_t es = small_launch(s, st);
    if (es != cudaSuccess) return cuda_fail(es, "small_launch");
    return 0;
  }
  if (use_mid(p, z_all)) {     // 160 < N <= 512: one cluster launch instead of the tiled kernels
    SmallArgs s = make_small(p, z_all, labels_all);
    s.row_stats = row_stats; s.partials = partials; s.loss_out = loss_out;
    bool taken = false;
    cudaError_t es = mid_launch(s, st, &taken);
    if (es != cudaSuccess) return cuda_fail(es, "mid_launch");
    if (taken) return 0;
  }
  if (use_tc(p, false)) {
    const char* err = "";
    int rc = tc_forward(p, z_all, labels_all, row_stats, partials, loss_out, workspace, st, &err, 0, mem_filled);
    if (rc) return fail(rc, "tc_forward: %s", err);
    return 0;
  }
  cudaError_t e = cudaMemsetAsync(workspace, 0, 256, st);
  if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(workspace)");
  FfmaArgs a = make_ffma(p, z_all, labels_all, workspace);
  a.row_stats = row_stats; a.partials = partials; a.loss_out = loss_out; a.mem_filled = mem_filled;
  e = ffma_forward(a, st);
  if (e != cudaSuccess) return cuda_fail(e, "ffma_forward");
  return 0;
}
}  // namespace

extern "C" {

int supcon_forward_rows(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                        float* row_stats, double* partials, float* loss_out, void* workspace,
                        size_t workspace_bytes, void* stream) {
  if (int rc = validate(p)) return rc;
  return forward_rows(p, z_all, labels_all, nullptr, row_stats, partials, loss_out, workspace, workspace_bytes,
                      stream, "supcon_forward_rows");
}

int supcon_forward_rows_memory(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                               const int32_t* mem_filled, float* row_stats, double* partials, float* loss_out,
                               void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = validate(p)) return rc;
  if (!(p->flags & SUPCON_FLAG_MEMORY_COLUMNS))
    return fail(SUPCON_E_INVALID, "supcon_forward_rows_memory needs SUPCON_FLAG_MEMORY_COLUMNS");
  return forward_rows(p, z_all, labels_all, mem_filled, row_stats, partials, loss_out, workspace, workspace_bytes,
                      stream, "supcon_forward_rows_memory");
}

int supcon_forward_rows_local(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                              void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = validate(p)) return rc;
  if (!z_all || !labels_all || !workspace) return fail(SUPCON_E_INVALID, "NULL buffer passed to supcon_forward_rows_local");
  if (workspace_bytes < workspace_need(p))
    return fail(SUPCON_E_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, workspace_need(p));
  if (!(use_tc(p, false) && tc_two_phase(p))) return 0;   // nothing to pre-compute: the second call does everything
  const char* err = "";
  int rc = tc_forward(p, z_all, labels_all, nullptr, nullptr, nullptr, workspace, reinterpret_cast<cudaStream_t>(stream),
                      &err, 1);
  if (rc) return fail(rc, "tc_forward(local columns): %s", err);
  return 0;
}

int supcon_forward_rows_remote(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                               float* row_stats, double* partials, void* workspace, size_t workspace_bytes,
                               void* stream) {
  if (int rc = validate(p)) return rc;
  if (!(use_tc(p, false) && tc_two_phase(p)))
    return supcon_forward_rows(p, z_all, labels_all, row_stats, partials, nullptr, workspace, workspace_bytes, stream);
  if (!z_all || !labels_all || !row_stats || !partials || !workspace)
    return fail(SUPCON_E_INVALID, "NULL buffer passed to supcon_forward_rows_remote");
  if (workspace_bytes < workspace_need(p))
    return fail(SUPCON_E_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, workspace_need(p));
  const char* err = "";
  int rc = tc_forward(p, z_all, labels_all, row_stats, partials, nullptr, workspace,
                      reinterpret_cast<cudaStream_t>(stream), &err, 2);
  if (rc) return fail(rc, "tc_forward(remote columns): %s", err);
  return 0;
}

int supcon_finalize(const supcon_problem_t* p, const double* partials_global, float* loss_out,
                    void* stream) {
  if (int rc = validate(p)) return rc;
  if (!partials_global || !loss_out) return fail(SUPCON_E_INVALID, "NULL buffer passed to supcon_finalize");
  finalize_kernel<<<1, 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      partials_global, loss_out, batch_columns(p), p->tau, p->alpha, p->lambda_uni, p->uni_t);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "finalize_kernel");
  return 0;
}

int supcon_finalize_sets(const supcon_problem_t* p, const double* partial_sets, int32_t n_sets,
                         double* partials_out, float* loss_out, void* stream) {
  if (int rc = validate(p)) return rc;
  if (!partial_sets || !partials_out || n_sets < 1)
    return fail(SUPCON_E_INVALID, "bad arguments to supcon_finalize_sets");
  if ((p->flags & SUPCON_FLAG_MEMORY_COLUMNS) && n_sets > 1)
    return fail(SUPCON_E_UNSUPPORTED, "SUPCON_FLAG_MEMORY_COLUMNS is single-rank: n_sets must be 1 (got %d)", n_sets);
  finalize_sets_kernel<<<1, 32, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      partial_sets, n_sets, partials_out, loss_out, batch_columns(p), p->tau, p->alpha, p->lambda_uni, p->uni_t);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "finalize_sets_kernel");
  return 0;
}

int supcon_backward_rows_local(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                               const float* stats_local, const double* partials_local, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (int rc = validate(p)) return rc;
  if (!(use_tc(p, true) && use_tc(p, false) && tc_bwd_two_phase(p))) return 0;   // _remote does everything
  if (!z_all || !labels_all || !stats_local || !partials_local || !workspace)
    return fail(SUPCON_E_INVALID, "NULL buffer passed to supcon_backward_rows_local");
  if (workspace_bytes < workspace_need(p))
    return fail(SUPCON_E_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, workspace_need(p));
  const char* err = "";
  int rc = tc_backward(p, z_all, labels_all, stats_local, partials_local, nullptr, nullptr, SUPCON_F32, workspace,
                       reinterpret_cast<cudaStream_t>(stream), &err, 1);
  if (rc) return fail(rc, "tc_backward(local columns): %s", err);
  return 0;
}

int supcon_backward_rows_remote(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                                const float* stats_all, const double* partials_global, const float* grad_out,
                                void* dz_out, int32_t dz_dtype, void* workspace, size_t workspace_bytes,
                                void* stream) {
  if (int rc = validate(p)) return rc;
  if (!(use_tc(p, true) && use_tc(p, false) && tc_bwd_two_phase(p)))
    return supcon_backward_rows(p, z_all, labels_all, stats_all, partials_global, grad_out, dz_out, dz_dtype,
                                workspace, workspace_bytes, stream);
  if (!z_all || !labels_all || !stats_all || !partials_global || !dz_out || !workspace)
    return fail(SUPCON_E_INVALID, "NULL buffer passed to supcon_backward_rows_remote");
  if (dz_dtype != SUPCON_F32 && dz_dtype != SUPCON_BF16)
    return fail(SUPCON_E_INVALID, "unknown dz_dtype %d", dz_dtype);
  if (workspace_bytes < workspace_need(p))
    return fail(SUPCON_E_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, workspace_need(p));
  const char* err = "";
  int rc = tc_backward(p, z_all, labels_all, stats_all, partials_global, grad_out, dz_out, dz_dtype, workspace,
                       reinterpret_cast<cudaStream_t>(stream), &err, 2);
  if (rc) return fail(rc, "tc_backward(remote columns): %s", err);
  return 0;
}

}  // extern "C"

namespace {
// supcon_backward_rows (mem_filled == NULL) and supcon_backward_rows_memory
int backward_rows(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all, const int32_t* mem_filled,
                  const float* stats_all, const double* partials_global, const float* grad_out, void* dz_out,
                  int32_t dz_dtype, void* workspace, size_t workspace_bytes, void* stream, const char* who) {
  if (!z_all || !labels_all || !stats_all || !partials_global || !dz_out)
    return fail(SUPCON_E_INVALID, "NULL buffer passed to %s", who);
  if (dz_dtype != SUPCON_F32 && dz_dtype != SUPCON_BF16)
    return fail(SUPCON_E_INVALID, "unknown dz_dtype %d", dz_dtype);
  if (use_tc(p, true)) {
    if (!workspace || workspace_bytes < workspace_need(p))
      return fail(SUPCON_E_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, workspace_need(p));
    const char* err = "";
    int rc = tc_backward(p, z_all, labels_all, stats_all, partials_global, grad_out, dz_out, dz_dtype, workspace,
                         reinterpret_cast<cudaStream_t>(stream), &err, 0, mem_filled);
    if (rc) return fail(rc, "tc_backward: %s", err);
    return 0;
  }
  if (!workspace || workspace_bytes < workspace_need(p))
    return fail(SUPCON_E_WORKSPACE, "workspace too small: %zu < %zu", workspace_bytes, workspace_need(p));
  FfmaArgs a = make_ffma(p, z_all, labels_all, workspace, /*backward=*/true);
  a.stats_all = stats_all;
  a.partials = const_cast<double*>(partials_global);
  a.grad_out = grad_out; a.dz_out = dz_out; a.mem_filled = mem_filled;
  cudaError_t e = ffma_backward(a, dz_dtype, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "ffma_backward");
  return 0;
}
}  // namespace

extern "C" {

int supcon_backward_rows(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                         const float* stats_all, const double* partials_global, const float* grad_out,
                         void* dz_out, int32_t dz_dtype, void* workspace, size_t workspace_bytes,
                         void* stream) {
  if (int rc = validate(p)) return rc;
  return backward_rows(p, z_all, labels_all, nullptr, stats_all, partials_global, grad_out, dz_out, dz_dtype,
                       workspace, workspace_bytes, stream, "supcon_backward_rows");
}

int supcon_backward_rows_memory(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                                const int32_t* mem_filled, const float* stats_all, const double* partials_global,
                                const float* grad_out, void* dz_out, int32_t dz_dtype, void* workspace,
                                size_t workspace_bytes, void* stream) {
  if (int rc = validate(p)) return rc;
  if (!(p->flags & SUPCON_FLAG_MEMORY_COLUMNS))
    return fail(SUPCON_E_INVALID, "supcon_backward_rows_memory needs SUPCON_FLAG_MEMORY_COLUMNS");
  return backward_rows(p, z_all, labels_all, mem_filled, stats_all, partials_global, grad_out, dz_out, dz_dtype,
                       workspace, workspace_bytes, stream, "supcon_backward_rows_memory");
}

int supcon_loss_and_grad(const supcon_problem_t* p, const void* z, const int32_t* labels, float* loss_out,
                         void* dz_out, int32_t dz_dtype, float* row_stats, double* partials,
                         void* workspace, size_t workspace_bytes, void* stream) {
  if (int rc = validate(p)) return rc;
  if (!owns_all_anchors(p))
    return fail(SUPCON_E_INVALID, "supcon_loss_and_grad needs the whole batch on one rank");
  if (!loss_out) return fail(SUPCON_E_INVALID, "loss_out is NULL");
  if (!z || !labels) return fail(SUPCON_E_INVALID, "NULL buffer passed to supcon_loss_and_grad");
  if (dz_out && dz_dtype != SUPCON_F32 && dz_dtype != SUPCON_BF16)
    return fail(SUPCON_E_INVALID, "unknown dz_dtype %d", dz_dtype);
  if (use_small(p, z)) {   // forward AND backward in a single cluster launch
    SmallArgs s = make_small(p, z, labels);
    s.row_stats = row_stats; s.partials = partials; s.loss_out = loss_out; s.dz_out = dz_out; s.dz_dtype = dz_dtype;
    cudaError_t es = small_launch(s, reinterpret_cast<cudaStream_t>(stream));
    if (es != cudaSuccess) return cuda_fail(es, "small_launch");
    return 0;
  }
  if (use_mid(p, z)) {     // forward AND backward of a mid-size batch in a single cluster launch
    SmallArgs s = make_small(p, z, labels);
    s.row_stats = row_stats; s.partials = partials; s.loss_out = loss_out; s.dz_out = dz_out; s.dz_dtype = dz_dtype;
    bool taken = false;
    cudaError_t es = mid_launch(s, reinterpret_cast<cudaStream_t>(stream), &taken);
    if (es != cudaSuccess) return cuda_fail(es, "mid_launch");
    if (taken) return 0;
  }
  int rc = supcon_forward_rows(p, z, labels, row_stats, partials, loss_out, workspace, workspace_bytes, stream);
  if (rc) return rc;
  if (dz_out)
    rc = supcon_backward_rows(p, z, labels, row_stats, partials, nullptr, dz_out, dz_dtype, workspace,
                              workspace_bytes, stream);
  return rc;
}

int supcon_label_keys(const void* labels, int32_t dtype, int32_t n, int32_t* keys_out, void* stream) {
  if (!labels || !keys_out || n < 1) return fail(SUPCON_E_INVALID, "bad arguments to supcon_label_keys");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int blocks = (n + 255) / 256;
  if (dtype == SUPCON_LABEL_I64) label_keys_kernel<long long><<<blocks, 256, 0, st>>>((const long long*)labels, n, keys_out);
  else if (dtype == SUPCON_LABEL_F32) label_keys_kernel<float><<<blocks, 256, 0, st>>>((const float*)labels, n, keys_out);
  else if (dtype == SUPCON_LABEL_F64) label_keys_kernel<double><<<blocks, 256, 0, st>>>((const double*)labels, n, keys_out);
  else return fail(SUPCON_E_INVALID, "unknown label dtype %d", dtype);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "label_keys_kernel");
  return 0;
}

int supcon_normalize_forward(const float* x, int32_t n, int32_t d, void* z_out, int32_t z_dtype,
                             float* norms_out, void* stream) {
  if (!x || !z_out || n < 1 || d < 1) return fail(SUPCON_E_INVALID, "bad arguments to supcon_normalize_forward");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int wpb = 8, blocks = (n + wpb - 1) / wpb;
  if (z_dtype == SUPCON_BF16)
    normalize_fwd_kernel<__nv_bfloat16><<<blocks, wpb * 32, 0, st>>>(x, n, d, (__nv_bfloat16*)z_out, norms_out);
  else if (z_dtype == SUPCON_F32)
    normalize_fwd_kernel<float><<<blocks, wpb * 32, 0, st>>>(x, n, d, (float*)z_out, norms_out);
  else return fail(SUPCON_E_INVALID, "unknown z_dtype %d", z_dtype);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "normalize_fwd_kernel");
  return 0;
}

int supcon_normalize_backward(const void* z, int32_t z_dtype, const float* norms, const void* dz,
                              int32_t dz_dtype, int32_t n, int32_t d, float* dx_out, void* stream) {
  if (!z || !norms || !dz || !dx_out || n < 1 || d < 1)
    return fail(SUPCON_E_INVALID, "bad arguments to supcon_normalize_backward");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int wpb = 8, blocks = (n + wpb - 1) / wpb;
  typedef __nv_bfloat16 bf;
  if (z_dtype == SUPCON_F32 && dz_dtype == SUPCON_F32)
    normalize_bwd_kernel<float, float><<<blocks, wpb * 32, 0, st>>>((const float*)z, norms, (const float*)dz, n, d, dx_out);
  else if (z_dtype == SUPCON_BF16 && dz_dtype == SUPCON_F32)
    normalize_bwd_kernel<bf, float><<<blocks, wpb * 32, 0, st>>>((const bf*)z, norms, (const float*)dz, n, d, dx_out);
  else if (z_dtype == SUPCON_F32 && dz_dtype == SUPCON_BF16)
    normalize_bwd_kernel<float, bf><<<blocks, wpb * 32, 0, st>>>((const float*)z, norms, (const bf*)dz, n, d, dx_out);
  else if (z_dtype == SUPCON_BF16 && dz_dtype == SUPCON_BF16)
    normalize_bwd_kernel<bf, bf><<<blocks, wpb * 32, 0, st>>>((const bf*)z, norms, (const bf*)dz, n, d, dx_out);
  else return fail(SUPCON_E_INVALID, "unknown dtype");
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return cuda_fail(e, "normalize_bwd_kernel");
  return 0;
}

static int head_pool_check(const void* hs, int32_t hs_dtype, int32_t batch, int32_t layers, int32_t feat,
                           int32_t frames, float dropout_p, const void* out, const char* who) {
  if (!hs || !out) return fail(SUPCON_E_INVALID, "NULL buffer passed to %s", who);
  if (hs_dtype != SUPCON_F32 && hs_dtype != SUPCON_BF16)
    return fail(SUPCON_E_INVALID, "%s: unknown hs_dtype %d (SUPCON_F32 or SUPCON_BF16)", who, hs_dtype);
  if (batch < 1 || layers < 1 || feat < 1 || frames < 1)
    return fail(SUPCON_E_INVALID, "%s: bad shape (%d, %d, %d, %d)", who, batch, layers, feat, frames);
  if (batch > 65535) return fail(SUPCON_E_UNSUPPORTED, "%s: batch %d > 65535", who, batch);
  if (!(dropout_p >= 0.f && dropout_p < 1.f)) return fail(SUPCON_E_INVALID, "%s: dropout_p must be in [0, 1)", who);
  if (head_pool_rows_per_block(feat, frames, hs_dtype) < 1)
    return fail(SUPCON_E_UNSUPPORTED, "%s: %d frames exceed the 12288 a block can stage", who, frames);
  return 0;
}

static int head_pool_fwd(const void* hs, int32_t hs_dtype, int32_t batch, int32_t layers, int32_t feat,
                         int32_t frames, float dropout_p, float negative_slope, const uint64_t* rng_state,
                         float* pooled_out, void* stream, const char* who) {
  if (int rc = head_pool_check(hs, hs_dtype, batch, layers, feat, frames, dropout_p, pooled_out, who)) return rc;
  HeadPoolArgs a{};
  a.hs = hs; a.hs_dtype = hs_dtype; a.pooled = pooled_out;
  a.rng_state = reinterpret_cast<const unsigned long long*>(rng_state);
  a.B = batch; a.K = layers; a.F = feat; a.T = frames;
  a.dropout_p = dropout_p; a.negative_slope = negative_slope;
  cudaError_t e = head_pool_forward(a, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "head_pool_fwd_kernel");
  return 0;
}

static int head_pool_bwd(const void* hs, int32_t hs_dtype, int32_t batch, int32_t layers, int32_t feat,
                         int32_t frames, float dropout_p, float negative_slope, const uint64_t* rng_state,
                         const float* dpooled, void* dhs_out, void* stream, const char* who) {
  if (int rc = head_pool_check(hs, hs_dtype, batch, layers, feat, frames, dropout_p, dhs_out, who)) return rc;
  if (!dpooled) return fail(SUPCON_E_INVALID, "NULL dpooled passed to %s", who);
  HeadPoolArgs a{};
  a.hs = hs; a.hs_dtype = hs_dtype; a.pooled = nullptr;
  a.rng_state = reinterpret_cast<const unsigned long long*>(rng_state);
  a.B = batch; a.K = layers; a.F = feat; a.T = frames;
  a.dropout_p = dropout_p; a.negative_slope = negative_slope;
  cudaError_t e = head_pool_backward(a, dpooled, dhs_out, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "head_pool_bwd_kernel");
  return 0;
}

int supcon_head_pool_forward_typed(const void* hs, int32_t hs_dtype, int32_t batch, int32_t layers, int32_t feat,
                                   int32_t frames, float dropout_p, float negative_slope, const uint64_t* rng_state,
                                   float* pooled_out, void* stream) {
  return head_pool_fwd(hs, hs_dtype, batch, layers, feat, frames, dropout_p, negative_slope, rng_state, pooled_out,
                       stream, "supcon_head_pool_forward_typed");
}

int supcon_head_pool_backward_typed(const void* hs, int32_t hs_dtype, int32_t batch, int32_t layers, int32_t feat,
                                    int32_t frames, float dropout_p, float negative_slope, const uint64_t* rng_state,
                                    const float* dpooled, void* dhs_out, void* stream) {
  return head_pool_bwd(hs, hs_dtype, batch, layers, feat, frames, dropout_p, negative_slope, rng_state, dpooled,
                       dhs_out, stream, "supcon_head_pool_backward_typed");
}

int supcon_head_pool_forward(const float* hs, int32_t batch, int32_t layers, int32_t feat, int32_t frames,
                             float dropout_p, float negative_slope, const uint64_t* rng_state, float* pooled_out,
                             void* stream) {
  return head_pool_fwd(hs, SUPCON_F32, batch, layers, feat, frames, dropout_p, negative_slope, rng_state, pooled_out,
                       stream, "supcon_head_pool_forward");
}

int supcon_head_pool_backward(const float* hs, int32_t batch, int32_t layers, int32_t feat, int32_t frames,
                              float dropout_p, float negative_slope, const uint64_t* rng_state,
                              const float* dpooled, float* dhs_out, void* stream) {
  return head_pool_bwd(hs, SUPCON_F32, batch, layers, feat, frames, dropout_p, negative_slope, rng_state, dpooled,
                       dhs_out, stream, "supcon_head_pool_backward");
}

int supcon_head_layer_mean_typed(const void* hs, int32_t hs_dtype, int32_t batch, int32_t layers, int32_t feat,
                                 int32_t frames, float* store_rows, void* stream) {
  const char* who = "supcon_head_layer_mean_typed";
  if (int rc = head_pool_check(hs, hs_dtype, batch, layers, feat, frames, 0.f, store_rows, who)) return rc;
  HeadPoolArgs a{};
  a.hs = hs; a.hs_dtype = hs_dtype;
  a.B = batch; a.K = layers; a.F = feat; a.T = frames;
  cudaError_t e = head_layer_mean(a, store_rows, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "head_layer_mean_kernel");
  return 0;
}

// the element type of a layer-mean store's rows: SUPCON_F32 or SUPCON_F16 (SUPCON_BF16 is an hs / z type only)
static int store_dtype_check(int32_t store_dtype, const char* who) {
  if (store_dtype != SUPCON_F32 && store_dtype != SUPCON_F16)
    return fail(SUPCON_E_INVALID, "%s: unknown store_dtype %d (SUPCON_F32 or SUPCON_F16)", who, store_dtype);
  return 0;
}

static int store_pool_fwd(const void* store, int32_t store_dtype, int64_t n_store, int32_t feat, int32_t frames,
                          const int64_t* idx, int32_t batch, float dropout_p, float negative_slope,
                          const uint64_t* rng_state, float* pooled_out, void* stream, const char* who) {
  if (int rc = store_dtype_check(store_dtype, who)) return rc;
  if (!idx) return fail(SUPCON_E_INVALID, "NULL idx passed to %s", who);
  if (n_store < 1) return fail(SUPCON_E_INVALID, "%s: bad store size %lld", who, (long long)n_store);
  if (int rc = head_pool_check(store, SUPCON_F32, batch, 1, feat, frames, dropout_p, pooled_out, who)) return rc;
  HeadPoolArgs a{};
  a.hs = store; a.pooled = pooled_out;
  a.rng_state = reinterpret_cast<const unsigned long long*>(rng_state);
  a.B = batch; a.F = feat; a.T = frames;
  a.dropout_p = dropout_p; a.negative_slope = negative_slope;
  cudaError_t e = head_store_pool_forward(a, store_dtype, reinterpret_cast<const long long*>(idx), n_store,
                                          reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "head_store_pool_fwd_kernel");
  return 0;
}

static int sharded_store_pool_fwd(const uint64_t* shard_bases, int32_t n_ranks, int32_t store_dtype,
                                  int64_t n_store, int32_t feat, int32_t frames, const int64_t* idx, int32_t batch,
                                  float dropout_p, float negative_slope, const uint64_t* rng_state,
                                  float* pooled_out, void* stream, const char* who) {
  if (int rc = store_dtype_check(store_dtype, who)) return rc;
  if (!idx) return fail(SUPCON_E_INVALID, "NULL idx passed to %s", who);
  if (n_ranks < 1) return fail(SUPCON_E_INVALID, "%s: bad rank count %d", who, n_ranks);
  if (n_store < n_ranks)
    return fail(SUPCON_E_INVALID, "%s: bad store size %lld for %d ranks", who, (long long)n_store, n_ranks);
  if (int rc = head_pool_check(shard_bases, SUPCON_F32, batch, 1, feat, frames, dropout_p, pooled_out, who)) return rc;
  HeadPoolArgs a{};
  a.pooled = pooled_out;
  a.rng_state = reinterpret_cast<const unsigned long long*>(rng_state);
  a.B = batch; a.F = feat; a.T = frames;
  a.dropout_p = dropout_p; a.negative_slope = negative_slope;
  cudaError_t e = head_sharded_store_pool_forward(a, store_dtype,
                                                  reinterpret_cast<const unsigned long long*>(shard_bases), n_ranks,
                                                  reinterpret_cast<const long long*>(idx), n_store,
                                                  reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "head_sharded_store_pool_fwd_kernel");
  return 0;
}

int supcon_head_store_pool_forward_typed(const void* store, int32_t store_dtype, int64_t n_store, int32_t feat,
                                         int32_t frames, const int64_t* idx, int32_t batch, float dropout_p,
                                         float negative_slope, const uint64_t* rng_state, float* pooled_out,
                                         void* stream) {
  return store_pool_fwd(store, store_dtype, n_store, feat, frames, idx, batch, dropout_p, negative_slope, rng_state,
                        pooled_out, stream, "supcon_head_store_pool_forward_typed");
}

int supcon_head_store_pool_forward(const float* store, int64_t n_store, int32_t feat, int32_t frames,
                                   const int64_t* idx, int32_t batch, float dropout_p, float negative_slope,
                                   const uint64_t* rng_state, float* pooled_out, void* stream) {
  return store_pool_fwd(store, SUPCON_F32, n_store, feat, frames, idx, batch, dropout_p, negative_slope, rng_state,
                        pooled_out, stream, "supcon_head_store_pool_forward");
}

int supcon_head_sharded_store_pool_forward_typed(const uint64_t* shard_bases, int32_t n_ranks, int32_t store_dtype,
                                                 int64_t n_store, int32_t feat, int32_t frames, const int64_t* idx,
                                                 int32_t batch, float dropout_p, float negative_slope,
                                                 const uint64_t* rng_state, float* pooled_out, void* stream) {
  return sharded_store_pool_fwd(shard_bases, n_ranks, store_dtype, n_store, feat, frames, idx, batch, dropout_p,
                                negative_slope, rng_state, pooled_out, stream,
                                "supcon_head_sharded_store_pool_forward_typed");
}

int supcon_head_sharded_store_pool_forward(const uint64_t* shard_bases, int32_t n_ranks, int64_t n_store,
                                           int32_t feat, int32_t frames, const int64_t* idx, int32_t batch,
                                           float dropout_p, float negative_slope, const uint64_t* rng_state,
                                           float* pooled_out, void* stream) {
  return sharded_store_pool_fwd(shard_bases, n_ranks, SUPCON_F32, n_store, feat, frames, idx, batch, dropout_p,
                                negative_slope, rng_state, pooled_out, stream, "supcon_head_sharded_store_pool_forward");
}

int supcon_peer_push(const supcon_peer_t* pe, const void* src0, size_t bytes0, uint64_t dst_off0, const void* src1,
                     size_t bytes1, uint64_t dst_off1, int32_t flag_id, int32_t wait_flag_id, int32_t include_self,
                     void* stream) {
  const char* err = "";
  if (int rc = peer_check(pe, &err)) return fail(rc, "supcon_peer_push: %s", err);
  if (!src0 || (bytes0 % 4) || (src1 && (bytes1 % 4)) || flag_id < 0 || flag_id >= SUPCON_PEER_NFLAGS ||
      wait_flag_id >= SUPCON_PEER_NFLAGS)
    return fail(SUPCON_E_INVALID, "bad arguments to supcon_peer_push");
  cudaError_t e = peer_push(*pe, src0, bytes0, dst_off0, src1, bytes1, dst_off1, flag_id, wait_flag_id, include_self,
                            reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "peer_push_kernel");
  return 0;
}

int supcon_peer_wait(const supcon_peer_t* pe, int32_t flag_id, void* stream) {
  const char* err = "";
  if (int rc = peer_check(pe, &err)) return fail(rc, "supcon_peer_wait: %s", err);
  if (flag_id < 0 || flag_id >= SUPCON_PEER_NFLAGS) return fail(SUPCON_E_INVALID, "bad flag id");
  cudaError_t e = peer_wait(*pe, flag_id, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "peer_wait_kernel");
  return 0;
}

int supcon_peer_end_step(const supcon_peer_t* pe, int32_t flag_id, void* stream) {
  const char* err = "";
  if (int rc = peer_check(pe, &err)) return fail(rc, "supcon_peer_end_step: %s", err);
  if (flag_id < 0 || flag_id >= SUPCON_PEER_NFLAGS) return fail(SUPCON_E_INVALID, "bad flag id");
  cudaError_t e = peer_end_step(*pe, flag_id, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "peer_end_step_kernel");
  return 0;
}

int supcon_topk_indices(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                        const float* row_stats, int32_t* idx_out, void* stream) {
  if (int rc = validate(p)) return rc;
  if (!z_all || !labels_all || !row_stats || !idx_out || p->topk < 1)
    return fail(SUPCON_E_INVALID, "bad arguments to supcon_topk_indices");
  if (use_tc(p, false))
    return fail(SUPCON_E_UNSUPPORTED,
                "supcon_topk_indices re-derives the sets with the exact fp32 Gram; statistics of the bf16 tensor path "
                "rank by the tcgen05 Gram -- pass SUPCON_FLAG_FORCE_EXACT to the forward and to this call");
  FfmaArgs a = make_ffma(p, z_all, labels_all, nullptr, false, /*use_plan=*/false);
  a.row_stats = const_cast<float*>(row_stats);
  cudaError_t e = ffma_topk_indices(a, idx_out, reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return cuda_fail(e, "ffma_topk_indices");
  return 0;
}

}  // extern "C"
