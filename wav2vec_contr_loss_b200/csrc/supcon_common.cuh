// Shared device helpers for the SupCon kernels (sm_100a).
//
// Math follows SURVEY.md Appendix A; reference citations are to
// JaskiratSudan/wav2vec_contr_loss loss.py.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "supcon_b200.h"

#ifndef SUPCON_INT_MAX
#define SUPCON_INT_MAX 2147483647
#endif

namespace supcon {

// fp32(1 - 1e-7) = 1 - 2^-23: the clamp bound the reference applies to an fp32
// Gram (loss.py:101-102; SURVEY Appendix C).
__device__ __forceinline__ float geo_hi() { return 0.99999988079071044921875f; }
#define SUPCON_PI_F 3.14159274101257324f
#define SUPCON_2_OVER_PI_F 0.636619772367581343f

// s(c) for geodesic similarity, op-for-op as loss.py:102-106 (no FMA contraction).
__device__ __forceinline__ float geodesic_sim(float c) {
  float ch = fminf(fmaxf(c, -geo_hi()), geo_hi());
  float theta = acosf(ch);
  float unit = __fsub_rn(1.0f, __fdiv_rn(theta, SUPCON_PI_F));
  return __fsub_rn(__fmul_rn(2.0f, unit), 1.0f);
}
// ds/dc: (2/pi)/sqrt(1-c^2) inside the clamp range (inclusive), 0 outside.
__device__ __forceinline__ float geodesic_slope(float c) {
  if (!(c >= -geo_hi() && c <= geo_hi())) return 0.0f;
  return SUPCON_2_OVER_PI_F * rsqrtf(fmaf(-c, c, 1.0f));
}
__device__ __forceinline__ float geodesic_slope_exact(float c) {
  if (!(c >= -geo_hi() && c <= geo_hi())) return 0.0f;
  return __fdiv_rn(SUPCON_2_OVER_PI_F, sqrtf(fmaf(-c, c, 1.0f)));
}

// Columns a kernel sweeps when the memory's fill level is read on the device (supcon_forward_rows_memory):
// n_rows + *mem_filled, or -1 when the count lies outside [0, n_total - n_rows] (the caller poisons its results
// with NaN and sweeps every column).  mem_filled == NULL: n_total, a full memory or none.
__device__ __forceinline__ int live_columns(const int32_t* mem_filled, int n_rows, int n_total) {
  if (mem_filled == nullptr) return n_total;
  const int f = *mem_filled;
  return (f >= 0 && f <= n_total - n_rows) ? n_rows + f : -1;
}

// Global coefficients of the backward pass, derived from the (all-reduced)
// partial sums exactly as loss.py:137-151 blends the two means.
struct GlobalCoef {
  float a_full;   // w_full  / (|A_f| tau)   (0 when A_f is empty)
  float a_mined;  // w_mined / (|A_m| tau)
  float cu;       // lambda * (-2t) / (M (m + 1e-8)), M = N(N-1)/2
  float loss;     // the scalar loss
};

// use_label_counts: take |A_f|, |A_m| from the label-derived GLOBAL counts (SUPCON_P_GCNT_*) that the tensor
// path's forward leaves in a rank's own partials, so coefficients are known before any exchange.
// n_batch: rows of the uniformity term (batch_columns(): n_total, or n_rows with SUPCON_FLAG_MEMORY_COLUMNS).
__device__ __forceinline__ GlobalCoef global_coef(const double* pg, int n_batch, float tau, float alpha,
                                                  float lambda_uni, float uni_t, bool use_label_counts = false) {
  GlobalCoef g;
  double cnt_f = pg[use_label_counts ? SUPCON_P_GCNT_FULL : SUPCON_P_CNT_FULL];
  double cnt_m = pg[use_label_counts ? SUPCON_P_GCNT_MINED : SUPCON_P_CNT_MINED];
  double main_loss = 0.0, wf = 0.0, wm = 0.0;
  if (cnt_f > 0.0) {
    double full = pg[SUPCON_P_SUM_FULL] / cnt_f;
    double mined;
    if (cnt_m > 0.0) {
      mined = pg[SUPCON_P_SUM_MINED] / cnt_m;
      wf = 1.0 - (double)alpha;
      wm = (double)alpha;
    } else {  // loss.py:142-143: mined falls back to full
      mined = full;
      wf = 1.0;
      wm = 0.0;
    }
    main_loss = (1.0 - (double)alpha) * full + (double)alpha * mined;
  }
  g.a_full = (cnt_f > 0.0) ? (float)(wf / (cnt_f * (double)tau)) : 0.0f;
  g.a_mined = (cnt_m > 0.0) ? (float)(wm / (cnt_m * (double)tau)) : 0.0f;
  g.cu = 0.0f;
  if (lambda_uni > 0.0f && n_batch > 1) {
    double pairs2 = (double)n_batch * (double)(n_batch - 1);
    double m = pg[SUPCON_P_SUM_W] / pairs2;
    main_loss += (double)lambda_uni * log(m + 1e-8);
    g.cu = (float)((double)lambda_uni * (-2.0 * (double)uni_t) / ((pairs2 * 0.5) * (m + 1e-8)));
  }
  g.loss = (float)main_loss;
  return g;
}

// Fixed-order block reduction of the per-row loss terms -> workspace; the last
// block to finish sums over blocks (fixed order, deterministic) into partials[]
// and optionally writes the scalar loss.  red = [5][rows] doubles in shared memory.
struct FinishArgs {
  double* block_partials;  // [gridDim.x][SUPCON_N_PARTIALS]
  unsigned* ticket;        // zero before the launch
  double* partials;        // [SUPCON_N_PARTIALS] out
  float* loss_out;         // optional
  int n_batch;             // rows of the uniformity term (global_coef)
  float tau, alpha, lambda_uni, uni_t;
};

// NV = number of per-row values reduced from `red` ([NV][rows] doubles); slots NV..7 of the block record are 0.
// `fixmax` (tensor path only) is stored in partials[SUPCON_P_FIXMAX] by the last block; other paths pass 0.
template <int NV = 5>
__device__ inline void block_partials_and_finish(const FinishArgs& a, const double* red, int rows,
                                                 double fixmax = 0.0) {
  __shared__ int is_last;
  const int tid = threadIdx.x;
  double* bp = a.block_partials + (int64_t)blockIdx.x * SUPCON_N_PARTIALS;
  if (tid < NV) {
    double s = 0.0;
    for (int r = 0; r < rows; ++r) s += red[tid * rows + r];
    bp[tid] = s;
  } else if (tid < SUPCON_N_PARTIALS) {
    bp[tid] = 0.0;
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    unsigned t = atomicAdd(a.ticket, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (tid < SUPCON_N_PARTIALS) {
    double s = 0.0;
    for (unsigned b = 0; b < gridDim.x; ++b)
      s += *((volatile double*)(a.block_partials + (int64_t)b * SUPCON_N_PARTIALS + tid));
    a.partials[tid] = (tid == SUPCON_P_FIXMAX) ? fixmax : s;
  }
  __syncthreads();
  if (tid == 0) {
    *a.ticket = 0u;
    if (a.loss_out) {
      GlobalCoef g = global_coef(a.partials, a.n_batch, a.tau, a.alpha, a.lambda_uni, a.uni_t);
      *a.loss_out = g.loss;
    }
  }
}

// ---- element access for fp32 / bf16 row-major matrices ----
template <typename T>
__device__ __forceinline__ float ld_elem(const T* p);
template <>
__device__ __forceinline__ float ld_elem<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float ld_elem<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}

// 4 consecutive elements starting at column k of row `row` (zero beyond d / invalid row)
template <typename T>
__device__ __forceinline__ float4 ld_row4(const T* base, int64_t row, bool row_ok, int k, int d, bool vec_ok) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (!row_ok) return v;
  const T* p = base + row * (int64_t)d + k;
  if (vec_ok && k + 3 < d) {
    if constexpr (sizeof(T) == 4) {
      v = __ldg(reinterpret_cast<const float4*>(p));
    } else {
      uint2 raw = __ldg(reinterpret_cast<const uint2*>(p));
      __nv_bfloat162 lo = *reinterpret_cast<__nv_bfloat162*>(&raw.x);
      __nv_bfloat162 hi = *reinterpret_cast<__nv_bfloat162*>(&raw.y);
      float2 a = __bfloat1622float2(lo), b = __bfloat1622float2(hi);
      v = make_float4(a.x, a.y, b.x, b.y);
    }
  } else {
    if (k + 0 < d) v.x = ld_elem<T>(p + 0);
    if (k + 1 < d) v.y = ld_elem<T>(p + 1);
    if (k + 2 < d) v.z = ld_elem<T>(p + 2);
    if (k + 3 < d) v.w = ld_elem<T>(p + 3);
  }
  return v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace supcon
