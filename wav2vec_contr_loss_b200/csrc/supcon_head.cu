// Producer of the loss's input: the compression head up to the Linear layer, fused with the time mean.
//
// Reference (compression_module.py:48-65, stage1_utils.py:122-123):
//     x   = LeakyReLU(Dropout(mean_k hs[b,k,f,t]))            (B, F, T)
//     seq = Linear(x^T)^T                                      (B, D, T)
//     z   = normalize(mean_t seq)                              (B, D)
// The Linear layer and the time mean are both linear, so  mean_t seq = W * (mean_t x) + bias : the per-frame
// GEMM over (B*T, F) collapses to one over (B, F), and everything left of it is ONE pass over hs:
//     pooled[b,f] = (1/T) sum_t LeakyReLU(Dropout((1/K) sum_k hs[b,k,f,t]))
// This file is that pass (forward) and its transpose (backward, only needed when the encoder is fine-tuned), and the
// same forward split in two for a frozen encoder: the layer mean written once per clip into a store, and the rest of
// the pass run on store rows gathered by index every epoch (one GPU's store, or one sharded over a node's GPUs).
// HBM-bound: the algorithmic traffic is hs read once (B*K*F*T elements: 1.3 GB of fp32 or 0.65 GB of bf16 at B = 64,
// K = 25, F = 1024, T = 199), the output is B*F*4 bytes.
//
// Element type of hs / dhs: fp32 or bf16 (the dtype of a bf16 encoder's output).  bf16 elements are widened to fp32
// exactly and everything after the load is the fp32 arithmetic in the same order, so a bf16 hs gives bit for bit the
// pooled values of its fp32 copy, and the bf16 dhs is the fp32 one rounded to nearest even.
//
// Layout: hs is (B, K, F, T) contiguous, T innermost.  For one b the (f, t) plane is contiguous, so a block takes
// `rows` consecutive feature rows = one contiguous run of rows*T elements per layer k (stride F*T between layers),
// reads it with 128-bit loads (4 floats or 8 bf16) when the run allows, keeps the activated values (fp32) in shared
// memory and reduces each row over t in a fixed order (deterministic, no atomics).
//
// Dropout: counter-based Philox4x32-10 keyed by a (seed, offset) pair read from DEVICE memory, so a captured CUDA
// graph draws a new mask every replay (the caller bumps the offset in-stream).  Element (b,f,t) uses word
// (i & 3) of the block i >> 2, i = (b*F + f)*T + t; the backward regenerates the same mask.
#include <type_traits>

#include <cuda_fp16.h>

#include "supcon_common.cuh"
#include "supcon_internal.h"

namespace supcon {
namespace {

constexpr int HP_THREADS = 256;

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

// multiplier applied by Dropout to element i: 0 or 1/(1-p)
__device__ __forceinline__ float dropout_scale(unsigned long long seed, unsigned long long offset, long long i,
                                               float p, float keep_scale) {
  const unsigned long long blk = (unsigned long long)i >> 2;
  const uint4 r = philox4x32_10(make_uint4((unsigned)blk, (unsigned)(blk >> 32), (unsigned)offset,
                                           (unsigned)(offset >> 32)),
                                make_uint2((unsigned)seed, (unsigned)(seed >> 32)));
  const int w = (int)(i & 3);
  const unsigned word = w == 0 ? r.x : (w == 1 ? r.y : (w == 2 ? r.z : r.w));
  const float u = (float)(word >> 8) * (1.0f / 16777216.0f);   // [0, 1)
  return u >= p ? keep_scale : 0.0f;
}

template <typename E>
struct RunView {            // the contiguous run of one block
  const E* base;            // hs + ((b*K)*F + f0)*T
  long long plane;          // F*T
  long long first_elem;     // (b*F + f0)*T : index of the run's first element in the (B,F,T) mask space
  int rows, len, f0, b;
};

template <typename E>
__device__ __forceinline__ RunView<E> run_of_block(const HeadPoolArgs& a) {
  RunView<E> v;
  v.b = blockIdx.y;
  v.f0 = blockIdx.x * a.rows_per_block;
  v.rows = min(a.rows_per_block, a.F - v.f0);
  v.len = v.rows * a.T;
  v.plane = (long long)a.F * a.T;
  v.base = static_cast<const E*>(a.hs) + ((long long)v.b * a.K) * v.plane + (long long)v.f0 * a.T;
  v.first_elem = ((long long)v.b * a.F + v.f0) * a.T;
  return v;
}

// one access of VEC elements of type E: 16 bytes (float4, or eight bf16 / fp16 in a uint4) or one element
template <typename E, int VEC>
struct Pack;
template <>
struct Pack<float, 4> { typedef float4 type; };
template <>
struct Pack<float, 1> { typedef float type; };
template <>
struct Pack<__nv_bfloat16, 8> { typedef uint4 type; };
template <>
struct Pack<__nv_bfloat16, 1> { typedef __nv_bfloat16 type; };
template <>
struct Pack<__half, 8> { typedef uint4 type; };
template <>
struct Pack<__half, 1> { typedef __half type; };

// the two bf16 of a 32-bit word widened to fp32 (exact): element 2i is the low half
__device__ __forceinline__ float bf16_lo(unsigned w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(unsigned w) { return __uint_as_float(w & 0xFFFF0000u); }
// and back, rounded to nearest even
__device__ __forceinline__ unsigned bf16x2_rn(float lo, float hi) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const unsigned*>(&h);
}

template <typename E, int VEC>
__device__ __forceinline__ void add_pack(float (&acc)[VEC], const typename Pack<E, VEC>::type& x) {
  if constexpr (VEC == 4) { acc[0] += x.x; acc[1] += x.y; acc[2] += x.z; acc[3] += x.w; }
  else if constexpr (VEC == 8) {
    acc[0] += bf16_lo(x.x); acc[1] += bf16_hi(x.x); acc[2] += bf16_lo(x.y); acc[3] += bf16_hi(x.y);
    acc[4] += bf16_lo(x.z); acc[5] += bf16_hi(x.z); acc[6] += bf16_lo(x.w); acc[7] += bf16_hi(x.w);
  }
  else if constexpr (std::is_same<E, float>::value) acc[0] += x;
  else acc[0] += __bfloat162float(x);
}

// sum over the K layers of VEC consecutive elements starting at run offset e, layers added in order k = 0..K-1;
// loads are issued eight layers at a time so that each thread keeps 8 x 16 bytes in flight
template <typename E, int VEC>
__device__ __forceinline__ void layer_sum(const RunView<E>& v, int K, int e, float (&acc)[VEC]) {
  typedef typename Pack<E, VEC>::type pack_t;
  constexpr int BATCH = 8;
#pragma unroll
  for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
  const E* p = v.base + e;
  int k = 0;
  for (; k + BATCH <= K; k += BATCH) {
    pack_t x[BATCH];
#pragma unroll
    for (int j = 0; j < BATCH; ++j) x[j] = __ldg(reinterpret_cast<const pack_t*>(p + (long long)(k + j) * v.plane));
#pragma unroll
    for (int j = 0; j < BATCH; ++j) add_pack<E, VEC>(acc, x[j]);
  }
  for (; k < K; ++k) add_pack<E, VEC>(acc, __ldg(reinterpret_cast<const pack_t*>(p + (long long)k * v.plane)));
}

// the two fp16 of a 32-bit word widened to fp32 (exact): element 2i is the low half
__device__ __forceinline__ float2 f16x2_to_float2(unsigned w) {
  return __half22float2(*reinterpret_cast<const __half2*>(&w));
}

// VEC consecutive values of a stored layer-mean row of element type S (fp32, or fp16 widened to fp32 exactly),
// starting at run offset e
template <typename S, int VEC>
__device__ __forceinline__ void stored_mean(const RunView<S>& v, int e, float (&x)[VEC]) {
  typedef typename Pack<S, VEC>::type pack_t;
  const pack_t q = __ldg(reinterpret_cast<const pack_t*>(v.base + e));
  if constexpr (VEC == 4) {
    x[0] = q.x; x[1] = q.y; x[2] = q.z; x[3] = q.w;
  } else if constexpr (VEC == 8) {
    const unsigned w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f = f16x2_to_float2(w[i]);
      x[2 * i] = f.x; x[2 * i + 1] = f.y;
    }
  } else if constexpr (std::is_same<S, float>::value) {
    x[0] = q;
  } else {
    x[0] = __half2float(q);
  }
}

// The forward of one block after its run is located: Dropout, LeakyReLU, and the time mean of each row.  STORED
// picks the source of the layer mean: false = the K-layer sum of hs times 1/K, true = a row of a layer-mean store
// (head_layer_mean_kernel wrote exactly that product, so both sources give the same bits).  The mask index is
// always the batch position's, so a gathered batch draws the mask of the same batch read from hs.
template <typename E, int VEC, bool STORED>
__device__ __forceinline__ void pool_run(const HeadPoolArgs& a, const RunView<E>& v) {
  extern __shared__ float act[];                      // [rows*T] activated values of this block's run
  const bool drop = a.dropout_p > 0.f && a.rng_state != nullptr;
  unsigned long long seed = 0, offset = 0;
  if (drop) { seed = a.rng_state[0]; offset = a.rng_state[1]; }
  const float inv_k = 1.0f / (float)a.K;
  const float keep_scale = drop ? 1.0f / (1.0f - a.dropout_p) : 1.0f;

  for (int e = threadIdx.x * VEC; e < v.len; e += HP_THREADS * VEC) {
    float acc[VEC];
    if constexpr (STORED) stored_mean<E, VEC>(v, e, acc);
    else layer_sum<E, VEC>(v, a.K, e, acc);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      float x = acc[i];
      if constexpr (!STORED) x *= inv_k;
      if (drop) x *= dropout_scale(seed, offset, v.first_elem + e + i, a.dropout_p, keep_scale);
      act[e + i] = x > 0.f ? x : x * a.negative_slope;
    }
  }
  __syncthreads();

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float inv_t = 1.0f / (float)a.T;
  for (int r = warp; r < v.rows; r += HP_THREADS / 32) {
    float s = 0.f;
    for (int t = lane; t < a.T; t += 32) s += act[r * a.T + t];
    s = warp_sum(s);
    if (lane == 0) a.pooled[(long long)v.b * a.F + v.f0 + r] = s * inv_t;
  }
}

template <typename E, int VEC>
__global__ void __launch_bounds__(HP_THREADS, 4) head_pool_fwd_kernel(HeadPoolArgs a) {
  pool_run<E, VEC, false>(a, run_of_block<E>(a));
}

// Gather-pool: batch position b reads store row idx[b] (idx on the device, so a captured graph takes new rows every
// replay; a.K = 1).  S is the store's element type (float, or __half widened exactly on the load).  row_of(row,
// plane) is the address of a row's (F, T) plane.  A row index outside [0, n_store) poisons pooled row b with NaN (the
// other rows stay exact); nothing is read for it.
template <typename S, int VEC, typename RowOf>
__device__ __forceinline__ void store_pool_run(const HeadPoolArgs& a, const long long* __restrict__ idx,
                                               long long n_store, RowOf row_of) {
  RunView<S> v = run_of_block<S>(a);
  const long long row = idx[v.b];
  if (row < 0 || row >= n_store) {
    for (int r = threadIdx.x; r < v.rows; r += HP_THREADS) a.pooled[(long long)v.b * a.F + v.f0 + r] = NAN;
    return;
  }
  v.base = row_of(row, v.plane) + (long long)v.f0 * a.T;
  pool_run<S, VEC, true>(a, v);
}

// a.hs = the (n_store, F, T) store of S
template <typename S, int VEC>
__global__ void __launch_bounds__(HP_THREADS, 4) head_store_pool_fwd_kernel(HeadPoolArgs a,
                                                                         const long long* __restrict__ idx,
                                                                         long long n_store) {
  store_pool_run<S, VEC>(a, idx, n_store, [&](long long row, long long plane) {
    return static_cast<const S*>(a.hs) + row * plane;
  });
}

// The store sharded over n_ranks GPUs: row i is local row i / n_ranks of the shard at bases[i % n_ranks], a device
// address in this process (its own shard, or a peer's mapped over NVLink); offsets are in elements of S
template <typename S, int VEC>
__global__ void __launch_bounds__(HP_THREADS, 4) head_sharded_store_pool_fwd_kernel(
    HeadPoolArgs a, const unsigned long long* __restrict__ bases, int n_ranks, const long long* __restrict__ idx,
    long long n_store) {
  store_pool_run<S, VEC>(a, idx, n_store, [&](long long row, long long plane) {
    return reinterpret_cast<const S*>(bases[row % n_ranks]) + (row / n_ranks) * plane;
  });
}

// store_rows[b] = (1/K) sum_k hs[b, k] in fp32, layers added in order: the layer mean of head_pool_fwd_kernel, bit
// for bit, written out instead of activated
template <typename E, int VEC>
__global__ void __launch_bounds__(HP_THREADS, 4) head_layer_mean_kernel(HeadPoolArgs a, float* __restrict__ rows) {
  const RunView<E> v = run_of_block<E>(a);
  const float inv_k = 1.0f / (float)a.K;
  float* out = rows + (long long)v.b * v.plane + (long long)v.f0 * a.T;
  for (int e = threadIdx.x * VEC; e < v.len; e += HP_THREADS * VEC) {
    float acc[VEC];
    layer_sum<E, VEC>(v, a.K, e, acc);
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[i] *= inv_k;
    if constexpr (VEC == 1) {
      out[e] = acc[0];
    } else {
#pragma unroll
      for (int i = 0; i < VEC; i += 4)
        *reinterpret_cast<float4*>(out + e + i) = make_float4(acc[i], acc[i + 1], acc[i + 2], acc[i + 3]);
    }
  }
}

// dhs[b,k,f,t] = dpooled[b,f] * (1/T) * LeakyReLU'(x) * dropout multiplier * (1/K), the same for every k; computed
// in fp32 and stored in E (bf16: round to nearest even)
template <typename E, int VEC>
__global__ void __launch_bounds__(HP_THREADS, 4) head_pool_bwd_kernel(HeadPoolArgs a, const float* __restrict__ dpooled,
                                                                   E* __restrict__ dhs) {
  const RunView<E> v = run_of_block<E>(a);
  const bool drop = a.dropout_p > 0.f && a.rng_state != nullptr;
  unsigned long long seed = 0, offset = 0;
  if (drop) { seed = a.rng_state[0]; offset = a.rng_state[1]; }
  const float inv_k = 1.0f / (float)a.K;
  const float keep_scale = drop ? 1.0f / (1.0f - a.dropout_p) : 1.0f;
  const float inv_kt = inv_k / (float)a.T;
  E* out = dhs + (v.base - static_cast<const E*>(a.hs));

  for (int e = threadIdx.x * VEC; e < v.len; e += HP_THREADS * VEC) {
    float acc[VEC], g[VEC];
    layer_sum<E, VEC>(v, a.K, e, acc);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const float m = drop ? dropout_scale(seed, offset, v.first_elem + e + i, a.dropout_p, keep_scale) : 1.0f;
      const float x = acc[i] * inv_k * m;
      const float up = dpooled[(long long)v.b * a.F + v.f0 + (e + i) / a.T];
      g[i] = up * inv_kt * m * (x > 0.f ? 1.0f : a.negative_slope);
    }
    E* q = out + e;
    if constexpr (VEC == 8) {
      const uint4 w = make_uint4(bf16x2_rn(g[0], g[1]), bf16x2_rn(g[2], g[3]), bf16x2_rn(g[4], g[5]),
                                 bf16x2_rn(g[6], g[7]));
      for (int k = 0; k < a.K; ++k) *reinterpret_cast<uint4*>(q + (long long)k * v.plane) = w;
    } else {
      for (int k = 0; k < a.K; ++k) {
        if constexpr (VEC == 4)
          *reinterpret_cast<float4*>(q + (long long)k * v.plane) = make_float4(g[0], g[1], g[2], g[3]);
        else if constexpr (std::is_same<E, float>::value)
          q[(long long)k * v.plane] = g[0];
        else
          q[(long long)k * v.plane] = __float2bfloat16_rn(g[0]);
      }
    }
  }
}

// 128-bit accesses need every run (and every layer plane) to start on a 16-byte boundary and to hold a multiple of
// `width` elements (four floats, eight bf16 or fp16) - including the shorter run of the last block of a row of blocks.
bool vector_ok(const HeadPoolArgs& a, const void* other, int width) {
  auto aligned = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; };
  const long long run = (long long)a.rows_per_block * a.T;
  const long long tail = (long long)(a.F % a.rows_per_block) * a.T;
  return aligned(a.hs) && (other == nullptr || aligned(other)) && ((long long)a.F * a.T) % width == 0 &&
         run % width == 0 && tail % width == 0;
}

}  // namespace

int head_pool_rows_per_block(int F, int T, int hs_dtype) {
  // 16 rows per block when they fit 48 KB of shared memory (T <= 768), fewer for longer clips; 0 = unsupported
  if (T < 1 || F < 1) return 0;
  int rows = 12288 / T;
  if (rows < 1) return 0;
  if (rows > 16) rows = 16;
  // keep runs a multiple of one 128-bit access for any T: four floats, eight 16-bit elements (from 8 rows up)
  if ((hs_dtype == SUPCON_BF16 || hs_dtype == SUPCON_F16) && rows >= 8) rows &= ~7;
  else if (rows > 4) rows &= ~3;
  return rows < F ? rows : F;
}

cudaError_t head_pool_forward(HeadPoolArgs a, cudaStream_t stream) {
  a.rows_per_block = head_pool_rows_per_block(a.F, a.T, a.hs_dtype);
  if (a.rows_per_block < 1) return cudaErrorInvalidValue;
  dim3 grid((a.F + a.rows_per_block - 1) / a.rows_per_block, a.B);
  const size_t smem = (size_t)a.rows_per_block * a.T * sizeof(float);
  if (a.hs_dtype == SUPCON_BF16) {
    if (vector_ok(a, nullptr, 8))
      head_pool_fwd_kernel<__nv_bfloat16, 8><<<grid, HP_THREADS, smem, stream>>>(a);
    else
      head_pool_fwd_kernel<__nv_bfloat16, 1><<<grid, HP_THREADS, smem, stream>>>(a);
  } else if (vector_ok(a, nullptr, 4)) {
    head_pool_fwd_kernel<float, 4><<<grid, HP_THREADS, smem, stream>>>(a);
  } else {
    head_pool_fwd_kernel<float, 1><<<grid, HP_THREADS, smem, stream>>>(a);
  }
  return cudaGetLastError();
}

cudaError_t head_layer_mean(HeadPoolArgs a, float* rows, cudaStream_t stream) {
  a.rows_per_block = head_pool_rows_per_block(a.F, a.T, a.hs_dtype);
  if (a.rows_per_block < 1) return cudaErrorInvalidValue;
  dim3 grid((a.F + a.rows_per_block - 1) / a.rows_per_block, a.B);
  if (a.hs_dtype == SUPCON_BF16) {
    if (vector_ok(a, rows, 8))
      head_layer_mean_kernel<__nv_bfloat16, 8><<<grid, HP_THREADS, 0, stream>>>(a, rows);
    else
      head_layer_mean_kernel<__nv_bfloat16, 1><<<grid, HP_THREADS, 0, stream>>>(a, rows);
  } else if (vector_ok(a, rows, 4)) {
    head_layer_mean_kernel<float, 4><<<grid, HP_THREADS, 0, stream>>>(a, rows);
  } else {
    head_layer_mean_kernel<float, 1><<<grid, HP_THREADS, 0, stream>>>(a, rows);
  }
  return cudaGetLastError();
}

cudaError_t head_store_pool_forward(HeadPoolArgs a, int store_dtype, const long long* idx, long long n_store,
                                    cudaStream_t stream) {
  a.K = 1;
  a.hs_dtype = store_dtype;
  a.rows_per_block = head_pool_rows_per_block(a.F, a.T, a.hs_dtype);
  if (a.rows_per_block < 1) return cudaErrorInvalidValue;
  dim3 grid((a.F + a.rows_per_block - 1) / a.rows_per_block, a.B);
  const size_t smem = (size_t)a.rows_per_block * a.T * sizeof(float);
  if (store_dtype == SUPCON_F16) {
    if (vector_ok(a, nullptr, 8))
      head_store_pool_fwd_kernel<__half, 8><<<grid, HP_THREADS, smem, stream>>>(a, idx, n_store);
    else
      head_store_pool_fwd_kernel<__half, 1><<<grid, HP_THREADS, smem, stream>>>(a, idx, n_store);
  } else if (vector_ok(a, nullptr, 4)) {
    head_store_pool_fwd_kernel<float, 4><<<grid, HP_THREADS, smem, stream>>>(a, idx, n_store);
  } else {
    head_store_pool_fwd_kernel<float, 1><<<grid, HP_THREADS, smem, stream>>>(a, idx, n_store);
  }
  return cudaGetLastError();
}

cudaError_t head_sharded_store_pool_forward(HeadPoolArgs a, int store_dtype, const unsigned long long* bases,
                                            int n_ranks, const long long* idx, long long n_store,
                                            cudaStream_t stream) {
  a.hs = nullptr;           // the shard bases are on the device: 16-byte alignment is the caller's promise
  a.K = 1;
  a.hs_dtype = store_dtype;
  a.rows_per_block = head_pool_rows_per_block(a.F, a.T, a.hs_dtype);
  if (a.rows_per_block < 1) return cudaErrorInvalidValue;
  dim3 grid((a.F + a.rows_per_block - 1) / a.rows_per_block, a.B);
  const size_t smem = (size_t)a.rows_per_block * a.T * sizeof(float);
  if (store_dtype == SUPCON_F16) {
    if (vector_ok(a, nullptr, 8))
      head_sharded_store_pool_fwd_kernel<__half, 8><<<grid, HP_THREADS, smem, stream>>>(a, bases, n_ranks, idx,
                                                                                         n_store);
    else
      head_sharded_store_pool_fwd_kernel<__half, 1><<<grid, HP_THREADS, smem, stream>>>(a, bases, n_ranks, idx,
                                                                                         n_store);
  } else if (vector_ok(a, nullptr, 4)) {
    head_sharded_store_pool_fwd_kernel<float, 4><<<grid, HP_THREADS, smem, stream>>>(a, bases, n_ranks, idx,
                                                                                      n_store);
  } else {
    head_sharded_store_pool_fwd_kernel<float, 1><<<grid, HP_THREADS, smem, stream>>>(a, bases, n_ranks, idx,
                                                                                      n_store);
  }
  return cudaGetLastError();
}

cudaError_t head_pool_backward(HeadPoolArgs a, const float* dpooled, void* dhs, cudaStream_t stream) {
  a.rows_per_block = head_pool_rows_per_block(a.F, a.T, a.hs_dtype);
  if (a.rows_per_block < 1) return cudaErrorInvalidValue;
  dim3 grid((a.F + a.rows_per_block - 1) / a.rows_per_block, a.B);
  if (a.hs_dtype == SUPCON_BF16) {
    __nv_bfloat16* d = static_cast<__nv_bfloat16*>(dhs);
    if (vector_ok(a, dhs, 8))
      head_pool_bwd_kernel<__nv_bfloat16, 8><<<grid, HP_THREADS, 0, stream>>>(a, dpooled, d);
    else
      head_pool_bwd_kernel<__nv_bfloat16, 1><<<grid, HP_THREADS, 0, stream>>>(a, dpooled, d);
  } else if (vector_ok(a, dhs, 4)) {
    head_pool_bwd_kernel<float, 4><<<grid, HP_THREADS, 0, stream>>>(a, dpooled, static_cast<float*>(dhs));
  } else {
    head_pool_bwd_kernel<float, 1><<<grid, HP_THREADS, 0, stream>>>(a, dpooled, static_cast<float*>(dhs));
  }
  return cudaGetLastError();
}

}  // namespace supcon
