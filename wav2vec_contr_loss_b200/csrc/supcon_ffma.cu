// Exact fp32 (CUDA-core FFMA) SupCon path: any N, any d, any labels, any z.
//
// This is the 1e-5-parity path (TF32/bf16 tensor math cannot meet 1e-5 at
// tau = 0.07, SURVEY H5) and the route for shapes the tcgen05 path does not
// take.  Forward sweeps the column tiles of a 64-row block keeping only O(N)
// row statistics; backward recomputes the tiles and forms
//     dz_i = sum_j (G_ij + G_ji) z_j
// from those statistics, so no N x N matrix ever reaches HBM.
//
// The dot product of rows i and j is accumulated in one fp32 chain over
// k = 0..d-1 in the same order everywhere, so c_ij == c_ji bit-for-bit and the
// backward sees exactly the similarities the forward ranked (needed for the
// hard-negative membership test; SURVEY H3).
#include "supcon_common.cuh"
#include "supcon_internal.h"

namespace supcon {

namespace {

constexpr int BM = 64;        // rows per CTA
constexpr int BN = 64;        // columns per sweep step
constexpr int KC = 32;        // k chunk staged in shared memory
constexpr int LDT = KC + 4;   // padded chunk stride (floats): conflict-free float4 reads
constexpr int LDS_ = BN + 4;  // padded stride of the 64x64 tiles
constexpr int NT = 256;
constexpr int DC = 256;       // dz columns per CTA in the backward

// ---- 64x64 tile of dot products; thread (tx,ty) owns rows ty+16i, cols tx+16j ----
template <typename T>
__device__ __forceinline__ void gram_tile(const T* __restrict__ z, int d, bool vec_ok, int row0, int row_end,
                                          int col0, int n_total, float* As, float* Bs, float (&acc)[4][4],
                                          float* nrm_r, float* nrm_c, bool want_norms) {
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float nr = 0.f, nc = 0.f;
  for (int k0 = 0; k0 < d; k0 += KC) {
#pragma unroll
    for (int it = 0; it < (BM * KC / 4) / NT; ++it) {
      int idx = tid + it * NT;
      int r = idx >> 3, q = idx & 7;
      int gr = row0 + r, gc = col0 + r;
      float4 va = ld_row4<T>(z, gr, gr < row_end, k0 + 4 * q, d, vec_ok);
      float4 vb = ld_row4<T>(z, gc, gc < n_total, k0 + 4 * q, d, vec_ok);
      *reinterpret_cast<float4*>(&As[r * LDT + 4 * q]) = va;
      *reinterpret_cast<float4*>(&Bs[r * LDT + 4 * q]) = vb;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < KC; kk += 4) {
      float4 a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(&As[(ty + 16 * i) * LDT + kk]);
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = *reinterpret_cast<const float4*>(&Bs[(tx + 16 * j) * LDT + kk]);
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float c = acc[i][j];
          c = fmaf(a[i].x, b[j].x, c);
          c = fmaf(a[i].y, b[j].y, c);
          c = fmaf(a[i].z, b[j].z, c);
          c = fmaf(a[i].w, b[j].w, c);
          acc[i][j] = c;
        }
    }
    if (want_norms && tid < 2 * BM) {  // squared norms, same chain order for every CTA
      const float* src = (tid < BM) ? &As[tid * LDT] : &Bs[(tid - BM) * LDT];
      float s = (tid < BM) ? nr : nc;
#pragma unroll
      for (int kk = 0; kk < KC; ++kk) s = fmaf(src[kk], src[kk], s);
      if (tid < BM) nr = s; else nc = s;
    }
    __syncthreads();
  }
  if (want_norms) {
    if (tid < BM) nrm_r[tid] = nr;
    else if (tid < 2 * BM) nrm_c[tid - BM] = nc;
  }
}

// row-state of the online softmax held by each of the 4 threads of a row
struct RowAcc {
  float m, sum_all, sum_pos_e, sum_pos_s, wsum;
  int npos, nneg;
};

__device__ __forceinline__ float rescale(float m_old, float m_new) {
  return (m_old == -INFINITY) ? 0.f : expf(m_old - m_new);
}

template <typename T>
__global__ void __launch_bounds__(NT) ffma_fwd_kernel(FfmaArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* As = reinterpret_cast<float*>(smem_raw);
  float* Bs = As + BM * LDT;
  float* Ss = Bs + BN * LDT;
  float* Ws = Ss + BM * LDS_;
  float* nrm_r = Ws + BM * LDS_;
  float* nrm_c = nrm_r + BM;
  int* lab_c = reinterpret_cast<int*>(nrm_c + BN);
  int* cnt = lab_c + BN;
  double* red = reinterpret_cast<double*>(cnt + BM);  // [5][BM]
  float* lv = reinterpret_cast<float*>(red + 5 * BM);  // [BM][kcap]
  int* li = reinterpret_cast<int*>(lv + BM * a.kcap);

  const T* z = reinterpret_cast<const T*>(a.z);
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int row0 = a.row_offset + blockIdx.x * BM;
  const int row_end = a.row_offset + a.n_rows;
  const bool geo = a.similarity == SUPCON_GEODESIC;
  const bool uni = a.lambda_uni > 0.f;
  const bool mine = a.mine != 0;
  // columns [n_cols, n_total) are absent (a memory that is not full yet); bad: the fill level is out of range
  const int n_live = live_columns(a.mem_filled, a.n_rows, a.n_total);
  const bool bad = n_live < 0;
  const int n_cols = bad ? a.n_total : n_live;

  // phase-2 mapping: 4 threads per row, thread q takes columns q, q+4, ...
  const int pr = tid >> 2, pq = tid & 3;
  const int gi = row0 + pr;
  const bool row_ok = gi < row_end;
  const int lab_r = row_ok ? a.labels[gi] : 0;

  RowAcc st;
  st.m = -INFINITY; st.sum_all = 0.f; st.sum_pos_e = 0.f; st.sum_pos_s = 0.f; st.wsum = 0.f;
  st.npos = 0; st.nneg = 0;

  // merged row results (valid in all 4 threads of a row after round 0)
  float M = -INFINITY, sum_all = 0.f, sum_pos_e = 0.f, sum_pos_s = 0.f, wsum = 0.f;
  int npos = 0, nneg = 0;
  // hard-negative selection state.  Selection runs in rounds of at most kcap
  // entries; round r only admits negatives ranked strictly after the last
  // entry (bound_v, bound_i) of round r-1 in (value desc, index asc) order.
  float sum_top = 0.f, bound_v = INFINITY;
  int bound_i = -1;
  int rounds_total = 1;

  // column range of this CTA (blockIdx.y = column split; one split = the whole sweep)
  const int split = blockIdx.y;
  const int c_lo = (int)(((int64_t)a.col_tiles * split) / a.splits) * BN;
  const int c_hi = min(n_cols, (int)(((int64_t)a.col_tiles * (split + 1)) / a.splits) * BN);

  float acc[4][4];
  for (int round = 0; round < rounds_total; ++round) {
    const bool first = round == 0;
    const int Kr = mine ? min(a.kcap, a.topk - round * a.kcap) : 0;
    const bool row_mines = mine && row_ok && (first || nneg > a.topk);
    if (tid < BM) cnt[tid] = 0;
    __syncthreads();
    for (int col0 = c_lo; col0 < c_hi; col0 += BN) {
      gram_tile<T>(z, a.d, a.vec_ok, row0, row_end, col0, n_cols, As, Bs, acc, nrm_r, nrm_c, uni && first);
      if (tid < BN) lab_c[tid] = (col0 + tid < n_cols) ? a.labels[col0 + tid] : 0;
      __syncthreads();  // norms + labels visible
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          int r = ty + 16 * i, c = tx + 16 * j;
          float cv = acc[i][j];
          Ss[r * LDS_ + c] = geo ? geodesic_sim(cv) : cv;
          if (uni && first) {
            float d2 = fmaxf(nrm_r[r] + nrm_c[c] - 2.f * cv, 0.f);
            Ws[r * LDS_ + c] = expf(-a.uni_t * d2);
          }
        }
      __syncthreads();

      // ---- row statistics over this tile (round 0 only) ----
      if (first) {
        float tmax = -INFINITY;
#pragma unroll 4
        for (int t = 0; t < BN / 4; ++t) {
          int c = pq + 4 * t, gj = col0 + c;
          if (row_ok && gj < n_cols && gj != gi) tmax = fmaxf(tmax, __fdiv_rn(Ss[pr * LDS_ + c], a.tau));
        }
        if (tmax > st.m) {
          float f = rescale(st.m, tmax);
          st.sum_all *= f; st.sum_pos_e *= f; st.m = tmax;
        }
#pragma unroll 4
        for (int t = 0; t < BN / 4; ++t) {
          int c = pq + 4 * t, gj = col0 + c;
          if (row_ok && gj < n_cols && gj != gi) {
            float s = Ss[pr * LDS_ + c];
            float e = expf(__fdiv_rn(s, a.tau) - st.m);
            st.sum_all += e;
            if (lab_c[c] == lab_r) { st.npos++; st.sum_pos_e += e; st.sum_pos_s += s; }
            else st.nneg++;
            if (uni && gj < a.n_batch) st.wsum += Ws[pr * LDS_ + c];   // memory columns: no uniformity
          }
        }
      }
      // ---- hard-negative candidates ----
      if (mine) {
        bool cand = false;
        int have = 0;
        float thr = -INFINITY;
        if (row_mines) {
          have = cnt[pr];
          thr = (have >= Kr) ? lv[pr * a.kcap + Kr - 1] : -INFINITY;
#pragma unroll 4
          for (int t = 0; t < BN / 4; ++t) {
            int c = pq + 4 * t, gj = col0 + c;
            if (gj < n_cols && lab_c[c] != lab_r) {
              float s = Ss[pr * LDS_ + c];
              bool elig = (s < bound_v) || (s == bound_v && gj > bound_i);
              if (elig && (have < Kr || s > thr)) cand = true;
            }
          }
        }
        unsigned any = __ballot_sync(0xffffffffu, cand);
        bool row_any = (any >> ((tid & 31) & ~3)) & 0xFu;
        if (row_any && pq == 0) {
          // sorted insert, (value desc, index asc): columns are visited in index
          // order and an equal value never displaces an earlier one.
          float* v = lv + pr * a.kcap;
          int* ix = li + pr * a.kcap;
          int cn = have;
          for (int c = 0; c < BN; ++c) {
            int gj = col0 + c;
            if (gj >= n_cols || lab_c[c] == lab_r) continue;
            float s = Ss[pr * LDS_ + c];
            if (!((s < bound_v) || (s == bound_v && gj > bound_i))) continue;
            int p;
            if (cn < Kr) p = cn++;
            else if (s > v[Kr - 1]) p = Kr - 1;
            else continue;
            while (p > 0 && v[p - 1] < s) { v[p] = v[p - 1]; ix[p] = ix[p - 1]; --p; }
            v[p] = s; ix[p] = gj;
          }
          cnt[pr] = cn;
        }
      }
      __syncthreads();  // tile buffers are rewritten by the next gram_tile
    }

    if (first) {  // merge the 4 threads of each row
      M = st.m;
      M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, 1));
      M = fmaxf(M, __shfl_xor_sync(0xffffffffu, M, 2));
      float f = rescale(st.m, M);
      sum_all = st.sum_all * f; sum_pos_e = st.sum_pos_e * f; sum_pos_s = st.sum_pos_s; wsum = st.wsum;
      npos = st.npos; nneg = st.nneg;
#pragma unroll
      for (int o = 1; o <= 2; o <<= 1) {
        sum_all += __shfl_xor_sync(0xffffffffu, sum_all, o);
        sum_pos_e += __shfl_xor_sync(0xffffffffu, sum_pos_e, o);
        sum_pos_s += __shfl_xor_sync(0xffffffffu, sum_pos_s, o);
        wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
        npos += __shfl_xor_sync(0xffffffffu, npos, o);
        nneg += __shfl_xor_sync(0xffffffffu, nneg, o);
      }
      int more = (mine && row_ok && nneg > a.topk && a.topk > a.kcap) ? 1 : 0;
      if (__syncthreads_or(more)) rounds_total = (a.topk + a.kcap - 1) / a.kcap;
      if (a.splits > 1) {
        // column-split launch: leave this range's partial record (+ its candidate list); the merge kernel
        // combines the ranges (online-max merge) and finishes the loss
        if (pq == 0 && row_ok) {
          const int64_t rec = (int64_t)split * a.rows_pad + (gi - a.row_offset);
          float* out = a.part + rec * 8;
          out[0] = M; out[1] = sum_all; out[2] = sum_pos_e; out[3] = sum_pos_s; out[4] = wsum;
          reinterpret_cast<int*>(out)[5] = npos; reinterpret_cast<int*>(out)[6] = nneg;
          const int c = mine ? cnt[pr] : 0;
          reinterpret_cast<int*>(out)[7] = c;
          for (int t = 0; t < c; ++t) {
            a.lv_part[rec * a.kcap + t] = lv[pr * a.kcap + t];
            a.li_part[rec * a.kcap + t] = li[pr * a.kcap + t];
          }
        }
        return;
      }
    }
    if (mine) {
      // close this round: fold its list into sum_top, publish the new bound to the row's threads
      if (pq == 0 && row_ok && nneg > a.topk) {
        const float* v = lv + pr * a.kcap;
        for (int t = 0; t < Kr; ++t) sum_top += expf(__fdiv_rn(v[t], a.tau) - M);
        bound_v = v[Kr - 1];
        bound_i = li[pr * a.kcap + Kr - 1];
      }
      bound_v = __shfl_sync(0xffffffffu, bound_v, (tid & 31) & ~3);
      bound_i = __shfl_sync(0xffffffffu, bound_i, (tid & 31) & ~3);
    }
    __syncthreads();
  }

  if (pq == 0) {
    double l_full = 0.0, c_full = 0.0, l_mined = 0.0, c_mined = 0.0, w = 0.0;
    if (row_ok) {
      float lse = M + logf(sum_all);
      float lse_m = lse, thr_val = -INFINITY;
      int thr_idx = SUPCON_INT_MAX;
      if (mine && nneg > a.topk) {
        lse_m = M + logf(sum_pos_e + sum_top);
        thr_val = bound_v;
        thr_idx = bound_i;
      } else if (a.topk < 1) {
        thr_val = INFINITY; thr_idx = -1;
      }
      float pos_mean = (npos > 0) ? __fdiv_rn(__fdiv_rn(sum_pos_s, a.tau), (float)npos) : 0.f;
      float* so = a.row_stats + (int64_t)(gi - a.row_offset) * SUPCON_STATS_STRIDE;
      so[SUPCON_ST_LSE] = lse;
      so[SUPCON_ST_LSE_M] = lse_m;
      reinterpret_cast<int*>(so)[SUPCON_ST_NPOS] = npos;
      reinterpret_cast<int*>(so)[SUPCON_ST_NNEG] = nneg;
      so[SUPCON_ST_THR_VAL] = thr_val;
      reinterpret_cast<int*>(so)[SUPCON_ST_THR_IDX] = thr_idx;
      so[SUPCON_ST_WSUM] = wsum;
      so[SUPCON_ST_POS_MEAN] = pos_mean;
      if (npos > 0) {
        l_full = (double)(lse - pos_mean); c_full = 1.0;
        if (nneg > 0 && a.topk >= 1) { l_mined = (double)(lse_m - pos_mean); c_mined = 1.0; }
      }
      w = (double)wsum;
      if (bad) {   // fill level out of range: NaN loss (c_full = 1 so that the loss reads the NaN sum)
        so[SUPCON_ST_LSE] = so[SUPCON_ST_LSE_M] = NAN;
        l_full = l_mined = w = NAN; c_full = 1.0;
      }
    }
    red[0 * BM + pr] = l_full; red[1 * BM + pr] = c_full; red[2 * BM + pr] = l_mined;
    red[3 * BM + pr] = c_mined; red[4 * BM + pr] = w;
  }
  __syncthreads();
  FinishArgs fa{a.block_partials, a.ticket, a.partials, a.loss_out, a.n_batch, a.tau, a.alpha, a.lambda_uni, a.uni_t};
  block_partials_and_finish(fa, red, BM);
}

// combine the column splits of ffma_fwd_kernel: online-max merge of the sums, (value desc, index asc) merge of
// the candidate lists, then the same row statistics / loss partials as the single-sweep kernel
__global__ void __launch_bounds__(128) ffma_fwd_merge_kernel(FfmaArgs a) {
  __shared__ double red[5 * 128];
  const int lr = blockIdx.x * 128 + threadIdx.x;
  double l_full = 0.0, c_full = 0.0, l_mined = 0.0, c_mined = 0.0, w = 0.0;
  if (lr < a.n_rows) {
    float M = -INFINITY;
    for (int s = 0; s < a.splits; ++s) M = fmaxf(M, a.part[((int64_t)s * a.rows_pad + lr) * 8]);
    float sum_all = 0.f, sum_pos_e = 0.f, sum_pos_s = 0.f, wsum = 0.f;
    int npos = 0, nneg = 0;
    for (int s = 0; s < a.splits; ++s) {
      const float* rec = a.part + ((int64_t)s * a.rows_pad + lr) * 8;
      const float f = (rec[0] == -INFINITY) ? 0.f : expf(rec[0] - M);
      sum_all += rec[1] * f; sum_pos_e += rec[2] * f; sum_pos_s += rec[3]; wsum += rec[4];
      npos += reinterpret_cast<const int*>(rec)[5]; nneg += reinterpret_cast<const int*>(rec)[6];
    }
    const float lse = M + logf(sum_all);
    float lse_m = lse, thr_val = -INFINITY;
    int thr_idx = SUPCON_INT_MAX;
    if (a.mine && nneg > a.topk) {
      const int K = a.topk;   // <= kcap <= 128 when the sweep is split
      float mv[128];
      int mi[128];
      int cnt = 0;
      for (int s = 0; s < a.splits; ++s) {
        const int64_t rec = (int64_t)s * a.rows_pad + lr;
        const int c = reinterpret_cast<const int*>(a.part + rec * 8)[7];
        for (int e = 0; e < c; ++e) {
          const float v = a.lv_part[rec * a.kcap + e];
          const int ix = a.li_part[rec * a.kcap + e];
          int p;
          if (cnt < K) p = cnt++;
          else if (v > mv[K - 1] || (v == mv[K - 1] && ix < mi[K - 1])) p = K - 1;
          else break;
          while (p > 0 && (mv[p - 1] < v || (mv[p - 1] == v && mi[p - 1] > ix))) { mv[p] = mv[p - 1]; mi[p] = mi[p - 1]; --p; }
          mv[p] = v; mi[p] = ix;
        }
      }
      float sum_top = 0.f;
      for (int e = 0; e < K; ++e) sum_top += expf(__fdiv_rn(mv[e], a.tau) - M);
      lse_m = M + logf(sum_pos_e + sum_top);
      thr_val = mv[K - 1];
      thr_idx = mi[K - 1];
    } else if (a.topk < 1) {
      thr_val = INFINITY; thr_idx = -1;
    }
    const float pos_mean = (npos > 0) ? __fdiv_rn(__fdiv_rn(sum_pos_s, a.tau), (float)npos) : 0.f;
    float* so = a.row_stats + (int64_t)lr * SUPCON_STATS_STRIDE;
    so[SUPCON_ST_LSE] = lse; so[SUPCON_ST_LSE_M] = lse_m;
    reinterpret_cast<int*>(so)[SUPCON_ST_NPOS] = npos; reinterpret_cast<int*>(so)[SUPCON_ST_NNEG] = nneg;
    so[SUPCON_ST_THR_VAL] = thr_val; reinterpret_cast<int*>(so)[SUPCON_ST_THR_IDX] = thr_idx;
    so[SUPCON_ST_WSUM] = wsum; so[SUPCON_ST_POS_MEAN] = pos_mean;
    if (npos > 0) {
      l_full = (double)(lse - pos_mean); c_full = 1.0;
      if (nneg > 0 && a.topk >= 1) { l_mined = (double)(lse_m - pos_mean); c_mined = 1.0; }
    }
    w = (double)wsum;
    if (live_columns(a.mem_filled, a.n_rows, a.n_total) < 0) {   // as in ffma_fwd_kernel
      so[SUPCON_ST_LSE] = so[SUPCON_ST_LSE_M] = NAN;
      l_full = l_mined = w = NAN; c_full = 1.0;
    }
  }
  red[0 * 128 + threadIdx.x] = l_full; red[1 * 128 + threadIdx.x] = c_full; red[2 * 128 + threadIdx.x] = l_mined;
  red[3 * 128 + threadIdx.x] = c_mined; red[4 * 128 + threadIdx.x] = w;
  __syncthreads();
  FinishArgs fa{a.block_partials, a.ticket, a.partials, a.loss_out, a.n_batch, a.tau, a.alpha, a.lambda_uni, a.uni_t};
  block_partials_and_finish(fa, red, 128);
}

// sum the column splits of ffma_bwd_kernel, add the uniformity diagonal term, scale by grad_out, convert
template <typename T, typename TO>
__global__ void __launch_bounds__(256) ffma_bwd_reduce_kernel(FfmaArgs a) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)a.n_rows * a.d) return;
  const int lr = (int)(idx / a.d), dd = (int)(idx % a.d);
  float v = 0.f;
  for (int s = 0; s < a.splits; ++s) v += a.dz_part[((int64_t)s * a.rows_pad + lr) * a.d + dd];
  const GlobalCoef g = global_coef(a.partials, a.n_batch, a.tau, a.alpha, a.lambda_uni, a.uni_t);
  const int gi = a.row_offset + lr;
  if (g.cu != 0.f)
    v = fmaf(g.cu * a.stats_all[(int64_t)gi * SUPCON_STATS_STRIDE + SUPCON_ST_WSUM],
             ld_elem<T>(reinterpret_cast<const T*>(a.z) + (int64_t)gi * a.d + dd), v);
  v *= a.grad_out ? *a.grad_out : 1.0f;
  if (live_columns(a.mem_filled, a.n_rows, a.n_total) < 0) v = NAN;
  TO* out = reinterpret_cast<TO*>(a.dz_out);
  if constexpr (sizeof(TO) == 4) out[idx] = v;
  else out[idx] = __float2bfloat16(v);
}

// ---------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------
__device__ __forceinline__ void load_coef(const FfmaArgs& a, const GlobalCoef& g, int gidx, bool ok, float* f,
                                          int* n, int slot, int stride) {
  // layout: f[0]=lse f[1]=rm f[2]=af f[3]=am f[4]=bp f[5]=thr ; n[0]=thr_idx n[1]=lab
  float lse = 0.f, rm = 0.f, af = 0.f, am = 0.f, bp = 0.f, thr = INFINITY;
  int ti = -1, lab = 0;
  if (ok && gidx >= a.n_batch) {
    // memory column (SUPCON_FLAG_MEMORY_COLUMNS): its label decides the row side's positives, but it has no
    // statistics and no column-side term; lse = +inf makes its exp(s/tau - lse) exactly 0
    lse = INFINITY;
    lab = a.labels[gidx];
    ok = false;
  }
  if (ok) {
    const float* s = a.stats_all + (int64_t)gidx * SUPCON_STATS_STRIDE;
    const int* si = reinterpret_cast<const int*>(s);
    int npos = si[SUPCON_ST_NPOS], nneg = si[SUPCON_ST_NNEG];
    lse = s[SUPCON_ST_LSE];
    bool in_f = npos > 0;
    bool in_m = in_f && nneg > 0 && a.topk >= 1;
    af = in_f ? g.a_full : 0.f;
    am = in_m ? g.a_mined : 0.f;
    rm = (am != 0.f) ? expf(lse - s[SUPCON_ST_LSE_M]) : 0.f;
    bp = in_f ? __fdiv_rn(af + am, (float)npos) : 0.f;
    thr = s[SUPCON_ST_THR_VAL];
    ti = si[SUPCON_ST_THR_IDX];
    lab = a.labels[gidx];
  }
  f[0 * stride + slot] = lse; f[1 * stride + slot] = rm; f[2 * stride + slot] = af;
  f[3 * stride + slot] = am; f[4 * stride + slot] = bp; f[5 * stride + slot] = thr;
  n[0 * stride + slot] = ti; n[1 * stride + slot] = lab;
}

template <typename T, typename TO>
__global__ void __launch_bounds__(NT) ffma_bwd_kernel(FfmaArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* As = reinterpret_cast<float*>(smem_raw);
  float* Bs = As + BM * LDT;
  float* Hs = Bs + BN * LDT;         // [BM][LDS_]
  float* Zs = Hs + BM * LDS_;        // [BN][DC]
  float* nrm_r = Zs + BN * DC;
  float* nrm_c = nrm_r + BM;
  float* rf = nrm_c + BN;            // [6][BM]
  float* cf = rf + 6 * BM;           // [6][BN]
  int* rn = reinterpret_cast<int*>(cf + 6 * BN);  // [2][BM]
  int* cn = rn + 2 * BM;                          // [2][BN]

  const T* z = reinterpret_cast<const T*>(a.z);
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const int row0 = a.row_offset + blockIdx.x * BM;
  const int row_end = a.row_offset + a.n_rows;
  const int dc0 = blockIdx.y * DC;
  const bool geo = a.similarity == SUPCON_GEODESIC;
  const GlobalCoef g = global_coef(a.partials, a.n_batch, a.tau, a.alpha, a.lambda_uni, a.uni_t);
  const bool uni = g.cu != 0.f;
  const bool mining = g.a_mined != 0.f;
  const int n_live = live_columns(a.mem_filled, a.n_rows, a.n_total);
  const int n_cols = n_live < 0 ? a.n_total : n_live;   // columns [n_cols, n_total) are absent

  if (tid < BM) load_coef(a, g, row0 + tid, row0 + tid < row_end, rf, rn, tid, BM);

  float dz[4][16];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int e = 0; e < 16; ++e) dz[i][e] = 0.f;

  const int split = blockIdx.z;
  const int c_lo = (int)(((int64_t)a.col_tiles * split) / a.splits) * BN;
  const int c_hi = min(n_cols, (int)(((int64_t)a.col_tiles * (split + 1)) / a.splits) * BN);
  float acc[4][4];
  for (int col0 = c_lo; col0 < c_hi; col0 += BN) {
    gram_tile<T>(z, a.d, a.vec_ok, row0, row_end, col0, n_cols, As, Bs, acc, nrm_r, nrm_c, uni);
    if (tid < BN) load_coef(a, g, col0 + tid, col0 + tid < n_cols, cf, cn, tid, BN);
    // stage Z_J[:, dc0:dc0+DC] (fp32) for the H.Z product
    for (int idx = tid; idx < BN * (DC / 4); idx += NT) {
      int r = idx / (DC / 4), q = idx % (DC / 4);
      int gc = col0 + r;
      float4 v = ld_row4<T>(z, gc, gc < n_cols, dc0 + 4 * q, a.d, a.vec_ok);
      *reinterpret_cast<float4*>(&Zs[r * DC + 4 * q]) = v;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int r = ty + 16 * i, c = tx + 16 * j;
        const int gi = row0 + r, gj = col0 + c;
        float h = 0.f;
        if (gi < row_end && gj < n_cols && gi != gj) {
          const float cv = acc[i][j];
          const float s = geo ? geodesic_sim(cv) : cv;
          const float lg = __fdiv_rn(s, a.tau);
          const float e_r = expf(lg - rf[0 * BM + r]);
          const float e_c = expf(lg - cf[0 * BN + c]);
          const bool pos = rn[1 * BM + r] == cn[1 * BN + c];
          h = rf[2 * BM + r] * e_r + cf[2 * BN + c] * e_c;
          if (mining) {
            bool mem_r = pos || s > rf[5 * BM + r] || (s == rf[5 * BM + r] && gj <= rn[0 * BM + r]);
            bool mem_c = pos || s > cf[5 * BN + c] || (s == cf[5 * BN + c] && gi <= cn[0 * BN + c]);
            if (mem_r) h = fmaf(rf[3 * BM + r] * rf[1 * BM + r], e_r, h);
            if (mem_c) h = fmaf(cf[3 * BN + c] * cf[1 * BN + c], e_c, h);
          }
          if (pos) h -= rf[4 * BM + r] + cf[4 * BN + c];
          if (geo) h *= geodesic_slope_exact(cv);
          if (uni && gj < a.n_batch) {   // memory columns: no uniformity
            float d2 = fmaxf(nrm_r[r] + nrm_c[c] - 2.f * cv, 0.f);
            h = fmaf(-g.cu, expf(-a.uni_t * d2), h);
          }
        }
        Hs[r * LDS_ + c] = h;
      }
    __syncthreads();
    // dz[rows][dd] += H[rows][:] . Z_J[:][dd]
#pragma unroll 2
    for (int jj = 0; jj < BN; jj += 4) {
      float4 h4[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) h4[i] = *reinterpret_cast<const float4*>(&Hs[(ty + 16 * i) * LDS_ + jj]);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float4 zv[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) zv[q] = *reinterpret_cast<const float4*>(&Zs[(jj + u) * DC + 4 * tx + 64 * q]);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float hv = (u == 0) ? h4[i].x : (u == 1) ? h4[i].y : (u == 2) ? h4[i].z : h4[i].w;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            dz[i][4 * q + 0] = fmaf(hv, zv[q].x, dz[i][4 * q + 0]);
            dz[i][4 * q + 1] = fmaf(hv, zv[q].y, dz[i][4 * q + 1]);
            dz[i][4 * q + 2] = fmaf(hv, zv[q].z, dz[i][4 * q + 2]);
            dz[i][4 * q + 3] = fmaf(hv, zv[q].w, dz[i][4 * q + 3]);
          }
        }
      }
    }
    __syncthreads();
  }

  if (a.splits > 1) {   // raw partial sums of this column range; ffma_bwd_reduce_kernel finishes them
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int gi = row0 + ty + 16 * i;
      if (gi >= row_end) continue;
      float* prow = a.dz_part + ((int64_t)split * a.rows_pad + (gi - a.row_offset)) * a.d;
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int dd = dc0 + 4 * tx + 64 * q + e;
          if (dd < a.d) prow[dd] = dz[i][4 * q + e];
        }
    }
    return;
  }
  const float gscale = n_live < 0 ? NAN : (a.grad_out ? *a.grad_out : 1.0f);
  TO* out = reinterpret_cast<TO*>(a.dz_out);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gi = row0 + ty + 16 * i;
    if (gi >= row_end) continue;
    float wdiag = 0.f;
    if (uni) wdiag = g.cu * a.stats_all[(int64_t)gi * SUPCON_STATS_STRIDE + SUPCON_ST_WSUM];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int dd = dc0 + 4 * tx + 64 * q + e;
        if (dd >= a.d) continue;
        float v = dz[i][4 * q + e];
        if (uni) v = fmaf(wdiag, ld_elem<T>(z + (int64_t)gi * a.d + dd), v);
        v *= gscale;
        if constexpr (sizeof(TO) == 4) out[(int64_t)(gi - a.row_offset) * a.d + dd] = v;
        else out[(int64_t)(gi - a.row_offset) * a.d + dd] = __float2bfloat16(v);
      }
  }
}

// hard-negative index sets (diagnostic): ascending column order, -1 padded
template <typename T>
__global__ void __launch_bounds__(NT) ffma_topk_idx_kernel(FfmaArgs a, int32_t* idx_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* As = reinterpret_cast<float*>(smem_raw);
  float* Bs = As + BM * LDT;
  float* Ss = Bs + BN * LDT;
  int* lab_c = reinterpret_cast<int*>(Ss + BM * LDS_);
  const T* z = reinterpret_cast<const T*>(a.z);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int row0 = a.row_offset + blockIdx.x * BM;
  const int row_end = a.row_offset + a.n_rows;
  const bool geo = a.similarity == SUPCON_GEODESIC;
  int filled = 0;
  float thr = 0.f; int thr_idx = 0, lab_r = 0;
  const int gi = row0 + tid;
  const bool owner = tid < BM && gi < row_end;
  if (owner) {
    const float* s = a.row_stats + (int64_t)(gi - a.row_offset) * SUPCON_STATS_STRIDE;
    thr = s[SUPCON_ST_THR_VAL];
    thr_idx = reinterpret_cast<const int*>(s)[SUPCON_ST_THR_IDX];
    lab_r = a.labels[gi];
  }
  float acc[4][4];
  for (int col0 = 0; col0 < a.n_total; col0 += BN) {
    gram_tile<T>(z, a.d, a.vec_ok, row0, row_end, col0, a.n_total, As, Bs, acc, nullptr, nullptr, false);
    if (tid < BN) lab_c[tid] = (col0 + tid < a.n_total) ? a.labels[col0 + tid] : 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j)
        Ss[(ty + 16 * i) * LDS_ + tx + 16 * j] = geo ? geodesic_sim(acc[i][j]) : acc[i][j];
    __syncthreads();
    if (owner) {
      for (int c = 0; c < BN; ++c) {
        int gj = col0 + c;
        if (gj >= a.n_total || lab_c[c] == lab_r) continue;
        float s = Ss[tid * LDS_ + c];
        if ((s > thr || (s == thr && gj <= thr_idx)) && filled < a.topk)
          idx_out[(int64_t)(gi - a.row_offset) * a.topk + filled++] = gj;
      }
    }
    __syncthreads();
  }
  if (owner)
    for (; filled < a.topk; ++filled) idx_out[(int64_t)(gi - a.row_offset) * a.topk + filled] = -1;
}

size_t fwd_smem_bytes(int kcap) {
  size_t f = (size_t)(BM * LDT + BN * LDT + 2 * BM * LDS_ + BM + BN) * 4 + (size_t)(BN + BM) * 4;
  f = (f + 7) & ~(size_t)7;
  f += 5 * BM * sizeof(double);
  f += (size_t)BM * kcap * 8;
  return f;
}
size_t bwd_smem_bytes() {
  return (size_t)(BM * LDT + BN * LDT + BM * LDS_ + BN * DC + BM + BN + 6 * BM + 6 * BN) * 4 +
         (size_t)(2 * BM + 2 * BN) * 4;
}
size_t topk_smem_bytes() { return (size_t)(BM * LDT + BN * LDT + BM * LDS_) * 4 + BN * 4; }

template <typename K>
cudaError_t set_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

}  // namespace

int ffma_kcap() { return 128; }

namespace {
int ffma_num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}
size_t up256(size_t x) { return (x + 255) / 256 * 256; }
}  // namespace

// Column splits: with 64-row blocks a mid-size batch (N ~ 1k) gives only a handful of CTAs, so the column
// sweep is cut into ranges (blockIdx.y / .z) until ~2 CTAs per SM exist; partial records / partial dz go
// through the workspace and a merge / reduce kernel.
FfmaPlan ffma_plan(const supcon_problem_t* p) {
  FfmaPlan pl;
  const int row_blocks = (p->n_rows + BM - 1) / BM;
  pl.col_tiles = (p->n_total + BN - 1) / BN;
  pl.rows_pad = row_blocks * BM;
  const bool mine = p->alpha != 0.f && p->topk >= 1;
  const int topk = p->topk < 0 ? 0 : p->topk;
  pl.kcap = mine ? (topk < ffma_kcap() ? topk : ffma_kcap()) : 0;
  const int dchunks = (p->d + DC - 1) / DC;
  const int max_s = pl.col_tiles / 4 > 0 ? pl.col_tiles / 4 : 1;
  int sf = (2 * ffma_num_sms()) / row_blocks;
  int sb = (2 * ffma_num_sms()) / (row_blocks * dchunks);
  if (mine && topk > ffma_kcap()) sf = 1;   // multi-round selection needs the whole sweep in one CTA
  pl.fwd_splits = sf < 1 ? 1 : (sf > max_s ? max_s : sf);
  pl.bwd_splits = sb < 1 ? 1 : (sb > max_s ? max_s : sb);
  if (pl.fwd_splits > 64) pl.fwd_splits = 64;
  if (pl.bwd_splits > 64) pl.bwd_splits = 64;
  pl.merge_blocks = (p->n_rows + 127) / 128;
  size_t off = 256;
  const int finish_blocks = row_blocks > pl.merge_blocks ? row_blocks : pl.merge_blocks;
  pl.off_block_partials = off; off += up256((size_t)finish_blocks * SUPCON_N_PARTIALS * sizeof(double));
  pl.off_part = off; off += up256(pl.fwd_splits > 1 ? (size_t)pl.fwd_splits * pl.rows_pad * 8 * 4 : 0);
  pl.off_lv = off; off += up256(pl.fwd_splits > 1 ? (size_t)pl.fwd_splits * pl.rows_pad * pl.kcap * 4 : 0);
  pl.off_li = off; off += up256(pl.fwd_splits > 1 ? (size_t)pl.fwd_splits * pl.rows_pad * pl.kcap * 4 : 0);
  pl.off_dz = off; off += up256(pl.bwd_splits > 1 ? (size_t)pl.bwd_splits * pl.rows_pad * p->d * 4 : 0);
  pl.total_bytes = off;
  return pl;
}

size_t ffma_workspace_bytes(const supcon_problem_t* p) { return ffma_plan(p).total_bytes; }

void ffma_bind_plan(FfmaArgs& a, const FfmaPlan& pl, void* workspace, bool backward) {
  char* ws = reinterpret_cast<char*>(workspace);
  a.ticket = reinterpret_cast<unsigned*>(ws);
  a.block_partials = reinterpret_cast<double*>(ws + pl.off_block_partials);
  a.part = reinterpret_cast<float*>(ws + pl.off_part);
  a.lv_part = reinterpret_cast<float*>(ws + pl.off_lv);
  a.li_part = reinterpret_cast<int*>(ws + pl.off_li);
  a.dz_part = reinterpret_cast<float*>(ws + pl.off_dz);
  a.col_tiles = pl.col_tiles;
  a.rows_pad = pl.rows_pad;
  a.splits = backward ? pl.bwd_splits : pl.fwd_splits;
}

cudaError_t ffma_forward(const FfmaArgs& a, cudaStream_t stream) {
  dim3 grid((a.n_rows + BM - 1) / BM, a.splits);
  const size_t smem = fwd_smem_bytes(a.kcap);
  cudaError_t e;
  if (a.z_dtype == SUPCON_BF16) {
    if ((e = set_smem(ffma_fwd_kernel<__nv_bfloat16>, smem)) != cudaSuccess) return e;
    ffma_fwd_kernel<__nv_bfloat16><<<grid, NT, smem, stream>>>(a);
  } else {
    if ((e = set_smem(ffma_fwd_kernel<float>, smem)) != cudaSuccess) return e;
    ffma_fwd_kernel<float><<<grid, NT, smem, stream>>>(a);
  }
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if (a.splits > 1) {
    ffma_fwd_merge_kernel<<<(a.n_rows + 127) / 128, 128, 0, stream>>>(a);
    e = cudaGetLastError();
  }
  return e;
}

cudaError_t ffma_backward(const FfmaArgs& a, int dz_dtype, cudaStream_t stream) {
  dim3 grid((a.n_rows + BM - 1) / BM, (a.d + DC - 1) / DC, a.splits);
  const size_t smem = bwd_smem_bytes();
  const int rblocks = (int)(((int64_t)a.n_rows * a.d + 255) / 256);
  cudaError_t e;
#define SUPCON_LAUNCH_BWD(TI, TO)                                              \
  do {                                                                         \
    if ((e = set_smem(ffma_bwd_kernel<TI, TO>, smem)) != cudaSuccess) return e; \
    ffma_bwd_kernel<TI, TO><<<grid, NT, smem, stream>>>(a);                    \
    if (a.splits > 1) ffma_bwd_reduce_kernel<TI, TO><<<rblocks, 256, 0, stream>>>(a); \
  } while (0)
  if (a.z_dtype == SUPCON_BF16) {
    if (dz_dtype == SUPCON_BF16) SUPCON_LAUNCH_BWD(__nv_bfloat16, __nv_bfloat16);
    else SUPCON_LAUNCH_BWD(__nv_bfloat16, float);
  } else {
    if (dz_dtype == SUPCON_BF16) SUPCON_LAUNCH_BWD(float, __nv_bfloat16);
    else SUPCON_LAUNCH_BWD(float, float);
  }
#undef SUPCON_LAUNCH_BWD
  return cudaGetLastError();
}

cudaError_t ffma_topk_indices(const FfmaArgs& a, int32_t* idx_out, cudaStream_t stream) {
  const int blocks = (a.n_rows + BM - 1) / BM;
  const size_t smem = topk_smem_bytes();
  cudaError_t e;
  if (a.z_dtype == SUPCON_BF16) {
    if ((e = set_smem(ffma_topk_idx_kernel<__nv_bfloat16>, smem)) != cudaSuccess) return e;
    ffma_topk_idx_kernel<__nv_bfloat16><<<blocks, NT, smem, stream>>>(a, idx_out);
  } else {
    if ((e = set_smem(ffma_topk_idx_kernel<float>, smem)) != cudaSuccess) return e;
    ffma_topk_idx_kernel<float><<<blocks, NT, smem, stream>>>(a, idx_out);
  }
  return cudaGetLastError();
}

}  // namespace supcon
