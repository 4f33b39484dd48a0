// Single-launch SupCon forward + backward for MID-SIZE batches, 160 < N <= 320 -- the reference's own default
// batch (stage1_config.py:22 BATCH_SIZE = 256) in its own dtype (fp32).  Same plan as supcon_small.cu (one
// thread-block cluster, exact fp32 FFMA dot products in one fixed k-order, warp-per-row statistics, row
// statistics exchanged through distributed shared memory between two cluster barriers, then H rows and dz rows)
// with two differences that lift the size limit:
//   * only the CTA's OWN rows of z are staged in shared memory; the columns stream from global memory (z is
//     <= 512 KB and L2-resident: every CTA reads it twice), so shared memory no longer has to hold all of z;
//   * the cluster has 16 CTAs (non-portable size; 8 when the device cannot co-schedule 16), up to 32 rows each.
// At these sizes the tiled exact path needs 5 launches and ~180 us (N = 256); this kernel is one launch and takes
// 107 us (N = 256, profiles/r02_small_batch_times.md).  Keeping two loads in flight by hand made it slower (125 us).
//
// c_ij is accumulated as ONE fma chain over k = 0..d-1, so c_ij == c_ji bit for bit and the backward's
// hard-negative membership test (threshold value + index) sees exactly the forward's values.
#include <cooperative_groups.h>

#include "supcon_common.cuh"
#include "supcon_internal.h"

namespace cg = cooperative_groups;

namespace supcon {
namespace {

constexpr int MNT = 256;     // threads per CTA
constexpr int MMAXR = 32;    // owned rows per CTA
constexpr int MMAXN = 320;   // columns (measured: from ~384 rows on the tiled kernels' many CTAs are as fast)
constexpr int MCOLS = MMAXN / 32;   // columns per lane in the statistics phase

struct MidLayout {
  int ld, np;
  size_t off_z, off_c, off_h, off_nrm, off_lab, off_stats_local, off_stats_all, off_part, total;
};

__host__ __device__ inline MidLayout mid_layout(int n, int d, int rows) {
  MidLayout L;
  L.ld = d + 4;
  L.np = (n + 31) / 32 * 32;
  size_t o = 0;
  L.off_z = o; o += (size_t)rows * L.ld * 4;          // own rows only
  L.off_c = o; o += (size_t)rows * L.np * 4;
  L.off_h = o; o += (size_t)rows * L.np * 4;
  L.off_nrm = o; o += (size_t)L.np * 4;
  L.off_lab = o; o += (size_t)L.np * 4;
  L.off_stats_local = o; o += (size_t)rows * SUPCON_STATS_STRIDE * 4;
  L.off_stats_all = o; o += (size_t)L.np * SUPCON_STATS_STRIDE * 4;
  o = (o + 7) & ~(size_t)7;
  L.off_part = o; o += SUPCON_N_PARTIALS * sizeof(double);
  L.total = o;
  return L;
}

template <typename T, typename TO>
__global__ void __launch_bounds__(MNT, 1) mid_kernel(SmallArgs a) {
  extern __shared__ __align__(16) unsigned char smem[];
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank();
  const int SC = (int)cluster.num_blocks();
  const int n = a.n, d = a.d;
  const int R = (n + SC - 1) / SC;
  const MidLayout L = mid_layout(n, d, R);
  float* zs = reinterpret_cast<float*>(smem + L.off_z);      // own rows [R][ld]
  float* cs = reinterpret_cast<float*>(smem + L.off_c);      // dot products of owned rows [R][np]
  float* hs = reinterpret_cast<float*>(smem + L.off_h);      // H rows [R][np]
  float* nrm = reinterpret_cast<float*>(smem + L.off_nrm);
  int* lab = reinterpret_cast<int*>(smem + L.off_lab);
  float* st_local = reinterpret_cast<float*>(smem + L.off_stats_local);
  float* st_all = reinterpret_cast<float*>(smem + L.off_stats_all);
  double* part = reinterpret_cast<double*>(smem + L.off_part);

  const T* z = reinterpret_cast<const T*>(a.z);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int r0 = rank * R;
  const int nrows = max(0, min(R, n - r0));
  const bool geo = a.similarity == SUPCON_GEODESIC;
  const bool uni = a.lambda_uni > 0.f;
  const bool mine = a.mine != 0;

  // ---- A0: stage the own rows (fp32) and all labels ----
  for (int idx = tid; idx < nrows * (d / 4); idx += MNT) {
    const int r = idx / (d / 4), q = idx % (d / 4);
    *reinterpret_cast<float4*>(&zs[r * L.ld + 4 * q]) = ld_row4<T>(z, r0 + r, true, 4 * q, d, true);
  }
  for (int j = tid; j < L.np; j += MNT) lab[j] = j < n ? a.labels[j] : 0;
  __syncthreads();

  // ---- A2: dot products c[r][j] of the owned rows against every column (streamed from global / L2);
  //      thread = column; one fma chain over k per (r, j); the squared norm of the column rides along ----
  for (int j = tid; j < L.np; j += MNT) {
    float acc[MMAXR];
#pragma unroll
    for (int r = 0; r < MMAXR; ++r) acc[r] = 0.f;
    float nj = 0.f;
    if (j < n) {
      for (int k = 0; k < d; k += 4) {
        const float4 b = ld_row4<T>(z, j, true, k, d, true);
        nj = fmaf(b.x, b.x, nj); nj = fmaf(b.y, b.y, nj); nj = fmaf(b.z, b.z, nj); nj = fmaf(b.w, b.w, nj);
#pragma unroll
        for (int r = 0; r < MMAXR; ++r) {
          if (r < nrows) {
            const float4 av = *reinterpret_cast<const float4*>(&zs[r * L.ld + k]);
            float c = acc[r];
            c = fmaf(av.x, b.x, c); c = fmaf(av.y, b.y, c); c = fmaf(av.z, b.z, c); c = fmaf(av.w, b.w, c);
            acc[r] = c;
          }
        }
      }
    }
    nrm[j] = nj;
#pragma unroll
    for (int r = 0; r < MMAXR; ++r)
      if (r < R) cs[r * L.np + j] = acc[r];
  }
  __syncthreads();

  // ---- B: row statistics, one warp per owned row ----
  double acc_full = 0.0, acc_cf = 0.0, acc_mined = 0.0, acc_cm = 0.0, acc_w = 0.0;
  const int ncq = L.np / 32;
  for (int r = warp; r < nrows; r += MNT / 32) {
    const int gi = r0 + r;
    const int lab_r = lab[gi];
    float sv[MCOLS];
    float m = -INFINITY;
#pragma unroll
    for (int q = 0; q < MCOLS; ++q) {
      const int j = lane + 32 * q;
      sv[q] = -INFINITY;
      if (q < ncq && j < n && j != gi) {
        const float c = cs[r * L.np + j];
        sv[q] = geo ? geodesic_sim(c) : c;
        m = fmaxf(m, __fdiv_rn(sv[q], a.tau));
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float sum_all = 0.f, sum_pos_e = 0.f, sum_pos_s = 0.f, wsum = 0.f;
    int npos = 0, nneg = 0;
    unsigned negmask = 0;
#pragma unroll
    for (int q = 0; q < MCOLS; ++q) {
      const int j = lane + 32 * q;
      if (q < ncq && j < n && j != gi) {
        const float e = expf(__fdiv_rn(sv[q], a.tau) - m);
        sum_all += e;
        if (lab[j] == lab_r) { npos++; sum_pos_e += e; sum_pos_s += sv[q]; }
        else { nneg++; negmask |= 1u << q; }
        if (uni) {
          const float d2 = fmaxf(nrm[gi] + nrm[j] - 2.f * cs[r * L.np + j], 0.f);
          wsum += expf(-a.uni_t * d2);
        }
      }
    }
    sum_all = warp_sum(sum_all); sum_pos_e = warp_sum(sum_pos_e); sum_pos_s = warp_sum(sum_pos_s);
    wsum = warp_sum(wsum);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      npos += __shfl_xor_sync(0xffffffffu, npos, o);
      nneg += __shfl_xor_sync(0xffffffffu, nneg, o);
    }
    const float lse = m + logf(sum_all);
    float lse_m = lse, thr_val = -INFINITY;
    int thr_idx = SUPCON_INT_MAX;
    if (mine && nneg > a.topk) {
      // K rounds of warp arg-max over the not-yet-selected negatives, order (value desc, index asc)
      float sum_top = 0.f;
      unsigned avail = negmask;
      for (int round = 0; round < a.topk; ++round) {
        float bv = -INFINITY;
        int bj = SUPCON_INT_MAX;
#pragma unroll
        for (int q = 0; q < MCOLS; ++q)
          if ((avail >> q) & 1u) {
            const int j = lane + 32 * q;
            if (sv[q] > bv || (sv[q] == bv && j < bj)) { bv = sv[q]; bj = j; }
          }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
          if (ov > bv || (ov == bv && oj < bj)) { bv = ov; bj = oj; }
        }
        if ((bj & 31) == lane) avail &= ~(1u << (bj >> 5));
        sum_top += expf(__fdiv_rn(bv, a.tau) - m);
        thr_val = bv; thr_idx = bj;
      }
      lse_m = m + logf(sum_pos_e + sum_top);
    } else if (a.topk < 1) {
      thr_val = INFINITY; thr_idx = -1;
    }
    if (lane == 0) {
      const float pos_mean = npos > 0 ? __fdiv_rn(__fdiv_rn(sum_pos_s, a.tau), (float)npos) : 0.f;
      float* so = st_local + r * SUPCON_STATS_STRIDE;
      so[SUPCON_ST_LSE] = lse; so[SUPCON_ST_LSE_M] = lse_m;
      reinterpret_cast<int*>(so)[SUPCON_ST_NPOS] = npos; reinterpret_cast<int*>(so)[SUPCON_ST_NNEG] = nneg;
      so[SUPCON_ST_THR_VAL] = thr_val; reinterpret_cast<int*>(so)[SUPCON_ST_THR_IDX] = thr_idx;
      so[SUPCON_ST_WSUM] = wsum; so[SUPCON_ST_POS_MEAN] = pos_mean;
      if (a.row_stats) {
        float* go = a.row_stats + (int64_t)gi * SUPCON_STATS_STRIDE;
#pragma unroll
        for (int w = 0; w < SUPCON_STATS_STRIDE; ++w) go[w] = so[w];
      }
      if (npos > 0) {
        acc_full += (double)(lse - pos_mean); acc_cf += 1.0;
        if (nneg > 0 && a.topk >= 1) { acc_mined += (double)(lse_m - pos_mean); acc_cm += 1.0; }
      }
      acc_w += (double)wsum;
    }
  }
  {
    __shared__ double wred[MNT / 32][5];
    if (lane == 0) {
      wred[warp][0] = acc_full; wred[warp][1] = acc_cf; wred[warp][2] = acc_mined; wred[warp][3] = acc_cm;
      wred[warp][4] = acc_w;
    }
    __syncthreads();
    if (tid < SUPCON_N_PARTIALS) {
      double s = 0.0;
      if (tid < 5)
        for (int w = 0; w < MNT / 32; ++w) s += wred[w][tid];
      part[tid] = s;
    }
  }
  cluster.sync();  // C: statistics and partials of every CTA are complete

  // ---- gather through distributed shared memory ----
  for (int idx = tid; idx < n * SUPCON_STATS_STRIDE; idx += MNT) {
    const int i = idx / SUPCON_STATS_STRIDE, w = idx % SUPCON_STATS_STRIDE;
    const float* remote = cluster.map_shared_rank(st_local, i / R);
    st_all[idx] = remote[(i % R) * SUPCON_STATS_STRIDE + w];
  }
  __shared__ double gpart[SUPCON_N_PARTIALS];
  if (tid < SUPCON_N_PARTIALS) {
    double s = 0.0;
    for (int c = 0; c < SC; ++c) s += cluster.map_shared_rank(part, c)[tid];   // rank order: deterministic
    gpart[tid] = s;
  }
  __syncthreads();
  cluster.sync();  // nobody may leave (or reuse st_local/part) while peers still read them
  const GlobalCoef g = global_coef(gpart, n, a.tau, a.alpha, a.lambda_uni, a.uni_t);
  if (rank == 0 && tid == 0) {
    if (a.loss_out) *a.loss_out = g.loss;
    if (a.partials)
      for (int w = 0; w < SUPCON_N_PARTIALS; ++w) a.partials[w] = gpart[w];
  }
  if (!a.dz_out) return;

  // ---- D1: H rows ----
  const bool mining = g.a_mined != 0.f;
  for (int idx = tid; idx < nrows * L.np; idx += MNT) {
    const int r = idx / L.np, j = idx % L.np;
    const int gi = r0 + r;
    float h = 0.f;
    if (j < n && j != gi) {
      const float* si = st_all + gi * SUPCON_STATS_STRIDE;
      const float* sj = st_all + j * SUPCON_STATS_STRIDE;
      const int npos_i = reinterpret_cast<const int*>(si)[SUPCON_ST_NPOS], nneg_i = reinterpret_cast<const int*>(si)[SUPCON_ST_NNEG];
      const int npos_j = reinterpret_cast<const int*>(sj)[SUPCON_ST_NPOS], nneg_j = reinterpret_cast<const int*>(sj)[SUPCON_ST_NNEG];
      const float af_i = npos_i > 0 ? g.a_full : 0.f, af_j = npos_j > 0 ? g.a_full : 0.f;
      const float am_i = (npos_i > 0 && nneg_i > 0 && a.topk >= 1) ? g.a_mined : 0.f;
      const float am_j = (npos_j > 0 && nneg_j > 0 && a.topk >= 1) ? g.a_mined : 0.f;
      const float cv = cs[r * L.np + j];
      const float s = geo ? geodesic_sim(cv) : cv;
      const float lg = __fdiv_rn(s, a.tau);
      const float e_r = expf(lg - si[SUPCON_ST_LSE]), e_c = expf(lg - sj[SUPCON_ST_LSE]);
      const bool pos = lab[gi] == lab[j];
      h = af_i * e_r + af_j * e_c;
      if (mining) {
        const float thr_i = si[SUPCON_ST_THR_VAL], thr_j = sj[SUPCON_ST_THR_VAL];
        const int ti = reinterpret_cast<const int*>(si)[SUPCON_ST_THR_IDX], tj = reinterpret_cast<const int*>(sj)[SUPCON_ST_THR_IDX];
        const bool mem_r = pos || s > thr_i || (s == thr_i && j <= ti);
        const bool mem_c = pos || s > thr_j || (s == thr_j && gi <= tj);
        if (mem_r && am_i != 0.f) h = fmaf(am_i * expf(si[SUPCON_ST_LSE] - si[SUPCON_ST_LSE_M]), e_r, h);
        if (mem_c && am_j != 0.f) h = fmaf(am_j * expf(sj[SUPCON_ST_LSE] - sj[SUPCON_ST_LSE_M]), e_c, h);
      }
      if (pos) {
        const float bp_i = npos_i > 0 ? __fdiv_rn(af_i + am_i, (float)npos_i) : 0.f;
        const float bp_j = npos_j > 0 ? __fdiv_rn(af_j + am_j, (float)npos_j) : 0.f;
        h -= bp_i + bp_j;
      }
      if (geo) h *= geodesic_slope_exact(cv);
      if (g.cu != 0.f) {
        const float d2 = fmaxf(nrm[gi] + nrm[j] - 2.f * cv, 0.f);
        h = fmaf(-g.cu, expf(-a.uni_t * d2), h);
      }
    }
    hs[idx] = h;
  }
  __syncthreads();

  // ---- D2: dz rows = H z (+ uniformity diagonal); thread = output column, z read coalesced from global ----
  const float gscale = a.grad_out ? *a.grad_out : 1.0f;
  TO* out = reinterpret_cast<TO*>(a.dz_out);
  for (int dd = tid; dd < d; dd += MNT) {
    float acc[MMAXR];
#pragma unroll
    for (int r = 0; r < MMAXR; ++r) acc[r] = 0.f;
    for (int j = 0; j < L.np; j += 4) {
      float zv[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) zv[u] = (j + u < n) ? ld_elem<T>(z + (int64_t)(j + u) * d + dd) : 0.f;
#pragma unroll
      for (int r = 0; r < MMAXR; ++r) {
        if (r < nrows) {
          const float4 h4 = *reinterpret_cast<const float4*>(&hs[r * L.np + j]);
          float v = acc[r];
          v = fmaf(h4.x, zv[0], v); v = fmaf(h4.y, zv[1], v); v = fmaf(h4.z, zv[2], v); v = fmaf(h4.w, zv[3], v);
          acc[r] = v;
        }
      }
    }
#pragma unroll
    for (int r = 0; r < MMAXR; ++r) {
      if (r < nrows) {
        const int gi = r0 + r;
        float v = acc[r];
        if (g.cu != 0.f) v = fmaf(g.cu * st_all[gi * SUPCON_STATS_STRIDE + SUPCON_ST_WSUM], zs[r * L.ld + dd], v);
        v *= gscale;
        if constexpr (sizeof(TO) == 4) out[(int64_t)gi * d + dd] = v;
        else out[(int64_t)gi * d + dd] = __float2bfloat16(v);
      }
    }
  }
}

template <typename TI, typename TO>
cudaError_t launch_mid(const SmallArgs& a, int cluster_ctas, size_t smem, cudaStream_t stream, bool query_only,
                       int* max_clusters) {
  cudaError_t e = cudaFuncSetAttribute(mid_kernel<TI, TO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  if (cluster_ctas > 8) {
    e = cudaFuncSetAttribute(mid_kernel<TI, TO>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess) return e;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(cluster_ctas, 1, 1);
  cfg.blockDim = dim3(MNT, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster_ctas; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (query_only) return cudaOccupancyMaxActiveClusters(max_clusters, mid_kernel<TI, TO>, &cfg);
  return cudaLaunchKernelEx(&cfg, mid_kernel<TI, TO>, a);
}

template <typename TI, typename TO>
int pick_cluster(const SmallArgs& a) {
  // 16 CTAs when the device can co-schedule such a cluster (asked once per instantiation), else 8 (N <= 256)
  static int can16 = -1;
  if (can16 < 0) {
    int mc = 0;
    const size_t smem = mid_layout(MMAXN, a.d, MMAXN / 16).total;
    cudaError_t e = launch_mid<TI, TO>(a, 16, smem, 0, true, &mc);
    if (e != cudaSuccess) { cudaGetLastError(); mc = 0; }
    can16 = mc > 0 ? 1 : 0;
  }
  if (can16) return 16;
  return a.n <= 8 * MMAXR ? 8 : 0;
}

}  // namespace

bool mid_supported(const supcon_problem_t* p, const void* z) {
  if (p->row_offset != 0 || p->n_rows != p->n_total) return false;
  if (p->n_total > MMAXN || p->n_total < 2) return false;
  if (p->d % 4 != 0 || p->d > 1024) return false;
  if ((reinterpret_cast<uintptr_t>(z) % 16) != 0) return false;
  const bool mine = p->alpha != 0.f && p->topk >= 1;
  if (mine && p->topk > 32 && p->topk < p->n_total - 1) return false;   // K rounds of arg-max: keep it short
  return mid_layout(p->n_total, p->d, MMAXR).total <= 224 * 1024;
}

int mid_cluster_ctas(const SmallArgs& a) {
  typedef __nv_bfloat16 bf;
  if (a.z_dtype == SUPCON_BF16) return a.dz_dtype == SUPCON_BF16 ? pick_cluster<bf, bf>(a) : pick_cluster<bf, float>(a);
  return a.dz_dtype == SUPCON_BF16 ? pick_cluster<float, bf>(a) : pick_cluster<float, float>(a);
}

cudaError_t mid_launch(const SmallArgs& a, cudaStream_t stream, bool* taken) {
  *taken = false;
  const int sc = mid_cluster_ctas(a);
  if (sc == 0) return cudaSuccess;
  const size_t smem = mid_layout(a.n, a.d, (a.n + sc - 1) / sc).total;
  cudaError_t e = cudaSuccess;
#define SUPCON_MID(TI, TO)                                                          \
  do {                                                                              \
    e = launch_mid<TI, TO>(a, sc, smem, stream, false, nullptr);                    \
    *taken = (e == cudaSuccess);                                                    \
  } while (0)
  if (a.z_dtype == SUPCON_BF16) {
    if (a.dz_dtype == SUPCON_BF16) SUPCON_MID(__nv_bfloat16, __nv_bfloat16);
    else SUPCON_MID(__nv_bfloat16, float);
  } else {
    if (a.dz_dtype == SUPCON_BF16) SUPCON_MID(float, __nv_bfloat16);
    else SUPCON_MID(float, float);
  }
#undef SUPCON_MID
  return e;
}

}  // namespace supcon
