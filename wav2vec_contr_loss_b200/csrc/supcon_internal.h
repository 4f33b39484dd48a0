// Internal launch interfaces between the C-ABI dispatcher and the kernel files.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "supcon_b200.h"

namespace supcon {

// Columns [0, n_batch) are the batch: they carry row statistics, get column-side gradient terms and enter the
// uniformity term (whose pair count is n_batch (n_batch - 1) / 2).  n_batch == n_total unless the problem has
// SUPCON_FLAG_MEMORY_COLUMNS, whose columns [n_rows, n_total) are a memory of constants.
inline int batch_columns(const supcon_problem_t* p) {
  return (p->flags & SUPCON_FLAG_MEMORY_COLUMNS) ? p->n_rows : p->n_total;
}

struct FfmaArgs {
  const void* z;             // [n_total][d]
  const int32_t* labels;     // [n_total]
  float* row_stats;          // fwd out / topk-idx in: [n_rows][STRIDE]
  const float* stats_all;    // bwd in: [n_total][STRIDE]
  double* partials;          // fwd: out [8]; bwd: in (global sums)
  float* loss_out;           // fwd: optional
  double* block_partials;    // workspace [blocks][8]
  unsigned* ticket;          // workspace counter (zero between launches)
  const float* grad_out;     // bwd: optional device scalar
  void* dz_out;              // bwd: [n_rows][d]
  int n_total, row_offset, n_rows, d;
  int n_batch;               // batch_columns(): columns from n_batch on are memory (no statistics, no uniformity)
  const int32_t* mem_filled; // device fill level of the memory (live_columns()); nullptr: all n_total columns
  int z_dtype, similarity, topk, kcap, mine, vec_ok;
  float tau, alpha, lambda_uni, uni_t;
  // column splits (ffma_plan): partial records / candidate lists / partial dz in the workspace
  int splits, col_tiles, rows_pad;
  float* part;      // [splits][rows_pad][8]
  float* lv_part;   // [splits][rows_pad][kcap]
  int* li_part;
  float* dz_part;   // [splits][rows_pad][d]
};

struct FfmaPlan {
  int fwd_splits, bwd_splits, col_tiles, rows_pad, kcap, merge_blocks;
  size_t off_block_partials, off_part, off_lv, off_li, off_dz, total_bytes;
};

int ffma_kcap();
FfmaPlan ffma_plan(const supcon_problem_t* p);
void ffma_bind_plan(FfmaArgs& a, const FfmaPlan& pl, void* workspace, bool backward);
size_t ffma_workspace_bytes(const supcon_problem_t* p);
cudaError_t ffma_forward(const FfmaArgs& a, cudaStream_t stream);
cudaError_t ffma_backward(const FfmaArgs& a, int dz_dtype, cudaStream_t stream);
cudaError_t ffma_topk_indices(const FfmaArgs& a, int32_t* idx_out, cudaStream_t stream);

// ---- bf16 tensor-core path (supcon_tc.cu) ----
struct TcSched {   // flattened (row block, column tile) work list cut into P contiguous CTA ranges
  int T;           // column tiles per row block
  int P;           // CTAs
  long long U;     // row_blocks * T
  // Column PANELS (backward at large N): the list is ordered (panel, row block, tile within the panel) instead of
  // (row block, tile), so that the CTAs running at the same time work on a few panels of z instead of all of it and
  // the Z_J tiles they stream stay in L2.  NP == 1: one panel = the plain row-major order.
  int RB;          // row blocks
  int NP;          // panels
  int Tp;          // tiles per panel (the last panel holds the remainder)
};
struct TcPlan {
  TcSched fwd_sched, bwd_sched;
  TcSched fwd_sched_local, fwd_sched_remote;   // two-phase forward (own columns first, then the others)
  TcSched bwd_sched_local, bwd_sched_remote;   // two-phase backward, likewise (64-column tiles)
  bool two_phase;
  int local_ct0, local_cts, slots_local;       // forward: own-column window in 128-column tiles
  int bwd_local_ct0, bwd_local_cts, bwd_slots_local;   // backward: the same window in 64-column tiles
  int n_pad, rows_pad, row_blocks, fwd_row_blocks, fwd_col_tiles, bwd_col_tiles, fwd_slots, bwd_slots, merge_blocks;
  int bwd_spp;                                 // backward: partial-record slots per column panel
  size_t off_block_partials, off_lab, off_nrm, off_colA, off_colAm, off_colB, off_colThr, off_colThrIdx,
      off_scalars, off_hkeys, off_hcounts, off_topk_v, off_topk_i, off_part, total_bytes;
  size_t off_hids, off_csum_part, off_csum;   // positives by linearity: class ids, per-block and total class sums
  size_t off_cls;                             // dense class id of every (padded) column, for the backward's reduce
  int csum_blocks;                            // blocks of tc_class_sum_kernel (256 columns each)
  uint32_t hash_size;
};
constexpr int TC_CMAX = 32;         // most classes the class-sum route handles (more: per-pair sums in the sweep)
constexpr int TC_FWD_PASSES = 2;    // passes the forward merge sums: the whole sweep, or own columns + the others
struct TcFwdArgs {
  const int32_t* lab_pad;
  const float* nrm_pad;
  const unsigned long long* hkeys;   // label -> class size table (tc_prep_fwd_kernel)
  const int* hcounts;
  uint32_t hmask;
  const unsigned* nrm2_max;          // bits of max_j |z_j|^2 over the columns swept so far (workspace header)
  // positives by linearity (cosine, no mining, whole forward): sum_{j in pos(i)} z_i.z_j = z_i . C[class_i] - |z_i|^2
  // with C[c] = sum of the rows of class c.  n_classes == nullptr: off.  plin_twin: this launch is the per-pair
  // kernel that only runs when there are more than TC_CMAX classes (its twin returns at once in that case).
  const int* n_classes;              // distinct labels seen by the label table (workspace header)
  const int* hids;                   // dense class id of every table slot
  const float* csum;                 // [TC_CMAX][256] class sums
  const void* z_rows;                // z (bf16), read by the merge for the rows' dot products with the class sums
  int plin_twin;
  float* part;       // [slots][rows_pad][8]
  float* topk_v;     // [splits][rows_pad][kcap]  per-split hard-negative candidates (mining)
  int32_t* topk_i;
  TcSched sched;
  int ct_base, ex_lo, ex_len, slot_base;
  // merge only: every pass whose partial records are summed (sched + first slot)
  int npass;
  TcSched msched[TC_FWD_PASSES];
  int mslot[TC_FWD_PASSES];
  int n_total, n_pad, row_offset, n_rows, rows_pad, topk, mine, kcap;
  float inv_tau, c1, c0, ut2;
  float m_limit;     // tau / 0.025: largest fixed maximum that cannot underflow a row's dominant terms
  const int32_t* mem_filled;   // device fill level of the memory (live_columns()); nullptr: all n_total columns
};
struct TcBwdPrepArgs {
  const float* stats;        // statistics of rows [stats_row0, ...): [..][STRIDE]
  int stats_row0;
  int j_lo, j_cnt;           // columns whose coefficients this launch computes
  int use_label_counts;      // |A_f|, |A_m| from the label-derived global counts (own partials, before any exchange)
  const double* partials;
  const int32_t* labels;
  float *colA, *colAm, *colB, *colThr;
  int32_t *colThrIdx, *lab_pad;
  // positives by linearity: dense class id of every column (hkeys == nullptr: not wanted)
  const unsigned long long* hkeys;
  const int* hids;
  uint32_t hmask;
  int32_t* cls_pad;
  float* scalars;
  int n_total, n_pad, topk;
  int n_batch;               // batch_columns(): columns from n_batch on are memory (zero coefficients, no statistics)
  int n_rows;
  const int32_t* mem_filled; // as in TcFwdArgs
  float tau, alpha, lambda_uni, uni_t;
};
struct TcBwdArgs {
  const int32_t* lab_pad;
  const float* nrm_pad;
  const float *colA, *colB;
  const float *colAm, *colThr;   // mining
  const int32_t* colThrIdx;
  const float* scalars;  // [0] = uniformity coefficient cu, [1] = exponent offset -M/tau log2(e)
  float* dz_part;        // [slots][rows_pad][256]
  TcSched sched;
  TcSched sched_b;       // reduce only: second pass of the two-phase backward (P == 0: none)
  int ct_base, ex_lo, ex_len, slot_base, slot_base_b;
  int spp;               // partial-record slots per panel of `sched`
  int n_total, n_pad, row_offset, n_rows, rows_pad;
  float c1, c0, ut2;
  // positives by linearity (cosine, no mining, single-phase backward): B is constant within a class, so
  // -sum_{j in pos(i)} (B_i + B_j) z_j = -2 B_i (C[class_i] - z_i) is added in fp32 by the reduce kernel and the
  // sweep forms H without the per-pair label compare.  n_classes == nullptr: off; plin_twin as in TcFwdArgs.
  const int* n_classes;
  const unsigned long long* hkeys;
  const int* hids;
  uint32_t hmask;
  const float* csum;     // [TC_CMAX][256]
  const int32_t* cls_pad;  // dense class id per column (tc_prep_bwd_kernel)
  int plin_twin;
  const int32_t* mem_filled;   // as in TcFwdArgs
};
TcPlan tc_plan(const supcon_problem_t* p);
bool tc_supported(const supcon_problem_t* p);
bool tc_two_phase(const supcon_problem_t* p);
bool tc_bwd_two_phase(const supcon_problem_t* p);
int tc_debug_plan(const supcon_problem_t* p, int32_t* out, int n_out);
int tc_debug_sched(int T, int P, long long U, int cta, int row_block, long long* range_begin, long long* range_end,
                   int* first_cta, int* last_cta);
// mem_filled (SUPCON_FLAG_MEMORY_COLUMNS, phase 0 only): device fill level of the memory; columns
// [n_rows + *mem_filled, n_total) are absent.  nullptr: every column is there.
int tc_forward(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all, float* row_stats,
               double* partials, float* loss_out, void* workspace, cudaStream_t stream, const char** err,
               int phase = 0, const int32_t* mem_filled = nullptr);
// phase: 0 = whole backward; 1 = only the columns this rank owns (`stats` = the rank's OWN statistics
// [n_rows][STRIDE], `partials` = its own forward partials; partial dz records, nothing else is written);
// 2 = all other columns (`stats` = everyone's, `partials` = the global sums) + reduce over both phases.
int tc_backward(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all, const float* stats,
                const double* partials, const float* grad_out, void* dz_out, int dz_dtype, void* workspace,
                cudaStream_t stream, const char** err, int phase = 0, const int32_t* mem_filled = nullptr);

// ---- exchange through peer memory (supcon_peer.cu) ----
int peer_check(const supcon_peer_t* pe, const char** err);
cudaError_t peer_push(const supcon_peer_t& pe, const void* src0, size_t bytes0, uint64_t off0, const void* src1,
                      size_t bytes1, uint64_t off1, int flag_id, int wait_flag_id, int include_self,
                      cudaStream_t stream);
cudaError_t peer_wait(const supcon_peer_t& pe, int flag_id, cudaStream_t stream);
cudaError_t peer_end_step(const supcon_peer_t& pe, int flag_id, cudaStream_t stream);

// ---- single-launch small-batch path (supcon_small.cu) ----
struct SmallArgs {
  const void* z;
  const int32_t* labels;
  float* row_stats;       // optional [n][STRIDE]
  double* partials;       // optional [8]
  float* loss_out;        // optional
  void* dz_out;           // optional [n][d]
  const float* grad_out;  // optional device scalar
  int n, d, z_dtype, dz_dtype, similarity, topk, mine;
  float tau, alpha, lambda_uni, uni_t;
};
bool small_supported(const supcon_problem_t* p, const void* z);
cudaError_t small_launch(const SmallArgs& a, cudaStream_t stream);

// ---- single-launch mid-size path, 160 < N <= 512 (supcon_mid.cu); *taken = false when the device cannot
//      co-schedule the cluster (the caller then uses the tiled kernels) ----
bool mid_supported(const supcon_problem_t* p, const void* z);
cudaError_t mid_launch(const SmallArgs& a, cudaStream_t stream, bool* taken);
// The route decisions below are shared with the test library's route report (supcon_debug_route); hidden, so that
// the product library exports nothing beyond its C ABI on their account.
#define SUPCON_HIDDEN __attribute__((visibility("hidden")))
// CTAs of the mid kernel's cluster on the current device: 16, 8, or 0 when it cannot take a.n rows
SUPCON_HIDDEN int mid_cluster_ctas(const SmallArgs& a);

// ---- route predicates of the dispatcher (supcon_api.cu) ----
SUPCON_HIDDEN bool use_tc(const supcon_problem_t* p, bool backward);     // tensor-core forward / backward
SUPCON_HIDDEN bool use_small(const supcon_problem_t* p, const void* z);  // single-launch small kernel
SUPCON_HIDDEN bool use_small_forward_rows(const supcon_problem_t* p, const void* z);   // ... in supcon_forward_rows
SUPCON_HIDDEN bool use_mid(const supcon_problem_t* p, const void* z);    // mid kernel (if mid_cluster_ctas > 0)
SUPCON_HIDDEN bool vec_ok(const void* z, const supcon_problem_t* p);     // tiled kernels: vector row loads
// tensor path: positives by linearity (class sums) in the forward / backward of this phase; the device still falls
// back to per-pair sums above TC_CMAX classes
SUPCON_HIDDEN bool tc_class_sums(const supcon_problem_t* p, bool backward, int phase);

// ---- producer of z: compression head up to the Linear layer, fused with the time mean (supcon_head.cu) ----
struct HeadPoolArgs {
  const void* hs;                       // [B][K][F][T] of hs_dtype
  float* pooled;                        // fwd out [B][F]
  const unsigned long long* rng_state;  // device {seed, offset}; NULL = no dropout
  int B, K, F, T;
  float dropout_p, negative_slope;
  int rows_per_block;                   // filled by the launcher
  int hs_dtype;                         // SUPCON_F32 | SUPCON_BF16: element type of hs and dhs (a store's: | F16)
};
int head_pool_rows_per_block(int F, int T, int hs_dtype);
cudaError_t head_pool_forward(HeadPoolArgs a, cudaStream_t stream);
cudaError_t head_layer_mean(HeadPoolArgs a, float* rows, cudaStream_t stream);   // rows [B][F][T] fp32
// a.hs = the (n_store, F, T) store of store_dtype (SUPCON_F32 | SUPCON_F16), idx = [B] store row of each batch
// position
cudaError_t head_store_pool_forward(HeadPoolArgs a, int store_dtype, const long long* idx, long long n_store,
                                    cudaStream_t stream);
// the same on a store sharded over n_ranks GPUs: row i at bases[i % n_ranks] + (i / n_ranks) * F * T elements
// (device table)
cudaError_t head_sharded_store_pool_forward(HeadPoolArgs a, int store_dtype, const unsigned long long* bases,
                                            int n_ranks, const long long* idx, long long n_store,
                                            cudaStream_t stream);
cudaError_t head_pool_backward(HeadPoolArgs a, const float* dpooled, void* dhs, cudaStream_t stream);

// tcgen05 building-block diagnostic (supcon_tc_debug.cu)
int tc_debug_tile(const void* z_bf16, int n, int d, int row_i, int row_j, float* s_out, float* o_out,
                  cudaStream_t stream, const char** err);

}  // namespace supcon
