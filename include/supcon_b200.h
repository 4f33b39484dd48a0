/*
 * supcon_b200.h -- C ABI of the B200-native supervised-contrastive loss path.
 *
 * Drop-in boundary for the Stage-1 objective of JaskiratSudan/wav2vec_contr_loss:
 * every entry point below replaces a piece of the reference's PyTorch
 * implementation (citations are relative to the reference repository root).
 * The reference is pure Python and has no FFI of its own; the binding a
 * maintainer adds is the ctypes stub shown in INTEGRATION.md (shipped as
 * wav2vec_contr_loss_b200/_cabi.py).
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless it says host
 *   - the caller owns all memory, including the workspace; the library never
 *     allocates or frees device memory and keeps no pointer after return
 *   - all work is issued asynchronously on `stream` (a cudaStream_t passed as
 *     void*); no host synchronisation; CUDA-graph capturable
 *   - return value: 0 = OK, >0 = cudaError_t, <0 = SUPCON_E_*; the message is
 *     available from supcon_last_error() (thread-local)
 *   - rows are "anchors"; a rank owns rows [row_offset, row_offset + n_rows) of
 *     the N x N similarity matrix and sees all n_total columns
 */
#ifndef SUPCON_B200_H_
#define SUPCON_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SUPCON_ABI_VERSION 3

/* element type of z / dz buffers */
#define SUPCON_F32 0
#define SUPCON_BF16 1
/* fp16: the element type of a layer-mean store's rows only (the store_dtype of the _store_pool_forward_typed entries);
 * every z / dz / hs dtype argument rejects it */
#define SUPCON_F16 2

/* similarity (reference loss.py:96-107) */
#define SUPCON_COSINE 0
#define SUPCON_GEODESIC 1

/* problem.flags */
#define SUPCON_FLAG_FORCE_EXACT 1u   /* never take the bf16 tensor-core path          */
#define SUPCON_FLAG_FORCE_TENSOR 2u  /* fail (SUPCON_E_UNSUPPORTED) instead of falling back */
#define SUPCON_FLAG_NO_SMALL 4u      /* do not use the single-launch small-batch kernel */
/* diagnostics: take the tensor path for one direction and the exact path for the other (not valid with
 * hard-negative mining: the two paths rank by different Gram arithmetic) */
#define SUPCON_FLAG_DEBUG_TC_FWD_ONLY 8u
#define SUPCON_FLAG_DEBUG_TC_BWD_ONLY 16u
/* Caller's promise that the rows of z are L2-normalised (what every caller of the reference passes,
 * stage1_utils.py:123): |z_i|^2 <= 1 + 2^-6.  Cosine similarity only reaches the bf16 tensor-core path under
 * this promise (its exponentials use one fixed maximum); without it z is taken as given on the exact path.
 * The promise is CHECKED on the device: max_i |z_i|^2 > tau / 0.025 makes the loss and dz NaN. */
#define SUPCON_FLAG_UNIT_ROWS 32u
/* The two-phase calls run beside this library's own (small) peer-push kernel, not beside a collective
 * library's kernel: their own-column phases use every SM instead of leaving some free for its channels. */
#define SUPCON_FLAG_PEER_EXCHANGE 64u
/* Tensor-core path, cosine similarity without mining: the positives' terms (sum of s_ij over a row's positives in
 * the forward, -sum (B_i + B_j) z_j in the backward) are linear in z_j and can be formed from per-class sums of
 * the rows, O(N d), instead of per pair in the sweep.  The library takes that route where it pays (single-phase
 * forward / backward of at least 2^30 pairs; at most 32 classes, decided on the device).  These two flags pin the
 * choice: CLASS_SUMS = also for small problems, NO_CLASS_SUMS = never. */
#define SUPCON_FLAG_CLASS_SUMS 128u
#define SUPCON_FLAG_NO_CLASS_SUMS 256u
/* supcon_backward_rows only: the caller's promise that `workspace` is the very buffer the supcon_forward_rows call
 * of the SAME problem used, untouched since.  The backward then takes the label table and the class sums the
 * forward left there instead of rebuilding them (three launches, ~40 us at N = 65536).  Without the flag the
 * backward needs nothing from the forward but the row statistics and partial sums. */
#define SUPCON_FLAG_WS_FROM_FORWARD 512u
/* Cross-batch memory (XBM): rows [0, n_rows) of z_all are the batch and its anchors; columns [n_rows, n_total) are
 * a memory of earlier batches' embeddings and labels.  Every anchor is contrasted against batch + memory (lse,
 * positives, negatives and the mined top-K run over all n_total columns), but only the batch carries statistics:
 *   - memory columns are constants: they get no gradient and no column-side term (H_ij = G_ij for j >= n_rows);
 *   - |A_f| and |A_m| count anchors only, and SUPCON_P_GCNT_* equal SUPCON_P_CNT_*;
 *   - the uniformity term stays over the batch's own pairs: log mean_{i<j<n_rows} exp(-t |z_i - z_j|^2), so its
 *     pair count comes from n_rows in supcon_finalize and everywhere else;
 *   - supcon_backward_rows reads stats_all as the anchors' [n_rows][STRIDE] statistics the forward wrote.
 * Requires row_offset == 0 and, when lambda_uni > 0, uni_t > 0 (SUPCON_E_INVALID otherwise).  Single rank only: the
 * two-phase _local / _remote calls treat the problem as not eligible, and supcon_finalize_sets with n_sets > 1
 * returns SUPCON_E_UNSUPPORTED.  With n_rows == n_total the loss is the plain loss; the problem still takes the tiled
 * kernels, never the single-launch small / mid ones, so that a separately issued forward and backward rank the hard
 * negatives with the same Gram arithmetic. */
#define SUPCON_FLAG_MEMORY_COLUMNS 1024u

/* error codes */
#define SUPCON_E_INVALID (-1)
#define SUPCON_E_UNSUPPORTED (-2)
#define SUPCON_E_WORKSPACE (-3)

/* per-row statistics written by the forward pass and consumed by the backward
 * pass: SUPCON_STATS_STRIDE 32-bit words per row, row-major. */
#define SUPCON_STATS_STRIDE 8
#define SUPCON_ST_LSE 0      /* f32  log sum_{j!=i} exp(s_ij/tau)                    */
#define SUPCON_ST_LSE_M 1    /* f32  same over positives + selected hard negatives   */
#define SUPCON_ST_NPOS 2     /* i32  |pos_i|                                         */
#define SUPCON_ST_NNEG 3     /* i32  |neg_i|                                         */
#define SUPCON_ST_THR_VAL 4  /* f32  similarity of the lowest-ranked selected negative
                                     (-inf when every negative is selected)          */
#define SUPCON_ST_THR_IDX 5  /* i32  its column index (INT32_MAX when all selected)  */
#define SUPCON_ST_WSUM 6     /* f32  sum_{j!=i} exp(-t |z_i - z_j|^2)                */
#define SUPCON_ST_POS_MEAN 7 /* f32  mean_{p in pos_i} s_ip/tau                      */

/* partial sums exchanged between ranks (doubles) */
#define SUPCON_N_PARTIALS 8
#define SUPCON_P_SUM_FULL 0
#define SUPCON_P_CNT_FULL 1
#define SUPCON_P_SUM_MINED 2
#define SUPCON_P_CNT_MINED 3
#define SUPCON_P_SUM_W 4
/* tensor path only (0 elsewhere); identical on every rank, so never summed across ranks: */
#define SUPCON_P_GCNT_FULL 5  /* |A_f| of the GLOBAL batch, derived from the gathered labels alone */
#define SUPCON_P_GCNT_MINED 6 /* |A_m| likewise                                                     */
#define SUPCON_P_FIXMAX 7     /* fixed maximum M the exponentials were taken against, exp((s - M)/tau):
                                 1 for unit rows, max_j |z_j|^2 otherwise, NaN = promise broken      */

typedef struct supcon_problem {
  int32_t n_total;    /* N: columns = global batch                                   */
  int32_t row_offset; /* first owned row                                             */
  int32_t n_rows;     /* owned rows                                                  */
  int32_t d;          /* embedding width                                             */
  int32_t z_dtype;    /* SUPCON_F32 | SUPCON_BF16                                    */
  int32_t similarity; /* SUPCON_COSINE | SUPCON_GEODESIC   (loss.py:21,30-32)        */
  int32_t topk;       /* topk_neg                           (loss.py:113)            */
  uint32_t flags;
  float tau;          /* temperature                        (loss.py:20,28)          */
  float alpha;        /* blend of full and mined loss       (loss.py:114,146)        */
  float lambda_uni;   /* uniformity_weight                  (loss.py:23,149-151)     */
  float uni_t;        /* uniformity_t                       (loss.py:24,93)          */
} supcon_problem_t;

int supcon_abi_version(void);
const char* supcon_last_error(void);

/* Bytes of scratch the calls below need for this problem (host out-param). */
int supcon_workspace_bytes(const supcon_problem_t* p, size_t* bytes_out);

/* Forward over the owned rows.  Replaces the similarity Gram, masks, the
 * per-anchor loop and the uniformity row sums: loss.py:96-107, :116-135, :77-93.
 *   z_all      [n_total][d]   labels_all [n_total] int32
 *   row_stats  [n_rows][SUPCON_STATS_STRIDE]      (out)
 *   partials   [SUPCON_N_PARTIALS] doubles         (out; this rank's sums)
 *   loss_out   optional; only when the rank owns every row (or with SUPCON_FLAG_MEMORY_COLUMNS, whose
 *              anchors are every row): the scalar loss (loss.py:137-153) is written by the same launch */
int supcon_forward_rows(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                        float* row_stats, double* partials, float* loss_out, void* workspace,
                        size_t workspace_bytes, void* stream);

/* Two-phase form of supcon_forward_rows for ranks that overlap the all-gather of z with compute:
 *   _local  sweeps only the columns this rank owns (rows [row_offset, row_offset + n_rows) of z_all and
 *           labels_all must be valid; nothing from other ranks is read) and leaves partial records in
 *           the workspace;
 *   _remote sweeps all other columns (the whole z_all / labels_all must be valid), merges both phases and
 *           writes row_stats / partials exactly as supcon_forward_rows would.
 * Both calls take the SAME workspace.  When the problem is not eligible (exact path, unaligned row block)
 * _local does nothing and _remote runs the whole forward. */
int supcon_forward_rows_local(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                              void* workspace, size_t workspace_bytes, void* stream);
int supcon_forward_rows_remote(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                               float* row_stats, double* partials, void* workspace, size_t workspace_bytes,
                               void* stream);

/* Scalar loss from globally summed partials (alpha blend, empty-set fall-backs,
 * uniformity term): loss.py:137-153. */
int supcon_finalize(const supcon_problem_t* p, const double* partials_global, float* loss_out,
                    void* stream);

/* Rank-ordered sum of the partial sums of `n_sets` ranks + the scalar loss in ONE launch (what the sharded
 * path runs after all-gathering every rank's partials): slots 0..4 are summed in set order (deterministic,
 * identical on all ranks), slots SUPCON_P_GCNT_* / SUPCON_P_FIXMAX are copied from set 0.
 *   partial_sets [n_sets][SUPCON_N_PARTIALS]   partials_out [SUPCON_N_PARTIALS]   loss_out optional */
int supcon_finalize_sets(const supcon_problem_t* p, const double* partial_sets, int32_t n_sets,
                         double* partials_out, float* loss_out, void* stream);

/* Backward for the owned rows (replaces autograd through loss.py:96-153):
 *   dz_i = grad_out * sum_j (G_ij + G_ji) z_j (+ uniformity), recomputing the
 *   similarity tiles; needs the statistics of ALL rows and the global partials.
 *   stats_all  [n_total][SUPCON_STATS_STRIDE]  (SUPCON_FLAG_MEMORY_COLUMNS: [n_rows][SUPCON_STATS_STRIDE], the
 *              anchors' statistics; memory columns have none)
 *   grad_out   device scalar (NULL = 1.0)
 *   dz_out     [n_rows][d] in dz_dtype */
int supcon_backward_rows(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                         const float* stats_all, const double* partials_global,
                         const float* grad_out, void* dz_out, int32_t dz_dtype, void* workspace,
                         size_t workspace_bytes, void* stream);

/* Two-phase form of supcon_backward_rows for ranks that overlap the exchange of row statistics with compute
 * (the symmetric formulation dz_i = sum_j (G_ij + G_ji) z_j needs the statistics of column j):
 *   _local  sweeps only the columns this rank owns, which need nothing but the rank's OWN statistics
 *           (stats_local [n_rows][STRIDE]) and its own forward partials (the global anchor counts in
 *           SUPCON_P_GCNT_* come from the gathered labels), and leaves partial dz records in the workspace;
 *           grad_out is not needed yet, so this can be issued right after the forward;
 *   _remote sweeps all other columns with everyone's statistics and the global partial sums, adds both
 *           phases, scales by grad_out and writes dz_out exactly as supcon_backward_rows would.
 * Both calls take the SAME workspace.  When the problem is not eligible (exact path, unaligned row block,
 * uniformity term: its coefficient needs the global sum) _local does nothing and _remote runs everything. */
int supcon_backward_rows_local(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                               const float* stats_local, const double* partials_local, void* workspace,
                               size_t workspace_bytes, void* stream);
int supcon_backward_rows_remote(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                                const float* stats_all, const double* partials_global, const float* grad_out,
                                void* dz_out, int32_t dz_dtype, void* workspace, size_t workspace_bytes,
                                void* stream);

/* supcon_forward_rows / supcon_backward_rows for a memory that is still filling, with its fill level in DEVICE
 * memory, so that one captured CUDA graph serves every fill level (a training step replayed as a graph while its
 * cross-batch memory fills).  Both need SUPCON_FLAG_MEMORY_COLUMNS (SUPCON_E_INVALID before any CUDA call without
 * it).  n_total is the CAPACITY, n_rows + memory size; the plan, the workspace and the route depend on it alone.
 *   mem_filled  DEVICE int32, read by the kernels only: columns [n_rows + *mem_filled, n_total) are absent.  They
 *               enter no sum, no count (|pos_i|, |neg_i|, the class sizes), no top-K list and not the fixed maximum,
 *               and they get no gradient.  Their rows of z_all must still hold finite values (the tensor path reads
 *               whole tiles).  A count outside [0, n_total - n_rows] makes the loss and dz NaN (no device fault).
 *               NULL = a full memory: the call is then supcon_forward_rows / supcon_backward_rows.
 * Results equal those of the plain calls with n_total = n_rows + *mem_filled on the same route, up to the order of
 * the column splits' sums.  On the tensor path the tiles of absent columns still run (masked): a call costs what a
 * full memory costs. */
int supcon_forward_rows_memory(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                               const int32_t* mem_filled, float* row_stats, double* partials, float* loss_out,
                               void* workspace, size_t workspace_bytes, void* stream);
int supcon_backward_rows_memory(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                                const int32_t* mem_filled, const float* stats_all, const double* partials_global,
                                const float* grad_out, void* dz_out, int32_t dz_dtype, void* workspace,
                                size_t workspace_bytes, void* stream);

/* ---- exchange between ranks through peer memory (NVLink / NVSwitch), see csrc/supcon_peer.cu -------------
 * The host maps every rank's exchange buffer into every process (a symmetric allocation, e.g.
 * torch.distributed._symmetric_memory) and describes it here.  All kernels are this library's own: plain
 * stores to peer addresses + per-rank step flags; no collective library call inside a step, CUDA-graph
 * capturable.  Replaces the all-gather of z / labels and of the row statistics (north_star's NCCL plan,
 * SURVEY 8e) where peer access exists; the NCCL path of distributed.py remains the fallback. */
#define SUPCON_PEER_MAX_WORLD 64
#define SUPCON_PEER_FLAG_Z 0      /* rows of z + labels of step e have landed          */
#define SUPCON_PEER_FLAG_STATS 1  /* row statistics + partial sums of step e have landed */
#define SUPCON_PEER_FLAG_DONE 2   /* rank has finished step e (its buffers may be overwritten) */
#define SUPCON_PEER_NFLAGS 3
/* bytes every buffer reserves at off_flags, zeroed once at set-up: int32 flags[NFLAGS][world] + 4 words, the first
 * of which is the push kernel's block ticket */
#define SUPCON_PEER_FLAG_BYTES(world) ((SUPCON_PEER_NFLAGS * (world) + 4) * 4)

typedef struct supcon_peer {
  int32_t rank, world;
  const uint64_t* peer_bases; /* DEVICE array [world]: base address of every rank's buffer as mapped in THIS
                                 process (peer_bases[rank] = the own buffer)                                 */
  uint64_t off_flags;         /* byte offset of the flag block inside each buffer                           */
  int32_t* epoch;             /* DEVICE int, rank-local: number of the current step, initialised to 1       */
  uint64_t mc_base;           /* multicast address of the buffers (NVSwitch writes one store into every rank's
                                 buffer: multimem.st), or 0: one unicast store per peer                      */
} supcon_peer_t;

/* Copy up to two byte ranges (sizes multiples of 4; src1 may be NULL) to the same offsets of EVERY peer's buffer
 * (and the own one if include_self), then set flag[flag_id][rank] = epoch in every buffer.
 * wait_flag_id >= 0: first wait until flag[wait_flag_id][p] >= epoch - 1 for all p (buffer reuse guard). */
int supcon_peer_push(const supcon_peer_t* pe, const void* src0, size_t bytes0, uint64_t dst_off0,
                     const void* src1, size_t bytes1, uint64_t dst_off1, int32_t flag_id, int32_t wait_flag_id,
                     int32_t include_self, void* stream);
/* One-block kernel: returns (on the stream) when flag[flag_id][p] >= epoch for every rank p. */
int supcon_peer_wait(const supcon_peer_t* pe, int32_t flag_id, void* stream);
/* End of a step: flag[flag_id][rank] = epoch in every buffer, then epoch += 1. */
int supcon_peer_end_step(const supcon_peer_t* pe, int32_t flag_id, void* stream);

/* Whole batch on one GPU: loss and (if dz_out != NULL) d loss / d z in as few
 * launches as the shape allows (one for small batches).  row_stats/partials
 * are scratch outputs as above. */
int supcon_loss_and_grad(const supcon_problem_t* p, const void* z, const int32_t* labels,
                         float* loss_out, void* dz_out, int32_t dz_dtype, float* row_stats,
                         double* partials, void* workspace, size_t workspace_bytes, void* stream);

/* Labels of any width -> the int32 class keys the kernels compare (loss.py:123 compares labels with ==; the
 * callers pass int64, stage1_utils.py:112): equal labels <-> equal keys.  One launch, replaces a dtype cast.
 * A label that 32 bits cannot hold losslessly (int64 outside int32, float64 that is not a float32) makes the
 * kernel report the row and trap -- a loud device fault instead of two classes silently merged.  -0.0 == +0.0;
 * every NaN row gets a key of its own (NaN equals nothing). */
#define SUPCON_LABEL_I64 1
#define SUPCON_LABEL_F32 2
#define SUPCON_LABEL_F64 3
int supcon_label_keys(const void* labels, int32_t dtype, int32_t n, int32_t* keys_out, void* stream);

/* Row L2 normalisation either side of the loss (stage1_utils.py:123,149):
 *   z = x / max(|x|, 1e-12);   dx = (dz - z (z.dz)) / max(|x|, 1e-12) */
int supcon_normalize_forward(const float* x, int32_t n, int32_t d, void* z_out, int32_t z_dtype,
                             float* norms_out, void* stream);
int supcon_normalize_backward(const void* z, int32_t z_dtype, const float* norms, const void* dz,
                              int32_t dz_dtype, int32_t n, int32_t d, float* dx_out, void* stream);

/* Producer of z (SURVEY 8f-N1): the compression head up to its Linear layer fused with the time mean
 * (compression_module.py:48-65 + the seq.mean(dim=-1) of stage1_utils.py:122-123).  Because the Linear layer and the
 * time mean commute, mean_t Linear(x_t) = Linear(mean_t x_t), and what is left of the head is one pass over hs:
 *   pooled[b][f] = (1/T) sum_t LeakyReLU(Dropout((1/K) sum_k hs[b][k][f][t]))
 * hs is (batch, layers, feat, frames) contiguous.  rng_state = device {seed, offset} (two 64-bit words) of the
 * counter-based dropout mask, or NULL / dropout_p == 0 for eval mode; the backward must be given the same values.
 * supcon_head_pool_backward writes d loss / d hs (same shape as hs) and is only needed when the encoder trains.
 * pooled_out and dpooled are fp32.
 *
 * hs_dtype (the _typed entry points) is the element type of hs and of dhs_out: SUPCON_F32, or SUPCON_BF16 for the
 * output of an encoder run in bf16, read as it is (no fp32 copy).  bf16 elements are widened to fp32 exactly and the
 * arithmetic after the load is the fp32 one, so pooled_out equals bit for bit that of the fp32 call on the widened
 * hs, and dhs_out is that call's fp32 dhs rounded to nearest even.  Any other hs_dtype returns SUPCON_E_INVALID.
 * supcon_head_pool_forward / _backward are the SUPCON_F32 case. */
int supcon_head_pool_forward_typed(const void* hs, int32_t hs_dtype, int32_t batch, int32_t layers, int32_t feat,
                                   int32_t frames, float dropout_p, float negative_slope, const uint64_t* rng_state,
                                   float* pooled_out /*[batch][feat]*/, void* stream);
int supcon_head_pool_backward_typed(const void* hs, int32_t hs_dtype, int32_t batch, int32_t layers, int32_t feat,
                                    int32_t frames, float dropout_p, float negative_slope, const uint64_t* rng_state,
                                    const float* dpooled /*[batch][feat]*/, void* dhs_out, void* stream);
int supcon_head_pool_forward(const float* hs, int32_t batch, int32_t layers, int32_t feat, int32_t frames,
                             float dropout_p, float negative_slope, const uint64_t* rng_state,
                             float* pooled_out /*[batch][feat]*/, void* stream);
int supcon_head_pool_backward(const float* hs, int32_t batch, int32_t layers, int32_t feat, int32_t frames,
                              float dropout_p, float negative_slope, const uint64_t* rng_state,
                              const float* dpooled /*[batch][feat]*/, float* dhs_out, void* stream);

/* Training the head on a frozen encoder from a store of its layer means, m[c] = (1/K) sum_k hs[c][k] (feat, frames)
 * fp32 per clip: everything of the head after the layer mean is recomputed from m every epoch, fresh dropout masks
 * included, without running the encoder again.
 *
 * supcon_head_layer_mean_typed writes store_rows[b] = (1/K) sum_k hs[b][k] for the batch's hs (hs_dtype as above);
 * store_rows is the store's row of the batch's first clip (store + slot0 * feat * frames).  The sum is in fp32 over
 * k = 0..K-1 in order, then times (1/K): the arithmetic of supcon_head_pool_forward_typed, bit for bit.
 *
 * supcon_head_store_pool_forward is supcon_head_pool_forward_typed on the store rows idx[0..batch) (int64, on the
 * device, so a captured graph takes new indices every replay):
 *   pooled[b][f] = (1/T) sum_t LeakyReLU(Dropout(store[idx[b]][f][t]))
 * The dropout mask of element (b, f, t) is the one supcon_head_pool_forward_typed draws for batch position b with the
 * same rng_state, so pooled_out equals bit for bit that call's on hs[idx[0..batch)].  An index outside [0, n_store)
 * writes NaN into its pooled row; the other rows are unaffected.  The store is a constant: there is no backward. */
int supcon_head_layer_mean_typed(const void* hs, int32_t hs_dtype, int32_t batch, int32_t layers, int32_t feat,
                                 int32_t frames, float* store_rows /*[batch][feat][frames]*/, void* stream);
int supcon_head_store_pool_forward(const float* store /*[n_store][feat][frames]*/, int64_t n_store, int32_t feat,
                                   int32_t frames, const int64_t* idx /*[batch]*/, int32_t batch, float dropout_p,
                                   float negative_slope, const uint64_t* rng_state,
                                   float* pooled_out /*[batch][feat]*/, void* stream);

/* supcon_head_sharded_store_pool_forward is supcon_head_store_pool_forward on a store sharded over the n_ranks GPUs
 * of one node: row i lives in the shard of rank i % n_ranks, at local row i / n_ranks (64-bit offsets).
 * shard_bases[r] (a device table of n_ranks addresses, so a captured graph reads it at every replay) is the address
 * of rank r's shard in the calling process: its own allocation, or a peer's mapped into it (CUDA IPC, symmetric
 * memory).  Every base must be 16-byte aligned and every shard hold ceil(n_store / n_ranks) rows of feat * frames
 * floats.  pooled_out equals bit for bit supcon_head_store_pool_forward's on a single store of the same n_store rows;
 * an index outside [0, n_store) writes NaN into its pooled row and reads nothing.  Returns SUPCON_E_INVALID, before
 * any CUDA call, for n_ranks < 1, n_store < n_ranks, a NULL table and the arguments the single-store call rejects. */
int supcon_head_sharded_store_pool_forward(const uint64_t* shard_bases /*device [n_ranks]*/, int32_t n_ranks,
                                           int64_t n_store, int32_t feat, int32_t frames,
                                           const int64_t* idx /*[batch]*/, int32_t batch, float dropout_p,
                                           float negative_slope, const uint64_t* rng_state,
                                           float* pooled_out /*[batch][feat]*/, void* stream);

/* store_dtype (the _typed entry points) is the element type of the store's rows: SUPCON_F32, or SUPCON_F16 for a
 * store kept at half the bytes.  fp16 elements are widened to fp32 exactly and the arithmetic after the load is the
 * fp32 one, so pooled_out equals bit for bit that of the SUPCON_F32 call on a store holding the widened values.
 * Shard offsets count elements of store_dtype.  Any other store_dtype, SUPCON_BF16 included, returns
 * SUPCON_E_INVALID before any CUDA call, as do the arguments the untyped entries reject.
 * supcon_head_store_pool_forward / supcon_head_sharded_store_pool_forward are the SUPCON_F32 case. */
int supcon_head_store_pool_forward_typed(const void* store /*[n_store][feat][frames]*/, int32_t store_dtype,
                                         int64_t n_store, int32_t feat, int32_t frames,
                                         const int64_t* idx /*[batch]*/, int32_t batch, float dropout_p,
                                         float negative_slope, const uint64_t* rng_state,
                                         float* pooled_out /*[batch][feat]*/, void* stream);
int supcon_head_sharded_store_pool_forward_typed(const uint64_t* shard_bases /*device [n_ranks]*/, int32_t n_ranks,
                                                 int32_t store_dtype, int64_t n_store, int32_t feat, int32_t frames,
                                                 const int64_t* idx /*[batch]*/, int32_t batch, float dropout_p,
                                                 float negative_slope, const uint64_t* rng_state,
                                                 float* pooled_out /*[batch][feat]*/, void* stream);

/* Diagnostics used by the parity tests: hard-negative index sets of the owned
 * rows, recomputed from the statistics (index ascending, -1 padded). */
int supcon_topk_indices(const supcon_problem_t* p, const void* z_all, const int32_t* labels_all,
                        const float* row_stats, int32_t* idx_out /*[n_rows][topk]*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SUPCON_B200_H_ */
