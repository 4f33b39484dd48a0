/* TEST-ONLY C entry points of libsupcon_b200_test.so (the product library and include/supcon_b200.h do not
 * carry them).  Used by tests/ and tools/ through tests/debug_lib.py. */
#ifndef SUPCON_DEBUG_H_
#define SUPCON_DEBUG_H_

#include "supcon_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

const char* supcon_debug_last_error(void);

/* tcgen05/TMA building blocks: for 128-row blocks I = row_i.., J = row_j.. of a bf16 matrix z [n][256] writes
 * S = Z_I Z_J^T ([128][128] fp32) and O = bf16(S) Z_J ([128][256] fp32). */
int supcon_debug_tc_tile(const void* z_bf16, int32_t n, int32_t d, int32_t row_i, int32_t row_j, float* s_out,
                         float* o_out, void* stream);

/* Host-only introspection of the tensor path's work distribution (no device work):
 *   supcon_debug_plan  out[0..15] = {fwd CTAs, fwd column tiles, fwd partial-record slots, bwd CTAs, bwd column
 *                      tiles, bwd slots, two-phase eligible, fwd own-column-phase CTAs, fwd other-column-phase
 *                      CTAs, fwd own-column-phase slots, forward (256-row) blocks, backward (128-row) blocks,
 *                      bwd own-column-phase CTAs, bwd other-column-phase CTAs, bwd own-column-phase slots,
 *                      bwd own-column tiles}
 *   supcon_debug_sched the contiguous unit range of one CTA and the first/last CTA touching a row block for a
 *                      flattened (row block, column tile) list of `units` = row_blocks * col_tiles entries */
int supcon_debug_plan(const supcon_problem_t* p, int32_t* out, int32_t n_out);
/* Host-only plan of the exact fp32 path (no device work): out[0..3] = {forward column splits, backward column
 * splits, top-K list capacity per row, selection rounds}; rounds = ceil(K / capacity) when mining, else 0. */
int supcon_debug_ffma_plan(const supcon_problem_t* p, int32_t* out, int32_t n_out);
/* Host-side route of a whole-batch problem, from the dispatcher's own predicates (no kernel runs):
 *   out[0] route of supcon_loss_and_grad, out[1] of supcon_forward_rows, out[2] of supcon_backward_rows
 *          (0 = small, 1 = mid, 2 = tensor, 3 = tiled exact; slots 0 and 1 name the forward's kernels, and with
 *          small / mid supcon_loss_and_grad's backward runs in the same launch; a mining supcon_forward_rows
 *          leaves the small kernel for the tiled ones, whose Gram its tiled backward recomputes);
 *   out[3] CTAs of the mid kernel's cluster when the mid kernel is eligible (16 or 8; 0: not eligible, or the device
 *          cannot co-schedule the cluster and the call falls through), -1 without a device (slots 0 and 1 then
 *          assume the cluster launches);
 *   out[4] the tiled kernels load rows as vectors (1) or element by element (0);
 *   out[5], out[6] the tensor forward / backward sum positives through class sums (host decision; above 32 classes
 *          the device still falls back to per-pair sums). */
int supcon_debug_route(const supcon_problem_t* p, const void* z, int32_t* out, int32_t n_out);
int supcon_debug_sched(int32_t col_tiles, int32_t ctas, int64_t units, int32_t cta, int32_t row_block,
                       int64_t* range_begin, int64_t* range_end, int32_t* first_cta, int32_t* last_cta);

#ifdef __cplusplus
}
#endif
#endif /* SUPCON_DEBUG_H_ */
