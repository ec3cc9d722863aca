/*
 * polara_b200 -- C-ABI of the B200-native factorization-and-scoring engine.
 *
 * The reference (evfro/polara, pure Python) has NO FFI of its own: its hot path
 * bottoms out in scipy/numpy/numba calls.  Each entry point below replaces one
 * of those call sites (cited per function; paths relative to the reference
 * checkout) and is what a ctypes binding on the reference side would bind --
 * see INTEGRATION.md for that binding.
 *
 * Conventions
 *   - every function returns an int status: 0 = OK, PB200_E* otherwise;
 *     pb200_last_error(ctx) gives the message.
 *   - all array arguments are DEVICE pointers (cudaMalloc'ed by the caller, e.g.
 *     torch tensors' data_ptr()) unless the name ends in _host.
 *   - work is enqueued on the context's stream; nothing synchronises unless noted.
 *   - CSR: indptr int64 [n_rows+1], indices int32 [nnz] (sorted within a row),
 *     values float32 [nnz].  Dense matrices are row-major float32 with an explicit
 *     leading dimension (ld, in elements).
 *   - sm_100a only.  No CPU fallback exists.
 */
#ifndef POLARA_B200_H
#define POLARA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PB200_OK 0
#define PB200_EINVAL 1   /* -> ValueError   */
#define PB200_ENOMEM 2   /* -> MemoryError  */
#define PB200_ECUDA 3    /* -> RuntimeError */
#define PB200_ENOTIMPL 4 /* -> NotImplementedError */

typedef struct pb200_ctx pb200_ctx;

/* candidate list entry produced by the scoring kernels */
typedef struct { float score; int32_t id; } pb200_cand;

int pb200_version(void);

/* stream: a cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream) or NULL
 * for the legacy default stream. */
int pb200_ctx_create(int device, void* stream, pb200_ctx** out);
int pb200_ctx_destroy(pb200_ctx* ctx);
/* later work is enqueued on `stream` (the caller orders it against earlier work on the previous stream). */
int pb200_ctx_set_stream(pb200_ctx* ctx, void* stream);
const char* pb200_last_error(pb200_ctx* ctx);
int pb200_ctx_sync(pb200_ctx* ctx);
/* development aid: prints the diagnostics a timed-out (trapped) kernel left in pinned host memory to stderr */
int pb200_debug_dump(pb200_ctx* ctx);
/* which scoring kernel pb200_score_topk uses: 0 = exact SIMT fp32 kernel,
 * 1 = tcgen05 (bf16 tensor-core filter + exact fp32 rescoring; same results). */
int pb200_set_score_kernel(pb200_ctx* ctx, int kind);
/* 1 (default): a user tile's sweep over the norm-ordered items stops at the first position where
 * ||e_u|| * ||v_pos|| (Cauchy-Schwarz) can no longer reach the user's seeded k-th best score -- results are unchanged
 * (the skipped pairs cannot enter a top-k list); 0: every (user, item) pair goes through the tensor-core filter. */
int pb200_set_prune(pb200_ctx* ctx, int on);
/* counters of the last scoring call (host array of 8 uint64):
 *  [0] kernels launched  [1] candidates rescored  [2] item tiles  [3] user tiles
 *  [4] duration of the last fused scoring kernel in microseconds (CUDA events on the
 *      context stream; synchronises)
 *  [5] (user tile x item tile) products the tensor-core sweep executed so far (cumulative over calls)
 *  [6] the same count had no sweep been cut short by the norm bound (pb200_set_prune)
 *  [7] non-zero: a kernel gave up on a barrier (diagnostic code) */
int pb200_get_stats(pb200_ctx* ctx, uint64_t* out8_host);

/* Row-sharded build (SURVEY.md 8e "Partitioning - build": users split across GPUs, one process per GPU).
 * The hook must replace the `count` elements at `dev_ptr` by their sum over all shards, ordered after prior work on
 * the context stream and before later work on it (e.g. ncclAllReduce on that stream, or torch.distributed.all_reduce
 * with the context stream current).  While a hook is installed pb200_rsvd and pb200_rescale treat their CSR
 * arguments as this rank's ROW BLOCK of the matrix: Gram matrices of user-side panels (f64, ell*ell), the
 * item-side panel A^T W (f32, n_cols*ell) and the column counts of pb200_rescale (i32, n_cols) go through it.
 * Every rank must make the same calls in the same order.  fn == NULL removes the hook.  Returns 0 on success. */
#define PB200_F32 0
#define PB200_F64 1
#define PB200_I32 2
typedef int (*pb200_reduce_fn)(void* user, void* dev_ptr, int64_t count, int dtype);
int pb200_set_reduce_hook(pb200_ctx* ctx, pb200_reduce_fn fn, void* user);

/* Item-sharded scoring (SURVEY.md 8e "Partitioning - scoring": every rank scores ALL users against its own item shard).
 * Between its probe pass and its sweep the tensor-core scoring path holds, per user, a lower bound of the user's final k-th
 * best score (the k-th best exact score among the shard's largest-norm unseen items).  A bound found on ANY shard holds for
 * the merged result, so the hook, called once per pb200_score_topk / pb200_score_topk_cands that the tensor-core path takes
 * (not by the CUDA-core kernel: pb200_set_score_kernel(0) or ranks above 509, which keep no such bounds; the choice depends
 * on the rank and the device only, so all ranks of a job agree) as fn(user, bounds, n_users, PB200_F32), must replace the
 * n_users floats at `bounds` by their elementwise MAXIMUM over all ranks (same ordering rules as the reduce hook; every rank
 * scores the same users in the same call order).  Shards whose items cannot reach another
 * shard's bound then stop their sweep early instead of producing candidates the merge would drop: results are unchanged.
 * Remove the hook (fn == NULL) before scoring calls that are not part of such a sharded job.  No reference counterpart. */
int pb200_set_bound_hook(pb200_ctx* ctx, pb200_reduce_fn fn, void* user);

/* A CSR matrix resident in HBM, optionally stored PANEL-MAJOR (pb200_csr_block_columns): the columns are cut into
 * n_panels panels of panel_cols columns, the nnz of panel 0 come first (rows in order, columns sorted), then panel 1, ...;
 * indptr has n_panels * n_rows + 1 entries (virtual row = panel * n_rows + row), indices are GLOBAL column ids.
 * n_panels == 1 is a plain CSR.  panel_ptr_host (HOST memory, n_panels + 1 entries, may be NULL when n_panels == 1)
 * holds the nnz offset at which each panel starts: the launch grids are sized from it without a device round trip. */
typedef struct {
    int64_t n_rows, n_cols, nnz;
    const int64_t* indptr;
    const int32_t* indices;
    const float* values;
    int32_t n_panels;
    int64_t panel_cols;
    const int64_t* panel_ptr_host;
} pb200_csr_view;

/* which SpMM kernel runs (all deterministic, same results up to the summation order of rows that straddle windows):
 *   3 (default) nnz windows per warp + 128-bit register gathers (a lane owns four columns; half a warp per nnz up to 64
 *               columns, a full warp up to 128): work split by nnz, carried row pieces added in order;
 *   4           the same with 32-bit gathers (a lane owns one column per 32-column group; also taken for operands that
 *               are not 16-byte aligned);
 *   1 / 2       dense rows of X staged in shared memory by cp.async.bulk (one UBLKCP per row) / by 16-byte cp.async --
 *               measured slower (the per-row copy issue is the bottleneck, DESIGN.md 3.2); operands that are not
 *               16-byte aligned fall back to 0;
 *   0           row-owned register gathers (round-1 kernel). */
int pb200_set_spmm_kernel(pb200_ctx* ctx, int kind);

/* Y[n_rows x ell] = A * X ; replaces csr_matrix.dot(ndarray) at
 * polara/recommender/models.py:860 (P.dot(V)) and the A x / A^T x products inside
 * scipy svds (models.py:844).  X is read up to column ell only (ldx >= ell); Y is written in whole groups of 32
 * columns, zero beyond ell (ldy >= ell rounded up to 32). */
int pb200_spmm(pb200_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz,
               const int64_t* indptr, const int32_t* indices, const float* values,
               const float* X, int64_t ldx, float* Y, int64_t ldy, int ell);

/* same product for a matrix view (plain or panel-major); with panels Y accumulates in panel order (deterministic). */
int pb200_spmm_csr(pb200_ctx* ctx, const pb200_csr_view* a, const float* X, int64_t ldx, float* Y, int64_t ldy, int ell);

/* Panel-major copy of a CSR matrix (see pb200_csr_view): a format conversion done once per build() so that the slice
 * of the dense operand one panel gathers from (panel_cols rows of X) stays resident in the 126 MB L2 while the nnz
 * stream through.  b_indptr [n_panels * n_rows + 1], b_indices/b_values [nnz] device; panel_ptr_host [n_panels + 1] HOST.
 * n_panels must equal ceil(n_cols / panel_cols).  Synchronises the stream (the panel offsets are returned to the host). */
int pb200_csr_block_columns(pb200_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz,
                            const int64_t* indptr, const int32_t* indices, const float* values,
                            int64_t panel_cols, int n_panels,
                            int64_t* b_indptr, int32_t* b_indices, float* b_values, int64_t* panel_ptr_host);

/* Device-side ingest of the triplets a Polara data model hands to a model: RecommenderData.to_coo (data.py:794-817:
 * idx intp [nnz x 2], val) and test_to_coo (data.py:835-862: user, item, feedback arrays) -> CSR with duplicates summed
 * and columns sorted; replaces coo_matrix(...).tocsr() at models.py:169-174 and csr_matrix((fdbk,(user,item))) at
 * models.py:208-210.  rows/cols: device int64 with element strides (idx[:, 0] / idx[:, 1] of a row-major [nnz x 2] array
 * have stride 2); vals: device float32/float64 (val_dtype PB200_F32 / PB200_F64) or NULL = all ones;
 * drop_zeros != 0 removes zero-valued triplets first (get_test_matrix, models.py:197-201);
 * require_sorted_rows != 0 makes decreasing row ids an error (PB200_EINVAL) -- the reference asserts that test triplets
 * are sorted by user (models.py:246).
 * Outputs: indptr_out [n_rows + 1], indices_out / values_out with room for nnz entries; *nnz_out_host (HOST) = entries
 * written.  Input already strictly increasing in (row, col) is converted without sorting.  Synchronises the stream. */
int pb200_coo_to_csr(pb200_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz,
                     const int64_t* rows, int64_t row_stride, const int64_t* cols, int64_t col_stride,
                     const void* vals, int val_dtype, int drop_zeros, int require_sorted_rows,
                     int64_t* indptr_out, int32_t* indices_out, float* values_out, int64_t* nnz_out_host);

/* x[i] += delta for i < count (device int64): re-bases the row pointers / user ids of a chunk of a larger matrix. */
int pb200_shift_i64(pb200_ctx* ctx, int64_t* x, int64_t count, int64_t delta);

/* CSR of A^T (= CSC of A), rows sorted; scipy's coo->csr/csc conversion at
 * models.py:169-174 plays this role on the CPU. */
int pb200_csr_transpose(pb200_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz,
                        const int64_t* indptr, const int32_t* indices, const float* values,
                        int64_t* t_indptr, int32_t* t_indices, float* t_values);

/* In place: values <- D_r^(row_scaling-1) A D_c^(col_scaling-1), D = diag(sqrt(nnz count))
 * ; polara/preprocessing/matrices.py:71-93 (binary=True) as called from
 * ScaledMatrixMixin.get_training_matrix, models.py:891-895. */
int pb200_rescale(pb200_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz,
                  const int64_t* indptr, const int32_t* indices, float* values,
                  double row_scaling, double col_scaling);

/* Truncated SVD by randomized subspace iteration; replaces
 * scipy.sparse.linalg.svds at models.py:844.  Needs both A (CSR) and A^T (CSR).
 *   V_out [n_cols x ldv]  right singular vectors, column j pairs with sigma_out[j]
 *   sigma_out [rank] float64, descending (models.py:846-855 ordering)
 *   U_out [n_rows x ldu] or NULL
 *   ell: subspace width (multiple of 32, > rank); max_iters: power iterations;
 *   tol: stop when the leading `rank` Ritz values move less than tol (relative)
 *   iters_done_host: host int, may be NULL. Synchronises the stream. */
int pb200_rsvd(pb200_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz,
               const int64_t* indptr, const int32_t* indices, const float* values,
               const int64_t* t_indptr, const int32_t* t_indices, const float* t_values,
               int rank, int ell, int max_iters, double tol, uint64_t seed,
               float* V_out, int64_t ldv, double* sigma_out, float* U_out, int64_t ldu,
               int* iters_done_host);

/* Same factorisation for matrix views (A and A^T may be panel-major).  info_host (HOST, 8 doubles, may be NULL):
 *   [0] subspace iterations done   [1] largest relative change of the leading `rank` Ritz values in the last iteration
 *   [2] upper bound of sin(largest principal angle) between the leading-`rank` right subspaces of the last two iterates
 *   [3] 1 if both fell below tol / vec_tol before max_iters, else 0 (the caller should warn: the factors are the best
 *       subspace found, not a converged one)
 * vec_tol <= 0 disables the subspace test. */
int pb200_rsvd_csr(pb200_ctx* ctx, const pb200_csr_view* A, const pb200_csr_view* At,
                   int rank, int ell, int max_iters, double tol, double vec_tol, uint64_t seed,
                   float* V_out, int64_t ldv, double* sigma_out, float* U_out, int64_t ldu, double* info_host);

/* Thin SVD pieces of a dense tall matrix M [n x c]: leading `rank` singular values
 * (sigma_out, float64, descending), left vectors U_out [n x ldu] and, if not NULL,
 * right vectors Vt_out [rank x c] (row-major).  Replaces svds() on the dense HOOI
 * unfoldings, polara/lib/tensor.py:71,75,79.  While a reduce hook is installed (pb200_set_reduce_hook) M is this rank's
 * block of ROWS: the c x c Gram matrix is summed over the ranks, sigma / Vt are global, U_out holds the rank's own rows
 * (the mode-0 step of a HOOI whose nnz are sharded by user). */
int pb200_tall_svd(pb200_ctx* ctx, const float* M, int64_t n, int c, int64_t ldm, int rank,
                   double* sigma_out, float* U_out, int64_t ldu, float* Vt_out);

/* Fused scores = E V^T  ->  seen-item masking -> per-row top-k; full score rows
 * never reach HBM.  Replaces the chain slice_recommendations (models.py:857-861,
 * the dgemm) -> downvote_seen_items (models.py:494-519) -> get_topk_elements
 * (models.py:522-564).
 *   E [m x lde] user embeddings (P V), V [n x ldv] item factors, r = rank
 *   seen_indptr/seen_indices: CSR of seen items per user (sorted, unique per row; ids in
 *       the OUTPUT id space, i.e. local item id + item_offset), NULL/NULL = filter_seen False
 *   out_ids int64 [m x k] (+ item_offset), out_scores float32 [m x k] or NULL.
 * Order: unseen items by (score desc, id asc); if fewer than k unseen items exist
 * the seen ones follow by (score desc, id asc) -- the order models.py:517-519 yields. */
int pb200_score_topk(pb200_ctx* ctx, const float* E, int64_t lde, const float* V, int64_t ldv,
                     int64_t m, int64_t n, int r,
                     const int64_t* seen_indptr, const int32_t* seen_indices,
                     int k, int64_t item_offset, int64_t* out_ids, float* out_scores);

/* Same, but stops at the per-row candidate list of THIS item shard:
 * out_cands [m x k] sorted, ids global (+item_offset), empty slots id=-1/score=-inf.
 * Used for item-factor sharding across GPUs. */
int pb200_score_topk_cands(pb200_ctx* ctx, const float* E, int64_t lde, const float* V, int64_t ldv,
                           int64_t m, int64_t n, int r,
                           const int64_t* seen_indptr, const int32_t* seen_indices,
                           int k, int64_t item_offset, pb200_cand* out_cands);

/* count empty entries {score = -inf, id = -1}: the padding rows of a candidate block that is exchanged between GPUs. */
int pb200_fill_empty_cands(pb200_ctx* ctx, pb200_cand* cands, int64_t count);

/* Merge `parts` sorted candidate lists per row: in [parts][m][k] -> ids/scores [m x k]. */
int pb200_merge_cands(pb200_ctx* ctx, const pb200_cand* in, int parts, int64_t m, int k,
                      int64_t* out_ids, float* out_scores);

/* Same merge on the rank that OWNS the rows after the exchange of an item-sharded job, completed with the reference's
 * seen-item fill-up (models.py:517-519): rows with fewer than k unseen candidates over all shards continue with their
 * seen items by (score desc, id asc), scored exactly from E [m x lde] (these rows' embeddings) and the WHOLE V [n x ldv].
 * in: parts lists of k entries per row, list p of row u at in[p * part_stride + u * k]; seen ids are global. */
int pb200_merge_cands_fill(pb200_ctx* ctx, const pb200_cand* in, int parts, int64_t part_stride, int64_t m, int k,
                           const float* E, int64_t lde, const float* V, int64_t ldv, int r, int64_t n,
                           const int64_t* seen_indptr, const int32_t* seen_indices,
                           int64_t* out_ids, float* out_scores);

/* out[a] = E[user_idx[a], :r] . V[item_idx[a], :r] for `count` (user, item) pairs (device int64 index arrays): the scores
 * of holdout items and of sampled unseen items in the sampled evaluation protocol -- inner_product_at
 * (polara/lib/sparse.py:58-72) as used by RandomSampleEvaluationSVDMixin (models.py:1095-1183).  Out-of-range indices
 * yield NaN.  The scores are the same canonical fp32 values the fused kernel ranks by. */
int pb200_gather_dot(pb200_ctx* ctx, const float* E, int64_t lde, int64_t m, const float* V, int64_t ldv, int64_t n,
                     int r, const int64_t* user_idx, const int64_t* item_idx, int64_t count, float* out);

/* Dense scores S [m x lds] = E V^T for a handful of users (the single-user path of
 * models.py:277-293 expects a dense score row). */
int pb200_score_dense(pb200_ctx* ctx, const float* E, int64_t lde, const float* V, int64_t ldv,
                      int64_t m, int64_t n, int r, float* S, int64_t lds);

/* Top-k of a caller's dense score block S [m x lds] (float32 / float64 by `dtype` = PB200_F32 / PB200_F64), for scores
 * that did not come from our factors: RecommenderModel.get_topk_elements, dense branch (models.py:561-563; topsort
 * 488-491).  With a seen CSR (int64 indptr [m+1], int32 sorted ids) the seen-item handling is fused in: unseen items by
 * (score desc, id asc), then -- if fewer than k are unseen -- the seen ones in the same order, i.e. what
 * downvote_seen_items (models.py:510-519) followed by get_topk_elements yields.  out_ids int64 [m x k]; out_scores
 * [m x k] in the input dtype or NULL.  k > n is an error (np.argpartition raises there). */
int pb200_topk_dense(pb200_ctx* ctx, const void* S, int dtype, int64_t lds, int64_t m, int64_t n,
                     const int64_t* seen_indptr, const int32_t* seen_indices, int k, int64_t* out_ids, void* out_scores);

/* In place on a dense score block: S[row, col] <- min(S) - (max(S at the seen pairs) - S[row, col]) - 1 for the nnz seen
 * pairs (rows / cols: device int64) -- RecommenderModel.downvote_seen_items, dense branch (models.py:510-519):
 * order-preserving push below the block minimum. */
int pb200_downvote_dense(pb200_ctx* ctx, void* S, int dtype, int64_t lds, int64_t m, int64_t n,
                         const int64_t* rows, const int64_t* cols, int64_t nnz);

/* res[i0,:,:] += val * U[i1,:] (x) W[i2,:] over all nnz of a 3-way COO tensor sorted
 * and grouped by mode-0 index (CSR-like: seg_ptr int64 [n0+1], i1/i2 int32 [nnz]);
 * out [n0 x ru*rw] row-major (ld = ldo).  Replaces dttm_seq/dttm_par,
 * polara/lib/sparse.py:203-234. */
int pb200_ttm(pb200_ctx* ctx, int64_t n0, int64_t nnz, const int64_t* seg_ptr,
              const int32_t* i1, const int32_t* i2, const float* values,
              const float* U, int ru, int64_t ldu, const float* W, int rw, int64_t ldw,
              float* out, int64_t ldo);

/* Same sum when the grouped mode has only a few huge segments (the feedback mode of the
 * user x item x feedback tensor): out[s, x*rb + y] = sum_{p in segment s} val_p A[ia_p,x] B[ib_p,y],
 * fp64 accumulation, deterministic.  seg_ptr int64 [n_seg+1] (device).  Synchronises the stream. */
int pb200_ttm_reduce(pb200_ctx* ctx, int n_seg, int64_t nnz, const int64_t* seg_ptr,
                     const int32_t* ia, const int32_t* ib, const float* values,
                     const float* A, int ra, int64_t lda, const float* B, int rb, int64_t ldb,
                     float* out, int64_t ldo);

/* Stable grouping of a 3-way COO tensor by one mode: nnz sorted by key (0..n_keys-1);
 * seg_ptr int64 [n_keys+1]; a_out/b_out/val_out = the other index arrays / values permuted.
 * arrange_indices (polara/lib/sparse.py:239-264) is the reference's host-side analogue. */
int pb200_coo_group(pb200_ctx* ctx, int64_t nnz, int64_t n_keys, const int32_t* key,
                    const int32_t* a, const int32_t* b, const float* val,
                    int64_t* seg_ptr, int32_t* a_out, int32_t* b_out, float* val_out);

/* ProbabilisticMF build (models.py:743-770 -> generalized_sgd_sweep, polara/lib/optimize.py:123-250), stratified:
 * users and items are cut into `strata` = B contiguous ranges (row_bounds / col_bounds, device int64 [B + 1], ascending,
 * first 0, last n_rows / n_cols; empty ranges allowed).  Sub-epoch s processes the blocks (b, (b + s) mod B),
 * b = 0..B-1, which share no user and no item; an epoch is the reference's sweep over the interactions permuted into
 * (s, b) block order, reference (row-major) order inside a block.  B = 1 is the reference's own order.
 * pb200_sgd_plan (once per build): from the training CSR (sorted, duplicates summed; zeros dropped by the caller) and
 * the indptr of its transpose, writes block_ptr int64 [B*B + 1] (block s*B + b starts at block_ptr[s*B + b]), the
 * permuted triplets users_out / items_out int32 [nnz], vals_out float32 [nnz], and the row / column nnz counts
 * row_cnt_out int32 [n_rows], col_cnt_out int32 [n_cols] (getnnz(axis=1/0)).  1 <= B <= min(n_rows, n_cols, 65535). */
int pb200_sgd_plan(pb200_ctx* ctx, int64_t n_rows, int64_t n_cols, int64_t nnz, const int64_t* indptr,
                   const int32_t* indices, const float* values, const int64_t* t_indptr, int strata,
                   const int64_t* row_bounds, const int64_t* col_bounds, int64_t* block_ptr,
                   int32_t* users_out, int32_t* items_out, float* vals_out, int32_t* row_cnt_out, int32_t* col_cnt_out);

/* One epoch of the plan's sweep, in place on the fp64 factors P [n_rows x ldp] and Q [n_cols x ldq] (row-major, rank
 * <= 512 columns used): err = a - P[m].Q[n]; P[m] += learn_rate * (err Q[n] - P[m] lambd / row_cnt[m]);
 * Q[n] += learn_rate * (err P[m] - Q[n] lambd / col_cnt[n]), both gradients from the old rows, fp64 without FMA
 * contraction.  *cum_error_host (HOST) = sum of err^2 (per block in processing order, then over blocks in (s, b)
 * order).  Deterministic: no atomics.  Synchronises the stream. */
int pb200_sgd_epoch(pb200_ctx* ctx, int strata, const int64_t* block_ptr, const int32_t* users, const int32_t* items,
                    const float* vals, const int32_t* row_cnt, const int32_t* col_cnt, double* P, int64_t ldp,
                    double* Q, int64_t ldq, int rank, double learn_rate, double lambd, double* cum_error_host);

#ifdef __cplusplus
}
#endif
#endif
