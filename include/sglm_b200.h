/*
 * sglm_b200.h — C ABI of libsglm_b200.so: the B200 (sm_100a) hot path of sGLM
 * (kimerein/sabatinilab-glm): lag/shift design-matrix gather, sufficient
 * statistics (X'X, X'y, X'WX ...), batched penalised-GLM solvers and scoring.
 *
 * The reference has no FFI — its boundary is the Python API of backend/sglm_pp.py,
 * backend/sglm.py and backend/sglm_cv.py, whose numerics are delegated to
 * scikit-learn.  Each entry point below names the reference interface whose
 * arithmetic it replaces (file:line relative to the reference tree; `sklearn/`
 * = scikit-learn 1.9.0 as called from backend/sglm.py:241).  The Python mirror
 * of the reference modules (sabatinilab-glm_b200/*.py) is the only caller;
 * INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - the caller allocates everything, including workspaces sized by the
 *     matching *_workspace_bytes();
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *     the call returns without synchronising;
 *   - return value: 0 = ok, <0 = SGLM_E_*; sglm_last_error() gives the text of
 *     the last failure on the calling thread; no C++ exception crosses the ABI;
 *   - entry points are re-entrant (no global mutable state) and honour the
 *     current CUDA device;
 *   - matrices are row-major with explicit leading dimensions counted in elements.
 */
#ifndef SGLM_B200_H
#define SGLM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGLM_OK 0
#define SGLM_E_INVALID_ARG (-1)
#define SGLM_E_SHAPE (-2)
#define SGLM_E_ALIGN (-3)
#define SGLM_E_WORKSPACE (-4)
#define SGLM_E_CUDA (-5)
#define SGLM_E_UNSUPPORTED (-6)

/* version = major*10000 + minor*100 + patch */
int sglm_version(void);
const char *sglm_last_error(void);

/* ------------------------------------------------------------------------- *
 * (a1-a3) lag / shift gather.  Replaces sglm_pp.timeshift / shift /
 * timeshift_multiple / concat_all_shifts (backend/sglm_pp.py:23-103, :298-357,
 * :436-457):   out[t, c] = X[t - col_shift[c], col_src[c]]  if that row exists,
 * else the 8-byte pattern `fill_bits` (np.nan = 0x7FF8000000000000).
 * The column map (col_src, col_shift) encodes block order, the all-columns
 * zero-shift block and keep_non_inx; it is built by the Python mirror.
 * Elements are moved as opaque 8-byte words (bit-exact, NaN payloads kept).
 * ------------------------------------------------------------------------- */
int sglm_timeshift_f64(const double *X, int64_t T, int32_t n_cols_in, int64_t ldx,
                       const int32_t *col_src, const int32_t *col_shift, int32_t n_cols_out,
                       uint64_t fill_bits, double *out, int64_t ldo, void *stream);

/* Same gather when the caller already knows min/max of col_shift (the Python mirror
 * builds the map, so it does): no device read-back, never synchronises the stream. */
int sglm_timeshift_f64_ranged(const double *X, int64_t T, int32_t n_cols_in, int64_t ldx,
                              const int32_t *col_src, const int32_t *col_shift,
                              int32_t n_cols_out, int32_t shift_min, int32_t shift_max,
                              uint64_t fill_bits, double *out, int64_t ldo, void *stream);

/* Row compaction that follows the gather in every caller (`dropna`,
 * er_refactored_from_scratch_cleanup.py:429; backend/test/test_sglm_ez.py:28):
 * out[r, :] = X[row_begin + r, :] for r < n_rows — a strided 2-D copy. */
int sglm_crop_rows_f64(const double *X, int64_t ldx, int64_t row_begin, int64_t n_rows,
                       int32_t n_cols, double *out, int64_t ldo, void *stream);

/* Fused dropna (the `dropna()` every driver applies between the lag builder and the fit,
 * er_refactored_from_scratch_cleanup.py:427-429; backend/test/test_sglm_ez.py:28):
 *   lag_valid_rows : valid[t] = 1 when row t of the lag design would hold no NaN — decided from the base
 *                    signals and the column map, the design is not built.  fill_is_nan != 0: rows whose source
 *                    row falls outside [0, T) are invalid (NaN padding).  summary3 (device int64[3]) =
 *                    {valid rows, first valid row, last valid row}.
 *   mask_compact_rows : ascending indices of the set rows of `valid` (rows must hold summary3[0] entries).
 *   timeshift_rows : the gather restricted to listed rows, out[r, c] = X[rows[r] - col_shift[c], col_src[c]].
 * When the valid rows are one contiguous range (no NaN in the base signals) the plain gather + a row view is used. */
int sglm_lag_valid_rows(const double *X, int64_t T, int32_t n_cols_in, int64_t ldx, const int32_t *col_src,
                        const int32_t *col_shift, int32_t n_cols_out, int32_t shift_min, int32_t shift_max,
                        int32_t fill_is_nan, uint8_t *valid, int64_t *summary3, void *stream);
/* Row mask of an index list (positions in [0, T); mask holds T rounded up to a multiple of 4 bytes, 4-byte
 * aligned): mask[t] = 1 for listed rows, *dup_flag = 1 when a row is listed twice.  With mask_compact_rows this
 * gives the sorted, duplicate-free test rows of a fold (backend/sglm_cv.py:106-110) without a sort. */
int sglm_index_mask_u8(const int64_t *idx, int64_t n_idx, uint8_t *mask, int64_t T, int32_t *dup_flag, void *stream);
/* Disjoint cells of overlapping row sets (the full data contain every test fold; random folds intersect —
 * GroupShuffleSplit, backend/sglm_pp.py:262-263) without a sort:
 *   rows_or_bit          : sig[t] |= 1 << bit for the rows listed in set `bit` (sig zeroed by the caller, <= 62 sets);
 *   cells_from_signatures: distinct signatures -> cell ids; `table` (device, 4104 bytes) = 256 keys (uint64, ~0 = empty
 *                          slot), 256 row counts (int64), {slots used, overflow flag} (int32); cell_of[t] = slot;
 *   match_compact_rows   : ascending rows of one cell (rows whose byte equals `match`). */
int sglm_rows_or_bit_u64(const int64_t *idx, int64_t n_idx, int32_t bit, uint64_t *sig, int64_t T, void *stream);
int sglm_cells_from_signatures(const uint64_t *sig, int64_t T, uint8_t *cell_of, void *table, void *stream);
int sglm_match_compact_rows(const uint8_t *ids, int64_t T, int32_t match, int64_t *rows, void *workspace,
                            size_t workspace_bytes, void *stream);
/* np.roll(y, shift) (the `roll` key of a parameter set, backend/sglm_cv.py:95-96): out[(i + shift) mod n] = y[i]. */
int sglm_roll_f64(const double *y, int64_t n, int64_t shift, double *out, void *stream);
size_t sglm_mask_compact_workspace_bytes(int64_t T);
int sglm_mask_compact_rows(const uint8_t *valid, int64_t T, int64_t *rows, void *workspace,
                           size_t workspace_bytes, void *stream);
int sglm_timeshift_rows_f64(const double *X, int64_t T, int32_t n_cols_in, int64_t ldx, const int32_t *col_src,
                            const int32_t *col_shift, int32_t n_cols_out, uint64_t fill_bits,
                            const int64_t *rows, int64_t n_rows, double *out, int64_t ldo, void *stream);

/* ------------------------------------------------------------------------- *
 * Sufficient statistics.  Replaces the X'X / X'y work that every sklearn fit
 * repeats per (fold, alpha) (sklearn/linear_model/_ridge.py:215-227,
 * _cd_fast.pyx:243-506 sweeps, _base.py:_preprocess_data) and the fancy-index
 * fold copies of backend/sglm_cv.py:106-110.
 *
 * For each weight set s:  G[s] = Z' diag(w_s) Z   with  Z = [X | Y | 1]
 * (n_aug = C + n_y + 1 columns), written as a full symmetric row-major matrix
 * G[s][i*ldg + j], ldg >= n_aug.  So G[:C,:C] = X'WX, G[:C, C+k] = X'W y_k,
 * G[:C, C+n_y] = sum w x,  G[C+k, C+k] = y_k'W y_k, G[n_aug-1, n_aug-1] = sum w.
 * W is [n_sets][ldw] (row counts / IRLS weights); a NULL W means unit weights
 * for every set.  ksplit_host[s] (host array, may be NULL) is the number of
 * K-chunks set s is split into.
 * ------------------------------------------------------------------------- */
size_t sglm_suffstats_workspace_bytes(int64_t T, int32_t C, int32_t n_y, int32_t n_sets,
                                      const int32_t *ksplit_host);
int sglm_suffstats_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y,
                       int64_t T, int32_t C, const double *W, int64_t ldw, int32_t n_sets,
                       const int32_t *ksplit_host, double *G, int64_t ldg, void *workspace,
                       size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------- *
 * Tensor-core Gram (tcgen05 kind::i8 + TMA + TMEM): the same statistics as
 * sglm_suffstats_f64 for 0/1 row sets, computed exactly in integers from signed
 * radix-128 digit planes of the fp64 columns (split / Ozaki scheme) and recombined in
 * fp64; columns that are exactly representable in fewer digits (0/1 event indicators)
 * only get the planes they need.  Two calls:
 *   analyze : device colE[n_aug] (scale exponents), colS[n_aug] (digit planes per column,
 *             1..8), flag != 0 when the data hold NaN/inf.  colmax_scratch: n_aug uint64.
 *   gram    : colS_host = host copy of colS; set_rows_host[s] = rows of set s; rows = device
 *             int64, the concatenated row lists of the sets, each padded with -1 to a multiple
 *             of 128.  G as in sglm_suffstats_f64.  use_check_gemm != 0 replaces the tcgen05
 *             GEMM by a CUDA-core integer GEMM (bit-identical results; validation only).
 *   plan_info: out4_host = {digit-plane rows S, positions, output tiles of 256x256, K parts}
 *             (issued int8 MACs = tiles * 256 * 256 * positions).
 * ------------------------------------------------------------------------- */
int sglm_gram_tc_analyze_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y,
                             int64_t T, int32_t C, int32_t *colE, int32_t *colS,
                             uint64_t *colmax_scratch, int32_t *flag, void *stream);
size_t sglm_gram_tc_workspace_bytes(int32_t n_aug, const int32_t *colS_host, int32_t n_sets,
                                    const int64_t *set_rows_host);
int sglm_gram_tc_plan_info(int32_t n_aug, const int32_t *colS_host, int32_t n_sets,
                           const int64_t *set_rows_host, int64_t *out4_host);
int sglm_gram_tc_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                     int32_t C, const int32_t *colE, const int32_t *colS, const int32_t *colS_host,
                     int32_t n_sets, const int64_t *set_rows_host, const int64_t *rows, double *G,
                     int64_t ldg, void *workspace, size_t workspace_bytes, int32_t use_check_gemm,
                     void *stream);

/* Weighted tensor-core Gram: rows of Z scaled by row_scale[t] (sqrt of a row weight: G = Z' diag(w) Z) and at
 * most max_planes digit planes per column (fewer than a column needs = digits rounded at the last plane: each
 * value off by at most 2^(E - 7 max_planes), i.e. 2^-(7 max_planes) of the column scale 2^E > max |z|; a
 * round-half-even tie at the last plane reaches it).  Replaces the X'WX of every Newton / IRLS step of the Poisson fit
 * (sklearn _glm/_newton_solver.py:315-359) as an APPROXIMATE Hessian; the gradient stays exact (sglm_xt_vec_f64). */
int sglm_gram_tc_analyze_scaled_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y,
                                    int64_t T, int32_t C, const double *row_scale, int32_t max_planes,
                                    int32_t *colE, int32_t *colS, uint64_t *colmax_scratch, int32_t *flag,
                                    void *stream);
int sglm_gram_tc_scaled_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                            int32_t C, const double *row_scale, const int32_t *colE, const int32_t *colS,
                            const int32_t *colS_host, int32_t n_sets, const int64_t *set_rows_host,
                            const int64_t *rows, double *G, int64_t ldg, void *workspace,
                            size_t workspace_bytes, void *stream);
/* out[c] = sum_t X[t][c] r[t] (X'r: the exact gradient of a GLM loss), one pass over X, deterministic. */
size_t sglm_xt_vec_workspace_bytes(int32_t C);
int sglm_xt_vec_f64(const double *X, int64_t ldx, const double *r, int64_t T, int32_t C, double *out,
                    void *workspace, size_t workspace_bytes, void *stream);

/* The same statistics from DISJOINT cells.  The row sets of a CV grid overlap (the full data contain every
 * test fold, random folds intersect); the partition they induce has n_cells cells, the int8 GEMM runs once over
 * every row (not once per set), and the Gram of output set o is the exact integer sum of the cells with
 * member_host[o * n_cells + c] != 0.  rows / cell_rows_host as rows / set_rows_host above; G holds n_out sets. */
size_t sglm_gram_tc_cells_workspace_bytes(int32_t n_aug, const int32_t *colS_host, int32_t n_cells,
                                          const int64_t *cell_rows_host, int32_t n_out);
int sglm_gram_tc_cells_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                           int32_t C, const int32_t *colE, const int32_t *colS, const int32_t *colS_host,
                           int32_t n_cells, const int64_t *cell_rows_host, const int64_t *rows, int32_t n_out,
                           const int32_t *member_host, double *G, int64_t ldg, void *workspace,
                           size_t workspace_bytes, int32_t use_check_gemm, void *stream);

/* Row-sharded form (one process per GPU, each holding a slice of the rows; SURVEY.md §8e "alternative"):
 *   colstats / exponents : the column analysis in two steps — every rank scans its rows (colmax_bits = bits of
 *              max |z| per column, col_lsb = lowest set bit per column), the ranks combine them (all-reduce max /
 *              min), and sglm_gram_tc_exponents derives the same colE / colS everywhere (colS: lowest set bits on
 *              entry, digit-plane counts on exit);
 *   cells_partial : slicing + int8 GEMM + cell sums of THIS rank's rows; the int64 plane Grams of the n_out row sets
 *              stay in the workspace at the offset sglm_gram_tc_cells_sgout reports (same offset and size on every
 *              rank: the digit-plane layout depends only on the combined analysis); the caller adds them over the
 *              ranks (ncclAllReduce int64 sum — exact, so the result has the bits of the one-GPU computation);
 *   cells_combine : fp64 recombination of the summed plane Grams -> G. */
int sglm_gram_tc_colstats_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                              int32_t C, uint64_t *colmax_bits, int32_t *col_lsb, void *stream);
int sglm_gram_tc_exponents(const uint64_t *colmax_bits, int32_t n_aug, int32_t max_planes, int32_t *colE,
                           int32_t *colS, int32_t *flag, void *stream);
int sglm_gram_tc_cells_sgout(int32_t n_aug, const int32_t *colS_host, int32_t n_cells, const int64_t *cell_rows_host,
                             int32_t n_out, uint64_t *offset_bytes, uint64_t *size_bytes);
int sglm_gram_tc_cells_partial_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                                   int32_t C, const int32_t *colE, const int32_t *colS, const int32_t *colS_host,
                                   int32_t n_cells, const int64_t *cell_rows_host, const int64_t *rows, int32_t n_out,
                                   const int32_t *member_host, void *workspace, size_t workspace_bytes, void *stream);
/* Row-sharded WEIGHTED Gram (the Hessian X' diag(w) X of a row-sharded GLM iteration), rows of Z scaled by row_scale:
 *   colstats_scaled : sglm_gram_tc_colstats_f64 with row_scale (NULL only when T == 0); the ranks combine (max / min),
 *                     then sglm_gram_tc_exponents with the Gram's max_planes;
 *   scaled_partial  : sglm_gram_tc_cells_partial_f64 with row_scale; finish with sglm_gram_tc_cells_combine_f64.
 * The int64 partials summed over ANY partition of the rows, then combined, are the bits of sglm_gram_tc_scaled_f64
 * over all rows. */
int sglm_gram_tc_colstats_scaled_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                                     int32_t C, const double *row_scale, uint64_t *colmax_bits, int32_t *col_lsb,
                                     void *stream);
int sglm_gram_tc_scaled_partial_f64(const double *X, int64_t ldx, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                                    int32_t C, const double *row_scale, const int32_t *colE, const int32_t *colS,
                                    const int32_t *colS_host, int32_t n_cells, const int64_t *cell_rows_host,
                                    const int64_t *rows, int32_t n_out, const int32_t *member_host, void *workspace,
                                    size_t workspace_bytes, void *stream);
int sglm_gram_tc_cells_combine_f64(int32_t C, int32_t n_y, const int32_t *colE, const int32_t *colS,
                                   const int32_t *colS_host, int32_t n_cells, const int64_t *cell_rows_host,
                                   int32_t n_out, double *G, int64_t ldg, void *workspace, size_t workspace_bytes,
                                   void *stream);

/* Lag designs WITHOUT the design matrix.  A column of a lag design (backend/sglm_pp.py:23-103 timeshift /
 * timeshift_multiple) is a base signal read at another row: Z[t, c] = base[t + off[c], src[c]].  Its digit planes are
 * the base signal's planes read at another position, so the statistics need neither the T x (P*L) fp64 design nor a
 * pass over it: the P base signals are sliced once, the K-major int8 operand is a byte gather from those planes
 * (tc_expand_kernel), the GEMM / cell sums / recombination are the ordinary ones.
 *   base       : device, the window of the base signals every column reads (n_u rows, row stride ldb);
 *   src / off  : host [C]; design row t of column c = window row t + off[c] (0 <= off[c], off[c] + T <= n_u);
 *   baseE / baseS (device) and baseS_host : scale exponents and digit planes of [base | 1] (P + 1 entries) over the
 *                window (sglm_gram_tc_colstats_f64 + sglm_gram_tc_exponents on the window); the caller gives every
 *                lag column the exponent and plane count of its base signal: colE[c] = baseE[src[c]], colS likewise;
 *                the entries of the response columns and the ones column (c >= C) come from the same two calls on Y.
 *   n_out == 0 : the row lists are the sets; n_out > 0: cells + membership (sglm_gram_tc_cells_f64);
 *   partial    : stop after the int64 plane Grams of the sets (row-sharded use), finish with
 *                sglm_gram_tc_cells_combine_f64 on the same workspace. */
typedef struct sglm_lag_design {
    const double *base;
    int64_t ldb;
    int64_t n_u;
    int32_t P;
    const int32_t *src_host;
    const int32_t *off_host;
    const int32_t *baseE;
    const int32_t *baseS;
    const int32_t *baseS_host;
} sglm_lag_design;
size_t sglm_gram_tc_lag_workspace_bytes(int32_t n_aug, const int32_t *colS_host, int32_t n_cells,
                                        const int64_t *cell_rows_host, int32_t n_out, int32_t P,
                                        const int32_t *baseS_host, int64_t n_u);
int sglm_gram_tc_lag_cells_f64(const sglm_lag_design *lag, const double *Y, int64_t ldy, int32_t n_y, int64_t T,
                               int32_t C, const int32_t *colE, const int32_t *colS, const int32_t *colS_host,
                               int32_t n_cells, const int64_t *cell_rows_host, const int64_t *rows, int32_t n_out,
                               const int32_t *member_host, double *G, int64_t ldg, void *workspace,
                               size_t workspace_bytes, int32_t partial, void *stream);

/* Index lists -> per-row multiplicities: counts[idx[i]] += 1 (the fold row sets of
 * backend/sglm_cv.py:106-110, X[idx_train,:] / X[idx_test,:]).  counts must be zeroed. */
int sglm_index_counts_f64(const int64_t *idx, int64_t n_idx, double *counts, int64_t T,
                          void *stream);

/* Centred problem from augmented statistics (sklearn _base.py:_preprocess_data +
 * _pre_fit): with A = A_plus - A_minus (A_minus may be NULL), n = A[1,1],
 * xbar = A[:C,1]/n, ybar = A[y,1]/n:
 *   Qc = A[:C,:C] - n xbar xbar',  qc = A[:C,y] - n xbar ybar,  yyc = A[y,y] - n ybar^2
 * (fit_intercept = 0: no centring, xbar = ybar = 0).  diag[i] = Qc[i,i] (compact copy for
 * the coordinate-descent kernel).  scal = {yyc, n, ybar, sum_y}. */
int sglm_center_stats_f64(const double *A_plus, const double *A_minus, int64_t ldg, int32_t C,
                          int32_t n_y, int32_t y_col, int32_t fit_intercept, double *Qc,
                          int64_t ldq, double *qc, double *xbar, double *diag, double *scal,
                          void *stream);

/* ------------------------------------------------------------------------- *
 * (a6) batched Gram coordinate descent — ElasticNet / Lasso.  Replaces
 * sklearn cd_fast.enet_coordinate_descent as reached from backend/sglm.py:106-110,
 * :241 (sklearn/linear_model/_cd_fast.pyx:243-506; Gram form :1095-1290):
 * cyclic order, soft threshold, trigger d_w_max/w_max <= tol, stop on
 * gap <= tol*yy, gap-safe screening (sklearn 1.9), cold or warm start.
 * One CTA per model, several models resident per SM; the sweep is blocked by 32 coordinates
 * (register/shuffle phase, then one streamed panel update of the rows that moved) with
 * iterates bit-identical to the sequential algorithm.
 *   prob_Q[p], prob_q[p], prob_diag[p] : device arrays of device pointers (Qc, qc,
 *   diag(Qc) from sglm_center_stats_f64); prob_yy[p] = yyc
 *   model m uses problem prob_of_model[m] with l1_reg[m] = alpha*l1_ratio*n and
 *   l2_reg[m] = alpha*(1-l1_ratio)*n  (_coordinate_descent.py:781-782).
 *   W[m*ldw + j] is in/out when warm_start & 1, else out (started from 0).  warm_start & 2: at least one sweep (the
 *   start is never returned on its duality gap alone; the sweep's largest move then decides).
 *   info[m*6 + {0..5}] = {gap, tol*yy, n_iter, n_row_updates, n_blocks_visited, share of time in the register phase}.
 * ------------------------------------------------------------------------- */
int sglm_enet_cd_gram_f64(const double *const *prob_Q, const double *const *prob_q,
                          const double *const *prob_diag, const double *prob_yy, int64_t ldq, int32_t C,
                          const int32_t *prob_of_model, const double *l1_reg,
                          const double *l2_reg, const double *tol, const int32_t *max_iter,
                          int32_t n_models, int32_t warm_start, int32_t do_screening,
                          double *W, int64_t ldw, double *info, void *stream);

/* Same fits, same iterates (a6), second-generation layout: one thread-block CLUSTER of
 * cluster_size CTAs per GROUP of group_size models that share a problem (fold).  The
 * coordinate blocks (w, Qw slice, register phase) are split over the cluster's CTAs, block
 * deltas travel as records through distributed shared memory, the panel update of a record
 * overlaps the next block's register phase (look-ahead), and a moved row of Q is loaded once
 * for all models of the group.
 *   group g uses problem prob_of_group[g]; its models are model_of_slot[g*group_size + s]
 *   (index into l1_reg / l2_reg / tol / max_iter, row of W and info; -1 = empty slot).
 *   Q pointers must be 16-byte aligned and ldq even.  Other arguments as above.
 *   prob_tmap: device array (64-byte aligned) of one TMA descriptor per problem, encoded on the host by
 *   sglm_enet_cd_cluster_encode_tmaps (Q_dev_ptrs = the same device pointers as prob_Q, as host values)
 *   into n_prob * sglm_enet_cd_cluster_tmap_bytes() bytes and copied to the device by the caller.
 *   group_stats (may be NULL): [n_groups][2] = {rows of Q the group's cluster loaded (a moved row is loaded once
 *   for all models of the group: 8*C bytes each), coordinate-block records processed} — measurement only.
 * sglm_enet_cd_cluster_supported(group_size, cluster_size) -> 1 if that shape is compiled in. */
int sglm_enet_cd_cluster_supported(int32_t group_size, int32_t cluster_size);
size_t sglm_enet_cd_cluster_tmap_bytes(void);
/* shared memory per CTA of that shape for C columns (must stay <= 227 KB; 0 = shape not compiled in) */
size_t sglm_enet_cd_cluster_smem_bytes(int32_t group_size, int32_t cluster_size, int32_t C);
int sglm_enet_cd_cluster_encode_tmaps(const uint64_t *Q_dev_ptrs, int32_t n_prob, int32_t C, int64_t ldq, void *out);
int sglm_enet_cd_cluster_f64(const double *const *prob_Q, const double *const *prob_q,
                             const double *const *prob_diag, const double *prob_yy, int64_t ldq, int32_t C,
                             const int32_t *prob_of_group, const int32_t *model_of_slot,
                             const double *l1_reg, const double *l2_reg, const double *tol,
                             const int32_t *max_iter, int32_t n_groups, int32_t group_size,
                             int32_t cluster_size, int32_t warm_start, int32_t do_screening,
                             double *W, int64_t ldw, double *info, const void *prob_tmap,
                             double *group_stats, void *stream);

/* ------------------------------------------------------------------------- *
 * (a7, a8) batched Cholesky solve — Ridge / OLS.  Replaces sklearn
 * _ridge._solve_cholesky (sklearn/linear_model/_ridge.py:215-227) and the
 * full-rank case of LinearRegression (_base.py:700-756):
 *   (Qc + alpha[k] I) w_k = qc   for k < n_alpha, one CTA per alpha.
 * work holds n_alpha * (C+1) * ldq doubles.  status[k]: bit 0 = not positive definite
 * (a pivot <= 0), bit 1 = a pivot at rounding-noise level (<= 1e-11 of the largest diagonal
 * entry: numerically rank deficient; the solve still completes).
 * ------------------------------------------------------------------------- */
size_t sglm_ridge_workspace_bytes(int32_t C, int64_t ldq, int32_t n_alpha);
int sglm_ridge_solve_f64(const double *Qc, int64_t ldq, const double *qc, int32_t C,
                         const double *alpha, int32_t n_alpha, double *W, int64_t ldw,
                         int32_t *status, void *work, size_t work_bytes, void *stream);
/* (a8) minimum-norm least squares for numerically rank-deficient normal equations — what scipy.linalg.lstsq(X, y,
 * cond = rcond) returns inside sklearn's LinearRegression (_base.py:750-753; reached from backend/sglm.py:96-101 when
 * alpha == 0): singular values of the centred X below rcond * s_max are dropped.  One-sided Jacobi on Qc = Xc'Xc, on
 * the device.  Runs only when (*status & status_mask) != 0 (*status: device int32 from sglm_ridge_solve_f64), overwrites
 * w and clears *status; returns at once otherwise — no host synchronisation either way.  shift = alpha > 0 solves the
 * Ridge system (Qc + alpha I) w = qc the same way (sklearn's SVD fallback for a failed Cholesky, _ridge.py:_solve_svd). */
size_t sglm_ols_minnorm_workspace_bytes(int32_t C);
int sglm_ols_minnorm_f64(const double *Qc, int64_t ldq, const double *qc, int32_t C, double rcond, double shift,
                         int32_t status_mask, int32_t *status, double *w, void *work, size_t work_bytes, void *stream);
/* x = (L L')^-1 rhs with the Cholesky factor of system k that sglm_ridge_solve_f64 left in `work`
 * (a solve without a second factorisation: chord iterations of the Poisson Newton solver). */
int sglm_chol_solve_f64(const void *work, int64_t ldq, int32_t C, int32_t k, const double *rhs, double *out,
                        void *stream);

/* Intercepts and augmented evaluation vectors (sklearn _set_intercept,
 * _coordinate_descent.py:1281):  b[m] = ybar[p] - xbar[p].w_m  (0 if xbar NULL)
 *   V[m] = [-w_m | e_{y_col} | -b_m]  so that  RSS(set) = V[m]' G[set] V[m]. */
int sglm_finalize_models_f64(const double *W, int64_t ldw, int32_t C, int32_t n_y,
                             const int32_t *y_col_of_model, const double *const *xbar_of_model,
                             const double *ybar_of_model, int32_t n_models, double *intercept,
                             double *V, int64_t ldv, void *stream);

/* (a11) scores from statistics: out[m] = V[m]' A V[m]  (A symmetric n x n). */
int sglm_quadform_f64(const double *A, int64_t lda, int32_t n, const double *V, int64_t ldv,
                      int32_t n_models, double *out, void *stream);
/* Row-split form for few models: partial[s * n_models + m] = sum over the rows of split s of v_m[i] (A v_m)[i];
 * the caller adds the n_splits partial sums in order. */
int sglm_quadform_split_f64(const double *A, int64_t lda, int32_t n, const double *V, int64_t ldv,
                            int32_t n_models, int32_t n_splits, double *partial, void *stream);

/* ------------------------------------------------------------------------- *
 * (a10, a11) explicit-matrix paths: GLM.predict / neg_mse_score / r2_score /
 * get_residuals (backend/sglm.py:150-184, :314-347).  link: 0 identity, 1 log.
 *   predict: out[t] = g^-1(X[t,:].w + b)
 *   score:   sums[0..7] = { n, sum r^2, sum y, sum y^2, sum y*eta, sum mu,
 *                           sum y log y, sum r }   with r = y - g^-1(eta), every term
 *            weighted by the row multiplicity rw[t] (NULL = 1; selects a fold)
 *            (resid may be NULL; else resid[t] = r).  ws: sglm_score_workspace_bytes().
 * ------------------------------------------------------------------------- */
int sglm_predict_f64(const double *X, int64_t ldx, int64_t T, int32_t C, const double *w,
                     const double *b_dev, int32_t link, double *out, void *stream);
size_t sglm_score_workspace_bytes(void);
int sglm_score_f64(const double *X, int64_t ldx, const double *y, const double *rw, int64_t T,
                   int32_t C, const double *w, const double *b_dev, int32_t link, double *resid,
                   double *sums, void *workspace, void *stream);

/* ------------------------------------------------------------------------- *
 * (a9) Poisson IRLS step.  Replaces one iteration of the TweedieRegressor(power=1)
 * optimisation (sklearn/linear_model/_glm/glm.py:185-339; Newton form
 * _glm/_newton_solver.py) for objective mean(mu - y*eta) + alpha/2 |w|^2:
 *   eta = X w + b, mu = exp(eta), weight[t] = rw[t]*mu, z[t] = eta + (y-mu)/mu,
 *   sums[0..3] = { sum rw*(mu - y*eta), sum rw*mu, sum rw, sum rw*y }.
 * rw (row multiplicity, may be NULL = 1) selects the fold.  The weighted
 * statistics of [X | z | 1] then come from sglm_suffstats_f64 and the Newton
 * system from sglm_center_stats_f64 + sglm_ridge_solve_f64.
 * ------------------------------------------------------------------------- */
int sglm_poisson_irls_prepare_f64(const double *X, int64_t ldx, const double *y, const double *rw,
                                  int64_t T, int32_t C, const double *w, const double *b_dev,
                                  double *weight, double *z, double *sums, void *workspace,
                                  void *stream);

/* ------------------------------------------------------------------------- *
 * The same two passes for the Tweedie family of `power` with log link (scikit-learn
 * TweedieRegressor(power=p) / HalfTweedieLoss; reference backend/sglm.py:112-117:
 * 'Poisson' p = 1, 'Gamma' p = 2, 'Tweedie' any p).  power must be 1 or > 1, else
 * SGLM_E_UNSUPPORTED before any CUDA call.  power = 1 computes exactly what
 * sglm_score_f64 (link 1) / sglm_poisson_irls_prepare_f64 compute.
 *   score_glm:         sums[0..7] = { n, sum r^2, sum y, sum y^2, s4, s5, s6, sum r },
 *                      r = y - mu; the deviance terms s4..s6 are
 *                        p = 1: { y*eta, mu, y log y };  p = 2: { eta, y/mu, log y };
 *                        other p: { y mu^(1-p), mu^(2-p), y^(2-p) }.
 *   glm_irls_prepare:  weight[t] = rw[t] * mu^(2-p) (Fisher weight), z[t] = eta + (y-mu)/mu,
 *                      sums[0..3] = { sum rw*loss, sum weight, sum rw, sum rw*y } with the
 *                      unit loss mu - y eta (p = 1), eta + y/mu (p = 2),
 *                      mu^(2-p)/(2-p) - y mu^(1-p)/(1-p) (other p).
 * ------------------------------------------------------------------------- */
int sglm_score_glm_f64(const double *X, int64_t ldx, const double *y, const double *rw, int64_t T,
                       int32_t C, const double *w, const double *b_dev, double power, double *resid,
                       double *sums, void *workspace, void *stream);
int sglm_glm_irls_prepare_f64(const double *X, int64_t ldx, const double *y, const double *rw,
                              int64_t T, int32_t C, const double *w, const double *b_dev, double power,
                              double *weight, double *z, double *sums, void *workspace, void *stream);

/* ------------------------------------------------------------------------- *
 * Steps either side of the lag builder, for data already on the device (SURVEY.md §8f-3):
 *   col_moments + zscore_apply : sglm_pp.zscore (backend/sglm_pp.py:105-118): (X - mean) / std per column; ddof 0 =
 *                   numpy std (ndarray input), 1 = pandas std (DataFrame input); skipna as pandas does.
 *   diff1         : one first difference of the listed columns (sglm_pp.diff, :120-190; the n-th difference is n
 *                   calls, the way np.diff computes it — bit-exact).
 *   rolling_minmax: sglm_pp.detrend_data (:522-545): pandas rolling(window, center=True).apply(lambda_min_max) —
 *                   the window's element (W+1)//2 - 1 scaled by the window's 5 % / 95 % quantiles (linear
 *                   interpolation); NaN where the window leaves its group segment or holds a NaN or +-inf
 *                   (pandas' rolling counts +-inf as missing).  col_moments: sd is NaN when at most ddof values
 *                   remain (an all-NaN column with skipna, one value with ddof 1).
 * ------------------------------------------------------------------------- */
size_t sglm_col_moments_workspace_bytes(int64_t T, int32_t C);
int sglm_col_moments_f64(const double *X, int64_t ldx, int64_t T, int32_t C, int32_t ddof, int32_t skipna,
                         double *mean, double *sd, void *workspace, size_t workspace_bytes, void *stream);
int sglm_zscore_apply_f64(const double *X, int64_t ldx, int64_t T, int32_t C, const double *mean, const double *sd,
                          double *out, int64_t ldo, void *stream);
int sglm_diff1_f64(const double *X, int64_t ldx, int64_t T, const int32_t *cols, int32_t n_cols, double *out,
                   int64_t ldo, void *stream);
int sglm_rolling_minmax_f64(const double *x, int64_t n, const int64_t *seg_lo, const int64_t *seg_hi, int32_t window,
                            double *out, void *stream);

/* Batched triangular solves with cached factors: out[s] = (L_s L_s')^-1 rhs[s] for every system s with
 * flags[s] == 1 (flags may be NULL); L_of[s] = factor left by sglm_ridge_solve_f64 (work + k (C+1) ldq doubles). */
int sglm_chol_solve_batched_f64(const double *const *L_of, int64_t ldq, int32_t C, const double *rhs, double *out,
                                int64_t ld, const int32_t *flags, int32_t n_systems, void *stream);

/* ------------------------------------------------------------------------- *
 * (a9, batched) Poisson grid: all (fold, alpha) fits of a sweep advance together.  Replaces the per-(fold, alpha)
 * TweedieRegressor(power=1).fit calls of backend/sglm.py:112-115, :241 (sklearn _glm/glm.py:185-339).  One
 * iteration of the whole batch of B models (columns of Wt [C][ldb], ldb % 64 == 0):
 *   sglm_pb_eta_f64       Eta [T][ldb] = X Wt                        (fp64 GEMM: X read once for all models)
 *   sglm_pb_epilogue_f64  mode 0: Eta <- R = rw (exp(Eta + b) - y) in place, sums [B][4] =
 *                                 {sum rw (mu - y eta), sum rw mu, sum rw, sum rw (mu - y)};
 *                         mode 1: sums [B][2][8] = the sglm_score_f64 sums for the row weights rw_a / rw_b
 *                         (Y [T][ldy] response columns, ycol[m]; RW [n_w][ldrw] row-weight vectors, rw id -1 = all
 *                         rows, rw_b id -2 = no rows; models with status != 0 are skipped in mode 0)
 *   sglm_pb_xt_r_f64      Gw [C][ldb] = X' R                         (fp64 GEMM, deterministic split over T)
 *   sglm_pb_step_f64      per model: objective check / step halving, rhs = H~ w - g, batched triangular solves
 *                         with the cached factors L_of[m] of (H~ + alpha n I), intercept, convergence test.
 *                         state_host: the solver state (device pointers and sizes) as sglm_pb_state_words()
 *                         64-bit words — see PbState in csrc/poisson_batch.cu; built by _engine.py.
 * H~ = X' diag(rw mu_ref) X of one reference model per fold comes from sglm_gram_tc_scaled_f64 (tcgen05). */
/* Quadratic forms of MANY vectors: out[m] = v_m' A v_m with the vectors as the columns of Vt [n][ldb] (ldb % 64 == 0,
 * columns >= n_models zero): one fp64 GEMM Y = A Vt (A read once per 64 vectors) + column dots in 16 fixed row chunks
 * (deterministic).  Y [n][ldb] and part [16][n_models] are caller buffers.  The scores of a CV grid from the
 * statistics (RSS(model, row set) = v' G[set] v; the reference: three prediction passes per fit, backend/sglm.py:305-312). */
int sglm_quadform_gemm_f64(const double *A, int64_t lda, int32_t n, const double *Vt, int64_t ldb, int32_t n_models,
                           double *Y, double *part, double *out, void *stream);
size_t sglm_pb_gemm_tn_workspace_bytes(int64_t T, int32_t C, int64_t ldb);
int sglm_pb_eta_f64(const double *X, int64_t ldx, int64_t T, int32_t C, const double *Wt, int64_t ldb, double *Eta,
                    void *stream);
int sglm_pb_xt_r_f64(const double *X, int64_t ldx, int64_t T, int32_t C, const double *R, int64_t ldb, double *Gw,
                     void *workspace, size_t workspace_bytes, void *stream);
size_t sglm_pb_epilogue_workspace_bytes(int64_t T, int32_t n_models);
int sglm_pb_epilogue_f64(double *Eta, int64_t ldb, int32_t n_models, int64_t T, const double *Y, int64_t ldy,
                         const int32_t *ycol, const double *RW, int64_t ldrw, const int32_t *rw_a,
                         const int32_t *rw_b, const double *b, const int32_t *status, int32_t mode, double *sums,
                         void *workspace, size_t workspace_bytes, void *stream);
/* sglm_pb_epilogue_f64 for the Tweedie family of `power` (1, or > 1 — else SGLM_E_UNSUPPORTED before any CUDA call;
 * log link): mode 0 writes R = rw dloss/deta = rw mu^(1-p) (mu - y) and sums [B][4] = {sum rw loss, sum rw mu^(2-p),
 * sum rw, sum R}; mode 1 the sglm_score_glm_f64 sums.  power = 1 is sglm_pb_epilogue_f64.
 * RW is not checked: a model with rw_a (or, in mode 1, rw_b) >= 0 reads RW row rw_a, so RW = NULL is only valid
 * when T = 0 or every id is negative.  T = 0 (an empty row slice) accepts Eta = Y = NULL and writes zero sums; the
 * same holds for X / R of sglm_pb_xt_r_f64 (Gw = 0), X / r of sglm_xt_vec_f64 (out = 0) and X / y / resid / weight /
 * z of sglm_score_glm_f64 and sglm_glm_irls_prepare_f64.  sglm_pb_xt_r_f64 needs R and its workspace 16-byte
 * aligned. */
int sglm_glm_epilogue_f64(double *Eta, int64_t ldb, int32_t n_models, int64_t T, const double *Y, int64_t ldy,
                          const int32_t *ycol, const double *RW, int64_t ldrw, const int32_t *rw_a,
                          const int32_t *rw_b, const double *b, const int32_t *status, double power, int32_t mode,
                          double *sums, void *workspace, size_t workspace_bytes, void *stream);
/* out[e] = parts[0][e] + parts[1][e] + ... in that order (parts [n_parts][n_elem]): the fixed-order sum of per-rank
 * fp64 partials gathered in rank order, so every rank of a row-sharded batch holds the same bits. */
int sglm_reduce_parts_f64(const double *parts, int64_t n_elem, int32_t n_parts, double *out, void *stream);
int sglm_pb_state_words(void);
int sglm_pb_step_f64(const uint64_t *state_host, const double *const *L_of, void *stream);
/* Elastic-net models in the batch (l1_ratio[m] = r > 0, l1_ratio [B]; the objective check adds alpha r |w|_1 and the
 * ridge weight becomes alpha (1 - r)): sglm_pb_step_f64 in which the models enet_models[0 .. n_enet) take a proximal-Newton
 * step — after the chord solve (which gives their ridge solution for the gap's yy), a warm-started
 * sglm_enet_cd_gram_f64 solve of  1/2 w'Qw - rhs'w + (alpha r n / hs)|w|_1 + 1/2 (alpha (1 - r) n / hs)|w|^2
 * replaces their new iterate.  L_of[m] of such a model factors (H~ + alpha (1 - r) n I).  workspace: 16-byte aligned,
 * sglm_pb_enet_workspace_bytes(C, ldw, n_enet) bytes; info [6 n_enet] = the inner solves' CD info (info[6k + 2]:
 * sweeps; 0 for a model that took no step).  Arguments are checked before any CUDA call. */
size_t sglm_pb_enet_workspace_bytes(int32_t C, int64_t ldw, int32_t n_enet);
int sglm_pb_step_enet_f64(const uint64_t *state_host, const double *const *L_of, const double *l1_ratio,
                          const int32_t *enet_models, int32_t n_enet, void *workspace, size_t workspace_bytes,
                          double *info, void *stream);

/* ------------------------------------------------------------------------- *
 * Measurement probe (bench.py; no reference counterpart): reads `n_doubles` doubles
 * `repeats` times with the access pattern of the coordinate-descent panel (16-byte
 * loads, 8 in flight per thread).  A buffer that fits L2 measures the L2 -> SM read
 * bandwidth, one far larger than L2 the HBM read bandwidth; the caller times it.
 * ------------------------------------------------------------------------- */
/* Issue rate of tcgen05.mma kind::i8 (operands resident in shared memory, one CTA per SM): int8 MACs issued =
 * *n_ctas_host * iters * 8 * 128 * 256 * 32; the denominator of the Gram GEMM's tensor-pipe fraction. */
int sglm_probe_mma_i8(int32_t iters, int64_t *n_ctas_host, void *stream);
int sglm_probe_read_f64(const double *buf, int64_t n_doubles, int32_t repeats, int32_t ctas_per_sm,
                        double *sink, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SGLM_B200_H */
