/*
 * slic_b200.h - C ABI of the B200-native FINCH / nearest-neighbour hot path.
 *
 * The reference (rvl-lab-utoronto/video_similarity_search) is pure Python: it has no FFI layer,
 * its module-level functions are the boundary.  This header is what a binding for that path
 * would call instead of numpy / scipy / scikit-learn; every entry point names the reference
 * lines it replaces (paths relative to the reference root).  INTEGRATION.md shows the ctypes
 * stub a maintainer adds on the reference side.
 *
 * Conventions
 *   - every function returns 0 (SLIC_OK) or a negative slic_status; the message for the last
 *     failure on the calling thread is slic_last_error().  Nothing throws across the boundary.
 *   - pointers named *_dev are device pointers on the current CUDA device; the *_host entry
 *     points at the end take host buffers and do their own transfers.
 *   - all device work is ordered on `stream` (a cudaStream_t passed as void*; NULL = the legacy
 *     default stream); temporaries come from the stream-ordered allocator, so no call blocks the
 *     host except where a result is returned through a host pointer (documented per call).
 *   - dtype: SLIC_F32 or SLIC_F64 - the arithmetic type of the reference at that call site
 *     (float32 at FINCH level 0, float64 at levels >= 1: clustering/finch.py:62,131).
 *   - matrices are dense row-major; indices / labels on the device are int32.
 *   - there is no CPU fallback: without an sm_100 device the calls fail with SLIC_ERR_NO_DEVICE.
 */
#ifndef SLIC_B200_H
#define SLIC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLIC_ABI_VERSION 1

#define SLIC_F32 0
#define SLIC_F64 1

#define SLIC_METRIC_COSINE 0
#define SLIC_METRIC_EUCLIDEAN 1

typedef enum slic_status {
    SLIC_OK = 0,
    SLIC_ERR_INVALID_ARG = -1,
    SLIC_ERR_CUDA = -2,
    SLIC_ERR_UNSUPPORTED = -3,
    SLIC_ERR_NO_DEVICE = -4,
    SLIC_ERR_OVERFLOW = -5
} slic_status;

typedef void* slic_stream_t; /* cudaStream_t */

/* ---- library ---------------------------------------------------------------------------- */
int slic_abi_version(void);
const char* slic_last_error(void);
/* SLIC_OK only if the current device is compute capability 10.x (B200 / sm_100a). */
int slic_require_device(void);
/* Number of CUDA kernels this library has launched in this process (monotonic). */
int64_t slic_launch_count(void);
/* Measurement hooks: with profiling enabled every launch of the tensor-core screen kernel is
 * bracketed by CUDA events on its own stream; slic_last_screen_time waits for the most recent
 * one and returns its duration and its algorithmic work (2 * nq * n * d_pad flop). */
int slic_profile_screen(int32_t enable);
int slic_last_screen_time(float* ms_out, double* flop_out);
/* Flop the tensor cores EXECUTED in that launch: equal to the algorithmic figure for rectangular searches; about
 * half of it for self-searches, which compute only the tiles on or right of the diagonal of the symmetric score
 * matrix (plus a small pre-pass) and filter each of them along rows and along columns. */
int slic_last_screen_exec_flop(double* flop_out);

/* Pipeline trace of the screen kernel (diagnostic): while enabled every launch adds, summed over its CTAs,
 * [0] cycles the TMA producer waited for a free smem stage, [1] cycles the MMA issuer waited for a free
 * accumulator (epilogue-bound), [2] for operands (TMA/L2-bound), [3] MMA issuer total, [4] cycles epilogue
 * warp 0 waited for a complete accumulator (MMA-bound), [5] epilogue warp 0 total, [6] 32-column chunks with
 * at least one candidate row and [7] chunks examined, [8] cycles the MMA issuer waited for its next unit id (scheduler,
 * pre-pass hand-over), [9] the same for epilogue warp 0, [10] units processed, [11] spare.  counters_out_host
 * (optional, [12]) receives the counters accumulated so far; they are then reset.  enable = 0 releases the buffer. */
int slic_screen_trace(int32_t enable, uint64_t* counters_out_host);

/* ---- K1 prep: row normalisation --------------------------------------------------------- */
/* sklearn cosine_similarity's normalize step behind clustering/finch.py:27, evaluate.py:213,
 * iic_retrieve_clips.py:295:  norm_i = sqrt(sum_k x_ik^2) (0 -> 1),  unit_i = x_i / norm_i in
 * `dtype`.  Optionally also emits the f16 copy (row stride d_pad, zero padded; d_pad % 64 == 0)
 * that the tensor-core screen reads.  unit_dev / norms_dev / unit_f16_dev may each be NULL. */
int slic_normalize_rows(const void* x_dev, int64_t n, int32_t d, int32_t dtype,
                        void* unit_dev, void* norms_dev,
                        uint16_t* unit_f16_dev, int32_t d_pad, slic_stream_t stream);

/* coclr_classify.py:788-789 (SURVEY.md 8f rank 4): out = x - x.mean(dim=0, keepdim=True) for a float32 [n, d] matrix.
 * Column sums in float64 (deterministic), mean rounded to float32 before the subtraction as torch holds it.
 * out_dev may alias x_dev; means_out_dev [d] is optional. */
int slic_center_columns(const float* x_dev, int64_t n, int32_t d, float* out_dev, float* means_out_dev,
                        slic_stream_t stream);

/* ---- K1 exact: brute-force first neighbour in the reference dtype ------------------------ */
/* clustering/finch.py:27-29 (pairwise_distances + fill_diagonal + argmin) without the n x n
 * matrix: for query row r (database row r + self_offset when self_offset >= 0, which is then
 * excluded) the column with the smallest clip(1 - <q_r, x_j>, 0, 2); ties -> lowest j.
 * Products are accumulated in float64.  q_rows_dev (optional) lists the query rows to process
 * (indices into q_unit_dev); outputs are indexed by position in that list.  */
int slic_nn_exact_top1(const void* q_unit_dev, const int32_t* q_rows_dev, int64_t nq,
                       const void* x_unit_dev, int64_t n, int32_t d, int32_t dtype,
                       int64_t self_offset, int32_t* idx_out_dev, void* dist_out_dev,
                       slic_stream_t stream);

/* ---- K1 tensor-core screen + exact re-rank ------------------------------------------------ */
/* The same first-neighbour search as slic_nn_exact_top1, done as a f16 tcgen05 GEMM with a
 * fused per-row candidate filter (scores never leave the SM) followed by an exact re-rank of
 * the surviving candidates in `dtype`.  eps is the screen's error allowance: every column whose
 * f16 score is within eps of the row's best is re-ranked (eps <= 0 selects the provable
 * default 2^-7 + 2^-11).  Rows whose candidate list overflowed are finished by the exact kernel, so the
 * result never depends on the screen's precision.  q_* may equal x_* (FINCH self-search). */
int slic_nn_top1(const void* q_unit_dev, const uint16_t* q_f16_dev, int64_t nq,
                 const void* x_unit_dev, const uint16_t* x_f16_dev, int64_t n,
                 int32_t d, int32_t d_pad, int32_t dtype, int64_t self_offset, float eps,
                 int32_t* idx_out_dev, void* dist_out_dev, int32_t* stats_out_dev /* [4] or NULL:
                 candidates re-ranked, rows finished by the exact kernel, list compactions, 0 */,
                 slic_stream_t stream);

/* Multi-GPU share of the level-0 self-search (clustering/finch.py:27-29 on N rows, spread over the GPUs of one box).
 * The score matrix of a self-search is symmetric: only the 256 x 256 tiles on or right of its diagonal are computed
 * and each is filtered along its rows and along its columns.  Process `part` of `parts` screens a contiguous
 * 1 / parts share (by tile count) of that triangle (plus a small pre-pass over all rows) and re-ranks its candidates exactly, so it holds, for EVERY row,
 * the best neighbour among the pairs it saw.  keys_out_dev [n + 1] (uint64):
 *   keys[i] = (float32 distance bits << 32) | neighbour index   (0x7fffffff7fffffff: no candidate seen for row i)
 *   keys[n] = 1, or 0 if this part's candidate log overflowed (its keys are then incomplete)
 * An element-wise MIN over the parts' arrays - one all-reduce over NCCL / NVLink - yields every row's first
 * neighbour with np.argmin's tie rule (smallest distance, then lowest index) and tells every process whether the
 * result is complete; slic_unpack_neighbor_keys splits it.  Needs n >= 16384 (SLIC_ERR_UNSUPPORTED below).
 *
 * The candidate filter of a row keeps what lies within eps of the best score seen for that row SO FAR; a part that sees
 * 1 / parts of the tiles alone learns those bests slowly and logs (and re-ranks) far too much.  Two-phase use:
 *   slic_sym_row_bests      part p screens its 1 / parts of the ROWS against 16 sampled column tiles and returns, for
 *                           those rows, the best screened score in a signed-comparable int32 form (INT32-lowest elsewhere);
 *   all-reduce MAX          of that [n] int32 array over the parts (4 n bytes);
 *   slic_nn_top1_sym_part   with row_bests_dev = the merged array: thresholds for ALL rows from the first tile on, no
 *                           pre-pass of its own.  row_bests_dev = NULL: single-phase (own pre-pass over all rows). */
int slic_sym_row_bests(const float* unit_dev, const uint16_t* unit_f16_dev, int64_t n, int32_t d, int32_t d_pad,
                       int32_t part, int32_t parts, int32_t* bests_out_dev, slic_stream_t stream);
int slic_nn_top1_sym_part(const float* unit_dev, const uint16_t* unit_f16_dev, int64_t n, int32_t d,
                          int32_t d_pad, int32_t part, int32_t parts, const int32_t* row_bests_dev, float eps,
                          uint64_t* keys_out_dev, int32_t* stats_out_dev /* [4] or NULL, as slic_nn_top1 */,
                          slic_stream_t stream);
/* keys [n] (merged) -> idx_out [n] int32, dist_out [n] float32; status_out_dev[0] = rows without a neighbour. */
int slic_unpack_neighbor_keys(const uint64_t* keys_dev, int64_t n, int32_t* idx_out_dev,
                              float* dist_out_dev, int32_t* status_out_dev, slic_stream_t stream);

/* Test hook, host only (no device work): the unit list the symmetric screen would execute for a self-search of n rows
 * as part `part` of `parts` - mode 0: pre-pass + triangle share, 1: row-bests pre-pass only, 2: triangle share only,
 * 3: fused (own rows' pre-pass + triangle share, the multi-GPU kernel); gated_chunks > 0: with upload gates
 * (slic_finch_host); col_tile: column-tile width of the kernel, 128 (A-resident kernels, d_pad <= 512) or 256.
 * units_out_host [capacity, 6] int32 (optional) receives per unit {row unit, first column tile, tile count, tile stride,
 * gate or -1, column-direction flag}; a unit covers the 256-row x col_tile-column tiles (row unit, first + k * stride),
 * k < count.  Lets a CPU test check that the parts tile the triangle exactly. */
int slic_debug_sym_plan(int64_t n, int32_t part, int32_t parts, int32_t mode, int32_t gated_chunks, int32_t col_tile,
                        int32_t* units_out_host, int64_t capacity, int64_t* num_units_out_host);

/* Debug / test hook: raw f16-screen scores of one 128 x 256 tile region, written as float
 * [nq, n] (small shapes only).  Lets the tests check the tcgen05 path element by element. */
int slic_screen_scores_debug(const uint16_t* q_f16_dev, int64_t nq, const uint16_t* x_f16_dev,
                             int64_t n, int32_t d_pad, float* out_dev, slic_stream_t stream);

/* ---- K1 dense / top-k (retrieval) ------------------------------------------------------- */
/* evaluate.py:208-223 (get_distance_matrix), iic_retrieve_clips.py:295: dense [nq, n] distance
 * matrix in `dtype`.  cosine: inputs are unit rows, out = clip(1 - s, 0, 2); euclidean: inputs
 * are raw rows, out = sqrt(max(|q|^2 + |x|^2 - 2 s, 0)) evaluated in float64 (as sklearn does).  same_matrix != 0
 * zeroes the diagonal exactly as sklearn does for Y is None. */
int slic_distance_matrix(const void* q_dev, int64_t nq, const void* x_dev, int64_t n,
                         int32_t d, int32_t dtype, int32_t metric, int32_t same_matrix,
                         void* out_dev, int64_t ld_out, slic_stream_t stream);

/* evaluate.py:226-231 (get_closest_data_mat), iic_retrieve_clips.py:296: the k smallest entries
 * of every row of a dense [nq, n] matrix, ascending (ties -> lowest column).  */
int slic_rows_topk(const void* dist_dev, int64_t nq, int64_t n, int64_t ld, int32_t dtype,
                   int32_t k, int32_t* idx_out_dev, void* val_out_dev, slic_stream_t stream);

/* Fused form of the two calls above (no [nq, n] matrix in HBM beyond one row block):
 * top-k cosine neighbours of unit query rows among unit database rows. */
int slic_topk_cosine(const void* q_unit_dev, int64_t nq, const void* x_unit_dev, int64_t n,
                     int32_t d, int32_t dtype, int32_t k, int64_t self_offset,
                     int32_t* idx_out_dev, void* dist_out_dev, slic_stream_t stream);

/* The same top-k search on the tensor cores: f16 tcgen05 screen with a fused per-row candidate
 * filter (a column survives iff its screened score is within eps of the row's running k-th best),
 * then exact evaluation in `dtype` and a (distance, column) sort of the survivors.  Results are
 * those of slic_topk_cosine (rows the screen cannot settle are finished by the exact kernels);
 * k <= 64.  stats_out_dev as in slic_nn_top1. */
int slic_topk_cosine_tc(const void* q_unit_dev, const uint16_t* q_f16_dev, int64_t nq,
                        const void* x_unit_dev, const uint16_t* x_f16_dev, int64_t n,
                        int32_t d, int32_t d_pad, int32_t dtype, int32_t k, int64_t self_offset,
                        float eps, int32_t* idx_out_dev, void* dist_out_dev,
                        int32_t* stats_out_dev, slic_stream_t stream);

/* evaluate.py:287-307 (get_topk_acc), iic_retrieve_clips.py:298-306: hits[m] = number of query
 * rows whose label occurs among the labels of their first ks[m] neighbours. */
int slic_hit_at_k(const int32_t* topk_idx_dev, int64_t nq, int32_t k_stride,
                  const int64_t* q_labels_dev, const int64_t* x_labels_dev,
                  const int32_t* ks_dev, int32_t num_ks, int32_t* hits_out_dev,
                  slic_stream_t stream);

/* ---- K2: first-neighbour graph components ------------------------------------------------- */
/* clustering/finch.py:40-47 + 50-55 (sparse (P+I)(P+I)^T, optional min_sim cut,
 * scipy connected_components(directed, weak)) on the nn[] array itself.
 * Labels are numbered by smallest member index, exactly as scipy numbers them.
 *   use_filter == 0: plain components of {i - nn[i]}.
 *   use_filter != 0: a link survives iff weight * distance <= min_sim, weight 2 for mutual first
 *     neighbours, 1 otherwise; rows sharing a first neighbour are linked iff their own distance
 *     <= min_sim (needs unit rows + dist_nn in `dtype`).
 * num_clust_out_dev receives the component count (device int32).  Entries of nn_dev outside [0, n) are
 * never followed; if there are any, num_clust_out_dev[0] comes back as MINUS their number (the
 * reference raises on such an index, finch.py:41-43). */
int slic_finch_components(const int32_t* nn_dev, int64_t n, int32_t use_filter, double min_sim,
                          const void* unit_dev, int32_t d, int32_t dtype, const void* dist_nn_dev,
                          int32_t* labels_out_dev, int32_t* num_clust_out_dev,
                          slic_stream_t stream);

/* clustering/finch.py:142-144: min_sim = max(orig_dist * adj) evaluated on the explicit link
 * list (direct links, weight 2 when mutual; sibling pairs, weight 1).  float32 result on device. */
int slic_finch_min_sim(const int32_t* nn_dev, int64_t n, const void* unit_dev, int32_t d,
                       int32_t dtype, const void* dist_nn_dev, float* min_sim_out_dev,
                       slic_stream_t stream);

/* clustering/finch.py:85-94 (update_adj, used by req_numclust): the linked pair (direct link or
 * sibling pair) with the smallest distance; pair_out_dev[0] < pair_out_dev[1]. */
int slic_finch_closest_link(const int32_t* nn_dev, int64_t n, const void* unit_dev, int32_t d,
                            int32_t dtype, const void* dist_nn_dev, int32_t* pair_out_dev,
                            slic_stream_t stream);

/* ---- K3: label composition + per-cluster means -------------------------------------------- */
/* clustering/finch.py:74-79 (get_merge): out[i] = u[prev[i]] (prev == NULL: out = u). */
int slic_compose_labels(const int32_t* prev_dev, const int32_t* u_dev, int64_t n,
                        int32_t* out_dev, slic_stream_t stream);

/* clustering/finch.py:58-71 (cool_mean): float64 mean of the float32 rows of every cluster,
 * labels dense 0..num_clust-1.  Deterministic: rows are summed in ascending index order. */
int slic_segmented_mean(const float* data_dev, const int32_t* labels_dev, int64_t n, int32_t d,
                        int32_t num_clust, double* out_dev, slic_stream_t stream);

/* The same reduction with the float64 SUMS and the row counts kept, so that the next FINCH level can be formed
 * from this one instead of from the N original rows: the clusters of level l+1 are unions of clusters of level l
 * (get_merge composes the labels, finch.py:74-79), hence sums_{l+1}[c] = sum of sums_l[p] over u[p] == c.
 * means_out_dev (optional) = sums / counts - the matrix cool_mean returns (finch.py:58-71). */
int slic_cluster_sums(const float* data_dev, const int32_t* labels_dev, int64_t n, int32_t d,
                      int32_t num_clust, double* sums_out_dev, int32_t* counts_out_dev,
                      double* means_out_dev, slic_stream_t stream);
/* labels_dev[p] in [0, num_clust) is the level-(l+1) cluster of level-l cluster p (the `u` of get_clust). */
int slic_merge_cluster_sums(const double* sums_prev_dev, const int32_t* counts_prev_dev,
                            const int32_t* labels_dev, int64_t n_prev, int32_t d, int32_t num_clust,
                            double* sums_out_dev, int32_t* counts_out_dev, double* means_out_dev,
                            slic_stream_t stream);

/* ---- K6: spherical k-means (clustering/cluster_masks.py fit_cluster, method='spherical_kmeans') ----------- */
/* spherecluster SphericalKMeans(...).fit(X) over scikit-learn 0.22 helpers; the algorithm is restated in
 * oracle/kmeans_oracle.py.  The random draws come from the caller, so that a binding reproduces any RNG's sequence.
 *
 * k-means++ seeding (_k_init) of the unit rows unit_dev [n, d] float32: first_id is the first seed, uniforms_host
 * [(k - 1) * L] the L draws of each later step in order (L = 2 + int(log(k)) in the reference, 1 <= L <= 32).  Every
 * step reads the rows once for all L candidates; sqdist(a, b) = max(|a|^2 + |b|^2 - 2 a.b, 0) in float64, rounded to
 * float32; potentials in float64, fixed order.  seeds_out_dev [k] int32 (row indices). */
int slic_kmeans_plusplus(const float* unit_dev, int64_t n, int32_t d, int32_t k, int64_t first_id,
                         const double* uniforms_host, int32_t L, int32_t* seeds_out_dev, slic_stream_t stream);
/* The whole fit of the raw rows x_dev [n, d] float32 (rows are L2-normalised first): n_init runs of seeding, Lloyd
 * (at most max_iter iterations, stop when the float64 centre shift <= mean(var(unit, axis=0)) * tol) and the final
 * E-step; the run with the smallest inertia is kept.  init_dev [k, d] float32 (optional, normalised before use; needs
 * n_init == 1) replaces the seeding; otherwise first_ids_host [n_init] and uniforms_host [n_init, (k - 1) * L] are
 * the draws of each run.  Outputs: labels_out_dev [n] int32, centers_out_dev [k, d] float32 (unit rows),
 * *inertia_out_host, *n_iter_out_host, stats_out_host [4] int64 (optional): candidates the screen re-ranked, rows
 * its exact finisher settled, candidate-list compactions, assignments run on the screen - summed over iterations.
 * Refuses n < k, k < 1, n_init < 1, max_iter < 1 with SLIC_ERR_INVALID_ARG before any device work.  Blocks until the
 * outputs are in place (one status read-back per few iterations). */
int slic_spherical_kmeans(const float* x_dev, int64_t n, int32_t d, int32_t k, const float* init_dev,
                          const int64_t* first_ids_host, const double* uniforms_host, int32_t L, int32_t n_init,
                          int32_t max_iter, double tol, int32_t* labels_out_dev, float* centers_out_dev,
                          double* inertia_out_host, int32_t* n_iter_out_host, int64_t* stats_out_host,
                          slic_stream_t stream);

/* ---- K4: label-equality masks and grouping ------------------------------------------------ */
/* models/infoNCE.py:281-283, loss/triplet_loss.py:136-142,254-261,291-297:
 * out[i, prepend + j] = (a[i] == b[j]) ^ negate as one byte per entry (torch.bool layout),
 * row stride nb + prepend; with prepend_ones the first column is 1 (the UberNCE self column). */
int slic_label_mask_u8(const int64_t* a_dev, int64_t na, const int64_t* b_dev, int64_t nb,
                       int32_t prepend_ones, int32_t negate, uint8_t* out_dev,
                       slic_stream_t stream);
/* Same mask, bit-packed: word w of row i holds columns 32w..32w+31 (bit j = column 32w + j),
 * row stride words_per_row = ceil(nb / 32) uint32. */
int slic_label_mask_bits(const int64_t* a_dev, int64_t na, const int64_t* b_dev, int64_t nb,
                         int32_t negate, uint32_t* out_dev, slic_stream_t stream);

/* online_train.py:648-652: cluster assignments back in the unshuffled order of the dataset,
 *   out[positions[i]] = values[i]  for i = 0..n-1 IN ORDER (a dataset index the sampler repeated keeps the LAST value),
 * slots nobody wrote = fill (the reference leaves None there).  out_of_range_dev[0] = positions outside [0, n_out). */
int slic_scatter_last_wins(const int32_t* values_dev, const int64_t* positions_dev, int64_t n,
                           int64_t n_out, int32_t fill, int32_t* out_dev, int32_t* out_of_range_dev,
                           slic_stream_t stream);

/* np.unique(labels, return_inverse=True) for int32 labels of any sign (sklearn's check_clusterings / contingency_matrix
 * behind online_train.py:634,640; datasets/triplets_dataset.py:99-104 for non-dense labels): dense_out[i] = rank of
 * labels[i] among the distinct values (ascending), uniq_out [capacity n, optional] = the distinct values,
 * num_out_dev[0] = how many.  Stable radix sort of (label, row), boundary flags, scan. */
int slic_dense_labels(const int32_t* labels_dev, int64_t n, int32_t* dense_out_dev, int32_t* uniq_out_dev,
                      int32_t* num_out_dev, slic_stream_t stream);

/* ---- cluster-quality scores (SURVEY.md 8f rank 3) ----------------------------------------- */
/* online_train.py:633-642 calls sklearn's normalized_mutual_info_score and adjusted_mutual_info_score on the true
 * labels and the FINCH labels.  This entry computes their ingredients on the device, following sklearn's arithmetic
 * (metrics/cluster/_supervised.py mutual_info_score + entropy, _expected_mutual_info_fast.pyx):
 *   out_dev[0] mutual information (nats)   [1] entropy of labels_true   [2] entropy of labels_pred
 *   out_dev[3] expected mutual information (0 unless want_emi)   [4], [5] number of non-empty classes / clusters
 * Labels must lie in [0, num_true) / [0, num_pred) (empty classes are allowed); a label outside is never counted
 * (no out-of-bounds write): all six outputs become NaN except out_dev[4] = -(number of such labels).
 * num_true * num_pred <= 2^28 cells (SLIC_ERR_UNSUPPORTED above).  The final ratios (and sklearn's special cases) are host arithmetic on these six numbers. */
int slic_cluster_metrics(const int32_t* labels_true_dev, const int32_t* labels_pred_dev, int64_t n,
                         int32_t num_true, int32_t num_pred, int32_t want_emi, double* out_dev,
                         slic_stream_t stream);

/* datasets/triplets_dataset.py:99-104 (label_to_indices) as CSR: order[] lists the rows of label
 * 0, then label 1, ... (ascending row index inside a label, what np.where yields);
 * offsets[c]..offsets[c+1] delimit label c.  Labels must lie in [0, num_labels). */
int slic_group_by_label(const int32_t* labels_dev, int64_t n, int32_t num_labels,
                        int32_t* order_out_dev, int32_t* offsets_out_dev, slic_stream_t stream);

/* ---- the whole hierarchy in one call ---------------------------------------------------------- */
/* clustering/finch.py:108-167 (FINCH without the req_clust refinement): level loop, exit rules
 * (:151-163), min_sim mode (:142-144, only when level 0 had dense distances), label composition
 * and float64 centroids, all on `stream`; the host reads one int per level.
 *   nn0_dev == NULL : level 0 is searched here (normalise + tcgen05 screen + exact re-rank, or the
 *                     exact kernel below 2048 rows); dense distances "exist" iff n <= 70 000 (:30).
 *   nn0_dev != NULL : level-0 first neighbours supplied - FINCH's initial_rank (dist0/unit0 NULL,
 *                     level0_dense 0) or an external search such as the row-sharded multi-GPU one
 *                     (dist0_dev [n] float32, unit0_dev [n, d] float32, level0_dense as above).
 * labels_out_dev: room for [n, capacity] int32; on return its first n * P entries are the [n, P]
 * C-contiguous matrix `c` of the reference (column l = partition l).  It may also be the device view
 * of page-locked host memory (cudaHostAlloc / a pinned torch tensor: the same address under unified
 * addressing): the matrix is then written over PCIe by the last kernel of the hierarchy and is on
 * the host when the call returns - no copy after the level count is known.  num_clust_out_host
 * [capacity], *num_levels_out_host = P.  SLIC_ERR_OVERFLOW if the hierarchy has more than
 * `capacity` levels. */
/* clustering/finch.py:19 (FLANN_THRESHOLD = 70000, a module constant): the row count above which the
 * reference holds no dense distances (no min_sim filter at that level).  Default 70000. */
int slic_set_flann_threshold(int64_t rows);

int slic_finch(const float* data_dev, int64_t n, int32_t d,
               const int32_t* nn0_dev, const float* dist0_dev, const float* unit0_dev,
               int32_t level0_dense, int32_t ensure_early_exit, int32_t capacity,
               int32_t* labels_out_dev, int32_t* num_clust_out_host, int32_t* num_levels_out_host,
               float* min_sim_out_host /* or NULL */, int32_t* has_min_sim_out_host /* or NULL */,
               slic_stream_t stream);

/* ---- host-buffer entry points (do their own H2D / D2H; block until the result is in place) -- */
/* clustering/finch.py:22-29 for a float32/float64 host matrix: first neighbour + distance. */
int slic_first_neighbors_host(const void* x_host, int64_t n, int32_t d, int32_t dtype,
                              int32_t* nn_out_host, void* dist_out_host);


/* FINCH(data, initial_rank, distance='cosine', ensure_early_exit) for a float32 host matrix
 * (numpy memory, pageable or pinned): the call a binding makes in place of clustering/finch.py:108.
 * The host -> device copy is cut into row chunks that are normalised as they land while the
 * level-0 tensor-core screen, launched first, consumes them (see csrc/finch_driver.cu), so the
 * PCIe transfer is hidden behind the O(N^2 D) stage.  initial_rank_host: NULL or [n] int64.
 * labels_out_host: room for [n, capacity] int32 (capacity <= 64); filled as [n, P] C-contiguous
 * (page-locked memory is written by the device directly, pageable memory through a device buffer
 * and a copy).  Blocks until the labels are in place. */
int slic_finch_host(const float* x_host, int64_t n, int32_t d, const int64_t* initial_rank_host,
                    int32_t ensure_early_exit, int32_t capacity, int32_t* labels_out_host,
                    int32_t* num_clust_out_host, int32_t* num_levels_out_host,
                    float* min_sim_out_host /* or NULL */, int32_t* has_min_sim_out_host /* or NULL */);

/* Host -> device copy on `stream` for callers that hold their device memory themselves: a pinned source goes straight to
 * cudaMemcpyAsync; a pageable one (a plain numpy array, what clustering/cluster_masks.py:80 produces) is staged in 32 MB
 * pieces through pinned buffers filled by 8 host threads, the DMA of one piece overlapping the staging of the next
 * (about 3x the rate of the driver's own single-threaded staging).  Returns once the last piece has been enqueued. */
int slic_copy_to_device(void* dst_dev, const void* src_host, int64_t bytes, slic_stream_t stream);

/* Upload / search overlap of slic_finch_host.  The pipelined path launches the persistent screen kernel BEFORE the
 * embeddings have arrived and needs the upload stream's small kernels to become resident next to it - true on an
 * otherwise idle B200, not promised by CUDA in general.  enable = 0: always upload first, then search (use this under
 * MPS / time slicing or when other work shares the device); 1: overlap whenever the resource check passes;
 * -1 (default): overlap unless the environment shows serialised launches (CUDA_LAUNCH_BLOCKING, compute-sanitizer,
 * Nsight tools) or SLIC_UPLOAD_OVERLAP=0.  A gate that stays shut for ~3 s makes the kernel give up without trapping;
 * the call then repeats the search after the upload (same result) and keeps the overlap off for the process. */
int slic_set_upload_overlap(int32_t enable);

/* ---- multi-GPU (one box, NVLink peer memory; csrc/comm.cu) ---------------------------------------------
 * The reference clusters on rank 0 only while the other DDP ranks wait at a barrier (online_train.py:619-627, 660-662).
 * Here the level-0 first-neighbour stage (clustering/finch.py:27-29) is shared by up to 8 GPUs of the box, every GPU
 * holding the full matrix; no collective library is on the data path - the ranks publish row bests into each other's
 * memory from inside the screen kernel and merge their (distance, neighbour) keys with one kernel reading peer memory. */
typedef struct slic_comm slic_comm_t;
#define SLIC_COMM_HANDLE_BYTES 64

/* (a) ONE PROCESS FOR ALL GPUS - the drop-in for the unmodified call site `c, num_clust, req_c = FINCH(data)` on rank 0:
 * slic_comm_create enables peer access among `devices` (device 0 of the list runs levels >= 1) and starts one worker
 * thread per device; max_rows bounds N of later calls (12 bytes of device memory per row and device).
 * slic_finch_multi = slic_finch_host on the group: every device uploads 1 / G of the rows and forwards them to its peers
 * over NVLink (copy engines), all devices share the level-0 search, labels come back from device 0.  Inputs the group
 * cannot share (initial_rank_host given, N < 16384, N > max_rows, one device) run on device 0 alone - same results.
 * slic_comm_last_timeline: ms_out_host[3] = {upload + forward, normalise + search, whole call} of the last call (CUDA
 * events on device 0). */
int slic_comm_create(const int32_t* devices, int32_t num_devices, int64_t max_rows, slic_comm_t** comm_out);
int slic_finch_multi(slic_comm_t* comm, const float* x_host, int64_t n, int32_t d, const int64_t* initial_rank_host,
                     int32_t ensure_early_exit, int32_t capacity, int32_t* labels_out_host,
                     int32_t* num_clust_out_host, int32_t* num_levels_out_host,
                     float* min_sim_out_host /* or NULL */, int32_t* has_min_sim_out_host /* or NULL */);
int slic_comm_last_timeline(slic_comm_t* comm, float* ms_out_host);
int slic_comm_destroy(slic_comm_t* comm);

/* (b) ONE PROCESS PER GPU (torch.distributed jobs): every rank creates its window on its current device and receives a
 * 64-byte CUDA IPC handle; the host side exchanges the handles (any transport) and every rank maps its peers' windows
 * with slic_comm_connect(all_handles = world x 64 bytes, in rank order).  slic_comm_nn_top1 is then called by EVERY rank
 * with the same normalised matrix (slic_normalize_rows: unit_dev [n, d] float32, f16_dev [n, d_pad]), n >= 16384: on
 * return (stream-ordered, no host synchronisation) idx_out_dev / dist_out_dev [n] hold the first neighbour and float32
 * cosine distance of every row - identical on every rank and to slic_nn_top1 on one GPU - and status_out_dev[2] =
 * {rows left without a neighbour, 1 if some rank's search was incomplete}; if either is non-zero the caller repeats the
 * search another way (degenerate inputs only). */
int slic_comm_window_create(int64_t max_rows, slic_comm_t** comm_out, void* ipc_handle_out /* 64 bytes */);
int slic_comm_connect(slic_comm_t* comm, int32_t rank, int32_t world, const void* all_handles);
int slic_comm_nn_top1(slic_comm_t* comm, const float* unit_dev, const uint16_t* f16_dev, int64_t n, int32_t d,
                      int32_t d_pad, int32_t* idx_out_dev, float* dist_out_dev, int32_t* status_out_dev,
                      slic_stream_t stream);

/* slic_finch on the group: the whole hierarchy of the device-resident [n, d] float32 matrix, called by EVERY rank with
 * the same matrix; level 0 through slic_comm_nn_top1's data path, everything after it replicated on every rank, one
 * host synchronisation at the end.  Outputs as slic_finch (labels_out_dev: [n, capacity] on this rank's device). */
int slic_comm_finch(slic_comm_t* comm, const float* data_dev, int64_t n, int32_t d, int32_t ensure_early_exit,
                    int32_t capacity, int32_t* labels_out_dev, int32_t* num_clust_out_host,
                    int32_t* num_levels_out_host, float* min_sim_out_host /* or NULL */,
                    int32_t* has_min_sim_out_host /* or NULL */, slic_stream_t stream);

/* Diagnostic timeline of slic_finch_host (CUDA events): enable, run a call, then read ms_out_host[4] =
 * {start -> first copy begins, upload duration, start -> level-0 search done, start -> labels copied back}. */
int slic_host_trace(int32_t enable, float* ms_out_host);

#ifdef __cplusplus
}
#endif
#endif /* SLIC_B200_H */
