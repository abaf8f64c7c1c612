/*
 * sqfa_b200 -- C ABI of the B200-native (sm_100a) SQFA hot paths.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types. Every pointer is a
 * DEVICE pointer unless the name ends in `_host`. Every function enqueues work on `stream`
 * (a cudaStream_t passed as void*; NULL = legacy default stream), never synchronises, never
 * allocates or frees device memory (callers pass workspaces sized by the *_workspace_bytes
 * queries) and returns 0 on success, a positive cudaError_t value on a CUDA failure or a negative
 * SQFA_E_* code on invalid arguments. `sqfa_last_error()` returns a human-readable message for
 * the last failure on the calling thread.
 *
 * Reference interfaces replaced (paths under /root/reference/src/sqfa/):
 *   HP1  statistics.py:8-54   class_statistics      -> sqfa_label_max, sqfa_bucket_labels,
 *        statistics.py:97-124 sample_covariance        sqfa_class_sums, sqfa_class_means,
 *        statistics.py:57-94  oas_covariance           sqfa_class_gram, sqfa_stats_epilogue
 *                                                  (all of them in one call: sqfa_class_statistics)
 *   HP2  linalg.py:19-45      conjugate_matrix      -> sqfa_project_fwd / sqfa_project_bwd
 *        model.py:172-237     transform_scatters / transform -> sqfa_project_fwd / sqfa_transform
 *        linalg.py:48-70      generalized_eigenvalues  \
 *        distances.py:46-237  affine_invariant(_sq), fisher_rao_lower_bound(_sq),
 *                             log_euclidean(_sq)        > sqfa_class_factor + sqfa_pair_distances
 *        _optim.py:16-30,90-96 closure loss + guard + autograd backward /
 */
#ifndef SQFA_B200_H_
#define SQFA_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* sqfa_stream_t; /* cudaStream_t */

#define SQFA_E_INVALID (-1)     /* bad argument (null pointer, negative size, unsupported shape) */
#define SQFA_E_WORKSPACE (-2)   /* workspace too small */
#define SQFA_E_UNSUPPORTED (-3) /* e.g. matrix size m > SQFA_MAX_M */

#define SQFA_MAX_M 64 /* largest SPD matrix the pair kernels accept (k+1 for Fisher-Rao) */

/* estimator argument of sqfa_stats_epilogue (reference: estimator="empirical" | "oas") */
#define SQFA_EST_EMPIRICAL 0
#define SQFA_EST_OAS 1
#define SQFA_EST_PACKED_GRAM 16 /* OR-ed in: the gram argument is the packed upper-tile list (below) */
#define SQFA_EST_CENTRED_SUMS 32 /* OR-ed in (sqfa_stats_epilogue): the shift argument holds the class sums of
                                    (x - s) for the s the Gram was centred on, and d = sums / n_c */

/* `accumulate` argument of sqfa_class_gram: a bit set */
#define SQFA_GRAM_ACCUMULATE 1 /* add to the existing content (streaming / chunked input) */
#define SQFA_GRAM_PACKED 2     /* write the packed list of upper tiles instead of (C, D, D) */

/* distance selector of the pair kernels */
#define SQFA_DIST_AFFINE_INVARIANT 0 /* distances.py:70-89  sqrt(sum log^2 lambda + 1e-6)      */
#define SQFA_DIST_FISHER_RAO_LB 1    /* distances.py:210-237 sqrt(AI^2(E_i,E_j)/2 + 1e-6)       */
#define SQFA_DIST_LOG_EUCLIDEAN 2    /* distances.py:119-138 sqrt(|logA - logB|_F^2 + 1e-6)     */
/* Bures-Wasserstein between SPD matrices (an extension, not reference API):
 *   d^2 = tr A + tr B - 2 tr((B^1/2 A B^1/2)^1/2), clamped at 0; sqrt(d^2 + 1e-6). m <= 34, else SQFA_E_UNSUPPORTED;
 *   no eig_out. */
#define SQFA_DIST_BURES_WASSERSTEIN 3
/* 2-Wasserstein between Gaussians: |mu_A - mu_B|^2 + Bures-Wasserstein^2 of the covariances. Closures only
 * (sqfa_fused_loss, sqfa_fused_loss_sharded, sqfa_closure_eval; M required, m = n_filters): sqfa_class_factor
 * and sqfa_pair_distances take no means and reject it. */
#define SQFA_DIST_WASSERSTEIN_GAUSSIAN 4
/* Distances between Gaussians under the mean covariance M = (Sigma_i + Sigma_j) / 2 of the pair, d = mu_i - mu_j,
 * x = d^T M^-1 d (distances.py:240-393). Closures only (sqfa_fused_loss, sqfa_fused_loss_sharded,
 * sqfa_closure_eval; M required, n_filters <= 32); the per-matrix entry points reject them, and
 * sqfa_gauss_pair_distances evaluates these distances pair by pair.
 *   SQFA_DIST_MAHALANOBIS    sqrt(x + 1e-6), or x with SQFA_DIST_SQUARED
 *   SQFA_DIST_BHATTACHARYYA  B = x / 8 + (logdet M - (logdet Sigma_i + logdet Sigma_j) / 2) / 2
 *   SQFA_DIST_HELLINGER      sqrt(1 - exp(-B) + 1e-6), no clamp
 * SQFA_DIST_SQUARED with Bhattacharyya or Hellinger is rejected. */
#define SQFA_DIST_MAHALANOBIS 5
#define SQFA_DIST_BHATTACHARYYA 6
#define SQFA_DIST_HELLINGER 7
/* add SQFA_DIST_SQUARED to get the squared variants (no sqrt, no epsilon) */
#define SQFA_DIST_SQUARED 16

int sqfa_version(void);
/* hash of the sources the library was built from (sqfa_b200/build.py); loaders compare it with the
 * sources they ship with and refuse a stale build */
const char* sqfa_build_id(void);
const char* sqfa_last_error(void);
/* number of SMs of the current device (grid sizing); <= 0 on failure */
int sqfa_device_sm_count(void);

/* ---------------------------------------------------------------------------------------------
 * HP1: class_statistics (statistics.py:8-54)
 * ------------------------------------------------------------------------------------------- */

/* max(labels) -> *out_max (int64; -1 when n == 0 or all labels negative).
 * Reference: `n_classes = int(torch.max(labels) + 1)` statistics.py:29.
 * out_max may be device memory or MAPPED PINNED HOST memory: the kernel stores the result there
 * itself, so the host can wait on an event recorded behind the call and read the value without a
 * device-to-host copy (which would queue behind bulk transfers of other streams on the copy engine). */
int sqfa_label_max(const int64_t* labels, int64_t n, int64_t* out_max, sqfa_stream_t stream);

/* Stable bucketing of rows by label (statistics.py:37, `(labels == i).nonzero()` for every i).
 *   perm    [n]     row ids sorted by class, ascending inside a class (== stable argsort);
 *                   rows with label outside [0, n_classes) come last (bucket n_classes)
 *   offsets [C+2]   offsets[c] = start of class c in perm, offsets[C] = start of dropped rows,
 *                   offsets[C+1] = n
 *   counts  [C+1]   class sizes, counts[C] = dropped rows
 * n must be < 2^31. */
size_t sqfa_bucket_workspace_bytes(int64_t n, int32_t n_classes);
int sqfa_bucket_labels(const int64_t* labels, int64_t n, int32_t n_classes, int64_t* counts, int64_t* offsets,
                       int32_t* perm, void* ws, size_t ws_bytes, sqfa_stream_t stream);

/* Per-class column sums  sums[c][j] (+)= sum_{i in c} (X[i][j] - shift[c][j])   (shift may be NULL).
 * X is row-major with row stride ldx (floats). ws: sqfa_class_sums_workspace_bytes. */
size_t sqfa_class_sums_workspace_bytes(int64_t n, int32_t n_dim, int32_t n_classes);
int sqfa_class_sums(const float* X, int64_t ldx, const int32_t* perm, const int64_t* offsets, const float* shift,
                    int64_t n, int32_t n_dim, int32_t n_classes, float* sums, int accumulate, void* ws,
                    size_t ws_bytes, sqfa_stream_t stream);

/* means[c][j] = sums[c][j] / counts[c] (+ shift[c][j])   (statistics.py:40; 0/0 = NaN when empty) */
int sqfa_class_means(const float* sums, const int64_t* counts, const float* shift, int32_t n_dim,
                     int32_t n_classes, float* means, sqfa_stream_t stream);

/* Segmented Gram on the tensor cores (tcgen05, 3xTF32):
 *   gram[c] (+)= sum_{i in c} (x_i - shift_c)(x_i - shift_c)^T        (statistics.py:119-120)
 * Only the upper triangle of every gram[c] (D x D, row-major) is defined on return.
 *   accumulate 0: gram is overwritten (zeroed, then summed); SQFA_GRAM_ACCUMULATE: added to the
 *              existing content (streaming / chunked input). SQFA_GRAM_PACKED: gram is not
 *              (C, D, D) but the list of the 256 x 256 tiles that intersect the upper triangle,
 *              [class][tile (tm <= tn, row-major over the upper triangle)][256][256] floats,
 *              sqfa_gram_packed_floats(n_dim, n_classes) in total -- the buffer a multi-device
 *              caller all-reduces (54 % of C D^2 at D = 3072); sqfa_stats_epilogue reads it with
 *              SQFA_EST_PACKED_GRAM. Entries of edge tiles beyond D are never written or read.
 *   chain_rows samples per tensor-core accumulation chain (0 = default 512). Every chain starts
 *              from a zero accumulator and is added to gram with fp32 red.global.add, which bounds
 *              the accumulator truncation bias of the tensor core (see DESIGN.md).
 *   n          number of rows of X (sizes the K split of small problems; no rows beyond the
 *              class offsets are read)
 *   done, n_groups, reserve_sms
 *              overlap of a multi-device caller's collective with this kernel: with done != NULL
 *              (int32 [n_groups], zeroed by the caller) the jobs run in class order, classes are
 *              split into n_groups contiguous groups (class c belongs to group c n_groups / n_classes;
 *              groups may be empty when n_groups > n_classes)
 *              and done[g] is incremented once per (job, CTA, epilogue warp) after the job's tile has
 *              been stored and fenced; when done[g] reaches sqfa_class_gram_group_signals(..., g)
 *              all tiles of group g are final, so a stream memory operation (cuStreamWaitValue32)
 *              on ANOTHER stream can release the all-reduce of that group's slice of gram while this
 *              kernel still computes the next groups. reserve_sms SMs are left out of the grid for
 *              that collective's kernels. done == NULL: largest class first, all SMs.
 *   first_class
 *              with done != NULL the class order starts at this class and wraps around
 *              (first_class, ..., C - 1, 0, ..., first_class - 1): a rank that pushes every finished
 *              group to the group's owner (sqfa_peer_push) runs the classes it owns itself LAST, so
 *              its last transfer hides behind its own remaining work and the ranks' transfers are
 *              staggered over different peers. 0 otherwise.
 *   ws         sqfa_class_gram_workspace_bytes(n, n_dim, n_classes) bytes (device-side job plan). */
size_t sqfa_class_gram_workspace_bytes(int64_t n, int32_t n_dim, int32_t n_classes);
size_t sqfa_gram_packed_floats(int32_t n_dim, int32_t n_classes);
/* rows x columns of tensor-core accumulator the kernel executes per sample and class for this n_dim
 * (every upper tile is a full MMA tile): executed TF32 flop of a launch = 3 * 2 * n * this. */
int64_t sqfa_gram_executed_tile_area(int32_t n_dim);
int sqfa_class_gram(const float* X, int64_t ldx, const int32_t* perm, const int64_t* offsets, const float* shift,
                    int64_t n, int32_t n_dim, int32_t n_classes, float* gram, int accumulate, int chain_rows,
                    int32_t* done, int32_t n_groups, int32_t first_class, int32_t reserve_sms, void* ws,
                    size_t ws_bytes, sqfa_stream_t stream);
int64_t sqfa_class_gram_group_signals(int64_t n, int32_t n_dim, int32_t n_classes, int32_t n_groups, int32_t group);
/* Enqueue on `stream` a wait until *flag >= value (device memory; cuStreamWaitValue32): what gates a
 * collective on the counters above. No kernel is launched, no SM is occupied while waiting. */
int sqfa_stream_wait_geq(sqfa_stream_t stream, const int32_t* flag, int32_t value);

/* One-pass class means (the single-device sqfa_class_statistics runs these steps):
 *   sqfa_class_pilot_shift      shift[c][j] = mean of the first min(n_c, 32) rows of class c in bucket order
 *                               (0 for an empty class); rows added in a fixed order
 *   sqfa_class_gram_sums        sqfa_class_gram (shift, accumulate 0, no completion counters) whose
 *                               diagonal tiles also write class-sum partials of (x - shift) into
 *                               partials[n_classes][nsplit][n_dim], nsplit = sqfa_class_gram_sum_splits(...);
 *                               X is read once for both. The partials are zeroed by the call.
 *                               nsplit = 0: the Gram would be split into more than 16 K parts (classes of
 *                               ~10^5 rows); sqfa_class_gram_sums returns SQFA_E_UNSUPPORTED and
 *                               sqfa_class_statistics takes the two passes (sums, means, Gram on the means).
 *   sqfa_class_means_from_partials
 *                               sums[c][j] = sum over the nsplit partials (float64, in order), then
 *                               means[c][j] = sums[c][j] / counts[c] + shift[c][j]   (NaN when empty)
 * followed by sqfa_stats_epilogue(shift = sums, estimator | SQFA_EST_CENTRED_SUMS). The Gram needs a shift
 * close to the class mean, not the mean itself: the epilogue takes n d d^T (d = sums / n) off it. */
int32_t sqfa_class_gram_sum_splits(int64_t n, int32_t n_dim, int32_t n_classes);
int sqfa_class_pilot_shift(const float* X, int64_t ldx, const int32_t* perm, const int64_t* offsets, int32_t n_dim,
                           int32_t n_classes, float* shift, sqfa_stream_t stream);
int sqfa_class_gram_sums(const float* X, int64_t ldx, const int32_t* perm, const int64_t* offsets, const float* shift,
                         int64_t n, int32_t n_dim, int32_t n_classes, float* gram, float* partials, void* ws,
                         size_t ws_bytes, sqfa_stream_t stream);
int sqfa_class_means_from_partials(const float* partials, int32_t nsplit, const int64_t* counts, const float* shift,
                                   int32_t n_dim, int32_t n_classes, float* sums, float* means,
                                   sqfa_stream_t stream);

/* Class counts as two exact float32 words, out[c] = counts[c] / 2^20 and out[n_classes + c] = counts[c] mod
 * 2^20, so that a multi-device caller sums [class sums | counts] of its ranks in ONE float32 all-reduce;
 * sqfa_counts_unpack turns the summed words back into int64 (exact below 2^44 rows). */
int sqfa_counts_pack(const int64_t* counts, int32_t n_classes, float* out, sqfa_stream_t stream);
int sqfa_counts_unpack(const float* in, int32_t n_classes, int64_t* counts, sqfa_stream_t stream);

/* Statistics epilogue (statistics.py:43-47, 84-93, 116, 120-122):
 *   cov[c] = (gram[c] - n_c d d^T) / (n_c - ddof),  d = means[c] - shift[c]  (shift NULL -> d = 0)
 *   ddof = 1: unbiased estimate; ddof = 0: `assume_centered` (statistics.py:116)
 *   estimator == SQFA_EST_OAS applies the OAS shrinkage to cov
 *   sm[c]  = cov[c] + means[c] means[c]^T       (sm may be NULL)
 * Reads the upper triangle of gram, writes full symmetric cov and sm; cov may alias gram unless
 * gram is packed (estimator | SQFA_EST_PACKED_GRAM). */
size_t sqfa_stats_epilogue_workspace_bytes(int32_t n_classes);
int sqfa_stats_epilogue(const float* gram, const float* means, const float* shift, const int64_t* counts,
                        int32_t n_dim, int32_t n_classes, int estimator, int ddof, float* cov, float* sm, void* ws,
                        size_t ws_bytes, sqfa_stream_t stream);

/* Reduce-scatter of the Gram partials by class, fused into the producer and the consumer instead of a
 * collective kernel (SURVEY.md 8(e) row 1, "ReduceScatter by class"): every rank computes the packed
 * partial Gram of ALL classes from its rows (sqfa_class_gram with completion counters); as soon as the
 * classes owned by rank g are final, the copy engine pushes that slice into slot [source rank] of rank
 * g's receive buffer (peer-mapped memory; sqfa_peer_push behind sqfa_stream_wait_geq on a side stream:
 * no SM is used, the tensor cores keep working on the next group); after one barrier each rank runs
 *   sqfa_stats_epilogue_reduce: cov[c] = (sum_s partial_s[c] - n_c d d^T) / (n_c - ddof), ...
 * over ITS classes only, reading source s from `peer_slots + s * slot_stride` (s != self) or from its own
 * packed buffer `gram` (s == self), summed in ascending s (bit-reproducible). All buffers hold the
 * packed tile layout of SQFA_GRAM_PACKED for `n_classes` (the classes this rank owns). */
int sqfa_stats_epilogue_reduce(const float* gram, const float* peer_slots, int64_t slot_stride, int32_t n_sources,
                               int32_t self, const float* means, const float* shift, const int64_t* counts,
                               int32_t n_dim, int32_t n_classes, int estimator, int ddof, float* cov, float* sm,
                               void* ws, size_t ws_bytes, sqfa_stream_t stream);
/* cudaMemcpyAsync(dst, src, bytes) on `stream` (copy engine; dst may be peer-mapped device memory). */
int sqfa_peer_push(void* dst, const void* src, size_t bytes, sqfa_stream_t stream);

/* class_statistics in ONE call (statistics.py:8-54) for n rows resident on one device, in one pass over X
 * (two where sqfa_class_gram_sum_splits is 0, see above):
 * bucket the labels, pilot shift, Gram of the rows centred by it with the class sums on the side, means,
 * epilogue. It is exactly the sequence sqfa_bucket_labels -> sqfa_class_pilot_shift -> sqfa_class_gram_sums
 * -> sqfa_class_means_from_partials -> sqfa_stats_epilogue (shift = the pilot shift) enqueued on `stream`
 * from one host call (no host round trips between the steps); multi-device callers use the two-pass entry
 * points (sqfa_class_sums, sqfa_class_gram) and all-reduce the partial sums between them.
 *   means   (n_classes, n_dim)          out
 *   cov     (n_classes, n_dim, n_dim)   out (the Gram is accumulated here, then finalised in place)
 *   sm      (n_classes, n_dim, n_dim)   out, may be NULL
 *   counts [n_classes + 1], offsets [n_classes + 2], perm [n]   out, as in sqfa_bucket_labels */
size_t sqfa_class_statistics_workspace_bytes(int64_t n, int32_t n_dim, int32_t n_classes);
int sqfa_class_statistics(const float* X, int64_t ldx, const int64_t* labels, int64_t n, int32_t n_dim,
                          int32_t n_classes, int estimator, int ddof, float* means, float* cov, float* sm,
                          int64_t* counts, int64_t* offsets, int32_t* perm, void* ws, size_t ws_bytes,
                          sqfa_stream_t stream);

/* bfloat16 / float16 points (`elem` = SQFA_ELEM_BF16 or SQFA_ELEM_F16; any other code returns
 * SQFA_E_INVALID with sqfa_last_error set, and the workspace / signal queries return 0). Same contracts as
 * the float32 entry points they are named after; only X changes: `const void*` with row stride ldx in
 * ELEMENTS. Every element is widened to float32 as it is loaded and the kernels then do exactly what they
 * do for float32 points (same centring, tf32 hi/lo split, MMA order and epilogue): sums, means, counts,
 * Grams, covariances and Z are float32, and
 *   - sqfa_class_sums_h, sqfa_class_statistics_h (means, epilogue), and sqfa_class_gram_h wherever the
 *     float32 Gram runs without a K split, give the SAME BITS as the float32 entry points on a contiguous
 *     float32 copy of X;
 *   - elsewhere (K-split Grams, whose parts are summed with red.add in arrival order; transform) the
 *     results agree with that copy's to float32 rounding.
 * Rows aligned to 4 elements (8 bytes) are read with one 8-byte load per 4 columns, other rows element by
 * element. The Gram's K-split rule counts the bytes of a class's rows (2 per element), so the workspace
 * and completion-signal queries take `elem` too; everything else (label bucketing, sqfa_class_means,
 * sqfa_stats_epilogue, counts, peer pushes) is dtype-free and shared. */
#define SQFA_ELEM_BF16 1
#define SQFA_ELEM_F16 2
int sqfa_class_sums_h(const void* X, int64_t ldx, int32_t elem, const int32_t* perm, const int64_t* offsets,
                      const float* shift, int64_t n, int32_t n_dim, int32_t n_classes, float* sums, int accumulate,
                      void* ws, size_t ws_bytes, sqfa_stream_t stream);
size_t sqfa_class_gram_workspace_bytes_h(int64_t n, int32_t n_dim, int32_t n_classes, int32_t elem);
int sqfa_class_gram_h(const void* X, int64_t ldx, int32_t elem, const int32_t* perm, const int64_t* offsets,
                      const float* shift, int64_t n, int32_t n_dim, int32_t n_classes, float* gram, int accumulate,
                      int chain_rows, int32_t* done, int32_t n_groups, int32_t first_class, int32_t reserve_sms,
                      void* ws, size_t ws_bytes, sqfa_stream_t stream);
int64_t sqfa_class_gram_group_signals_h(int64_t n, int32_t n_dim, int32_t n_classes, int32_t n_groups, int32_t group,
                                        int32_t elem);
size_t sqfa_class_statistics_workspace_bytes_h(int64_t n, int32_t n_dim, int32_t n_classes, int32_t elem);
int32_t sqfa_class_gram_sum_splits_h(int64_t n, int32_t n_dim, int32_t n_classes, int32_t elem);
int sqfa_class_pilot_shift_h(const void* X, int64_t ldx, int32_t elem, const int32_t* perm, const int64_t* offsets,
                             int32_t n_dim, int32_t n_classes, float* shift, sqfa_stream_t stream);
int sqfa_class_gram_sums_h(const void* X, int64_t ldx, int32_t elem, const int32_t* perm, const int64_t* offsets,
                           const float* shift, int64_t n, int32_t n_dim, int32_t n_classes, float* gram,
                           float* partials, void* ws, size_t ws_bytes, sqfa_stream_t stream);
int sqfa_class_statistics_h(const void* X, int64_t ldx, int32_t elem, const int64_t* labels, int64_t n, int32_t n_dim,
                            int32_t n_classes, int estimator, int ddof, float* means, float* cov, float* sm,
                            int64_t* counts, int64_t* offsets, int32_t* perm, void* ws, size_t ws_bytes,
                            sqfa_stream_t stream);
/* Z = X F^T with bf16 / fp16 X and float32 F, Z (sqfa_transform; X staged in shared memory as it is) */
int sqfa_transform_h(const void* X, int64_t ldx, int32_t elem, const float* F, int64_t n, int32_t n_dim,
                     int32_t n_filters, float* Z, sqfa_stream_t stream);

/* float64 variants (the reference follows the dtype of `points`, statistics.py:28,32-34, and runs its
 * test-suite in float64): same contracts as the float32 entry points above, label bucketing is shared.
 * FP64 pipe (DFMA), 64 x 64 upper tiles, every reduction in a fixed order (bit-reproducible); no
 * workspace. gram is (C, D, D) with the upper triangle defined; cov must not alias gram. */
int sqfa_class_sums_f64(const double* X, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                        const double* shift, int64_t n, int32_t n_dim, int32_t n_classes, double* sums,
                        int accumulate, sqfa_stream_t stream);
int sqfa_class_means_f64(const double* sums, const int64_t* counts, const double* shift, int32_t n_dim,
                         int32_t n_classes, double* means, sqfa_stream_t stream);
int sqfa_class_gram_f64(const double* X, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                        const double* shift, int64_t n, int32_t n_dim, int32_t n_classes, double* gram,
                        int accumulate, sqfa_stream_t stream);
int sqfa_stats_epilogue_f64(const double* gram, const double* means, const double* shift, const int64_t* counts,
                            int32_t n_dim, int32_t n_classes, int estimator, int ddof, double* cov, double* sm,
                            sqfa_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * HP2: the per-iteration loss and its backward (model.py:190-220, 508-546; _optim.py:90-96)
 * ------------------------------------------------------------------------------------------- */

/* Projection  T[c] = F S[c]  (k x D),  Psi[c] = T[c] F^T (k x k),  mu'[c] = F m[c]  (k)
 * -- conjugate_matrix(S, F) linalg.py:41 and transform(means) model.py:236 in one pass over S.
 *   S [C][D][D] symmetric, M [C][D] or NULL, F [k][D], k <= 32
 *   T [C][k][D] saved for the backward, Psi [C][k][k], Mu [C][k] (only if M != NULL)
 *   ws: sqfa_project_workspace_bytes (shared by fwd and bwd) */
size_t sqfa_project_workspace_bytes(int32_t n_classes, int32_t n_dim, int32_t n_filters);
int sqfa_project_fwd(const float* S, const float* M, const float* F, int32_t n_classes, int32_t n_dim,
                     int32_t n_filters, float* T, float* Psi, float* Mu, void* ws, size_t ws_bytes,
                     sqfa_stream_t stream);

/* dF = sum_c ( (gPsi[c] + gPsi[c]^T) T[c] + gMu[c] m[c]^T )   (gMu and M may both be NULL):
 * analytic adjoint of sqfa_project_fwd w.r.t. F, replaces autograd through linalg.py:41 */
int sqfa_project_bwd(const float* gPsi, const float* gMu, const float* T, const float* M, int32_t n_classes,
                     int32_t n_dim, int32_t n_filters, float* dF, void* ws, size_t ws_bytes,
                     sqfa_stream_t stream);

/* Z = X F^T  (model.py:236, transform): X [n][D] row stride ldx, F [k][D], Z [n][k] */
int sqfa_transform(const float* X, int64_t ldx, const float* F, int64_t n, int32_t n_dim, int32_t n_filters,
                   float* Z, sqfa_stream_t stream);

/* Embedding (model.py:216-217 / 537-538 noise, distances.py:162-174 _embed_gaussian):
 *   dist AI / LE : E[c] = Psi[c] + noise I                              (m = k,  Mu unused)
 *   dist FR      : E[c] = [[Psi[c] + noise I + mu mu^T, mu],[mu^T, 1]]  (m = k + 1)
 * and its adjoint  (gPsi, gMu) <- gE  (gMu written only for FR). */
int sqfa_embed_fwd(const float* Psi, const float* Mu, float noise, int32_t n_classes, int32_t n_filters,
                   int32_t dist, float* E, sqfa_stream_t stream);
int sqfa_embed_bwd(const float* gE, const float* Mu, int32_t n_classes, int32_t n_filters, int32_t dist,
                   float* gPsi, float* gMu, sqfa_stream_t stream);

/* Per-class factorisation of the m x m SPD matrices E[c] (m <= SQFA_MAX_M), one warp per class:
 *   AI / FR: W[c] = [L | L^-1]  (Cholesky E = L L^T), 2 m^2 floats per class
 *   LE     : W[c] = [V | lambda | log lambda | logE] (2 m^2 + 2 m floats), one-sided Jacobi
 * Replaces spd_inv_sqrt (linalg.py:144-162) / spd_log (linalg.py:165-183). flag[0] is set to 1
 * if any matrix is not positive definite / has non-finite entries (0 otherwise). */
size_t sqfa_class_factor_floats(int32_t m, int32_t dist);
int sqfa_class_factor(const float* E, int32_t n_classes, int32_t m, int32_t dist, float* W, int32_t* flag,
                      sqfa_stream_t stream);

/* Pairwise distances d(A_a, B_b), one warp per pair (one-sided Jacobi on L_b^-1 L_a; replaces
 * generalized_eigenvalues linalg.py:48-70 + distances.py:46-237).
 *   Wa, Wb     outputs of sqfa_class_factor (same dist) for the n_a / n_b matrices
 *   triangular 1: self distances (n_a == n_b, Wa == Wb): only the strict lower triangle is
 *              evaluated, pairs p = i (i - 1) / 2 + j (i > j) for p in [pair_begin, pair_end);
 *              d(i,j) is written to (i,j) and (j,i) and the diagonal is set to d(i,i)
 *              (sqrt(1e-6), or 0 for the squared variants). The reference evaluates all C*C pairs
 *              and reads the lower triangle (_optim.py:94).
 *              0: all n_a * n_b pairs, p = a * n_b + b.
 *   dist_out   [n_a][n_b] or NULL
 *   loss       [2] or NULL: += { sum_p d_p , number of non-finite d_p }  (_optim.py:94, guard :16-30)
 *   gEa, gEb   [n][m][m] or both NULL: += w_p * d(d_p)/dE, w_p = weight * (gD ? gD[a][b] (+ gD[b][a]
 *              when triangular) : 1). For LE these are gradients w.r.t. the matrix logarithms
 *              (feed them to sqfa_class_factor_bwd). gEa == gEb is allowed.
 *   eig_out    [n_a][n_b][m] or NULL (AI / FR, triangular == 0 only): the generalized eigenvalues
 *              of (A_a, B_b) in descending order (generalized_eigenvalues, linalg.py:48-70)
 *   ws         needed when loss or gEa is given: sqfa_pair_distances_workspace_bytes(...) bytes,
 *              16-byte aligned. Sums are DETERMINISTIC: every warp stores the partial loss / gradient
 *              of its tile of pairs there and a second kernel adds them per class in a fixed order
 *              (no floating-point atomics), so results are bit-identical from run to run. */
size_t sqfa_pair_distances_workspace_bytes(int32_t n_a, int32_t n_b, int32_t m, int32_t dist, int32_t triangular,
                                           int64_t pair_begin, int64_t pair_end);
int sqfa_pair_distances(const float* Wa, const float* Wb, int32_t n_a, int32_t n_b, int32_t m, int32_t dist,
                        int32_t triangular, int64_t pair_begin, int64_t pair_end, float weight, const float* gD,
                        float* dist_out, float* loss, float* gEa, float* gEb, float* eig_out, void* ws,
                        size_t ws_bytes, sqfa_stream_t stream);

/* LE only: gE[c] += adjoint of logE = V log(Lambda) V^T applied to gLog[c] (Daleckii-Krein).
 * No-op for AI / FR, whose gradients sqfa_pair_distances accumulates directly on E. */
int sqfa_class_factor_bwd(const float* W, const float* gLog, int32_t n_classes, int32_t m, int32_t dist,
                          float* gE, sqfa_stream_t stream);

/* The whole closure body of the fitting loop (_optim.py:90-96) in one call, at fixed filters F:
 *   out[0] = -mean_{i>j} d(E_i, E_j) over pairs [pair_begin, pair_end) (scaled by 1/P of ALL pairs,
 *            so partial results of a sharded pair list add up), out[1] = # non-finite distances,
 *   out[2] = max |dF|,
 *   dF     = d out[0] / dF   (k x D),
 * with E_c = F S_c F^T + noise I (AI, LE) or its Calvo-Oller embedding with mu'_c = F m_c (FR).
 * Eight kernels on `stream` inside `ws` (16-byte aligned, sqfa_fused_loss_workspace_bytes for the same
 * pair range): projection (stream + finish), per-class embedding + factorisation, pair kernel,
 * per-class gradient reduction + embedding adjoint, projection adjoint. Deterministic. */
size_t sqfa_fused_loss_workspace_bytes(int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                                       int64_t pair_begin, int64_t pair_end);
int sqfa_fused_loss(const float* S, const float* M, const float* F, int32_t n_classes, int32_t n_dim,
                    int32_t n_filters, float noise, int32_t dist, int64_t pair_begin, int64_t pair_end, float* out,
                    float* dF, void* ws, size_t ws_bytes, sqfa_stream_t stream);

/* sqfa_fused_loss with the CLASSES and the PAIRS sharded over the ranks of a multi-device caller (AI and
 * FR; S, M hold all classes on every rank, a rank reads only its own), in three phases on the SAME
 * workspace with one small all-reduce (the caller's) after each of the first two:
 *   phase 0: projection of classes [class_begin, class_end): T_c and their slices of exchange span 0 =
 *            [per-chunk partials of Psi | of mu'] (zero elsewhere)          -> all-reduce span 0 (sum)
 *   phase 1: embedding + factorisation of all classes, pair kernel on [pair_begin, pair_end), per-class
 *            reduction and embedding adjoint: partial (gPsi, gMu) of all classes and
 *            {weight * sum d, #non-finite} in exchange span 1               -> all-reduce span 1 (sum)
 *   phase 2: projection adjoint over classes [class_begin, class_end) -> dF (k x D), the caller's share of
 *            d loss / dF                                                     -> all-reduce dF (sum)
 * After the second all-reduce the last 64 floats of span 1 start with {loss, #non-finite distances}.
 * The projection -- the only part that reads C D^2 floats -- and its adjoint shard with the classes, the
 * pair stage with the pairs; sqfa_fused_loss_exchange_span gives a span's byte offset and size in ws. */
int sqfa_fused_loss_exchange_span(int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                                  int64_t pair_begin, int64_t pair_end, int32_t which, size_t* offset_bytes,
                                  size_t* bytes);
int sqfa_fused_loss_sharded(int32_t phase, const float* S, const float* M, const float* F, int32_t n_classes,
                            int32_t n_dim, int32_t n_filters, float noise, int32_t dist, int32_t class_begin,
                            int32_t class_end, int64_t pair_begin, int64_t pair_end, float* dF, void* ws,
                            size_t ws_bytes, sqfa_stream_t stream);

/* The same evaluation at the RAW filter parameter W of a constrained model, constraint included
 * (constraints.py:17-141): F = W / |W| row-wise (SQFA_CONSTRAINT_SPHERE) or F = W
 * (SQFA_CONSTRAINT_NONE); grad = d out[0] / dW through the constraint's adjoint, with zero rows for
 * the first n_fixed filters (FixedFilters of the pairwise curriculum); out[2] = max |grad|, the
 * quantity L-BFGS tests first. out_host (may be NULL): MAPPED PINNED HOST memory [3] that receives a copy
 * of out from the last kernel, so the host needs an event wait and no device-to-host copy. One call per
 * closure evaluation of the fitting loop. */
#define SQFA_CONSTRAINT_NONE 0
#define SQFA_CONSTRAINT_SPHERE 1
int sqfa_closure_eval(const float* S, const float* M, const float* raw_filters, int32_t n_classes, int32_t n_dim,
                      int32_t n_filters, float noise, int32_t dist, int32_t constraint, int32_t n_fixed,
                      int64_t pair_begin, int64_t pair_end, float* out, float* out_host, float* grad, void* ws,
                      size_t ws_bytes, sqfa_stream_t stream);

/* sqfa_closure_eval in float64: S, M, raw_filters, out, out_host and grad are double. For
 * SQFA_DIST_AFFINE_INVARIANT and SQFA_DIST_FISHER_RAO_LB (each optionally + SQFA_DIST_SQUARED) and
 * n_filters <= 32; other codes and n_filters > 32 return SQFA_E_UNSUPPORTED (M is required for Fisher-Rao; the
 * mean-covariance distances have their own entry point, sqfa_gauss_closure_eval_f64).
 * `noise` points to ONE double in device memory (read by the kernels, so a captured graph picks up a new
 * value). As in float32, out[0] over a sub-range [pair_begin, pair_end) is scaled by 1/P of ALL pairs, so
 * the losses and gradients of disjoint ranges add up. Deterministic: no floating-point atomics. The
 * workspace query returns 0 for arguments the evaluation rejects. */
size_t sqfa_fused_loss_workspace_bytes_f64(int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                                           int64_t pair_begin, int64_t pair_end);
int sqfa_closure_eval_f64(const double* S, const double* M, const double* raw_filters, int32_t n_classes,
                          int32_t n_dim, int32_t n_filters, const double* noise, int32_t dist, int32_t constraint,
                          int32_t n_fixed, int64_t pair_begin, int64_t pair_end, double* out, double* out_host,
                          double* grad, void* ws, size_t ws_bytes, sqfa_stream_t stream);

/* The float64 closure of the mean-covariance distances: the same 18 parameters and contracts as
 * sqfa_closure_eval_f64, for SQFA_DIST_MAHALANOBIS (optionally + SQFA_DIST_SQUARED), SQFA_DIST_BHATTACHARYYA
 * and SQFA_DIST_HELLINGER. M is required, n_filters <= 32, constraint NONE or SPHERE. Every other code,
 * SQFA_DIST_SQUARED with Bhattacharyya or Hellinger and n_filters > 32 return SQFA_E_UNSUPPORTED (the codes of
 * sqfa_closure_eval_f64 with a message naming it); the workspace query returns 0 for them. */
size_t sqfa_gauss_closure_workspace_bytes_f64(int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                                              int64_t pair_begin, int64_t pair_end);
int sqfa_gauss_closure_eval_f64(const double* S, const double* M, const double* raw_filters, int32_t n_classes,
                                int32_t n_dim, int32_t n_filters, const double* noise, int32_t dist,
                                int32_t constraint, int32_t n_fixed, int64_t pair_begin, int64_t pair_end,
                                double* out, double* out_host, double* grad, void* ws, size_t ws_bytes,
                                sqfa_stream_t stream);

/* sqfa_fused_loss_sharded in float64: the classes and the pairs of a float64 closure sharded over the ranks of a
 * multi-device caller, with the same three phases, exchange spans and contracts (S, M hold all classes on every
 * rank, a rank reads only its own; F is the constrained filters, dF the rank's share of d loss / dF). For the codes
 * of sqfa_closure_eval_f64 and sqfa_gauss_closure_eval_f64: SQFA_DIST_AFFINE_INVARIANT, SQFA_DIST_FISHER_RAO_LB and
 * SQFA_DIST_MAHALANOBIS (each optionally + SQFA_DIST_SQUARED), SQFA_DIST_BHATTACHARYYA and SQFA_DIST_HELLINGER;
 * M is required for all but the affine-invariant distance, n_filters <= 32. `noise` points to ONE double in device
 * memory. ws: 16-byte aligned, at least the float64 workspace query of the code (sqfa_fused_loss_workspace_bytes_f64
 * or sqfa_gauss_closure_workspace_bytes_f64) for [pair_begin, pair_end). After the second all-reduce the last 64
 * doubles of span 1 start with {loss, #non-finite distances}. Deterministic: no floating-point atomics.
 * Other known codes and n_filters > 32 return SQFA_E_UNSUPPORTED; every check runs before any launch. */
int sqfa_fused_loss_exchange_span_f64(int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                                      int64_t pair_begin, int64_t pair_end, int32_t which, size_t* offset_bytes,
                                      size_t* bytes);
int sqfa_fused_loss_sharded_f64(int32_t phase, const double* S, const double* M, const double* F, int32_t n_classes,
                                int32_t n_dim, int32_t n_filters, const double* noise, int32_t dist,
                                int32_t class_begin, int32_t class_end, int64_t pair_begin, int64_t pair_end,
                                double* dF, void* ws, size_t ws_bytes, sqfa_stream_t stream);

/* Plug-in distances between Gaussians that use the mean covariance of the pair (distances.py:240-432),
 * one warp per pair (Cholesky of (Sigma_a + Sigma_b) / 2 in shared memory), all n_a * n_b pairs:
 *   SQFA_GAUSS_MAHALANOBIS_SQ  d^T M^-1 d                                             (:283-330)
 *   SQFA_GAUSS_BHATTACHARYYA   d^T M^-1 d / 8 + (logdet M - (logdet Sa + logdet Sb) / 2) / 2   (:240-280)
 * (mahalanobis :333-361, hellinger :364-393 and fisher_rao_same_cov :396-432 are scalar maps of these.)
 *   forward : gD == NULL, dist_out [n_a][n_b]
 *   backward: gD [n_a][n_b] = upstream gradient; g_sigma_a [n_a][k][k], g_mu_a [n_a][k], g_sigma_b, g_mu_b are
 *             OVERWRITTEN with the analytic gradients (per-pair partials in ws, summed per class in a fixed
 *             order); dist_out may be NULL.
 *   flag [1] or NULL: set to 1 if some matrix was not positive definite. k <= SQFA_MAX_M. */
#define SQFA_GAUSS_MAHALANOBIS_SQ 0
#define SQFA_GAUSS_BHATTACHARYYA 1
size_t sqfa_gauss_pair_workspace_bytes(int32_t n_a, int32_t n_b, int32_t k, int32_t want_grad);
int sqfa_gauss_pair_distances(const float* mu_a, const float* sigma_a, const float* mu_b, const float* sigma_b,
                              int32_t n_a, int32_t n_b, int32_t k, int32_t mode, const float* gD, float* dist_out,
                              float* g_sigma_a, float* g_mu_a, float* g_sigma_b, float* g_mu_b, void* ws,
                              size_t ws_bytes, int32_t* flag, sqfa_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Optimiser support (reference: torch.optim.LBFGS driven by fitting_loop, _optim.py:78-96)
 * ------------------------------------------------------------------------------------------- */

/* One L-BFGS iteration's "update memory + two-loop recursion" (torch/optim/lbfgs.py, no line search)
 * in one launch, same arithmetic in the same order:
 *   unless first:  y = g - prev_g,  s = t_prev * d,  ys = y.s;
 *                  if ys > 1e-10: append (y, s, 1/ys) to the history (dropping the oldest pair when
 *                  `history` pairs are held) and set H = ys / y.y
 *   q = -g; newest..oldest: al_i = ro_i s_i.q, q -= al_i y_i;  r = H q;
 *   oldest..newest: r += (al_i - ro_i y_i.r) s_i;   d = r;  prev_g = g      (first: d = -g, H = 1)
 * State owned by the caller, all device memory: prev_g, d [n]; S, Y [(history + 1) * n] (ring with
 * one spare row); ro [history + 1]; hdiag [1]; meta int32 [2] = {ring head, pairs held}.
 * param (may be NULL): the optimiser's fixed step is applied in the same launch, x += t d with
 * t = min(1, 1 / sum|g|) lr on the first iteration and lr afterwards, UNLESS g.d > -tolerance_change (the
 * test on which torch.optim.LBFGS stops before stepping) -- so a caller can enqueue the next loss /
 * gradient evaluation right behind this launch and wait once for both.
 * out_scalars [8] = {ys, g.d, max|d|, sum|g|, pairs held, t, step applied (0/1), -} may be device or
 * MAPPED PINNED HOST memory (the host then needs only an event wait to apply the stopping rules).
 * n <= sqfa_lbfgs_max_n() (the vector lives in the registers of one 8-CTA cluster),
 * history <= sqfa_lbfgs_max_history(); otherwise SQFA_E_UNSUPPORTED. */
int64_t sqfa_lbfgs_max_n(void);
int32_t sqfa_lbfgs_max_history(void);
int sqfa_lbfgs_direction(const float* g, float* prev_g, float* d, float* S, float* Y, float* ro, float* hdiag,
                         int32_t* meta, int64_t n, int32_t history, float t_prev, int first, float* param, float lr,
                         float tolerance_change, float* out_scalars, sqfa_stream_t stream);

/* The same update in float64, with the same arithmetic in the same order, for a float64 parameter
 * (every state buffer above in double; meta stays int32). The three host scalars are passed by
 * pointer: scalars_host [3] = {t_prev, lr, tolerance_change} is PLAIN HOST memory, read during the
 * call and not retained. out_scalars [8] has the layout above, in double, device or mapped pinned host
 * memory. n <= sqfa_lbfgs_max_n_f64() (8 doubles per thread of the cluster), history <=
 * sqfa_lbfgs_max_history(); otherwise SQFA_E_UNSUPPORTED. NULL pointers (param excepted), n <= 0 or
 * history < 1: SQFA_E_INVALID. */
int64_t sqfa_lbfgs_max_n_f64(void);
int sqfa_lbfgs_direction_f64(const double* g, double* prev_g, double* d, double* S, double* Y, double* ro,
                             double* hdiag, int32_t* meta, int64_t n, int32_t history, const double* scalars_host,
                             int first, double* param, double* out_scalars, sqfa_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SQFA_B200_H_ */
