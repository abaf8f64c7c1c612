// Internal launcher declarations shared by the .cu translation units and the C-ABI (capi.cu).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace sqfa {

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute: remember what was set on
// which device (a process may drive several), raise it when a launch needs more.
constexpr int kMaxDevices = 64;
template <typename Kernel>
inline cudaError_t ensure_dynamic_smem(Kernel kernel, int bytes, int (&set_bytes)[kMaxDevices]) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= kMaxDevices) dev = 0;
  if (set_bytes[dev] >= bytes) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) set_bytes[dev] = bytes;
  return e;
}

// warps per block of a one-warp-per-problem kernel: at most max_warps, fewer when the per-warp shared-memory
// scratch would not fit in 200 KB (large m)
inline int warps_for(int per_warp_bytes, int max_warps) {
  const int nw = (200 * 1024) / (per_warp_bytes > 0 ? per_warp_bytes : 1);
  return nw > max_warps ? max_warps : (nw < 1 ? 1 : nw);
}

// n elements of T rounded up to whole 256-byte granules (workspace offsets)
template <typename T>
inline size_t al(size_t n) {
  constexpr size_t g = 256 / sizeof(T);
  return (n + g - 1) & ~(g - 1);
}

// Element type of the data points X (same values as SQFA_ELEM_* of the C ABI); see elem.cuh.
enum ElemType { ELEM_F32 = 0, ELEM_BF16 = 1, ELEM_F16 = 2 };
inline int elem_bytes(int elem) { return elem == ELEM_F32 ? 4 : 2; }

// ---- bucket.cu (K1) ----
cudaError_t launch_label_max(const int64_t* labels, int64_t n, int64_t* out_max, cudaStream_t stream);
size_t bucket_workspace_bytes(int64_t n, int32_t C);
cudaError_t launch_bucket_labels(const int64_t* labels, int64_t n, int32_t C, int64_t* counts, int64_t* offsets,
                                 int32_t* perm, void* ws, size_t ws_bytes, cudaStream_t stream);

// ---- stats.cu (K2a, K3) ----
int class_sums_splits(int64_t n, int C, int D, int num_sms);
cudaError_t launch_class_sums(const void* X, int elem, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                              const float* shift, int64_t n, int D, int C, float* sums, int accumulate,
                              float* partial_ws, int nsplit, cudaStream_t stream);
cudaError_t launch_class_means(const float* sums, const int64_t* counts, const float* shift, int D, int C,
                               float* means, cudaStream_t stream);
cudaError_t launch_class_pilot_shift(const void* X, int elem, int64_t ldx, const int32_t* perm,
                                    const int64_t* offsets, int D, int C, float* shift, cudaStream_t stream);
// sums[c][j] = sum over s < nsplit of partial[c][s][j], in float64, s in order
cudaError_t launch_class_sums_finalize(const float* partial, int nsplit, int D, int C, float* sums,
                                       cudaStream_t stream);
cudaError_t launch_counts_pack(const int64_t* counts, int C, float* out, cudaStream_t stream);
cudaError_t launch_counts_unpack(const float* in, int C, int64_t* counts, cudaStream_t stream);
size_t stats_epilogue_workspace_bytes(int C);
// Partial Grams of the same classes held in several buffers (a rank's own packed tiles + the slots its
// peers pushed theirs into): source s is `gram` for s == self, else peers + s * stride. Summed in order.
struct GramSources {
  const float* peers;
  int64_t stride;  // floats between the slots of consecutive source ranks
  int n_src;       // 0 / 1: `gram` alone
  int self;
};
cudaError_t launch_stats_epilogue(const float* gram, int packed, const float* means, const float* shift,
                                  const int64_t* counts, int D, int C, int estimator, int ddof, float* cov, float* sm,
                                  void* ws, cudaStream_t stream, GramSources src = GramSources{nullptr, 0, 0, 0},
                                  int centred_sums = 0);

// ---- gram.cu (K2: tcgen05 cta_group::2 Gram on CTA pairs) ----
int gram_tiles_per_class(int D, int* TT_out);
int64_t gram_executed_tile_area(int D);
int gram_ksplit(int64_t n, int C, int D, int num_sms, int elem_size);
int gram_ksplit_launch(int64_t n, int C, int D, int packed, int num_sms, int elem_size);
size_t gram_workspace_bytes(int C, int D, int ksplit_max);
// sums != nullptr: the diagonal tiles' producers also write class-sum partials sums[C][4 KS][D] of (x - shift),
// KS = gram_ksplit_launch(...); class_sums_finalize with nsplit = 4 KS adds them up
cudaError_t launch_class_gram(const void* X, int elem, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                              const float* shift, int64_t n, int D, int C, float* gram, int accumulate, int packed,
                              int chain_rows, int32_t* done, int n_groups, int first_class, int reserve_sms, void* ws,
                              int num_sms, cudaStream_t stream, float* sums = nullptr);
size_t gram_packed_floats(int D, int C);  // floats of the packed upper-tile list (256 x 256 tiles)
}  // namespace sqfa

namespace sqfa {
// ---- project.cu (K4, K6, transform, embedding, constraint) ----
int project_nsplit(int C, int D, int k);
int project_nchunk(int D);
size_t project_workspace_bytes(int C, int D, int k);
size_t project_psipart_floats(int C, int D, int k);
size_t project_mupart_floats(int C, int D, int k);
// ---- project_tc.cu (K4 on the tensor cores for 8 < k <= 32) ----
bool project_tc_applicable(const float* S, const float* F, int D, int k);
cudaError_t launch_project_tc(const float* S, const float* F, int C, int D, int k, float* T, cudaStream_t st);
cudaError_t launch_project_partials(const float* S, const float* M, const float* F, int C, int D, int k, float* T,
                                    float* partial, float* PsiPart, float* MuPart, cudaStream_t st);
cudaError_t launch_project_fwd(const float* S, const float* M, const float* F, int C, int D, int k, float* T,
                               float* Psi, float* Mu, float* ws, cudaStream_t st);
cudaError_t launch_project_bwd(const float* gPsi, const float* gMu, const float* T, const float* M, int C, int D,
                               int k, float* dF, float* ws, cudaStream_t st);
// The closure's tail, shared by the float32 and float64 closures (T = float, double): class-split partials of the
// projection adjoint, then one block per filter sums them, applies the constraint's adjoint, zeroes the frozen rows
// and publishes max |grad| into out[2] (which the pair stage's reduce kernel zeroes) and out_host.
template <typename T>
int project_bwd_csplit(int C, int D);
template <typename Real>
cudaError_t launch_project_bwd_constrained(const Real* gPsi, const Real* gMu, const Real* T, const Real* M, int C,
                                           int D, int k, const Real* F, const Real* inv_norm, int sphere, int n_fixed,
                                           Real* grad, Real* out, Real* out_host, unsigned int* ticket, Real* ws,
                                           cudaStream_t st);
template <typename T>
cudaError_t launch_constraint_fwd(const T* Wraw, int D, int k, T* F, T* inv_norm, cudaStream_t st);
cudaError_t launch_transform(const void* X, int elem, int64_t ldx, const float* F, int64_t n, int D, int k, float* Z,
                             cudaStream_t st);
cudaError_t launch_embed_fwd(const float* Psi, const float* Mu, float noise, int C, int k, int fr, float* E,
                             cudaStream_t st);
cudaError_t launch_embed_bwd(const float* gE, const float* Mu, int C, int k, int fr, float* gPsi, float* gMu,
                             cudaStream_t st);

// ---- pairs.cu (K5) ----
// A launch of the pair kernels covers the R x R tiles of block rows bi0 .. bi1 of the pair matrix
// (lower triangle for self distances); local tile t = global tile - tile0.
struct PairTiles {
  int R, tri, nbj, bi0, bi1;
  int64_t tile0, ntiles;
};
struct PairArgs {
  const float* Wa;
  const float* Wb;
  int nA, nB, m, dist, tri;
  int64_t pair_begin, pair_end;
  float weight;
  const float* gD;
  float* dist_out;
  float* eig_out;
  float* rowpart;   // [ntiles][R][m*m] per-tile partial gradients of the row classes (LE: one factor per pair)
  float* colpart;   // [ntiles][R][m*m] ... of the column classes
  float* losspart;  // [ntiles][2] {sum of distances, non-finite count}
  const float* Mu;  // Gaussian Wasserstein: class means [nA][k] (rows and columns are the same classes)
  int k;
  float* pwpart;    // Gaussian Wasserstein: [ntiles][R][R] per-pair factor of the means gradient
  PairTiles T;
};
struct PairWorkspace {
  size_t rowpart, colpart, losspart, pwpart, total_floats;  // offsets in floats
  PairTiles T;
};
PairTiles make_pair_tiles(int nA, int nB, int tri, int64_t pair_begin, int64_t pair_end, int R);
PairWorkspace pair_workspace(int nA, int nB, int m, int dist, int tri, int64_t pair_begin, int64_t pair_end);
size_t class_factor_floats(int m, int dist);
cudaError_t launch_class_factor(const float* E, int C, int m, int dist, float* W, int32_t* flag, cudaStream_t st);
cudaError_t launch_class_prepare(const float* PsiPart, const float* MuPart, int nchunk, float noise, int C, int k,
                                 int dist, float* Mu, float* E, float* W, int32_t* flag, cudaStream_t st);
cudaError_t launch_pair_distances(const float* Wa, const float* Wb, int nA, int nB, int m, int dist, int tri,
                                  int64_t pair_begin, int64_t pair_end, float weight, const float* gD,
                                  float* dist_out, float* loss, float* gEa, float* gEb, float* eig_out, float* ws,
                                  cudaStream_t st);
cudaError_t launch_pair_closure(const float* W, int C, int m, int dist, int64_t pair_begin, int64_t pair_end,
                                float weight, const float* Mu, int k, float* out, float* gPsi, float* gMu, float* gLog,
                                float* ws, cudaStream_t st);
// Per class c < C: dLoss/dE_c summed from the per-tile row / column partials in a fixed order, then the adjoint
// of the embedding -> (gPsi, gMu); out = {weight * sum d, #non-finite, 0}. T = float, double.
template <typename T>
cudaError_t launch_pair_reduce_closure(const PairTiles& tiles, int C, int m, int k, int fr, const T* rowpart,
                                       const T* colpart, const T* losspart, T weight, const T* Mu, T* out, T* gPsi,
                                       T* gMu, cudaStream_t st);
cudaError_t launch_class_factor_bwd(const float* W, const float* gLog, int C, int m, int dist, float* gE,
                                    cudaStream_t st);
}  // namespace sqfa

namespace sqfa {
// ---- closure.cu ----
size_t fused_loss_workspace_bytes(int C, int D, int k, int dist, int64_t pair_begin, int64_t pair_end);
void fused_loss_exchange_span(int C, int D, int k, int dist, int64_t pair_begin, int64_t pair_end, int which,
                              size_t* offset_bytes, size_t* bytes);
cudaError_t launch_fused_loss_sharded(int phase, const float* S, const float* M, const float* F, int C, int D, int k,
                                      float noise, int dist, int c0, int c1, int64_t pair_begin, int64_t pair_end,
                                      float* dF, float* ws, cudaStream_t st);
cudaError_t launch_fused_loss(const float* S, const float* M, const float* filters, int C, int D, int k, float noise,
                              int dist, int constraint, int n_fixed, int64_t pair_begin, int64_t pair_end, float* out,
                              float* out_host, float* grad, float* ws, cudaStream_t st);
// ---- closure64.cu (float64 closures, k <= 32: affine-invariant / Fisher-Rao lower bound, and the mean-covariance
// distances of gauss.cu; one workspace layout, sized by the distance code) ----
size_t fused_loss_workspace_bytes_f64(int C, int D, int k, int dist, int64_t pair_begin, int64_t pair_end);
cudaError_t launch_closure_f64(const double* S, const double* M, const double* raw_filters, int C, int D, int k,
                               const double* noise, int dist, int constraint, int n_fixed, int64_t pair_begin,
                               int64_t pair_end, double* out, double* out_host, double* grad, double* ws,
                               cudaStream_t st);
cudaError_t launch_gauss_closure_f64(const double* S, const double* M, const double* raw_filters, int C, int D, int k,
                                     const double* noise, int dist, int constraint, int n_fixed, int64_t pair_begin,
                                     int64_t pair_end, double* out, double* out_host, double* grad, double* ws,
                                     cudaStream_t st);
// the class- and pair-sharded closure of closure.cu in float64, for every code of the two closures above
void fused_loss_exchange_span_f64(int C, int D, int k, int dist, int64_t pair_begin, int64_t pair_end, int which,
                                  size_t* offset_bytes, size_t* bytes);
cudaError_t launch_fused_loss_sharded_f64(int phase, const double* S, const double* M, const double* F, int C, int D,
                                          int k, const double* noise, int dist, int c0, int c1, int64_t pair_begin,
                                          int64_t pair_end, double* dF, double* ws, cudaStream_t st);
}  // namespace sqfa


namespace sqfa {
// ---- lbfgs.cu (device-side L-BFGS direction update) ----
int lbfgs_max_n();
int lbfgs_max_history();
cudaError_t launch_lbfgs_direction(const float* g, float* prev_g, float* d, float* S, float* Y, float* ro, float* hdiag,
                                   int32_t* meta, int64_t n, int history, float t_prev, int first, float* param,
                                   float lr, float tol_change, float* out, cudaStream_t stream);
// the same update in float64, n <= lbfgs_max_n_f64()
int lbfgs_max_n_f64();
cudaError_t launch_lbfgs_direction_f64(const double* g, double* prev_g, double* d, double* S, double* Y, double* ro,
                                       double* hdiag, int32_t* meta, int64_t n, int history, double t_prev, int first,
                                       double* param, double lr, double tol_change, double* out, cudaStream_t stream);
}  // namespace sqfa

namespace sqfa {
// ---- stats64.cu (float64 variants of K2a, K2, K3) ----
cudaError_t launch_class_sums_f64(const double* X, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                                  const double* shift, int D, int C, double* sums, int accumulate, cudaStream_t st);
cudaError_t launch_class_means_f64(const double* sums, const int64_t* counts, const double* shift, int D, int C,
                                   double* means, cudaStream_t st);
cudaError_t launch_class_gram_f64(const double* X, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                                  const double* shift, int D, int C, double* gram, int accumulate, cudaStream_t st);
cudaError_t launch_stats_epilogue_f64(const double* gram, const double* means, const double* shift,
                                      const int64_t* counts, int D, int C, int estimator, int ddof, double* cov,
                                      double* sm, cudaStream_t st);
}  // namespace sqfa

namespace sqfa {
// ---- gauss.cu (mean-covariance distances between Gaussians: Mahalanobis, Bhattacharyya) ----
size_t gauss_workspace_floats(int nA, int nB, int k, int want_grad);
cudaError_t launch_gauss_pairs(const float* muA, const float* SigA, const float* muB, const float* SigB, int nA,
                               int nB, int k, int mode, const float* gD, float* dist_out, float* gSigA, float* gMuA,
                               float* gSigB, float* gMuB, float* ws, int32_t* flag_out, cudaStream_t st);
// closure codes SQFA_DIST_MAHALANOBIS / BHATTACHARYYA / HELLINGER
__host__ __device__ inline bool is_gauss_closure(int dist) { return (dist & 15) >= 5 && (dist & 15) <= 7; }
__host__ __device__ inline bool gauss_closure_needs_logdet(int dist) { return (dist & 15) == 6 || (dist & 15) == 7; }
// workspace of the pair stage in elements of the closure's scalar type (the same count in float32 and float64)
size_t gauss_closure_workspace_elems(int C, int k, int64_t pair_begin, int64_t pair_end);
// float32: noise by value; float64: noise from one device double
cudaError_t launch_gauss_closure_class(const float* PsiPart, const float* MuPart, int nchunk, float noise, int C, int k,
                                       int dist, float* Psi, float* Mu, float* logdet, float* Sinv, int32_t* flag,
                                       cudaStream_t st);
cudaError_t launch_gauss_closure_class(const double* PsiPart, const double* MuPart, int nchunk, const double* noise,
                                       int C, int k, int dist, double* Psi, double* Mu, double* logdet, double* Sinv,
                                       int32_t* flag, cudaStream_t st);
cudaError_t launch_gauss_closure_pairs(const float* Psi, const float* Mu, const float* logdet, const float* Sinv, int C,
                                       int k, int dist, int64_t pair_begin, int64_t pair_end, float weight, float* out,
                                       float* gPsi, float* gMu, float* ws, cudaStream_t st);
cudaError_t launch_gauss_closure_pairs(const double* Psi, const double* Mu, const double* logdet, const double* Sinv,
                                       int C, int k, int dist, int64_t pair_begin, int64_t pair_end, double weight,
                                       double* out, double* gPsi, double* gMu, double* ws, cudaStream_t st);
}  // namespace sqfa
