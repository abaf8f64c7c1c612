// extern "C" boundary of libsqfa_b200.so -- see include/sqfa_b200.h for the contract.
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cuda_runtime.h>

#include "../../include/sqfa_b200.h"
#include "sqfa_internal.h"

namespace {

thread_local char g_err[512] = "";

int fail_arg(const char* fn, const char* what, int code = SQFA_E_INVALID) {
  snprintf(g_err, sizeof(g_err), "%s: %s", fn, what);
  return code;
}

int wrap(const char* fn, cudaError_t e) {
  if (e == cudaSuccess) return 0;
  snprintf(g_err, sizeof(g_err), "%s: CUDA error %d (%s)", fn, (int)e, cudaGetErrorString(e));
  return (int)e;
}

inline cudaStream_t S(sqfa_stream_t s) { return static_cast<cudaStream_t>(s); }

int sm_count_cached() {
  static int sms[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return -1;
  if (sms[dev] == 0) {
    int v = 0;
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
    sms[dev] = v;
  }
  return sms[dev];
}

// element code of the *_h entry points -> sqfa::ElemType; -1 (with sqfa_last_error set) if unknown
int half_elem(const char* fn, int32_t elem) {
  if (elem == SQFA_ELEM_BF16) return sqfa::ELEM_BF16;
  if (elem == SQFA_ELEM_F16) return sqfa::ELEM_F16;
  snprintf(g_err, sizeof(g_err), "%s: unknown element code %d (SQFA_ELEM_BF16 = 1, SQFA_ELEM_F16 = 2)", fn, (int)elem);
  return -1;
}

int class_sums_impl(const char* fn, const void* X, int elem, int64_t ldx, const int32_t* perm,
                    const int64_t* offsets, const float* shift, int64_t n, int32_t n_dim, int32_t n_classes,
                    float* sums, int accumulate, void* ws, size_t ws_bytes, sqfa_stream_t stream);
int class_gram_impl(const char* fn, const void* X, int elem, int64_t ldx, const int32_t* perm,
                    const int64_t* offsets, const float* shift, int64_t n, int32_t n_dim, int32_t n_classes,
                    float* gram, int accumulate, int chain_rows, int32_t* done, int32_t n_groups,
                    int32_t first_class, int32_t reserve_sms, void* ws, size_t ws_bytes, sqfa_stream_t stream,
                    float* sum_partials = nullptr);
int class_pilot_shift_impl(const char* fn, const void* X, int elem, int64_t ldx, const int32_t* perm,
                           const int64_t* offsets, int32_t n_dim, int32_t n_classes, float* shift, sqfa_stream_t stream);
int32_t class_gram_sum_splits(int64_t n, int32_t n_dim, int32_t n_classes, int elem);
size_t class_gram_ws(int64_t n, int32_t n_dim, int32_t n_classes, int elem);
int64_t class_gram_signals(int64_t n, int32_t n_dim, int32_t n_classes, int32_t n_groups, int32_t group, int elem);
size_t class_statistics_ws(int64_t n, int32_t n_dim, int32_t n_classes, int elem);
int class_statistics_impl(const char* fn, const void* X, int elem, int64_t ldx, const int64_t* labels, int64_t n,
                          int32_t n_dim, int32_t n_classes, int estimator, int ddof, float* means, float* cov,
                          float* sm, int64_t* counts, int64_t* offsets, int32_t* perm, void* ws, size_t ws_bytes,
                          sqfa_stream_t stream);

}  // namespace

extern "C" {

#ifndef SQFA_BUILD_ID
#define SQFA_BUILD_ID "unknown"
#endif

int sqfa_version(void) { return 200; }
const char* sqfa_build_id(void) { return SQFA_BUILD_ID; }
const char* sqfa_last_error(void) { return g_err; }
int sqfa_device_sm_count(void) { return sm_count_cached(); }

// --------------------------------------------------------------------------------------------- HP1
int sqfa_label_max(const int64_t* labels, int64_t n, int64_t* out_max, sqfa_stream_t stream) {
  if (n < 0 || out_max == nullptr || (n > 0 && labels == nullptr)) return fail_arg(__func__, "bad argument");
  return wrap(__func__, sqfa::launch_label_max(labels, n, out_max, S(stream)));
}

size_t sqfa_bucket_workspace_bytes(int64_t n, int32_t n_classes) {
  return sqfa::bucket_workspace_bytes(n < 0 ? 0 : n, n_classes);
}

int sqfa_bucket_labels(const int64_t* labels, int64_t n, int32_t n_classes, int64_t* counts, int64_t* offsets,
                       int32_t* perm, void* ws, size_t ws_bytes, sqfa_stream_t stream) {
  if (n < 0 || n_classes < 0 || counts == nullptr || offsets == nullptr || ws == nullptr ||
      (n > 0 && (labels == nullptr || perm == nullptr)))
    return fail_arg(__func__, "bad argument");
  if (n >= ((int64_t)1 << 31)) return fail_arg(__func__, "n must be < 2^31", SQFA_E_UNSUPPORTED);
  if (ws_bytes < sqfa::bucket_workspace_bytes(n, n_classes))
    return fail_arg(__func__, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_bucket_labels(labels, n, n_classes, counts, offsets, perm, ws, ws_bytes, S(stream)));
}

size_t sqfa_class_sums_workspace_bytes(int64_t n, int32_t n_dim, int32_t n_classes) {
  const int sms = sm_count_cached();
  const int ns = sqfa::class_sums_splits(n, n_classes, n_dim, sms > 0 ? sms : 148);
  return (size_t)ns * (size_t)(n_classes > 0 ? n_classes : 1) * (size_t)(n_dim > 0 ? n_dim : 1) * sizeof(float);
}

int sqfa_class_sums(const float* X, int64_t ldx, const int32_t* perm, const int64_t* offsets, const float* shift,
                    int64_t n, int32_t n_dim, int32_t n_classes, float* sums, int accumulate, void* ws,
                    size_t ws_bytes, sqfa_stream_t stream) {
  return class_sums_impl(__func__, X, sqfa::ELEM_F32, ldx, perm, offsets, shift, n, n_dim, n_classes, sums,
                         accumulate, ws, ws_bytes, stream);
}

int sqfa_class_sums_h(const void* X, int64_t ldx, int32_t elem, const int32_t* perm, const int64_t* offsets,
                      const float* shift, int64_t n, int32_t n_dim, int32_t n_classes, float* sums, int accumulate,
                      void* ws, size_t ws_bytes, sqfa_stream_t stream) {
  const int e = half_elem(__func__, elem);
  if (e < 0) return SQFA_E_INVALID;
  return class_sums_impl(__func__, X, e, ldx, perm, offsets, shift, n, n_dim, n_classes, sums, accumulate, ws,
                         ws_bytes, stream);
}

int sqfa_class_means(const float* sums, const int64_t* counts, const float* shift, int32_t n_dim,
                     int32_t n_classes, float* means, sqfa_stream_t stream) {
  if (sums == nullptr || counts == nullptr || means == nullptr || n_dim <= 0 || n_classes < 0)
    return fail_arg(__func__, "bad argument");
  return wrap(__func__, sqfa::launch_class_means(sums, counts, shift, n_dim, n_classes, means, S(stream)));
}

size_t sqfa_class_gram_workspace_bytes(int64_t n, int32_t n_dim, int32_t n_classes) {
  return class_gram_ws(n, n_dim, n_classes, sqfa::ELEM_F32);
}

size_t sqfa_class_gram_workspace_bytes_h(int64_t n, int32_t n_dim, int32_t n_classes, int32_t elem) {
  const int e = half_elem(__func__, elem);
  return e < 0 ? 0 : class_gram_ws(n, n_dim, n_classes, e);
}

int64_t sqfa_gram_executed_tile_area(int32_t n_dim) {
  return n_dim > 0 ? sqfa::gram_executed_tile_area(n_dim) : 0;
}

size_t sqfa_gram_packed_floats(int32_t n_dim, int32_t n_classes) {
  if (n_dim <= 0 || n_classes <= 0) return 0;
  return sqfa::gram_packed_floats(n_dim, n_classes);
}

int sqfa_class_gram(const float* X, int64_t ldx, const int32_t* perm, const int64_t* offsets, const float* shift,
                    int64_t n, int32_t n_dim, int32_t n_classes, float* gram, int accumulate, int chain_rows,
                    int32_t* done, int32_t n_groups, int32_t first_class, int32_t reserve_sms, void* ws,
                    size_t ws_bytes, sqfa_stream_t stream) {
  return class_gram_impl(__func__, X, sqfa::ELEM_F32, ldx, perm, offsets, shift, n, n_dim, n_classes, gram, accumulate,
                         chain_rows, done, n_groups, first_class, reserve_sms, ws, ws_bytes, stream);
}

int sqfa_class_gram_h(const void* X, int64_t ldx, int32_t elem, const int32_t* perm, const int64_t* offsets,
                      const float* shift, int64_t n, int32_t n_dim, int32_t n_classes, float* gram, int accumulate,
                      int chain_rows, int32_t* done, int32_t n_groups, int32_t first_class, int32_t reserve_sms,
                      void* ws, size_t ws_bytes, sqfa_stream_t stream) {
  const int e = half_elem(__func__, elem);
  if (e < 0) return SQFA_E_INVALID;
  return class_gram_impl(__func__, X, e, ldx, perm, offsets, shift, n, n_dim, n_classes, gram, accumulate, chain_rows,
                         done, n_groups, first_class, reserve_sms, ws, ws_bytes, stream);
}

int64_t sqfa_class_gram_group_signals(int64_t n, int32_t n_dim, int32_t n_classes, int32_t n_groups, int32_t group) {
  return class_gram_signals(n, n_dim, n_classes, n_groups, group, sqfa::ELEM_F32);
}

int64_t sqfa_class_gram_group_signals_h(int64_t n, int32_t n_dim, int32_t n_classes, int32_t n_groups, int32_t group,
                                        int32_t elem) {
  const int e = half_elem(__func__, elem);
  return e < 0 ? 0 : class_gram_signals(n, n_dim, n_classes, n_groups, group, e);
}

int32_t sqfa_class_gram_sum_splits(int64_t n, int32_t n_dim, int32_t n_classes) {
  return class_gram_sum_splits(n, n_dim, n_classes, sqfa::ELEM_F32);
}

int32_t sqfa_class_gram_sum_splits_h(int64_t n, int32_t n_dim, int32_t n_classes, int32_t elem) {
  const int e = half_elem(__func__, elem);
  return e < 0 ? 0 : class_gram_sum_splits(n, n_dim, n_classes, e);
}

int sqfa_class_pilot_shift(const float* X, int64_t ldx, const int32_t* perm, const int64_t* offsets, int32_t n_dim,
                           int32_t n_classes, float* shift, sqfa_stream_t stream) {
  return class_pilot_shift_impl(__func__, X, sqfa::ELEM_F32, ldx, perm, offsets, n_dim, n_classes, shift, stream);
}

int sqfa_class_pilot_shift_h(const void* X, int64_t ldx, int32_t elem, const int32_t* perm, const int64_t* offsets,
                             int32_t n_dim, int32_t n_classes, float* shift, sqfa_stream_t stream) {
  const int e = half_elem(__func__, elem);
  if (e < 0) return SQFA_E_INVALID;
  return class_pilot_shift_impl(__func__, X, e, ldx, perm, offsets, n_dim, n_classes, shift, stream);
}

int sqfa_class_gram_sums(const float* X, int64_t ldx, const int32_t* perm, const int64_t* offsets, const float* shift,
                         int64_t n, int32_t n_dim, int32_t n_classes, float* gram, float* partials, void* ws,
                         size_t ws_bytes, sqfa_stream_t stream) {
  if (partials == nullptr || shift == nullptr) return fail_arg(__func__, "bad argument");
  if (class_gram_sum_splits(n, n_dim, n_classes, sqfa::ELEM_F32) == 0)
    return fail_arg(__func__, "K split too deep for class-sum partials", SQFA_E_UNSUPPORTED);
  return class_gram_impl(__func__, X, sqfa::ELEM_F32, ldx, perm, offsets, shift, n, n_dim, n_classes, gram, 0, 0,
                         nullptr, 0, 0, 0, ws, ws_bytes, stream, partials);
}

int sqfa_class_gram_sums_h(const void* X, int64_t ldx, int32_t elem, const int32_t* perm, const int64_t* offsets,
                           const float* shift, int64_t n, int32_t n_dim, int32_t n_classes, float* gram,
                           float* partials, void* ws, size_t ws_bytes, sqfa_stream_t stream) {
  const int e = half_elem(__func__, elem);
  if (e < 0) return SQFA_E_INVALID;
  if (partials == nullptr || shift == nullptr) return fail_arg(__func__, "bad argument");
  if (class_gram_sum_splits(n, n_dim, n_classes, e) == 0)
    return fail_arg(__func__, "K split too deep for class-sum partials", SQFA_E_UNSUPPORTED);
  return class_gram_impl(__func__, X, e, ldx, perm, offsets, shift, n, n_dim, n_classes, gram, 0, 0, nullptr, 0, 0, 0,
                         ws, ws_bytes, stream, partials);
}

int sqfa_class_means_from_partials(const float* partials, int32_t nsplit, const int64_t* counts, const float* shift,
                                   int32_t n_dim, int32_t n_classes, float* sums, float* means,
                                   sqfa_stream_t stream) {
  if (partials == nullptr || nsplit <= 0 || counts == nullptr || shift == nullptr || sums == nullptr ||
      means == nullptr || n_dim <= 0 || n_classes < 0)
    return fail_arg(__func__, "bad argument");
  const cudaError_t e = sqfa::launch_class_sums_finalize(partials, nsplit, n_dim, n_classes, sums, S(stream));
  if (e != cudaSuccess) return wrap(__func__, e);
  return wrap(__func__, sqfa::launch_class_means(sums, counts, shift, n_dim, n_classes, means, S(stream)));
}

// cuStreamWaitValue32 through the runtime's driver entry point lookup (no link dependency on libcuda)
int sqfa_stream_wait_geq(sqfa_stream_t stream, const int32_t* flag, int32_t value) {
  if (flag == nullptr) return fail_arg(__func__, "bad argument");
  typedef int (*wait_fn)(cudaStream_t, unsigned long long, unsigned int, unsigned int);
  static wait_fn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuStreamWaitValue32", &p, cudaEnableDefault, &q);
    if (e != cudaSuccess || p == nullptr || q != cudaDriverEntryPointSuccess)
      return fail_arg(__func__, "cuStreamWaitValue32 is not available", SQFA_E_UNSUPPORTED);
    fn = reinterpret_cast<wait_fn>(p);
  }
  const int rc = fn(S(stream), (unsigned long long)reinterpret_cast<uintptr_t>(flag), (unsigned int)value,
                    0u /* CU_STREAM_WAIT_VALUE_GEQ */);
  if (rc != 0) {
    snprintf(g_err, sizeof(g_err), "%s: cuStreamWaitValue32 failed with CUresult %d", __func__, rc);
    return 1000 + rc;
  }
  return 0;
}

int sqfa_counts_pack(const int64_t* counts, int32_t n_classes, float* out, sqfa_stream_t stream) {
  if (n_classes < 0 || (n_classes > 0 && (counts == nullptr || out == nullptr))) return fail_arg(__func__, "bad argument");
  return wrap(__func__, sqfa::launch_counts_pack(counts, n_classes, out, S(stream)));
}
int sqfa_counts_unpack(const float* in, int32_t n_classes, int64_t* counts, sqfa_stream_t stream) {
  if (n_classes < 0 || (n_classes > 0 && (counts == nullptr || in == nullptr))) return fail_arg(__func__, "bad argument");
  return wrap(__func__, sqfa::launch_counts_unpack(in, n_classes, counts, S(stream)));
}

size_t sqfa_stats_epilogue_workspace_bytes(int32_t n_classes) {
  return sqfa::stats_epilogue_workspace_bytes(n_classes);
}

int sqfa_stats_epilogue(const float* gram, const float* means, const float* shift, const int64_t* counts,
                        int32_t n_dim, int32_t n_classes, int estimator, int ddof, float* cov, float* sm, void* ws,
                        size_t ws_bytes, sqfa_stream_t stream) {
  const int packed = estimator & SQFA_EST_PACKED_GRAM;
  const int centred_sums = estimator & SQFA_EST_CENTRED_SUMS;
  estimator &= ~(SQFA_EST_PACKED_GRAM | SQFA_EST_CENTRED_SUMS);
  if (gram == nullptr || means == nullptr || counts == nullptr || cov == nullptr || n_dim <= 0 || n_classes < 0 ||
      (estimator != SQFA_EST_EMPIRICAL && estimator != SQFA_EST_OAS) || (ddof != 0 && ddof != 1) ||
      (packed && cov == gram) || (centred_sums && shift == nullptr))
    return fail_arg(__func__, "bad argument");
  if (estimator == SQFA_EST_OAS && (ws == nullptr || ws_bytes < sqfa::stats_epilogue_workspace_bytes(n_classes)))
    return fail_arg(__func__, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_stats_epilogue(gram, packed, means, shift, counts, n_dim, n_classes, estimator,
                                                    ddof, cov, sm, ws, S(stream), sqfa::GramSources{nullptr, 0, 0, 0},
                                                    centred_sums ? 1 : 0));
}

int sqfa_stats_epilogue_reduce(const float* gram, const float* peer_slots, int64_t slot_stride, int32_t n_sources,
                               int32_t self, const float* means, const float* shift, const int64_t* counts,
                               int32_t n_dim, int32_t n_classes, int estimator, int ddof, float* cov, float* sm,
                               void* ws, size_t ws_bytes, sqfa_stream_t stream) {
  if (gram == nullptr || peer_slots == nullptr || means == nullptr || counts == nullptr || cov == nullptr ||
      n_dim <= 0 || n_classes < 0 || n_sources < 1 || n_sources > 64 || self < 0 || self >= n_sources ||
      slot_stride < (int64_t)sqfa::gram_packed_floats(n_dim, n_classes) ||
      (estimator != SQFA_EST_EMPIRICAL && estimator != SQFA_EST_OAS) || (ddof != 0 && ddof != 1))
    return fail_arg(__func__, "bad argument");
  if (estimator == SQFA_EST_OAS && (ws == nullptr || ws_bytes < sqfa::stats_epilogue_workspace_bytes(n_classes)))
    return fail_arg(__func__, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_stats_epilogue(gram, 1, means, shift, counts, n_dim, n_classes, estimator, ddof,
                                                    cov, sm, ws, S(stream),
                                                    sqfa::GramSources{peer_slots, slot_stride, n_sources, self}));
}

// Copy-engine push: no kernel, no SM. With `dst` a peer-mapped address (CUDA IPC / symmetric memory) the
// bytes travel over NVLink while this device's SMs keep computing.
int sqfa_peer_push(void* dst, const void* src, size_t bytes, sqfa_stream_t stream) {
  if ((dst == nullptr || src == nullptr) && bytes > 0) return fail_arg(__func__, "bad argument");
  if (bytes == 0) return 0;
  return wrap(__func__, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, S(stream)));
}

}  // extern "C"

// --------------------------------------------------------------------------------------------- HP2
extern "C" {

size_t sqfa_project_workspace_bytes(int32_t n_classes, int32_t n_dim, int32_t n_filters) {
  if (n_classes <= 0 || n_dim <= 0 || n_filters <= 0) return 256;
  return sqfa::project_workspace_bytes(n_classes, n_dim, n_filters);
}

int sqfa_project_fwd(const float* S_, const float* M, const float* F, int32_t n_classes, int32_t n_dim,
                     int32_t n_filters, float* T, float* Psi, float* Mu, void* ws, size_t ws_bytes,
                     sqfa_stream_t stream) {
  if (S_ == nullptr || F == nullptr || T == nullptr || Psi == nullptr || ws == nullptr || n_classes < 0 ||
      n_dim <= 0 || n_filters <= 0 || (M != nullptr && Mu == nullptr))
    return fail_arg(__func__, "bad argument");
  if (n_filters > 32) return fail_arg(__func__, "n_filters must be <= 32", SQFA_E_UNSUPPORTED);
  if (ws_bytes < sqfa_project_workspace_bytes(n_classes, n_dim, n_filters))
    return fail_arg(__func__, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_project_fwd(S_, M, F, n_classes, n_dim, n_filters, T, Psi, Mu,
                                                 static_cast<float*>(ws), S(stream)));
}

int sqfa_project_bwd(const float* gPsi, const float* gMu, const float* T, const float* M, int32_t n_classes,
                     int32_t n_dim, int32_t n_filters, float* dF, void* ws, size_t ws_bytes,
                     sqfa_stream_t stream) {
  if (gPsi == nullptr || T == nullptr || dF == nullptr || ws == nullptr || n_classes < 0 || n_dim <= 0 ||
      n_filters <= 0 || ((gMu == nullptr) != (M == nullptr)))
    return fail_arg(__func__, "bad argument");
  if (n_filters > 32) return fail_arg(__func__, "n_filters must be <= 32", SQFA_E_UNSUPPORTED);
  if (ws_bytes < sqfa_project_workspace_bytes(n_classes, n_dim, n_filters))
    return fail_arg(__func__, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_project_bwd(gPsi, gMu, T, M, n_classes, n_dim, n_filters, dF,
                                                 static_cast<float*>(ws), S(stream)));
}

int sqfa_transform(const float* X, int64_t ldx, const float* F, int64_t n, int32_t n_dim, int32_t n_filters,
                   float* Z, sqfa_stream_t stream) {
  if (n < 0 || n_dim <= 0 || n_filters <= 0 || F == nullptr || (n > 0 && (X == nullptr || Z == nullptr)) ||
      ldx < n_dim)
    return fail_arg(__func__, "bad argument");
  return wrap(__func__, sqfa::launch_transform(X, sqfa::ELEM_F32, ldx, F, n, n_dim, n_filters, Z, S(stream)));
}

int sqfa_transform_h(const void* X, int64_t ldx, int32_t elem, const float* F, int64_t n, int32_t n_dim,
                     int32_t n_filters, float* Z, sqfa_stream_t stream) {
  const int e = half_elem(__func__, elem);
  if (e < 0) return SQFA_E_INVALID;
  if (n < 0 || n_dim <= 0 || n_filters <= 0 || F == nullptr || (n > 0 && (X == nullptr || Z == nullptr)) ||
      ldx < n_dim)
    return fail_arg(__func__, "bad argument");
  return wrap(__func__, sqfa::launch_transform(X, e, ldx, F, n, n_dim, n_filters, Z, S(stream)));
}

static int dist_ok(int32_t dist) {
  const int b = dist & 15;
  if ((dist & SQFA_DIST_SQUARED) && (b == SQFA_DIST_BHATTACHARYYA || b == SQFA_DIST_HELLINGER))
    return 0;  // the reference has no squared form of these
  return (dist & ~(15 | SQFA_DIST_SQUARED)) == 0 &&
         (b == SQFA_DIST_AFFINE_INVARIANT || b == SQFA_DIST_FISHER_RAO_LB || b == SQFA_DIST_LOG_EUCLIDEAN ||
          b == SQFA_DIST_BURES_WASSERSTEIN || b == SQFA_DIST_WASSERSTEIN_GAUSSIAN || sqfa::is_gauss_closure(dist));
}

// distances whose closure reads the class means
static int dist_uses_means(int32_t dist) {
  const int b = dist & 15;
  return b == SQFA_DIST_FISHER_RAO_LB || b == SQFA_DIST_WASSERSTEIN_GAUSSIAN || sqfa::is_gauss_closure(dist);
}

// The mean-covariance codes exist for closures only: the per-matrix entry points have no means and no
// pair-mean covariance. Returns 0 or the fail_arg code.
static int check_not_gauss_closure(const char* fn, int32_t dist) {
  if (sqfa::is_gauss_closure(dist))
    return fail_arg(fn, "SQFA_DIST_MAHALANOBIS / BHATTACHARYYA / HELLINGER are closure codes: evaluate these "
                        "distances with sqfa_gauss_pair_distances");
  return 0;
}

// Bures-Wasserstein runs in the column-pair kernel only (m <= 34); the Gaussian form needs means, which the
// per-matrix entry points do not take. Returns 0 or the fail_arg code.
static int check_bw_matrices(const char* fn, int32_t dist, int32_t m) {
  const int b = dist & 15;
  if (b == SQFA_DIST_WASSERSTEIN_GAUSSIAN)
    return fail_arg(fn, "SQFA_DIST_WASSERSTEIN_GAUSSIAN needs class means: use SQFA_DIST_BURES_WASSERSTEIN on the "
                        "covariances and add |mu_A - mu_B|^2");
  if (b == SQFA_DIST_BURES_WASSERSTEIN && m > 34)
    return fail_arg(fn, "Bures-Wasserstein supports m <= 34", SQFA_E_UNSUPPORTED);
  return 0;
}

int sqfa_embed_fwd(const float* Psi, const float* Mu, float noise, int32_t n_classes, int32_t n_filters,
                   int32_t dist, float* E, sqfa_stream_t stream) {
  const int fr = (dist & 15) == SQFA_DIST_FISHER_RAO_LB;
  if (!dist_ok(dist) || Psi == nullptr || E == nullptr || n_classes < 0 || n_filters <= 0 || (fr && Mu == nullptr))
    return fail_arg(__func__, "bad argument");
  if (const int rc = check_not_gauss_closure(__func__, dist)) return rc;
  return wrap(__func__, sqfa::launch_embed_fwd(Psi, Mu, noise, n_classes, n_filters, fr, E, S(stream)));
}

int sqfa_embed_bwd(const float* gE, const float* Mu, int32_t n_classes, int32_t n_filters, int32_t dist,
                   float* gPsi, float* gMu, sqfa_stream_t stream) {
  const int fr = (dist & 15) == SQFA_DIST_FISHER_RAO_LB;
  if (!dist_ok(dist) || gE == nullptr || gPsi == nullptr || n_classes < 0 || n_filters <= 0 ||
      (fr && (Mu == nullptr || gMu == nullptr)))
    return fail_arg(__func__, "bad argument");
  if (const int rc = check_not_gauss_closure(__func__, dist)) return rc;
  return wrap(__func__, sqfa::launch_embed_bwd(gE, Mu, n_classes, n_filters, fr, gPsi, gMu, S(stream)));
}

size_t sqfa_class_factor_floats(int32_t m, int32_t dist) { return sqfa::class_factor_floats(m, dist); }

int sqfa_class_factor(const float* E, int32_t n_classes, int32_t m, int32_t dist, float* W, int32_t* flag,
                      sqfa_stream_t stream) {
  if (!dist_ok(dist) || E == nullptr || W == nullptr || flag == nullptr || n_classes < 0 || m <= 0)
    return fail_arg(__func__, "bad argument");
  if (const int rc = check_not_gauss_closure(__func__, dist)) return rc;
  if (m > SQFA_MAX_M) return fail_arg(__func__, "m exceeds SQFA_MAX_M", SQFA_E_UNSUPPORTED);
  if (const int rc = check_bw_matrices(__func__, dist, m)) return rc;
  return wrap(__func__, sqfa::launch_class_factor(E, n_classes, m, dist, W, flag, S(stream)));
}

size_t sqfa_pair_distances_workspace_bytes(int32_t n_a, int32_t n_b, int32_t m, int32_t dist, int32_t triangular,
                                           int64_t pair_begin, int64_t pair_end) {
  if (n_a <= 0 || n_b <= 0 || m <= 0 || !dist_ok(dist) || sqfa::is_gauss_closure(dist)) return 256;
  return sqfa::pair_workspace(n_a, n_b, m, dist, triangular ? 1 : 0, pair_begin, pair_end).total_floats *
             sizeof(float) + 256;
}

int sqfa_pair_distances(const float* Wa, const float* Wb, int32_t n_a, int32_t n_b, int32_t m, int32_t dist,
                        int32_t triangular, int64_t pair_begin, int64_t pair_end, float weight, const float* gD,
                        float* dist_out, float* loss, float* gEa, float* gEb, float* eig_out, void* ws,
                        size_t ws_bytes, sqfa_stream_t stream) {
  if (!dist_ok(dist) || Wa == nullptr || Wb == nullptr || n_a < 0 || n_b < 0 || m <= 0 ||
      (triangular && (n_a != n_b || Wa != Wb)) || ((gEa == nullptr) != (gEb == nullptr)) ||
      (eig_out != nullptr && (triangular || (dist & 15) == SQFA_DIST_LOG_EUCLIDEAN)))
    return fail_arg(__func__, "bad argument");
  if (const int rc = check_not_gauss_closure(__func__, dist)) return rc;
  if (const int rc = check_bw_matrices(__func__, dist, m)) return rc;
  if (eig_out != nullptr && (dist & 15) == SQFA_DIST_BURES_WASSERSTEIN)
    return fail_arg(__func__, "eig_out is not defined for Bures-Wasserstein");
  const int64_t P = triangular ? (int64_t)n_a * (n_a - 1) / 2 : (int64_t)n_a * n_b;
  if (pair_begin < 0 || pair_end > P || pair_begin > pair_end) return fail_arg(__func__, "bad pair range");
  if (m > SQFA_MAX_M) return fail_arg(__func__, "m exceeds SQFA_MAX_M", SQFA_E_UNSUPPORTED);
  const bool needs_ws = (loss != nullptr || gEa != nullptr) && pair_end > pair_begin;
  if (needs_ws && (ws == nullptr || (reinterpret_cast<uintptr_t>(ws) & 15) != 0 ||
                   ws_bytes < sqfa_pair_distances_workspace_bytes(n_a, n_b, m, dist, triangular, pair_begin, pair_end)))
    return fail_arg(__func__, "workspace missing, misaligned or too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_pair_distances(Wa, Wb, n_a, n_b, m, dist, triangular ? 1 : 0, pair_begin,
                                                    pair_end, weight, gD, dist_out, loss, gEa, gEb, eig_out,
                                                    static_cast<float*>(ws), S(stream)));
}

int sqfa_class_factor_bwd(const float* W, const float* gLog, int32_t n_classes, int32_t m, int32_t dist,
                          float* gE, sqfa_stream_t stream) {
  if (!dist_ok(dist) || W == nullptr || gLog == nullptr || gE == nullptr || n_classes < 0 || m <= 0)
    return fail_arg(__func__, "bad argument");
  if (const int rc = check_not_gauss_closure(__func__, dist)) return rc;
  if (m > SQFA_MAX_M) return fail_arg(__func__, "m exceeds SQFA_MAX_M", SQFA_E_UNSUPPORTED);
  return wrap(__func__, sqfa::launch_class_factor_bwd(W, gLog, n_classes, m, dist, gE, S(stream)));
}

}  // extern "C"

extern "C" {

size_t sqfa_fused_loss_workspace_bytes(int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                                       int64_t pair_begin, int64_t pair_end) {
  if (n_classes <= 0 || n_dim <= 0 || n_filters <= 0 || !dist_ok(dist)) return 256;
  return sqfa::fused_loss_workspace_bytes(n_classes, n_dim, n_filters, dist, pair_begin, pair_end);
}

static int closure_common(const char* fn, const float* S_, const float* M, const float* filters, int32_t n_classes,
                          int32_t n_dim, int32_t n_filters, float noise, int32_t dist, int constraint, int n_fixed,
                          int64_t pair_begin, int64_t pair_end, float* out, float* out_host, float* grad, void* ws,
                          size_t ws_bytes, sqfa_stream_t stream) {
  const int base = dist & 15;
  if (!dist_ok(dist) || S_ == nullptr || filters == nullptr || out == nullptr || grad == nullptr || ws == nullptr ||
      n_classes <= 0 || n_dim <= 0 || n_filters <= 0 || (dist_uses_means(dist) && M == nullptr) ||
      n_fixed < 0 || n_fixed > n_filters || (reinterpret_cast<uintptr_t>(ws) & 15) != 0)
    return fail_arg(fn, "bad argument");
  const int m = base == SQFA_DIST_FISHER_RAO_LB ? n_filters + 1 : n_filters;
  if (n_filters > 32 || m > SQFA_MAX_M) return fail_arg(fn, "n_filters must be <= 32", SQFA_E_UNSUPPORTED);
  const int64_t P = (int64_t)n_classes * (n_classes - 1) / 2;
  if (pair_begin < 0 || pair_end > P || pair_begin > pair_end) return fail_arg(fn, "bad pair range");
  if (ws_bytes < sqfa_fused_loss_workspace_bytes(n_classes, n_dim, n_filters, dist, pair_begin, pair_end))
    return fail_arg(fn, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(fn, sqfa::launch_fused_loss(S_, M, filters, n_classes, n_dim, n_filters, noise, dist, constraint,
                                          n_fixed, pair_begin, pair_end, out, out_host, grad,
                                          static_cast<float*>(ws), S(stream)));
}

int sqfa_fused_loss(const float* S_, const float* M, const float* F, int32_t n_classes, int32_t n_dim,
                    int32_t n_filters, float noise, int32_t dist, int64_t pair_begin, int64_t pair_end, float* out,
                    float* dF, void* ws, size_t ws_bytes, sqfa_stream_t stream) {
  return closure_common(__func__, S_, M, F, n_classes, n_dim, n_filters, noise, dist, -1, 0, pair_begin, pair_end,
                        out, nullptr, dF, ws, ws_bytes, stream);
}

int sqfa_fused_loss_exchange_span(int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                                  int64_t pair_begin, int64_t pair_end, int32_t which, size_t* offset_bytes,
                                  size_t* bytes) {
  if (n_classes <= 0 || n_dim <= 0 || n_filters <= 0 || !dist_ok(dist) || (which != 0 && which != 1) ||
      offset_bytes == nullptr || bytes == nullptr)
    return fail_arg(__func__, "bad argument");
  sqfa::fused_loss_exchange_span(n_classes, n_dim, n_filters, dist, pair_begin, pair_end, which, offset_bytes, bytes);
  return 0;
}

int sqfa_fused_loss_sharded(int32_t phase, const float* S_, const float* M, const float* F, int32_t n_classes,
                            int32_t n_dim, int32_t n_filters, float noise, int32_t dist, int32_t class_begin,
                            int32_t class_end, int64_t pair_begin, int64_t pair_end, float* dF, void* ws,
                            size_t ws_bytes, sqfa_stream_t stream) {
  const int base = dist & 15;
  if (!dist_ok(dist) || S_ == nullptr || F == nullptr || ws == nullptr || n_classes <= 0 || n_dim <= 0 ||
      n_filters <= 0 || (dist_uses_means(dist) && M == nullptr) || phase < 0 || phase > 2 ||
      (phase == 2 && dF == nullptr) || class_begin < 0 || class_end > n_classes || class_begin > class_end ||
      (reinterpret_cast<uintptr_t>(ws) & 15) != 0)
    return fail_arg(__func__, "bad argument");
  if (base == SQFA_DIST_LOG_EUCLIDEAN)
    return fail_arg(__func__, "log-Euclidean closures shard their pairs only (sqfa_fused_loss)", SQFA_E_UNSUPPORTED);
  const int m = base == SQFA_DIST_FISHER_RAO_LB ? n_filters + 1 : n_filters;
  if (n_filters > 32 || m > SQFA_MAX_M) return fail_arg(__func__, "n_filters must be <= 32", SQFA_E_UNSUPPORTED);
  const int64_t P = (int64_t)n_classes * (n_classes - 1) / 2;
  if (pair_begin < 0 || pair_end > P || pair_begin > pair_end) return fail_arg(__func__, "bad pair range");
  if (ws_bytes < sqfa_fused_loss_workspace_bytes(n_classes, n_dim, n_filters, dist, pair_begin, pair_end))
    return fail_arg(__func__, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_fused_loss_sharded(phase, S_, M, F, n_classes, n_dim, n_filters, noise, dist,
                                                        class_begin, class_end, pair_begin, pair_end, dF,
                                                        static_cast<float*>(ws), S(stream)));
}

int sqfa_closure_eval(const float* S_, const float* M, const float* raw_filters, int32_t n_classes, int32_t n_dim,
                      int32_t n_filters, float noise, int32_t dist, int32_t constraint, int32_t n_fixed,
                      int64_t pair_begin, int64_t pair_end, float* out, float* out_host, float* grad, void* ws,
                      size_t ws_bytes, sqfa_stream_t stream) {
  if (constraint != SQFA_CONSTRAINT_NONE && constraint != SQFA_CONSTRAINT_SPHERE)
    return fail_arg(__func__, "constraint must be SQFA_CONSTRAINT_NONE or SQFA_CONSTRAINT_SPHERE");
  return closure_common(__func__, S_, M, raw_filters, n_classes, n_dim, n_filters, noise, dist, constraint, n_fixed,
                        pair_begin, pair_end, out, out_host, grad, ws, ws_bytes, stream);
}

// float64 closure: affine-invariant and Fisher-Rao lower bound (plain or squared) only
static int f64_dist_ok(int32_t dist) {
  const int b = dist & 15;
  return (dist & ~(15 | SQFA_DIST_SQUARED)) == 0 && (b == SQFA_DIST_AFFINE_INVARIANT || b == SQFA_DIST_FISHER_RAO_LB);
}

size_t sqfa_fused_loss_workspace_bytes_f64(int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                                           int64_t pair_begin, int64_t pair_end) {
  const int64_t P = (int64_t)n_classes * (n_classes - 1) / 2;
  if (n_classes <= 0 || n_dim <= 0 || n_filters <= 0 || n_filters > 32 || !f64_dist_ok(dist) || pair_begin < 0 ||
      pair_end > P || pair_begin > pair_end)
    return 0;
  return sqfa::fused_loss_workspace_bytes_f64(n_classes, n_dim, n_filters, dist, pair_begin, pair_end);
}

int sqfa_closure_eval_f64(const double* S_, const double* M, const double* raw_filters, int32_t n_classes,
                          int32_t n_dim, int32_t n_filters, const double* noise, int32_t dist, int32_t constraint,
                          int32_t n_fixed, int64_t pair_begin, int64_t pair_end, double* out, double* out_host,
                          double* grad, void* ws, size_t ws_bytes, sqfa_stream_t stream) {
  if (!f64_dist_ok(dist))
    return fail_arg(__func__, sqfa::is_gauss_closure(dist)
                                  ? "the float64 closure supports SQFA_DIST_AFFINE_INVARIANT and SQFA_DIST_FISHER_RAO_LB "
                                    "(optionally + SQFA_DIST_SQUARED); the mean-covariance distances take "
                                    "sqfa_gauss_closure_eval_f64"
                                  : "the float64 closure supports SQFA_DIST_AFFINE_INVARIANT and SQFA_DIST_FISHER_RAO_LB "
                                    "(optionally + SQFA_DIST_SQUARED)",
                    SQFA_E_UNSUPPORTED);
  if (constraint != SQFA_CONSTRAINT_NONE && constraint != SQFA_CONSTRAINT_SPHERE)
    return fail_arg(__func__, "constraint must be SQFA_CONSTRAINT_NONE or SQFA_CONSTRAINT_SPHERE");
  if (S_ == nullptr || raw_filters == nullptr || noise == nullptr || out == nullptr || grad == nullptr ||
      ws == nullptr || n_classes <= 0 || n_dim <= 0 || n_filters <= 0 || n_fixed < 0 || n_fixed > n_filters ||
      ((dist & 15) == SQFA_DIST_FISHER_RAO_LB && M == nullptr) || (reinterpret_cast<uintptr_t>(ws) & 15) != 0)
    return fail_arg(__func__, "bad argument");
  if (n_filters > 32) return fail_arg(__func__, "n_filters must be <= 32", SQFA_E_UNSUPPORTED);
  const int64_t P = (int64_t)n_classes * (n_classes - 1) / 2;
  if (pair_begin < 0 || pair_end > P || pair_begin > pair_end) return fail_arg(__func__, "bad pair range");
  if (ws_bytes < sqfa_fused_loss_workspace_bytes_f64(n_classes, n_dim, n_filters, dist, pair_begin, pair_end))
    return fail_arg(__func__, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_closure_f64(S_, M, raw_filters, n_classes, n_dim, n_filters, noise, dist,
                                                 constraint, n_fixed, pair_begin, pair_end, out, out_host, grad,
                                                 static_cast<double*>(ws), S(stream)));
}

// float64 closure of the mean-covariance distances: Mahalanobis (plain or squared), Bhattacharyya, Hellinger
static int gauss_f64_dist_ok(int32_t dist) {
  const int b = dist & 15;
  return (dist & ~(15 | SQFA_DIST_SQUARED)) == 0 && sqfa::is_gauss_closure(dist) &&
         (b == SQFA_DIST_MAHALANOBIS || (dist & SQFA_DIST_SQUARED) == 0);
}

size_t sqfa_gauss_closure_workspace_bytes_f64(int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                                              int64_t pair_begin, int64_t pair_end) {
  const int64_t P = (int64_t)n_classes * (n_classes - 1) / 2;
  if (n_classes <= 0 || n_dim <= 0 || n_filters <= 0 || n_filters > 32 || !gauss_f64_dist_ok(dist) ||
      pair_begin < 0 || pair_end > P || pair_begin > pair_end)
    return 0;
  return sqfa::fused_loss_workspace_bytes_f64(n_classes, n_dim, n_filters, dist, pair_begin, pair_end);
}

int sqfa_gauss_closure_eval_f64(const double* S_, const double* M, const double* raw_filters, int32_t n_classes,
                                int32_t n_dim, int32_t n_filters, const double* noise, int32_t dist,
                                int32_t constraint, int32_t n_fixed, int64_t pair_begin, int64_t pair_end,
                                double* out, double* out_host, double* grad, void* ws, size_t ws_bytes,
                                sqfa_stream_t stream) {
  if (f64_dist_ok(dist))
    return fail_arg(__func__, "SQFA_DIST_AFFINE_INVARIANT and SQFA_DIST_FISHER_RAO_LB take sqfa_closure_eval_f64",
                    SQFA_E_UNSUPPORTED);
  if (!gauss_f64_dist_ok(dist))
    return fail_arg(__func__, "the float64 mean-covariance closure supports SQFA_DIST_MAHALANOBIS (optionally + "
                              "SQFA_DIST_SQUARED), SQFA_DIST_BHATTACHARYYA and SQFA_DIST_HELLINGER",
                    SQFA_E_UNSUPPORTED);
  if (constraint != SQFA_CONSTRAINT_NONE && constraint != SQFA_CONSTRAINT_SPHERE)
    return fail_arg(__func__, "constraint must be SQFA_CONSTRAINT_NONE or SQFA_CONSTRAINT_SPHERE");
  if (S_ == nullptr || M == nullptr || raw_filters == nullptr || noise == nullptr || out == nullptr ||
      grad == nullptr || ws == nullptr || n_classes <= 0 || n_dim <= 0 || n_filters <= 0 || n_fixed < 0 ||
      n_fixed > n_filters || (reinterpret_cast<uintptr_t>(ws) & 15) != 0)
    return fail_arg(__func__, "bad argument");
  if (n_filters > 32) return fail_arg(__func__, "n_filters must be <= 32", SQFA_E_UNSUPPORTED);
  const int64_t P = (int64_t)n_classes * (n_classes - 1) / 2;
  if (pair_begin < 0 || pair_end > P || pair_begin > pair_end) return fail_arg(__func__, "bad pair range");
  if (ws_bytes < sqfa_gauss_closure_workspace_bytes_f64(n_classes, n_dim, n_filters, dist, pair_begin, pair_end))
    return fail_arg(__func__, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_gauss_closure_f64(S_, M, raw_filters, n_classes, n_dim, n_filters, noise, dist,
                                                       constraint, n_fixed, pair_begin, pair_end, out, out_host, grad,
                                                       static_cast<double*>(ws), S(stream)));
}

// sharded float64 closure: the codes of both float64 closures. Returns 0, or the fail_arg code for a code, n_filters
// or pair range the layout cannot take (checked before anything else reads the layout).
static int sharded_f64_check(const char* fn, int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                             int64_t pair_begin, int64_t pair_end) {
  if (!dist_ok(dist) || n_classes <= 0 || n_dim <= 0 || n_filters <= 0) return fail_arg(fn, "bad argument");
  if (!f64_dist_ok(dist) && !gauss_f64_dist_ok(dist))
    return fail_arg(fn, "the sharded float64 closure supports SQFA_DIST_AFFINE_INVARIANT, SQFA_DIST_FISHER_RAO_LB and "
                        "SQFA_DIST_MAHALANOBIS (each optionally + SQFA_DIST_SQUARED), SQFA_DIST_BHATTACHARYYA and "
                        "SQFA_DIST_HELLINGER",
                    SQFA_E_UNSUPPORTED);
  if (n_filters > 32) return fail_arg(fn, "n_filters must be <= 32", SQFA_E_UNSUPPORTED);
  const int64_t P = (int64_t)n_classes * (n_classes - 1) / 2;
  if (pair_begin < 0 || pair_end > P || pair_begin > pair_end) return fail_arg(fn, "bad pair range");
  return 0;
}

int sqfa_fused_loss_exchange_span_f64(int32_t n_classes, int32_t n_dim, int32_t n_filters, int32_t dist,
                                      int64_t pair_begin, int64_t pair_end, int32_t which, size_t* offset_bytes,
                                      size_t* bytes) {
  if ((which != 0 && which != 1) || offset_bytes == nullptr || bytes == nullptr)
    return fail_arg(__func__, "bad argument");
  if (const int rc = sharded_f64_check(__func__, n_classes, n_dim, n_filters, dist, pair_begin, pair_end)) return rc;
  sqfa::fused_loss_exchange_span_f64(n_classes, n_dim, n_filters, dist, pair_begin, pair_end, which, offset_bytes,
                                     bytes);
  return 0;
}

int sqfa_fused_loss_sharded_f64(int32_t phase, const double* S_, const double* M, const double* F, int32_t n_classes,
                                int32_t n_dim, int32_t n_filters, const double* noise, int32_t dist,
                                int32_t class_begin, int32_t class_end, int64_t pair_begin, int64_t pair_end,
                                double* dF, void* ws, size_t ws_bytes, sqfa_stream_t stream) {
  if (S_ == nullptr || F == nullptr || ws == nullptr || noise == nullptr || (dist_uses_means(dist) && M == nullptr) ||
      phase < 0 || phase > 2 || (phase == 2 && dF == nullptr) || class_begin < 0 || class_end > n_classes ||
      class_begin > class_end || (reinterpret_cast<uintptr_t>(ws) & 15) != 0)
    return fail_arg(__func__, "bad argument");
  if (const int rc = sharded_f64_check(__func__, n_classes, n_dim, n_filters, dist, pair_begin, pair_end)) return rc;
  if (ws_bytes < sqfa::fused_loss_workspace_bytes_f64(n_classes, n_dim, n_filters, dist, pair_begin, pair_end))
    return fail_arg(__func__, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_fused_loss_sharded_f64(phase, S_, M, F, n_classes, n_dim, n_filters, noise, dist,
                                                            class_begin, class_end, pair_begin, pair_end, dF,
                                                            static_cast<double*>(ws), S(stream)));
}

}  // extern "C"

extern "C" {

// ---- the whole of class_statistics for rows resident on one device, in one call ----
size_t sqfa_class_statistics_workspace_bytes(int64_t n, int32_t n_dim, int32_t n_classes) {
  return class_statistics_ws(n, n_dim, n_classes, sqfa::ELEM_F32);
}

size_t sqfa_class_statistics_workspace_bytes_h(int64_t n, int32_t n_dim, int32_t n_classes, int32_t elem) {
  const int e = half_elem(__func__, elem);
  return e < 0 ? 0 : class_statistics_ws(n, n_dim, n_classes, e);
}

int sqfa_class_statistics(const float* X, int64_t ldx, const int64_t* labels, int64_t n, int32_t n_dim,
                          int32_t n_classes, int estimator, int ddof, float* means, float* cov, float* sm,
                          int64_t* counts, int64_t* offsets, int32_t* perm, void* ws, size_t ws_bytes,
                          sqfa_stream_t stream) {
  return class_statistics_impl(__func__, X, sqfa::ELEM_F32, ldx, labels, n, n_dim, n_classes, estimator, ddof, means,
                               cov, sm, counts, offsets, perm, ws, ws_bytes, stream);
}

int sqfa_class_statistics_h(const void* X, int64_t ldx, int32_t elem, const int64_t* labels, int64_t n, int32_t n_dim,
                            int32_t n_classes, int estimator, int ddof, float* means, float* cov, float* sm,
                            int64_t* counts, int64_t* offsets, int32_t* perm, void* ws, size_t ws_bytes,
                            sqfa_stream_t stream) {
  const int e = half_elem(__func__, elem);
  if (e < 0) return SQFA_E_INVALID;
  return class_statistics_impl(__func__, X, e, ldx, labels, n, n_dim, n_classes, estimator, ddof, means, cov, sm,
                               counts, offsets, perm, ws, ws_bytes, stream);
}

}  // extern "C"

extern "C" {

int64_t sqfa_lbfgs_max_n(void) { return sqfa::lbfgs_max_n(); }
int32_t sqfa_lbfgs_max_history(void) { return sqfa::lbfgs_max_history(); }

int sqfa_lbfgs_direction(const float* g, float* prev_g, float* d, float* S_, float* Y, float* ro, float* hdiag,
                         int32_t* meta, int64_t n, int32_t history, float t_prev, int first, float* param, float lr,
                         float tolerance_change, float* out_scalars, sqfa_stream_t stream) {
  if (g == nullptr || prev_g == nullptr || d == nullptr || S_ == nullptr || Y == nullptr || ro == nullptr ||
      hdiag == nullptr || meta == nullptr || out_scalars == nullptr || n <= 0 || history < 1)
    return fail_arg(__func__, "bad argument");
  if (n > sqfa::lbfgs_max_n() || history > sqfa::lbfgs_max_history())
    return fail_arg(__func__, "vector or history too large for the single-cluster kernel", SQFA_E_UNSUPPORTED);
  return wrap(__func__, sqfa::launch_lbfgs_direction(g, prev_g, d, S_, Y, ro, hdiag, meta, n, history, t_prev,
                                                     first ? 1 : 0, param, lr, tolerance_change, out_scalars,
                                                     S(stream)));
}

int64_t sqfa_lbfgs_max_n_f64(void) { return sqfa::lbfgs_max_n_f64(); }

int sqfa_lbfgs_direction_f64(const double* g, double* prev_g, double* d, double* S_, double* Y, double* ro,
                             double* hdiag, int32_t* meta, int64_t n, int32_t history, const double* scalars_host,
                             int first, double* param, double* out_scalars, sqfa_stream_t stream) {
  if (g == nullptr || prev_g == nullptr || d == nullptr || S_ == nullptr || Y == nullptr || ro == nullptr ||
      hdiag == nullptr || meta == nullptr || scalars_host == nullptr || out_scalars == nullptr || n <= 0 ||
      history < 1)
    return fail_arg(__func__, "bad argument");
  if (n > sqfa::lbfgs_max_n_f64() || history > sqfa::lbfgs_max_history())
    return fail_arg(__func__, "vector or history too large for the single-cluster kernel", SQFA_E_UNSUPPORTED);
  // {t_prev, lr, tolerance_change}: read here and passed by value, so the caller may reuse the memory at once
  const double t_prev = scalars_host[0], lr = scalars_host[1], tolerance_change = scalars_host[2];
  return wrap(__func__, sqfa::launch_lbfgs_direction_f64(g, prev_g, d, S_, Y, ro, hdiag, meta, n, history, t_prev,
                                                         first ? 1 : 0, param, lr, tolerance_change, out_scalars,
                                                         S(stream)));
}

}  // extern "C"

extern "C" {

// --------------------------------------------------------------------------------- float64 hot path 1
int sqfa_class_sums_f64(const double* X, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                        const double* shift, int64_t n, int32_t n_dim, int32_t n_classes, double* sums,
                        int accumulate, sqfa_stream_t stream) {
  if (n < 0 || n_dim <= 0 || n_classes < 0 || offsets == nullptr || sums == nullptr ||
      (n > 0 && (X == nullptr || perm == nullptr)) || ldx < n_dim)
    return fail_arg(__func__, "bad argument");
  return wrap(__func__, sqfa::launch_class_sums_f64(X, ldx, perm, offsets, shift, n_dim, n_classes, sums, accumulate,
                                                    S(stream)));
}

int sqfa_class_means_f64(const double* sums, const int64_t* counts, const double* shift, int32_t n_dim,
                         int32_t n_classes, double* means, sqfa_stream_t stream) {
  if (sums == nullptr || counts == nullptr || means == nullptr || n_dim <= 0 || n_classes < 0)
    return fail_arg(__func__, "bad argument");
  return wrap(__func__, sqfa::launch_class_means_f64(sums, counts, shift, n_dim, n_classes, means, S(stream)));
}

int sqfa_class_gram_f64(const double* X, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                        const double* shift, int64_t n, int32_t n_dim, int32_t n_classes, double* gram,
                        int accumulate, sqfa_stream_t stream) {
  if (n < 0 || n_dim <= 0 || n_classes < 0 || offsets == nullptr || gram == nullptr ||
      (n > 0 && (X == nullptr || perm == nullptr)) || ldx < n_dim || (accumulate & ~SQFA_GRAM_ACCUMULATE))
    return fail_arg(__func__, "bad argument");
  if (n_classes > 65535) return fail_arg(__func__, "n_classes must be <= 65535", SQFA_E_UNSUPPORTED);
  return wrap(__func__, sqfa::launch_class_gram_f64(X, ldx, perm, offsets, shift, n_dim, n_classes, gram, accumulate,
                                                    S(stream)));
}

int sqfa_stats_epilogue_f64(const double* gram, const double* means, const double* shift, const int64_t* counts,
                            int32_t n_dim, int32_t n_classes, int estimator, int ddof, double* cov, double* sm,
                            sqfa_stream_t stream) {
  if (gram == nullptr || means == nullptr || counts == nullptr || cov == nullptr || cov == gram || n_dim <= 0 ||
      n_classes < 0 || (estimator != SQFA_EST_EMPIRICAL && estimator != SQFA_EST_OAS) || (ddof != 0 && ddof != 1))
    return fail_arg(__func__, "bad argument");
  return wrap(__func__, sqfa::launch_stats_epilogue_f64(gram, means, shift, counts, n_dim, n_classes, estimator, ddof,
                                                        cov, sm, S(stream)));
}

}  // extern "C"

extern "C" {

// ------------------------------------------------------------- plug-in distances between Gaussians
size_t sqfa_gauss_pair_workspace_bytes(int32_t n_a, int32_t n_b, int32_t k, int32_t want_grad) {
  if (n_a <= 0 || n_b <= 0 || k <= 0) return 1024;
  return sqfa::gauss_workspace_floats(n_a, n_b, k, want_grad) * sizeof(float);
}

int sqfa_gauss_pair_distances(const float* mu_a, const float* sigma_a, const float* mu_b, const float* sigma_b,
                              int32_t n_a, int32_t n_b, int32_t k, int32_t mode, const float* gD, float* dist_out,
                              float* g_sigma_a, float* g_mu_a, float* g_sigma_b, float* g_mu_b, void* ws,
                              size_t ws_bytes, int32_t* flag, sqfa_stream_t stream) {
  const bool grad = gD != nullptr;
  if (mu_a == nullptr || sigma_a == nullptr || mu_b == nullptr || sigma_b == nullptr || n_a < 0 || n_b < 0 || k <= 0 ||
      (mode != SQFA_GAUSS_MAHALANOBIS_SQ && mode != SQFA_GAUSS_BHATTACHARYYA) || ws == nullptr ||
      (!grad && dist_out == nullptr) ||
      (grad && (g_sigma_a == nullptr || g_mu_a == nullptr || g_sigma_b == nullptr || g_mu_b == nullptr)))
    return fail_arg(__func__, "bad argument");
  if (k > SQFA_MAX_M) return fail_arg(__func__, "k exceeds SQFA_MAX_M", SQFA_E_UNSUPPORTED);
  if (ws_bytes < sqfa_gauss_pair_workspace_bytes(n_a, n_b, k, grad ? 1 : 0))
    return fail_arg(__func__, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(__func__, sqfa::launch_gauss_pairs(mu_a, sigma_a, mu_b, sigma_b, n_a, n_b, k, mode, gD, dist_out,
                                                 g_sigma_a, g_mu_a, g_sigma_b, g_mu_b, static_cast<float*>(ws), flag,
                                                 S(stream)));
}

}  // extern "C"

// ------------------------------------------------------ shared bodies of the float32 and *_h entry points
namespace {

int class_sums_impl(const char* fn, const void* X, int elem, int64_t ldx, const int32_t* perm,
                    const int64_t* offsets, const float* shift, int64_t n, int32_t n_dim, int32_t n_classes,
                    float* sums, int accumulate, void* ws, size_t ws_bytes, sqfa_stream_t stream) {
  if (n < 0 || n_dim <= 0 || n_classes < 0 || offsets == nullptr || sums == nullptr || ws == nullptr ||
      (n > 0 && (X == nullptr || perm == nullptr)) || ldx < n_dim)
    return fail_arg(fn, "bad argument");
  const int sms = sm_count_cached();
  const int ns = sqfa::class_sums_splits(n, n_classes, n_dim, sms > 0 ? sms : 148);
  if (ws_bytes < (size_t)ns * (size_t)n_classes * (size_t)n_dim * sizeof(float))
    return fail_arg(fn, "workspace too small", SQFA_E_WORKSPACE);
  return wrap(fn, sqfa::launch_class_sums(X, elem, ldx, perm, offsets, shift, n, n_dim, n_classes, sums, accumulate,
                                          static_cast<float*>(ws), ns, S(stream)));
}

size_t class_gram_ws(int64_t n, int32_t n_dim, int32_t n_classes, int elem) {
  if (n_classes <= 0 || n_dim <= 0) return 256;
  const int sms = sm_count_cached();
  return sqfa::gram_workspace_bytes(
      n_classes, n_dim,
      sqfa::gram_ksplit(n < 0 ? 0 : n, n_classes, n_dim, sms > 0 ? sms : 148, sqfa::elem_bytes(elem)));
}

int class_gram_impl(const char* fn, const void* X, int elem, int64_t ldx, const int32_t* perm,
                    const int64_t* offsets, const float* shift, int64_t n, int32_t n_dim, int32_t n_classes,
                    float* gram, int accumulate, int chain_rows, int32_t* done, int32_t n_groups,
                    int32_t first_class, int32_t reserve_sms, void* ws, size_t ws_bytes, sqfa_stream_t stream,
                    float* sum_partials) {
  if (n_dim <= 0 || n_classes < 0 || offsets == nullptr || gram == nullptr || ws == nullptr || ldx < n_dim ||
      X == nullptr || perm == nullptr || (accumulate & ~(SQFA_GRAM_ACCUMULATE | SQFA_GRAM_PACKED)) ||
      (done != nullptr && (n_groups <= 0 || n_groups > 65536)) || reserve_sms < 0 || first_class < 0 ||
      (first_class > 0 && (done == nullptr || first_class >= n_classes)))
    return fail_arg(fn, "bad argument");
  if (n < 0) return fail_arg(fn, "bad argument");
  if (ws_bytes < class_gram_ws(n, n_dim, n_classes, elem)) return fail_arg(fn, "workspace too small", SQFA_E_WORKSPACE);
  if ((int64_t)n_classes * sqfa::gram_tiles_per_class(n_dim, nullptr) > (1ll << 30) / 4096)
    return fail_arg(fn, "too many (class, tile) jobs", SQFA_E_UNSUPPORTED);
  const int sms = sm_count_cached();
  if (sms <= 0) return fail_arg(fn, "no CUDA device");
  return wrap(fn, sqfa::launch_class_gram(X, elem, ldx, perm, offsets, shift, n, n_dim, n_classes, gram,
                                          accumulate & SQFA_GRAM_ACCUMULATE, accumulate & SQFA_GRAM_PACKED, chain_rows,
                                          done, n_groups, first_class, reserve_sms, ws, sms, S(stream), sum_partials));
}

int class_pilot_shift_impl(const char* fn, const void* X, int elem, int64_t ldx, const int32_t* perm,
                           const int64_t* offsets, int32_t n_dim, int32_t n_classes, float* shift, sqfa_stream_t stream) {
  if (X == nullptr || perm == nullptr || offsets == nullptr || shift == nullptr || n_dim <= 0 || n_classes < 0 ||
      ldx < n_dim)
    return fail_arg(fn, "bad argument");
  return wrap(fn, sqfa::launch_class_pilot_shift(X, elem, ldx, perm, offsets, n_dim, n_classes, shift, S(stream)));
}

// class-sum partials per class that sqfa_class_gram_sums writes: 4 sample quads x the launch's K parts; 0 when
// the Gram is split into more than kOnePassMaxKsplit K parts (classes of ~10^5 rows, the c5 shard): the partials
// would outgrow the workspace the two-pass sums use, and those shapes keep the two passes
constexpr int kOnePassMaxKsplit = 16;
int32_t class_gram_sum_splits(int64_t n, int32_t n_dim, int32_t n_classes, int elem) {
  if (n_dim <= 0 || n_classes <= 0) return 0;
  const int sms = sm_count_cached();
  const int ks = sqfa::gram_ksplit_launch(n < 0 ? 0 : n, n_classes, n_dim, 0, sms > 0 ? sms : 148, sqfa::elem_bytes(elem));
  return ks <= kOnePassMaxKsplit ? 4 * ks : 0;
}

int64_t class_gram_signals(int64_t n, int32_t n_dim, int32_t n_classes, int32_t n_groups, int32_t group, int elem) {
  if (n_dim <= 0 || n_classes <= 0 || n_groups <= 0 || n_groups > 65536 || group < 0 || group >= n_groups) return 0;
  const int sms = sm_count_cached();
  const int64_t ks = sqfa::gram_ksplit(n < 0 ? 0 : n, n_classes, n_dim, sms > 0 ? sms : 148, sqfa::elem_bytes(elem));
  int64_t classes = 0;  // classes c with c * n_groups / n_classes == group
  for (int c = 0; c < n_classes; ++c) classes += ((int64_t)c * n_groups) / n_classes == group ? 1 : 0;
  return classes * sqfa::gram_tiles_per_class(n_dim, nullptr) * ks * 8;  // 2 CTAs x 4 epilogue warps per job
}

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }
struct StatsWs { size_t bucket, sums_ws, sums, gram, epi, total; };
inline StatsWs stats_ws(int64_t n, int32_t D, int32_t C, int elem) {
  StatsWs w;
  w.bucket = align256(sqfa_bucket_workspace_bytes(n, C));
  // the one-pass path keeps the pilot shift and the Gram's class-sum partials where the two-pass sums kept theirs
  const size_t splits = (size_t)class_gram_sum_splits(n, D, C, elem);
  const size_t one_pass = splits == 0 ? 0
                                      : align256((size_t)C * (size_t)D * sizeof(float)) +
                                            splits * (size_t)C * (size_t)D * sizeof(float);
  const size_t two_pass = sqfa_class_sums_workspace_bytes(n, D, C);
  w.sums_ws = align256(one_pass > two_pass ? one_pass : two_pass);
  w.sums = align256((size_t)(C > 0 ? C : 1) * (size_t)(D > 0 ? D : 1) * sizeof(float));
  w.gram = align256(class_gram_ws(n, D, C, elem));
  w.epi = align256(sqfa_stats_epilogue_workspace_bytes(C));
  w.total = w.bucket + w.sums_ws + w.sums + w.gram + w.epi;
  return w;
}

size_t class_statistics_ws(int64_t n, int32_t n_dim, int32_t n_classes, int elem) {
  return stats_ws(n < 0 ? 0 : n, n_dim, n_classes, elem).total;
}

int class_statistics_impl(const char* fn, const void* X, int elem, int64_t ldx, const int64_t* labels, int64_t n,
                          int32_t n_dim, int32_t n_classes, int estimator, int ddof, float* means, float* cov,
                          float* sm, int64_t* counts, int64_t* offsets, int32_t* perm, void* ws, size_t ws_bytes,
                          sqfa_stream_t stream) {
  if (X == nullptr || labels == nullptr || means == nullptr || cov == nullptr || counts == nullptr ||
      offsets == nullptr || perm == nullptr || ws == nullptr || n <= 0 || n_dim <= 0 || n_classes <= 0)
    return fail_arg(fn, "bad argument");
  const StatsWs w = stats_ws(n, n_dim, n_classes, elem);
  if (ws_bytes < w.total) return fail_arg(fn, "workspace too small", SQFA_E_WORKSPACE);
  uint8_t* p = static_cast<uint8_t*>(ws);
  void* ws_bucket = p;
  float* shift = reinterpret_cast<float*>(p + w.bucket);
  float* partials = reinterpret_cast<float*>(p + w.bucket + align256((size_t)n_classes * (size_t)n_dim * sizeof(float)));
  float* sums = reinterpret_cast<float*>(p + w.bucket + w.sums_ws);
  void* ws_gram = p + w.bucket + w.sums_ws + w.sums;
  void* ws_epi = p + w.bucket + w.sums_ws + w.sums + w.gram;
  int rc = sqfa_bucket_labels(labels, n, n_classes, counts, offsets, perm, ws_bucket, w.bucket, stream);
  if (rc) return rc;
  // One pass over X: the Gram centres on a pilot shift s (the first rows of each class) and its diagonal
  // tiles write the class sums of x - s on the way; mean = s + sums / n, and the epilogue takes n d d^T,
  // d = mean - s, off the Gram. Failures name the step, as the step's own entry point would.
  const bool f32 = elem == sqfa::ELEM_F32;
  const int32_t splits = class_gram_sum_splits(n, n_dim, n_classes, elem);
  if (splits == 0) {  // deep K split: sums, means, then the Gram centred on the means
    rc = class_sums_impl(f32 ? "sqfa_class_sums" : "sqfa_class_sums_h", X, elem, ldx, perm, offsets, nullptr, n, n_dim,
                         n_classes, sums, 0, shift, w.sums_ws, stream);
    if (rc) return rc;
    rc = sqfa_class_means(sums, counts, nullptr, n_dim, n_classes, means, stream);
    if (rc) return rc;
    rc = class_gram_impl(f32 ? "sqfa_class_gram" : "sqfa_class_gram_h", X, elem, ldx, perm, offsets, means, n, n_dim,
                         n_classes, cov, 0, 0, nullptr, 0, 0, 0, ws_gram, w.gram, stream);
    if (rc) return rc;
    return sqfa_stats_epilogue(cov, means, nullptr, counts, n_dim, n_classes, estimator, ddof, cov, sm, ws_epi, w.epi,
                               stream);
  }
  rc = class_pilot_shift_impl(f32 ? "sqfa_class_pilot_shift" : "sqfa_class_pilot_shift_h", X, elem, ldx, perm,
                              offsets, n_dim, n_classes, shift, stream);
  if (rc) return rc;
  rc = class_gram_impl(f32 ? "sqfa_class_gram_sums" : "sqfa_class_gram_sums_h", X, elem, ldx, perm, offsets, shift, n,
                       n_dim, n_classes, cov, 0, 0, nullptr, 0, 0, 0, ws_gram, w.gram, stream, partials);
  if (rc) return rc;
  rc = sqfa_class_means_from_partials(partials, splits, counts, shift, n_dim, n_classes, sums, means, stream);
  if (rc) return rc;
  return sqfa_stats_epilogue(cov, means, sums, counts, n_dim, n_classes, estimator | SQFA_EST_CENTRED_SUMS, ddof, cov,
                             sm, ws_epi, w.epi, stream);
}

}  // namespace
