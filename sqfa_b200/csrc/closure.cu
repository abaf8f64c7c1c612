// The whole closure body of the SQFA fitting loop as ONE native call:
//   loss = -mean_{i>j} d(E_i, E_j),  E_c = embed(F S_c F^T + noise I [, F m_c]),  grad = dloss/d(filters)
// (reference: /root/reference/src/sqfa/_optim.py:90-96 -> model.py:190-220 / 508-546 ->
//  distances.py -> linalg.py and the autograd backward of all of it, including the filter
//  constraint constraints.py:37).
// It sequences the kernels of project.cu and pairs.cu on the caller's stream inside a caller-provided
// workspace -- 8 kernel launches (and one 8-byte memset of the flags), no atomics on floating-point sums:
//   constraint_fwd          F = W / |W|                                  (sphere constraint only)
//   project_stream          row-split partials of T_c = F S_c            (the one pass over C D^2 floats)
//   project_finish          T_c, per-chunk partials of Psi_c = T_c F^T and mu'_c = F m_c
//   class_prepare           Psi_c, mu'_c, E_c, factorisation W_c         (one warp per class)
//   pair kernel             distances + per-tile partial dLoss/dE        (one warp per tile of pairs)
//   pair_reduce             dLoss/dE_c in fixed order -> embedding adjoint (gPsi, gMu); loss
//   project_bwd             class-split partials of dLoss/dF
//   closure_finish          dLoss/dF, constraint adjoint -> grad, max |grad|
// Log-Euclidean adds le_grad + le_factor_bwd + embed_bwd between the pair kernel and project_bwd; the
// Gaussian Wasserstein distance projects the means too (no embedding) and adds le_grad for their gradient.
// The mean-covariance distances (Mahalanobis, Bhattacharyya, Hellinger) project the means and replace
// class_prepare / pair kernel / pair_reduce with the class, pair and reduce stages of gauss.cu.
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/sqfa_b200.h"
#include "sqfa_internal.h"

namespace sqfa {

namespace {

struct ClosureLayout {
  size_t F, inv_norm, T, Mu, E, W, logdet, sinv, gE, gLog, gPsi, gMu, red_out, flag, proj, psipart, mupart, pair,
      total;
};

ClosureLayout closure_layout(int C, int D, int k, int dist, int64_t pair_begin, int64_t pair_end) {
  const int base = dist & 15;
  const int m = (base == SQFA_DIST_FISHER_RAO_LB) ? k + 1 : k;
  const bool le = base == SQFA_DIST_LOG_EUCLIDEAN;
  const bool gauss = is_gauss_closure(dist);  // E holds Psi_c; no factorisation W
  const bool ld = gauss_closure_needs_logdet(dist);
  ClosureLayout L;
  size_t o = 0;
  L.F = o;        o += al<float>((size_t)k * D);
  L.inv_norm = o; o += al<float>(k);
  L.T = o;        o += al<float>((size_t)C * k * D);
  L.Mu = o;       o += al<float>((size_t)C * k);
  L.E = o;        o += al<float>((size_t)C * m * m);
  L.W = o;        o += gauss ? 0 : al<float>((size_t)C * class_factor_floats(m, dist));
  L.logdet = o;   o += ld ? al<float>(C) : 0;
  L.sinv = o;     o += ld ? al<float>((size_t)C * k * k) : 0;
  L.gE = o;       o += le ? al<float>((size_t)C * m * m) : 0;
  L.gLog = o;     o += le ? al<float>((size_t)C * m * m) : 0;
  L.gPsi = o;     o += al<float>((size_t)C * k * k);
  L.gMu = o;      o += al<float>((size_t)C * k);
  L.red_out = o;  o += al<float>(16);  // {loss, #non-finite, -} of a rank's pairs: [gPsi | gMu | red_out] is one exchange span
  L.flag = o;     o += al<float>(16);
  L.proj = o;     o += al<float>(project_workspace_bytes(C, D, k) / sizeof(float) + 1);
  L.psipart = o;  o += project_psipart_floats(C, D, k);
  L.mupart = o;   o += project_mupart_floats(C, D, k);
  L.pair = o;     o += al<float>(gauss ? gauss_closure_workspace_elems(C, k, pair_begin, pair_end)
                            : pair_workspace(C, C, m, dist, 1, pair_begin, pair_end).total_floats);
  L.total = o;
  return L;
}

}  // namespace

size_t fused_loss_workspace_bytes(int C, int D, int k, int dist, int64_t pair_begin, int64_t pair_end) {
  return closure_layout(C, D, k, dist, pair_begin, pair_end).total * sizeof(float);
}

// filters: the constrained filters F (constraint < 0), or the raw parameter (constraint 0 = none,
// 1 = sphere). grad: d out[0] / d filters.  out: {loss, #non-finite distances, max |grad|}; out_host (optional):
// the same three numbers in mapped pinned host memory, written by the last kernel.
cudaError_t launch_fused_loss(const float* S, const float* M, const float* filters, int C, int D, int k, float noise,
                              int dist, int constraint, int n_fixed, int64_t pair_begin, int64_t pair_end, float* out,
                              float* out_host, float* grad, float* ws, cudaStream_t st) {
  const int base = dist & 15;
  const bool fr = base == SQFA_DIST_FISHER_RAO_LB;
  const bool le = base == SQFA_DIST_LOG_EUCLIDEAN;
  const bool gauss = is_gauss_closure(dist);
  const bool means = fr || base == SQFA_DIST_WASSERSTEIN_GAUSSIAN || gauss;  // this distance uses the class means
  const int m = fr ? k + 1 : k;
  const ClosureLayout L = closure_layout(C, D, k, dist, pair_begin, pair_end);
  float* Fbuf = ws + L.F;
  float* inv_norm = ws + L.inv_norm;
  float* T = ws + L.T;
  float* Mu = ws + L.Mu;
  float* E = ws + L.E;
  float* W = ws + L.W;
  float* gE = ws + L.gE;
  float* gLog = ws + L.gLog;
  float* gPsi = ws + L.gPsi;
  float* gMu = ws + L.gMu;
  int32_t* flag = reinterpret_cast<int32_t*>(ws + L.flag);
  float* proj = ws + L.proj;
  float* PsiPart = ws + L.psipart;
  float* MuPart = ws + L.mupart;
  float* pairws = ws + L.pair;
  const float* Mfr = means ? M : nullptr;
  const int64_t P = (int64_t)C * (C - 1) / 2;
  const float weight = -1.0f / (float)(P > 0 ? P : 1);
  const int sphere = constraint == 1 ? 1 : 0;

  cudaError_t e;
  const float* F = filters;
  if (sphere) {
    if ((e = launch_constraint_fwd(filters, D, k, Fbuf, inv_norm, st)) != cudaSuccess) return e;
    F = Fbuf;
  }
  if ((e = launch_project_partials(S, Mfr, F, C, D, k, T, proj, PsiPart, means ? MuPart : nullptr, st)) != cudaSuccess)
    return e;
  if (gauss) {
    if ((e = launch_gauss_closure_class(PsiPart, MuPart, project_nchunk(D), noise, C, k, dist, E, Mu, ws + L.logdet,
                                        ws + L.sinv, flag, st)) != cudaSuccess)
      return e;
    if ((e = launch_gauss_closure_pairs(E, Mu, ws + L.logdet, ws + L.sinv, C, k, dist, pair_begin, pair_end, weight, out,
                                        gPsi, gMu, pairws, st)) != cudaSuccess)
      return e;
  } else {
    if ((e = launch_class_prepare(PsiPart, means ? MuPart : nullptr, project_nchunk(D), noise, C, k, dist, Mu, E, W,
                                  flag, st)) != cudaSuccess)
      return e;
    if ((e = launch_pair_closure(W, C, m, dist, pair_begin, pair_end, weight, Mu, k, out, gPsi, gMu, gLog, pairws,
                                 st)) != cudaSuccess)
      return e;
  }
  if (le) {
    if ((e = cudaMemsetAsync(gE, 0, (size_t)C * m * m * sizeof(float), st)) != cudaSuccess) return e;
    if ((e = launch_class_factor_bwd(W, gLog, C, m, dist, gE, st)) != cudaSuccess) return e;
    if ((e = launch_embed_bwd(gE, Mu, C, k, 0, gPsi, gMu, st)) != cudaSuccess) return e;
  }
  return launch_project_bwd_constrained(gPsi, means ? gMu : nullptr, T, Mfr, C, D, k, F, inv_norm, sphere, n_fixed, grad,
                                        out, out_host, reinterpret_cast<unsigned int*>(flag + 1), proj, st);
}

// ------------------------------------------------------------------------------------------------
// The same closure with the CLASSES and the PAIRS sharded over ranks (pair list of a large C, SURVEY.md
// section 8(e) row 2). Three phases; between them the caller all-reduces one small span of the workspace:
//   phase 0  projection of the caller's classes [c0, c1): T_c and their slices of the span
//            [PsiPart | MuPart] (zeroed elsewhere, so the sum over ranks assembles all classes)
//   phase 1  embedding + factorisation of ALL classes (C small problems, replicated), the pair kernel on the
//            caller's pairs, per-class reduction + embedding adjoint -> partial (gPsi, gMu) of all classes
//            and {weight * sum d, #non-finite} in the span [gPsi | gMu | red_out]
//   phase 2  projection adjoint over the caller's classes -> its share of dLoss/dF (summed by the caller)
// Nothing of size C D^2 is read twice across the ranks: the projection (the HBM-bound part) and its
// adjoint shard with the classes, the pair stage with the pairs.
void fused_loss_exchange_span(int C, int D, int k, int dist, int64_t pair_begin, int64_t pair_end, int which,
                              size_t* offset_bytes, size_t* bytes) {
  const ClosureLayout L = closure_layout(C, D, k, dist, pair_begin, pair_end);
  if (which == 0) {
    *offset_bytes = L.psipart * sizeof(float);
    *bytes = (L.pair - L.psipart) * sizeof(float);  // psipart and mupart are adjacent, pair follows
  } else {
    *offset_bytes = L.gPsi * sizeof(float);
    *bytes = (L.flag - L.gPsi) * sizeof(float);  // gPsi | gMu | red_out
  }
}

cudaError_t launch_fused_loss_sharded(int phase, const float* S, const float* M, const float* F, int C, int D, int k,
                                      float noise, int dist, int c0, int c1, int64_t pair_begin, int64_t pair_end,
                                      float* dF, float* ws, cudaStream_t st) {
  const int base = dist & 15;
  const bool fr = base == SQFA_DIST_FISHER_RAO_LB;
  const bool gauss = is_gauss_closure(dist);
  const bool means = fr || base == SQFA_DIST_WASSERSTEIN_GAUSSIAN || gauss;
  if (base == SQFA_DIST_LOG_EUCLIDEAN) return cudaErrorNotSupported;
  const int m = fr ? k + 1 : k;
  const ClosureLayout L = closure_layout(C, D, k, dist, pair_begin, pair_end);
  float* T = ws + L.T;
  float* Mu = ws + L.Mu;
  float* gPsi = ws + L.gPsi;
  float* gMu = ws + L.gMu;
  float* PsiPart = ws + L.psipart;
  float* MuPart = ws + L.mupart;
  float* proj = ws + L.proj;
  const float* Mfr = means ? M : nullptr;
  const int nchunk = project_nchunk(D);
  const int n_own = c1 > c0 ? c1 - c0 : 0;
  cudaError_t e;
  if (phase == 0) {
    if ((e = cudaMemsetAsync(PsiPart, 0, (L.pair - L.psipart) * sizeof(float), st)) != cudaSuccess) return e;
    if (n_own == 0) return cudaSuccess;
    return launch_project_partials(S + (size_t)c0 * D * D, means ? M + (size_t)c0 * D : nullptr, F, n_own, D, k,
                                   T + (size_t)c0 * k * D, proj, PsiPart + (size_t)c0 * nchunk * k * k,
                                   means ? MuPart + (size_t)c0 * nchunk * k : nullptr, st);
  }
  if (phase == 1) {
    const int64_t P = (int64_t)C * (C - 1) / 2;
    const float weight = -1.0f / (float)(P > 0 ? P : 1);
    if (gauss) {
      if ((e = launch_gauss_closure_class(PsiPart, MuPart, nchunk, noise, C, k, dist, ws + L.E, Mu, ws + L.logdet,
                                          ws + L.sinv, reinterpret_cast<int32_t*>(ws + L.flag), st)) != cudaSuccess)
        return e;
      return launch_gauss_closure_pairs(ws + L.E, Mu, ws + L.logdet, ws + L.sinv, C, k, dist, pair_begin, pair_end,
                                        weight, ws + L.red_out, gPsi, gMu, ws + L.pair, st);
    }
    if ((e = launch_class_prepare(PsiPart, means ? MuPart : nullptr, nchunk, noise, C, k, dist, Mu, ws + L.E, ws + L.W,
                                  reinterpret_cast<int32_t*>(ws + L.flag), st)) != cudaSuccess)
      return e;
    return launch_pair_closure(ws + L.W, C, m, dist, pair_begin, pair_end, weight, Mu, k, ws + L.red_out, gPsi, gMu,
                               nullptr, ws + L.pair, st);
  }
  // phase 2: (gPsi, gMu) are now the sums over all pairs
  return launch_project_bwd(gPsi + (size_t)c0 * k * k, means ? gMu + (size_t)c0 * k : nullptr, T + (size_t)c0 * k * D,
                            Mfr != nullptr ? Mfr + (size_t)c0 * D : nullptr, n_own, D, k, dF, proj, st);
}

}  // namespace sqfa
