// Pairwise distances between Gaussians that use the MEAN covariance of the pair -- the reference's other
// `distance_fun` plug-ins (/root/reference/src/sqfa/distances.py:240-432, SURVEY.md section 8(f) row 4):
//   mahalanobis_sq(a, b) = d^T M^-1 d,          d = mu_a - mu_b,  M = (Sigma_a + Sigma_b) / 2      (:283-330)
//   bhattacharyya(a, b)  = maha / 8 + (logdet M - (logdet Sigma_a + logdet Sigma_b) / 2) / 2      (:240-280)
// (mahalanobis, hellinger and fisher_rao_same_cov are scalar maps of these two, applied on the host side).
// The reference materialises (n_a, n_b, k, k) mean covariances and calls torch.linalg.inv / logdet on all
// of them; here one warp owns one pair: Cholesky M = L L^T in shared memory, z = L^-1 d, maha = |z|^2,
// logdet M = 2 sum log L_jj. The backward pass is analytic, with u = M^-1 d:
//   d maha / d mu_a = 2 u,  d maha / d mu_b = -2 u,  d maha / d Sigma_a = d maha / d Sigma_b = -u u^T / 2
//   d logdet M / d Sigma_a = M^-1 / 2,               d logdet Sigma_a / d Sigma_a = Sigma_a^-1
// Per-pair gradient partials are stored and summed per class in a fixed order (no float atomics).
// The second half of this file is the fitting closure of these distances (SQFA_DIST_MAHALANOBIS / BHATTACHARYYA /
// HELLINGER): strict lower triangle only, the scalar map inside, tile partials instead of per-pair ones.
#include <cfloat>
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/sqfa_b200.h"
#include "sqfa_internal.h"
#include "pair_tiles.cuh"

namespace sqfa {

namespace {

constexpr int GP_WARPS = 4;

__device__ __forceinline__ float gp_warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// in-place lower Cholesky of the k x k matrix M (row stride ld), one warp; returns logdet, sets ok. T = float, double.
template <typename T>
__device__ T gp_cholesky(T* M, int k, int ld, int lane, bool& ok) {
  T logdet = T(0);
  for (int j = 0; j < k; ++j) {
    T d = M[j * ld + j];
    for (int q = 0; q < j; ++q) d -= M[j * ld + q] * M[j * ld + q];
    if (!(d > T(0)) || !isfinite(d)) ok = false;
    const T ljj = sqrt(d);
    logdet += T(2) * log(ljj);
    __syncwarp();
    for (int i = j + 1 + lane; i < k; i += 32) {
      T v = M[i * ld + j];
      for (int q = 0; q < j; ++q) v -= M[i * ld + q] * M[j * ld + q];
      M[i * ld + j] = v / ljj;
    }
    if (lane == 0) M[j * ld + j] = ljj;
    __syncwarp();
  }
  return logdet;
}

// Linv (row stride ld) = L^-1 for lower triangular L, one column per lane
template <typename T>
__device__ void gp_tri_inverse(const T* L, T* Li, int k, int ld, int lane) {
  for (int c = lane; c < k; c += 32) {
    for (int i = 0; i < k; ++i) {
      T s = (i == c) ? T(1) : T(0);
      for (int q = c; q < i; ++q) s -= L[i * ld + q] * Li[q * ld + c];
      Li[i * ld + c] = (i < c) ? T(0) : s / L[i * ld + i];
    }
  }
  __syncwarp();
}

// logdet of the k x k SPD matrix staged in L (row stride ld) and, if Sinv_c != NULL, its inverse L^-T L^-1;
// one warp, Li is scratch. A failed Cholesky sets *flag. In float32 the logdet is left as the factorisation made
// it (NaN, or +-inf for a zero or infinite pivot); in float64 it is NaN, so every distance of the class is NaN.
template <typename T>
__device__ __forceinline__ void gp_logdet_inverse(T* L, T* Li, int k, int ld, int lane, T* logdet_c, T* Sinv_c,
                                                  int32_t* flag) {
  bool ok = true;
  const T ldv = gp_cholesky(L, k, ld, lane, ok);
  if (!ok && lane == 0) atomicOr(flag, 1);
  if (lane == 0) *logdet_c = (ok || sizeof(T) == sizeof(float)) ? ldv : T(NAN);
  if (Sinv_c != nullptr) {
    gp_tri_inverse(L, Li, k, ld, lane);
    for (int idx = lane; idx < k * k; idx += 32) {  // Sigma^-1 = L^-T L^-1
      const int r = idx / k, s = idx % k;
      T a = T(0);
      for (int q = (r > s ? r : s); q < k; ++q) a += Li[q * ld + r] * Li[q * ld + s];
      Sinv_c[idx] = a;
    }
  }
}

// per class: logdet Sigma_c and (optionally) Sigma_c^-1; one warp per class
__global__ void __launch_bounds__(GP_WARPS * 32)
gauss_class_kernel(const float* __restrict__ Sigma, int C, int k, float* __restrict__ logdet,
                   float* __restrict__ Sinv, int32_t* __restrict__ flag) {
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * GP_WARPS + warp;
  if (c >= C) return;
  const int ld = k + 1;
  float* L = sm + (size_t)warp * 2 * k * ld;
  float* Li = L + k * ld;
  for (int idx = lane; idx < k * k; idx += 32) L[(idx / k) * ld + idx % k] = Sigma[(int64_t)c * k * k + idx];
  __syncwarp();
  gp_logdet_inverse(L, Li, k, ld, lane, logdet + c, Sinv != nullptr ? Sinv + (int64_t)c * k * k : nullptr, flag);
}

// One warp per pair (a, b), a in [a0, a1), b in [0, nB). mode 0: mahalanobis_sq, 1: bhattacharyya.
// Forward: dist_out[a][b]. Backward (gD != NULL): per-pair partials, PER = k*k + k floats each,
//   rowpart[(a - a0) * nB + b] = gD[a][b] * (d dist / d Sigma_a | d dist / d mu_a)   (without the Sigma_a^-1 term)
//   colpart[(a - a0) * nB + b] = gD[a][b] * (d dist / d Sigma_b | d dist / d mu_b)
__global__ void __launch_bounds__(GP_WARPS * 32)
gauss_pair_kernel(const float* __restrict__ muA, const float* __restrict__ SigA, const float* __restrict__ muB,
                  const float* __restrict__ SigB, const float* __restrict__ ldA, const float* __restrict__ ldB, int nA,
                  int nB, int k, int mode, int a0, int a1, const float* __restrict__ gD, float* __restrict__ dist_out,
                  float* __restrict__ rowpart, float* __restrict__ colpart, int32_t* __restrict__ flag) {
  extern __shared__ float sm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * GP_WARPS + warp;
  if (t >= (int64_t)(a1 - a0) * nB) return;
  const int a = a0 + (int)(t / nB), b = (int)(t % nB);
  const int ld = k + 1;
  float* L = sm + (size_t)warp * (2 * k * ld + 3 * k);
  float* Li = L + k * ld;
  float* dvec = Li + k * ld;
  float* z = dvec + k;
  float* u = z + k;
  for (int idx = lane; idx < k * k; idx += 32)
    L[(idx / k) * ld + idx % k] = 0.5f * (SigA[(int64_t)a * k * k + idx] + SigB[(int64_t)b * k * k + idx]);
  for (int i = lane; i < k; i += 32) dvec[i] = muA[(int64_t)a * k + i] - muB[(int64_t)b * k + i];
  __syncwarp();
  bool ok = true;
  const float logdetM = gp_cholesky(L, k, ld, lane, ok);
  if (!ok && lane == 0) atomicOr(flag, 1);
  // z = L^-1 d (forward substitution; the inner sums are warp reductions)
  for (int j = 0; j < k; ++j) {
    float s = 0.f;
    for (int q = lane; q < j; q += 32) s += L[j * ld + q] * z[q];
    s = gp_warp_sum(s);
    if (lane == 0) z[j] = (dvec[j] - s) / L[j * ld + j];
    __syncwarp();
  }
  float maha = 0.f;
  for (int i = lane; i < k; i += 32) maha += z[i] * z[i];
  maha = gp_warp_sum(maha);
  if (dist_out != nullptr && lane == 0) {
    const float v = mode == 0 ? maha : 0.125f * maha + 0.5f * (logdetM - 0.5f * (ldA[a] + ldB[b]));
    dist_out[(int64_t)a * nB + b] = v;
  }
  if (gD == nullptr) return;
  // u = L^-T z (back substitution)
  for (int j = k - 1; j >= 0; --j) {
    float s = 0.f;
    for (int q = j + 1 + lane; q < k; q += 32) s += L[q * ld + j] * u[q];
    s = gp_warp_sum(s);
    if (lane == 0) u[j] = (z[j] - s) / L[j * ld + j];
    __syncwarp();
  }
  const float g = gD[(int64_t)a * nB + b];
  const int per = k * k + k;
  float* rp = rowpart + t * per;
  float* cp = colpart + t * per;
  // coefficients: dist = cm * maha + cl * logdet M (+ class terms handled per class)
  const float cm = mode == 0 ? 1.f : 0.125f, cl = mode == 0 ? 0.f : 0.5f;
  if (cl != 0.f) gp_tri_inverse(L, Li, k, ld, lane);
  for (int idx = lane; idx < k * k; idx += 32) {
    const int r = idx / k, s = idx % k;
    float v = -0.5f * cm * u[r] * u[s];
    if (cl != 0.f) {  // + cl * M^-1 / 2
      float minv = 0.f;
      for (int q = (r > s ? r : s); q < k; ++q) minv += Li[q * ld + r] * Li[q * ld + s];
      v += 0.5f * cl * minv;
    }
    rp[idx] = g * v;
    cp[idx] = g * v;
  }
  for (int i = lane; i < k; i += 32) {
    const float v = 2.f * cm * u[i] * g;
    rp[k * k + i] = v;
    cp[k * k + i] = -v;
  }
}

// gSigA[a] (=|+=) sum_b rowpart[a][b] (+ class term), gSigB[b] += sum_a colpart[a][b] over the chunk
// [a0, a1); block = class, thread = element of (Sigma | mu). Fixed order.
__global__ void __launch_bounds__(256)
gauss_reduce_kernel(const float* __restrict__ rowpart, const float* __restrict__ colpart, const float* __restrict__ gD,
                    const float* __restrict__ SinvA, const float* __restrict__ SinvB, int nA, int nB, int k, int mode,
                    int a0, int a1, float* gSigA, float* gMuA, float* gSigB, float* gMuB) {
  const int per = k * k + k;
  const int c = blockIdx.x;
  for (int e = threadIdx.x; e < per; e += 256) {
    if (c >= a0 && c < a1) {  // row side: class c of set A, complete for this chunk
      float s = 0.f, gsum = 0.f;
      const float* p = rowpart + (int64_t)(c - a0) * nB * per + e;
      for (int b = 0; b < nB; ++b) {
        s += p[(int64_t)b * per];
        if (mode == 1 && e < k * k) gsum += gD[(int64_t)c * nB + b];
      }
      if (mode == 1 && e < k * k) s -= 0.25f * gsum * SinvA[(int64_t)c * k * k + e];  // -(logdet Sigma_a) / 4
      if (e < k * k) gSigA[(int64_t)c * k * k + e] = s;
      else gMuA[(int64_t)c * k + (e - k * k)] = s;
    }
    if (c < nB) {  // column side: class c of set B accumulates over the chunks
      float s = 0.f, gsum = 0.f;
      for (int a = a0; a < a1; ++a) {
        s += colpart[((int64_t)(a - a0) * nB + c) * per + e];
        if (mode == 1 && e < k * k) gsum += gD[(int64_t)a * nB + c];
      }
      if (mode == 1 && e < k * k) s -= 0.25f * gsum * SinvB[(int64_t)c * k * k + e];
      if (e < k * k) gSigB[(int64_t)c * k * k + e] += s;
      else gMuB[(int64_t)c * k + (e - k * k)] += s;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Fitting closure of the mean-covariance distances (SQFA_DIST_MAHALANOBIS / BHATTACHARYYA / HELLINGER):
//   class stage   one warp per class: Psi_c = sum of the projection's chunk partials + noise I, mu'_c;
//                 Bhattacharyya / Hellinger also logdet Psi_c and Psi_c^-1 (gp_cholesky, gp_tri_inverse)
//   pair stage    a warp owns an R x R tile of the strict lower triangle; a group of G lanes (G = k rounded
//                 up to a power of two, the matrix padded with the identity) owns one pair, so 32 / G pairs
//                 run side by side. Lane r holds row r of M = (Psi_i + Psi_j) / 2 in registers; an in-place
//                 Gauss-Jordan sweep with the pivot rows broadcast by shuffles leaves row r of M^-1. Its
//                 pivots are the squared Cholesky pivots: their logs sum to logdet M, and a pivot that is not
//                 positive and finite makes the distance NaN (as a failed Cholesky does). u = M^-1 d and
//                 x = d^T u follow with G more shuffles.
//   reduce        per class, the tile partials of its block row and block column in a fixed order
// Per pair, with g = weight * d'(x or B) and (c_m, c_l) = (1, 0) for Mahalanobis, (1/8, 1/2) otherwise:
//   dL/dPsi_i = dL/dPsi_j = g (-c_m / 2 u u^T + c_l / 2 M^-1),   dL/dmu'_i = -dL/dmu'_j = 2 c_m g u,
// and the class term -1/4 Psi_c^-1 sum_o g(c, o) of the logdet Psi_c in B is added once per class.
// The three kernels are templates on the scalar type: float for the float32 closure (closure.cu), double for
// the float64 one (closure64.cu, launch_gauss_closure_f64; DESIGN.md section 19).
// ------------------------------------------------------------------------------------------------
constexpr int GC_WARPS = 4;
constexpr double GC_EPS = 1e-6;  // distances.py:29 EPSILON

// elements of one class slot of a tile partial: [dL/dPsi (k*k) | dL/dmu' (k) | sum of g]
__host__ __device__ inline int gc_slot_floats(int k) { return k * k + k + 1; }

// The closure's kernels are templates on the scalar type T = float, double. The float64 closure reads the noise
// from one device double (a captured graph picks up a new value), the float32 closure takes it by value.
__device__ __forceinline__ float gc_noise(float noise) { return noise; }
__device__ __forceinline__ double gc_noise(const double* noise) { return *noise; }
__device__ __forceinline__ float gc_nan(float) { return __int_as_float(0x7fffffff); }
__device__ __forceinline__ double gc_nan(double) { return __longlong_as_double(0x7fffffffffffffffll); }
__device__ __forceinline__ float gc_max(float) { return FLT_MAX; }
__device__ __forceinline__ double gc_max(double) { return DBL_MAX; }

template <typename Real>
struct GaussClosureArgs {
  const Real* Psi;     // [C][k][k]
  const Real* Mu;      // [C][k]
  const Real* logdet;  // [C] (Bhattacharyya / Hellinger)
  int C, k, dist, Q;    // a tile row is processed as Q batches of 32 / G pairs
  int64_t pair_begin, pair_end;
  Real weight;
  PairTiles T;
  Real* rowpart;   // [ntiles][R][slot]
  Real* colpart;   // [ntiles][R][slot]
  Real* losspart;  // [ntiles][2] {sum of distances, non-finite count}
};

template <int G, typename T>
__device__ __forceinline__ T gc_group_sum(T v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename T, typename Noise>
__global__ void __launch_bounds__(GP_WARPS * 32)
gauss_closure_class_kernel(const T* __restrict__ PsiPart, const T* __restrict__ MuPart, int nchunk, Noise noise_arg,
                           int C, int k, int want_logdet, T* __restrict__ Psi, T* __restrict__ Mu,
                           T* __restrict__ logdet, T* __restrict__ Sinv, int32_t* __restrict__ flag) {
  extern __shared__ __align__(16) unsigned char gc_class_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * GP_WARPS + warp;
  if (c >= C) return;
  const T noise = gc_noise(noise_arg);
  const int ld = k + 1;
  T* L = reinterpret_cast<T*>(gc_class_smem) + (size_t)warp * 2 * k * ld;
  T* Li = L + k * ld;
  for (int r = lane; r < k; r += 32) {  // chunks added in order, as class_prepare does
    T a = T(0);
    for (int ch = 0; ch < nchunk; ++ch) a += MuPart[((int64_t)c * nchunk + ch) * k + r];
    Mu[(int64_t)c * k + r] = a;
  }
  for (int idx = lane; idx < k * k; idx += 32) {
    T v = T(0);
    for (int ch = 0; ch < nchunk; ++ch) v += PsiPart[((int64_t)c * nchunk + ch) * k * k + idx];
    if (idx / k == idx % k) v += noise;
    Psi[(int64_t)c * k * k + idx] = v;
    L[(idx / k) * ld + idx % k] = v;
  }
  if (!want_logdet) return;
  __syncwarp();
  gp_logdet_inverse(L, Li, k, ld, lane, logdet + c, Sinv + (int64_t)c * k * k, flag);
}

// Where a lane keeps its row-slot accumulator racc[G + 2]: registers, or for double at G = 32 (where M's row
// alone takes 64 registers) a [G + 2][32] block of shared memory after the warp's column accumulators, one
// column per lane like colacc.
template <typename T, int G>
struct GcRowAcc {
  static constexpr bool in_smem = sizeof(T) == 8 && G == 32;
};

template <typename T, int G>
__host__ __device__ inline int gc_pair_smem_elems(int Q) {
  return (Q + (GcRowAcc<T, G>::in_smem ? 1 : 0)) * (G + 2) * 32;
}

template <typename T, int G, bool SMEM>
struct GcRowSlot;
template <typename T, int G>
struct GcRowSlot<T, G, false> {
  T v[G + 2];
  __device__ __forceinline__ GcRowSlot(T*, int, int) {}
  __device__ __forceinline__ T& operator[](int e) { return v[e]; }
};
template <typename T, int G>
struct GcRowSlot<T, G, true> {
  T* p;
  __device__ __forceinline__ GcRowSlot(T* colacc, int Q, int lane) : p(colacc + Q * (G + 2) * 32 + lane) {}
  __device__ __forceinline__ T& operator[](int e) { return p[e * 32]; }
};

template <typename T, int G>
__global__ void __launch_bounds__(GC_WARPS * 32)
gauss_closure_pair_kernel(const GaussClosureArgs<T> A) {
  constexpr int NP = 32 / G;  // pairs side by side in a warp
  extern __shared__ __align__(16) unsigned char gc_pair_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * GC_WARPS + warp;
  if (t >= A.T.ntiles) return;
  const int grp = lane / G, r = lane % G;
  const int k = A.k, Q = A.Q, R = A.T.R, base = A.dist & 15;
  const int per = gc_slot_floats(k);
  const bool bhat = base != SQFA_DIST_MAHALANOBIS;
  const T cm = bhat ? T(0.125) : T(1), cl = bhat ? T(0.5) : T(0);
  // column-slot accumulators [Q][G + 2][32]: every lane owns its own column, so no synchronisation
  constexpr int QR = GcRowAcc<T, G>::in_smem ? 1 : 0;  // batches of column slots that hold the row slot
  T* colacc = reinterpret_cast<T*>(gc_pair_smem) + (size_t)warp * (Q + QR) * (G + 2) * 32;
  for (int e = 0; e < Q * (G + 2); ++e) colacc[e * 32 + lane] = T(0);
  int bi, bj;
  decode_tile(A.T, t, bi, bj);
  T dsum = T(0), nbad = T(0);
  for (int ii = 0; ii < R; ++ii) {
    const int i = bi * R + ii;
    GcRowSlot<T, G, GcRowAcc<T, G>::in_smem> racc(colacc, Q, lane);
#pragma unroll
    for (int e = 0; e < G + 2; ++e) racc[e] = T(0);
    for (int q = 0; q < Q; ++q) {
      const int j = bj * R + q * NP + grp;
      const bool valid = pair_in_launch(i, j, A.C, A.C, 1, A.pair_begin, A.pair_end);
      const bool live = valid && r < k;
      T Mr[G];
      const T* pi = A.Psi + ((int64_t)i * k + r) * k;
      const T* pj = A.Psi + ((int64_t)j * k + r) * k;
#pragma unroll
      for (int l = 0; l < G; ++l) Mr[l] = (live && l < k) ? T(0.5) * (pi[l] + pj[l]) : (l == r ? T(1) : T(0));
      const T dv = live ? A.Mu[(int64_t)i * k + r] - A.Mu[(int64_t)j * k + r] : T(0);
      // Gauss-Jordan: after step p the rows hold [M^-1 of the leading p x p block | eliminated rest]
      T mypiv = T(1);
#pragma unroll
      for (int p = 0; p < G; ++p) {
        const T piv = __shfl_sync(0xffffffffu, Mr[p], p, G);
        const T pinv = T(1) / piv;
        const T f = Mr[p];
        const bool prow = r == p;
        if (prow) mypiv = piv;
#pragma unroll
        for (int l = 0; l < G; ++l) {
          const T pl = __shfl_sync(0xffffffffu, Mr[l], p, G) * pinv;
          if (l == p) Mr[l] = prow ? pinv : -f * pinv;
          else Mr[l] = prow ? pl : fma(-f, pl, Mr[l]);
        }
      }
      T u = T(0);  // u_r = (M^-1 d)_r
#pragma unroll
      for (int l = 0; l < G; ++l) u = fma(Mr[l], __shfl_sync(0xffffffffu, dv, l, G), u);
      const T x = gc_group_sum<G>(dv * u);
      const bool pos = mypiv > T(0) && mypiv <= gc_max(T(0));
      const bool ok = gc_group_sum<G>(pos ? T(0) : T(1)) == T(0);
      T pre = x;
      if (bhat) {
        const T ldM = gc_group_sum<G>(log(mypiv));  // padded rows: log 1 = 0
        pre = valid ? T(0.125) * x + T(0.5) * (ldM - T(0.5) * (A.logdet[i] + A.logdet[j])) : T(0);
      }
      if (!ok) pre = gc_nan(T(0));
      T dval, dmap;  // distance and its derivative w.r.t. x (Mahalanobis) or B
      if (base == SQFA_DIST_HELLINGER) {
        const T e = exp(-pre);
        dval = sqrt(T(1) - e + T(GC_EPS));
        dmap = T(0.5) * e / dval;
      } else if (base == SQFA_DIST_MAHALANOBIS && !(A.dist & SQFA_DIST_SQUARED)) {
        dval = sqrt(pre + T(GC_EPS));
        dmap = T(0.5) / dval;
      } else {
        dval = pre;
        dmap = T(1);
      }
      const T g = valid ? A.weight * dmap : T(0);
      if (valid && r == 0) {
        dsum += dval;
        if (!isfinite(dval)) nbad += T(1);
      }
      const T gu = g * u;
      T* ca = colacc + q * (G + 2) * 32 + lane;
#pragma unroll
      for (int l = 0; l < G; ++l) {
        const T ul = __shfl_sync(0xffffffffu, u, l, G);
        const T v = fma(T(0.5) * cl * g, Mr[l], T(-0.5) * cm * gu * ul);
        racc[l] += v;
        ca[l * 32] += v;
      }
      racc[G] += T(2) * cm * gu;
      ca[G * 32] -= T(2) * cm * gu;
      racc[G + 1] += g;
      ca[(G + 1) * 32] += g;
    }
    // row slot ii: sum over the NP pairs side by side (butterfly: every group ends with the same bits)
#pragma unroll
    for (int e = 0; e < G + 2; ++e)
#pragma unroll
      for (int o = G; o < 32; o <<= 1) racc[e] += __shfl_xor_sync(0xffffffffu, racc[e], o);
    if (grp == 0 && r < k) {
      T* rp = A.rowpart + (t * R + ii) * per;
#pragma unroll
      for (int l = 0; l < G; ++l)
        if (l < k) rp[r * k + l] = racc[l];
      rp[k * k + r] = racc[G];
      if (r == 0) rp[k * k + k] = racc[G + 1];
    }
  }
  if (r < k) {
    for (int q = 0; q < Q; ++q) {
      T* cp = A.colpart + (t * R + q * NP + grp) * per;
      const T* ca = colacc + q * (G + 2) * 32 + lane;
      for (int l = 0; l < k; ++l) cp[r * k + l] = ca[l * 32];
      cp[k * k + r] = ca[G * 32];
      if (r == 0) cp[k * k + k] = ca[(G + 1) * 32];
    }
  }
  dsum = warp_sum(dsum);
  nbad = warp_sum(nbad);
  if (lane == 0) {
    A.losspart[2 * t] = dsum;
    A.losspart[2 * t + 1] = nbad;
  }
}

// Per class c (blocks 0 .. C - 1): the slot partials of the tiles of its block row (ascending block column)
// and block column (ascending block row) -> gPsi[c] (+ the logdet class term), gMu[c]. Block C: out =
// {weight * sum d, #non-finite, 0} from the loss partials. Fixed order throughout.
template <typename T>
__global__ void __launch_bounds__(1024)
gauss_closure_reduce_kernel(const PairTiles Tl, int C, int k, int dist, const T* __restrict__ rowpart,
                            const T* __restrict__ colpart, const T* __restrict__ losspart,
                            const T* __restrict__ Sinv, T weight, T* __restrict__ out,
                            T* __restrict__ gPsi, T* __restrict__ gMu) {
  extern __shared__ __align__(16) unsigned char gc_reduce_smem[];
  T* sg = reinterpret_cast<T*>(gc_reduce_smem);  // the reduced slot of this class
  const int c = blockIdx.x;
  if (c == C) {
    T sum, bad;
    reduce_loss_partials(losspart, Tl.ntiles, sum, bad);
    if (threadIdx.x == 0) {
      out[0] = weight * sum;
      out[1] = bad;
      out[2] = T(0);  // max |grad|, filled by closure_finish_kernel
    }
    return;
  }
  const int per = gc_slot_floats(k), R = Tl.R, slot = c % R, bc = c / R;
  const int64_t pstride = (int64_t)R * per;
  for (int e = threadIdx.x; e < per; e += blockDim.x) {
    T a = T(0), b = T(0);
    if (bc >= Tl.bi0 && bc <= Tl.bi1) {  // row side: tiles (bc, 0 .. bc)
      const T* p = rowpart + ((int64_t)bc * (bc + 1) / 2 - Tl.tile0) * pstride + (int64_t)slot * per + e;
#pragma unroll 4
      for (int bj = 0; bj <= bc; ++bj) a += p[bj * pstride];
    }
    const int i0 = max(Tl.bi0, bc);  // column side: tiles (i0 .. bi1, bc)
#pragma unroll 4
    for (int bi = i0; bi <= Tl.bi1; ++bi)
      b += colpart[((int64_t)bi * (bi + 1) / 2 + bc - Tl.tile0) * pstride + (int64_t)slot * per + e];
    sg[e] = a + b;
  }
  __syncthreads();
  const bool bhat = gauss_closure_needs_logdet(dist);
  const T gsum = sg[k * k + k];
  for (int e = threadIdx.x; e < k * k + k; e += blockDim.x) {
    if (e < k * k) gPsi[(int64_t)c * k * k + e] = bhat ? sg[e] - T(0.25) * gsum * Sinv[(int64_t)c * k * k + e] : sg[e];
    else gMu[(int64_t)c * k + e - k * k] = sg[e];
  }
}

}  // namespace

size_t gauss_workspace_floats(int nA, int nB, int k, int want_grad) {
  // [logdet A | logdet B | Sinv A | Sinv B | flag | row partials | column partials (chunk of rows of A)]
  size_t f = (size_t)nA + nB + 64;
  if (want_grad) {
    f += ((size_t)nA + nB) * k * k;
    const size_t per = (size_t)k * k + k;
    size_t rows = (size_t)(16u << 20) / (per * (nB > 0 ? nB : 1));  // partials of a chunk: <= 2 x 64 MB
    if (rows < 1) rows = 1;
    if (rows > (size_t)nA) rows = nA;
    f += 2 * rows * nB * per;
  }
  return f + 256;
}

cudaError_t launch_gauss_pairs(const float* muA, const float* SigA, const float* muB, const float* SigB, int nA,
                               int nB, int k, int mode, const float* gD, float* dist_out, float* gSigA, float* gMuA,
                               float* gSigB, float* gMuB, float* ws, int32_t* flag_out, cudaStream_t st) {
  if (nA <= 0 || nB <= 0) return cudaSuccess;
  const bool grad = gD != nullptr;
  float* ldA = ws;
  float* ldB = ldA + nA;
  int32_t* flag = reinterpret_cast<int32_t*>(ldB + nB);
  float* SinvA = ldB + nB + 64;
  float* SinvB = SinvA + (grad ? (size_t)nA * k * k : 0);
  float* part = SinvB + (grad ? (size_t)nB * k * k : 0);
  const int ld = k + 1;
  cudaError_t e = cudaMemsetAsync(flag, 0, sizeof(int32_t), st);
  if (e != cudaSuccess) return e;
  {
    const int smem = GP_WARPS * 2 * k * ld * (int)sizeof(float);
    static int smem_set[kMaxDevices] = {0};
    if ((e = ensure_dynamic_smem(gauss_class_kernel, smem, smem_set)) != cudaSuccess) return e;
    const bool need_inv = grad && mode == 1;
    gauss_class_kernel<<<(nA + GP_WARPS - 1) / GP_WARPS, GP_WARPS * 32, smem, st>>>(SigA, nA, k, ldA,
                                                                                  need_inv ? SinvA : nullptr, flag);
    gauss_class_kernel<<<(nB + GP_WARPS - 1) / GP_WARPS, GP_WARPS * 32, smem, st>>>(SigB, nB, k, ldB,
                                                                                  need_inv ? SinvB : nullptr, flag);
  }
  const int smem = GP_WARPS * (2 * k * ld + 3 * k) * (int)sizeof(float);
  static int smem_set2[kMaxDevices] = {0};
  if ((e = ensure_dynamic_smem(gauss_pair_kernel, smem, smem_set2)) != cudaSuccess) return e;
  if (!grad) {
    const int64_t npairs = (int64_t)nA * nB;
    gauss_pair_kernel<<<(unsigned)((npairs + GP_WARPS - 1) / GP_WARPS), GP_WARPS * 32, smem, st>>>(
        muA, SigA, muB, SigB, ldA, ldB, nA, nB, k, mode, 0, nA, nullptr, dist_out, nullptr, nullptr, flag);
  } else {
    const size_t per = (size_t)k * k + k;
    size_t rows = (size_t)(16u << 20) / (per * nB);
    if (rows < 1) rows = 1;
    if (rows > (size_t)nA) rows = nA;
    float* rowpart = part;
    float* colpart = part + rows * nB * per;
    if ((e = cudaMemsetAsync(gSigB, 0, (size_t)nB * k * k * sizeof(float), st)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(gMuB, 0, (size_t)nB * k * sizeof(float), st)) != cudaSuccess) return e;
    const int nC = nA > nB ? nA : nB;
    for (int a0 = 0; a0 < nA; a0 += (int)rows) {
      const int a1 = a0 + (int)rows < nA ? a0 + (int)rows : nA;
      const int64_t npairs = (int64_t)(a1 - a0) * nB;
      gauss_pair_kernel<<<(unsigned)((npairs + GP_WARPS - 1) / GP_WARPS), GP_WARPS * 32, smem, st>>>(
          muA, SigA, muB, SigB, ldA, ldB, nA, nB, k, mode, a0, a1, gD, dist_out, rowpart, colpart, flag);
      gauss_reduce_kernel<<<nC, 256, 0, st>>>(rowpart, colpart, gD, SinvA, SinvB, nA, nB, k, mode, a0, a1, gSigA, gMuA,
                                              gSigB, gMuB);
    }
  }
  if (flag_out != nullptr) {
    if ((e = cudaMemcpyAsync(flag_out, flag, sizeof(int32_t), cudaMemcpyDeviceToDevice, st)) != cudaSuccess) return e;
  }
  return cudaGetLastError();
}

// ---- fitting closure of the mean-covariance distances ----
// group width G and tile edge R = (32 / G) Q: Q grows with the pair count while tiles stay plentiful, up to
// R = 16 / 8 / 4 at G <= 8 / 16 / 32, so that the partials (2 R (k^2 + k + 1) elements per tile of R^2 pairs) stay
// below the affine-invariant closure's. The float64 closure keeps the rule: its largest block, 4 warps at G = 32 and
// Q = 4, takes 170 KB of shared memory (gc_pair_smem_elems).
static int gc_group(int k) {
  int G = 2;
  while (G < k) G *= 2;
  return G;
}

static int gc_batches(int G, int64_t npairs) {
  const int np = 32 / G, qmax = G <= 2 ? 1 : (G == 4 ? 2 : 4);
  int Q = 1;
  while (Q < qmax && npairs / ((int64_t)(2 * Q * np) * (2 * Q * np)) >= 4096) Q *= 2;
  return Q;
}

struct GcWorkspace {
  size_t rowpart, colpart, losspart, total_floats;
  PairTiles T;
  int Q;
};

static GcWorkspace gc_workspace(int C, int k, int64_t pair_begin, int64_t pair_end) {
  GcWorkspace w;
  const int64_t npairs = pair_end > pair_begin ? pair_end - pair_begin : 0;
  const int G = gc_group(k);
  w.Q = gc_batches(G, npairs);
  w.T = make_pair_tiles(C, C, 1, pair_begin, pair_end, (32 / G) * w.Q);
  auto al = [](size_t n) { return (n + 63) & ~size_t(63); };
  const size_t part = (size_t)w.T.ntiles * w.T.R * gc_slot_floats(k);
  w.rowpart = 0;
  w.colpart = al(part);
  w.losspart = w.colpart + al(part);
  w.total_floats = w.losspart + al((size_t)2 * w.T.ntiles) + 64;
  return w;
}

size_t gauss_closure_workspace_elems(int C, int k, int64_t pair_begin, int64_t pair_end) {
  return gc_workspace(C, k, pair_begin, pair_end).total_floats;
}

template <typename T, typename Noise>
static cudaError_t launch_gc_class(const T* PsiPart, const T* MuPart, int nchunk, Noise noise, int C, int k, int dist,
                                   T* Psi, T* Mu, T* logdet, T* Sinv, int32_t* flag, cudaStream_t st) {
  cudaError_t e = cudaMemsetAsync(flag, 0, 2 * sizeof(int32_t), st);  // flag[1]: closure_finish's arrival ticket
  if (e != cudaSuccess || C <= 0) return e;
  const int smem = GP_WARPS * 2 * k * (k + 1) * (int)sizeof(T);
  static int smem_set[kMaxDevices] = {0};
  if ((e = ensure_dynamic_smem(gauss_closure_class_kernel<T, Noise>, smem, smem_set)) != cudaSuccess) return e;
  gauss_closure_class_kernel<T, Noise><<<(C + GP_WARPS - 1) / GP_WARPS, GP_WARPS * 32, smem, st>>>(
      PsiPart, MuPart, nchunk, noise, C, k, gauss_closure_needs_logdet(dist) ? 1 : 0, Psi, Mu, logdet, Sinv, flag);
  return cudaGetLastError();
}

cudaError_t launch_gauss_closure_class(const float* PsiPart, const float* MuPart, int nchunk, float noise, int C, int k,
                                       int dist, float* Psi, float* Mu, float* logdet, float* Sinv, int32_t* flag,
                                       cudaStream_t st) {
  return launch_gc_class(PsiPart, MuPart, nchunk, noise, C, k, dist, Psi, Mu, logdet, Sinv, flag, st);
}

cudaError_t launch_gauss_closure_class(const double* PsiPart, const double* MuPart, int nchunk, const double* noise,
                                       int C, int k, int dist, double* Psi, double* Mu, double* logdet, double* Sinv,
                                       int32_t* flag, cudaStream_t st) {
  return launch_gc_class(PsiPart, MuPart, nchunk, noise, C, k, dist, Psi, Mu, logdet, Sinv, flag, st);
}

template <typename T, int G>
static cudaError_t launch_gc_pair(const GaussClosureArgs<T>& A, cudaStream_t st) {
  const int smem = GC_WARPS * gc_pair_smem_elems<T, G>(A.Q) * (int)sizeof(T);
  static int smem_set[kMaxDevices] = {0};
  cudaError_t e = ensure_dynamic_smem(gauss_closure_pair_kernel<T, G>, smem, smem_set);
  if (e != cudaSuccess) return e;
  const unsigned blocks = (unsigned)((A.T.ntiles + GC_WARPS - 1) / GC_WARPS);
  gauss_closure_pair_kernel<T, G><<<blocks, GC_WARPS * 32, smem, st>>>(A);
  return cudaGetLastError();
}

template <typename T>
static cudaError_t launch_gc_pairs(const T* Psi, const T* Mu, const T* logdet, const T* Sinv, int C, int k, int dist,
                                   int64_t pair_begin, int64_t pair_end, T weight, T* out, T* gPsi, T* gMu, T* ws,
                                   cudaStream_t st) {
  const GcWorkspace W = gc_workspace(C, k, pair_begin, pair_end);
  GaussClosureArgs<T> A;
  A.Psi = Psi; A.Mu = Mu; A.logdet = logdet;
  A.C = C; A.k = k; A.dist = dist; A.Q = W.Q;
  A.pair_begin = pair_begin; A.pair_end = pair_end; A.weight = weight; A.T = W.T;
  A.rowpart = ws + W.rowpart; A.colpart = ws + W.colpart; A.losspart = ws + W.losspart;
  cudaError_t e = cudaSuccess;
  if (W.T.ntiles > 0) {
    switch (gc_group(k)) {
      case 2: e = launch_gc_pair<T, 2>(A, st); break;
      case 4: e = launch_gc_pair<T, 4>(A, st); break;
      case 8: e = launch_gc_pair<T, 8>(A, st); break;
      case 16: e = launch_gc_pair<T, 16>(A, st); break;
      case 32: e = launch_gc_pair<T, 32>(A, st); break;
      default: return cudaErrorNotSupported;
    }
    if (e != cudaSuccess) return e;
  }
  const int per = gc_slot_floats(k), passes = (per + 1023) / 1024;
  int nt = (((per + passes - 1) / passes) + 31) & ~31;
  if (nt < 128) nt = 128;
  gauss_closure_reduce_kernel<T><<<C + 1, nt, per * sizeof(T), st>>>(W.T, C, k, dist, A.rowpart, A.colpart, A.losspart,
                                                                     Sinv, weight, out, gPsi, gMu);
  return cudaGetLastError();
}

cudaError_t launch_gauss_closure_pairs(const float* Psi, const float* Mu, const float* logdet, const float* Sinv, int C,
                                       int k, int dist, int64_t pair_begin, int64_t pair_end, float weight, float* out,
                                       float* gPsi, float* gMu, float* ws, cudaStream_t st) {
  return launch_gc_pairs(Psi, Mu, logdet, Sinv, C, k, dist, pair_begin, pair_end, weight, out, gPsi, gMu, ws, st);
}

cudaError_t launch_gauss_closure_pairs(const double* Psi, const double* Mu, const double* logdet, const double* Sinv,
                                       int C, int k, int dist, int64_t pair_begin, int64_t pair_end, double weight,
                                       double* out, double* gPsi, double* gMu, double* ws, cudaStream_t st) {
  return launch_gc_pairs(Psi, Mu, logdet, Sinv, C, k, dist, pair_begin, pair_end, weight, out, gPsi, gMu, ws, st);
}

}  // namespace sqfa
