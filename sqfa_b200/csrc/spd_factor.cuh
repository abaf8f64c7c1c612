// The class stage of the fitting closure, shared by the float32 pair kernels (pairs.cu) and the float64
// closure (closure64.cu): assembly of E_c from the projection's chunk partials, and a warp-level Cholesky
// factorisation with the inverse of the factor. T = float or double.
#pragma once
#include <cstdint>
#include <type_traits>
#include <cuda_runtime.h>

namespace sqfa {
namespace {

// sum_{ch < nchunk} p[ch * stride], added in chunk order with eight loads in flight
template <typename T>
__device__ __forceinline__ T sum_chunks(const T* p, int nchunk, int stride) {
  T a = T(0);
  int ch = 0;
  for (; ch + 8 <= nchunk; ch += 8) {
    T u[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) u[q] = p[(int64_t)(ch + q) * stride];
#pragma unroll
    for (int q = 0; q < 8; ++q) a += u[q];
  }
  for (; ch < nchunk; ++ch) a += p[(int64_t)ch * stride];
  return a;
}

// E_c of class c, one warp (reference model.py:216-217 / 537-538, distances.py:162-174):
//   Psi_c = sum of its column-chunk partials, mu'_c likewise when MuPart is given (into mus and Mu[c]),
//   E_c = Psi_c + noise I, for Fisher-Rao (fr) the Calvo-Oller embedding
//   [[Psi_c + noise I + mu' mu'^T, mu'], [mu'^T, 1]].
// Es (m x m, m = k + fr) receives E_c, and Eg[c] (m x m per class) a copy unless Eg is the literal nullptr (a
// compile-time choice: the float32 closure keeps E, the float64 closure does not). The caller syncs the warp
// before reading Es.
template <typename T, typename EOut>
__device__ __forceinline__ void assemble_class_matrix(const T* PsiPart, const T* MuPart, int nchunk, T noise, int c,
                                                      int k, bool fr, T* Mu, T* mus, T* Es, EOut Eg, int lane) {
  const int m = fr ? k + 1 : k;
  if (MuPart != nullptr) {
    for (int r = lane; r < k; r += 32) {
      const T a = sum_chunks(MuPart + (int64_t)c * nchunk * k + r, nchunk, k);
      mus[r] = a;
      Mu[(int64_t)c * k + r] = a;
    }
    __syncwarp();
  }
  for (int idx = lane; idx < m * m; idx += 32) {
    const int r = idx / m, s = idx % m;
    T v;
    if (r < k && s < k) {
      v = sum_chunks(PsiPart + (int64_t)c * nchunk * k * k + r * k + s, nchunk, k * k);
      if (r == s) v += noise;
      if (fr) v = fma(mus[r], mus[s], v);
    } else if (r == k && s == k) {
      v = T(1);
    } else {
      v = mus[r < k ? r : s];
    }
    Es[idx] = v;
    if constexpr (!std::is_null_pointer_v<EOut>) Eg[(int64_t)c * m * m + idx] = v;
  }
}

// Cholesky E = L L^T and L^-1 of an m x m SPD matrix, one warp. La / Li: shared, row stride ld.
// Returns false (all lanes) if a pivot is not positive / finite.
template <typename T>
__device__ bool warp_cholesky_inverse(const T* __restrict__ E, T* La, T* Li, int m, int ld, int lane) {
  for (int idx = lane; idx < m * m; idx += 32) {
    const int r = idx / m, c = idx % m;
    La[r * ld + c] = E[idx];
    Li[r * ld + c] = T(0);
  }
  __syncwarp();
  bool ok = true;
  for (int j = 0; j < m; ++j) {
    T d = La[j * ld + j];
    for (int k = 0; k < j; ++k) d -= La[j * ld + k] * La[j * ld + k];
    if (!(d > T(0)) || !isfinite(d)) ok = false;
    const T ljj = sqrt(d);
    __syncwarp();
    for (int i = j + 1 + lane; i < m; i += 32) {
      T v = La[i * ld + j];
      for (int k = 0; k < j; ++k) v -= La[i * ld + k] * La[j * ld + k];
      La[i * ld + j] = v / ljj;
    }
    if (lane == 0) La[j * ld + j] = ljj;
    __syncwarp();
  }
  // inverse by forward substitution, one column per lane
  for (int c = lane; c < m; c += 32) {
    for (int i = 0; i < m; ++i) {
      T s = (i == c) ? T(1) : T(0);
      for (int k = 0; k < i; ++k) s -= La[i * ld + k] * Li[k * ld + c];
      Li[i * ld + c] = (i < c) ? T(0) : s / La[i * ld + i];
    }
  }
  __syncwarp();
  return ok;
}

}  // namespace
}  // namespace sqfa
