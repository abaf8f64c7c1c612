// Warp-level Cholesky factorisation with the inverse of the factor, shared by the float32 pair kernels
// (pairs.cu) and the float64 closure (closure64.cu). T = float or double.
#pragma once
#include <cuda_runtime.h>

namespace sqfa {
namespace {

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
