// Device helpers of the R x R pair tiles (PairTiles, sqfa_internal.h) shared by the pair kernels of
// pairs.cu, the mean-covariance closure of gauss.cu and the float64 closure of closure64.cu: tile
// decoding, the pair mask of a launch and the fixed-order reduction of the per-tile loss partials.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "sqfa_internal.h"

namespace sqfa {
namespace {

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// local tile t of the launch -> block row / block column
__device__ __forceinline__ void decode_tile(const PairTiles& T, int64_t t, int& bi, int& bj) {
  const int64_t gt = T.tile0 + t;
  if (T.tri) {
    long long b = (long long)((sqrt(8.0 * (double)gt + 1.0) - 1.0) * 0.5);
    while (b * (b + 1) / 2 > gt) --b;
    while ((b + 1) * (b + 2) / 2 <= gt) ++b;
    bi = (int)b;
    bj = (int)(gt - b * (b + 1) / 2);
  } else {
    bi = (int)(gt / T.nbj);
    bj = (int)(gt % T.nbj);
  }
}

// pair (i, j) of a tile: is it part of this launch, and which linear pair index does it have
__device__ __forceinline__ bool pair_in_launch(int i, int j, int nA, int nB, int tri, int64_t pair_begin,
                                               int64_t pair_end) {
  if (i >= nA || j >= nB || (tri && j >= i)) return false;
  const int64_t p = tri ? (int64_t)i * (i - 1) / 2 + j : (int64_t)i * nB + j;
  return p >= pair_begin && p < pair_end;
}

// fixed-order sum of the per-tile {sum of distances, non-finite count}: every thread sums a strided
// subset in ascending tile order, then a fixed tree over the block (any block size up to 1024)
template <typename T>
__device__ void reduce_loss_partials(const T* __restrict__ losspart, int64_t ntiles, T& sum, T& bad) {
  __shared__ T red[2][1024];
  const int nt = blockDim.x;
  T a = T(0), b = T(0);
  for (int64_t t = threadIdx.x; t < ntiles; t += nt) {
    a += losspart[2 * t];
    b += losspart[2 * t + 1];
  }
  red[0][threadIdx.x] = a;
  red[1][threadIdx.x] = b;
  __syncthreads();
  for (int o = 512; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o && (int)threadIdx.x + o < nt) {
      red[0][threadIdx.x] += red[0][threadIdx.x + o];
      red[1][threadIdx.x] += red[1][threadIdx.x + o];
    }
    __syncthreads();
  }
  sum = red[0][0];
  bad = red[1][0];
}

}  // namespace
}  // namespace sqfa
