// K4 / K6 / transform: everything in the closure that touches the D-dimensional data space.
//
//   project_fwd : T[c] = F S[c] (k x D), Psi[c] = T[c] F^T, mu'[c] = F m[c]
//                 = conjugate_matrix(S, F)  /root/reference/src/sqfa/linalg.py:41 (via
//                 model.py:187) and transform(means) model.py:236, in ONE streaming pass over the
//                 C*D*D statistics (HBM-bound: D*D*4 bytes per class, k/2 flop per byte).
//   project_bwd : dF = sum_c (gPsi[c] + gPsi[c]^T) T[c] + gMu[c] m[c]^T  -- the analytic adjoint of
//                 the above; S is symmetric so the saved T replaces a second pass over S
//                 (autograd in the reference re-reads S: _optim.py:95).
//   transform   : Z = X F^T  model.py:236 for user data (HBM-bound on X).
//   embed       : feature noise (model.py:216-217, 537-538) and the Calvo-Oller embedding
//                 (distances.py:162-174) with its adjoint.
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/sqfa_b200.h"
#include "elem.cuh"
#include "sqfa_internal.h"

namespace sqfa {

namespace {

constexpr int PS_WARPS = 4;
constexpr int PS_THREADS = PS_WARPS * 32;
constexpr int PS_COLS = PS_WARPS * 128;  // columns per block: one 128-column strip (float4 per lane) per warp
constexpr int PS_MAXROWS = 256;          // rows of S per block (F^T tile in shared memory)

// partial[split][c][f][j] = sum_{i in rows of split} F[f][i] * S[c][i][j]
// Every warp streams its own 128-column strip down the rows of the split (512 contiguous bytes per
// row and warp, R rows in flight per thread), so there is no cross-warp reduction: a thread's
// accumulators are final for its 4 columns. HBM-bound for k <= 8.
template <int KT>
__global__ void __launch_bounds__(PS_THREADS)
project_stream_kernel(const float* __restrict__ S, const float* __restrict__ F, int C, int D, int k, int rows,
                      int vec16, float* __restrict__ partial) {
  __shared__ __align__(16) float Fs[PS_MAXROWS][KT];  // F^T tile: [row i][filter]
  const int c = blockIdx.z, split = blockIdx.y;
  const int i0 = split * rows;
  const int i1 = min(D, i0 + rows);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  for (int idx = tid; idx < rows * KT; idx += PS_THREADS) {
    const int f = idx / rows, ii = idx % rows;  // consecutive threads read consecutive i: coalesced
    Fs[ii][f] = (i0 + ii < i1 && f < k) ? F[(int64_t)f * D + i0 + ii] : 0.f;
  }
  __syncthreads();
  const int col = blockIdx.x * PS_COLS + warp * 128 + 4 * lane;
  if (col >= D) return;
  // D % 4 == 0 and 16-byte aligned S / partial (checked by the launcher): col + 4 <= D and every
  // row start is 16-byte aligned; otherwise scalar accesses
  const bool vec = vec16 != 0;
  // accumulators packed over filter pairs: acc2[f/2][q] = (filter f, filter f+1) of column col+q,
  // so every update is ONE packed-fp32 FMA (fma.rn.f32x2): FMA issue binds this kernel for k >= 16
  float2 acc2[KT / 2][4];
#pragma unroll
  for (int f = 0; f < KT / 2; ++f)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc2[f][q] = make_float2(0.f, 0.f);
  const float* Sc = S + (int64_t)c * D * D + col;
  constexpr int R = (KT >= 32) ? 4 : 8;  // independent 16-byte loads in flight per thread
  for (int ib = i0; ib < i1; ib += R) {
    float4 v[R];
#pragma unroll
    for (int u = 0; u < R; ++u) {
      const int i = ib + u;
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < i1) {
        const float* p = Sc + (int64_t)i * D;
        if (vec) {
          v[u] = __ldg(reinterpret_cast<const float4*>(p));
        } else {
          v[u].x = __ldg(p);
          v[u].y = col + 1 < D ? __ldg(p + 1) : 0.f;
          v[u].z = col + 2 < D ? __ldg(p + 2) : 0.f;
          v[u].w = col + 3 < D ? __ldg(p + 3) : 0.f;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < R; ++u) {
      const float* fr = Fs[min(ib + u, i1 - 1) - i0];  // rows past the end carry v = 0
      const float2 vx = make_float2(v[u].x, v[u].x), vy = make_float2(v[u].y, v[u].y);
      const float2 vz = make_float2(v[u].z, v[u].z), vw = make_float2(v[u].w, v[u].w);
#pragma unroll
      for (int f = 0; f < KT; f += 4) {
        const float4 w = *reinterpret_cast<const float4*>(fr + f);
        const float2 w01 = make_float2(w.x, w.y), w23 = make_float2(w.z, w.w);
        acc2[f / 2][0] = __ffma2_rn(w01, vx, acc2[f / 2][0]);
        acc2[f / 2][1] = __ffma2_rn(w01, vy, acc2[f / 2][1]);
        acc2[f / 2][2] = __ffma2_rn(w01, vz, acc2[f / 2][2]);
        acc2[f / 2][3] = __ffma2_rn(w01, vw, acc2[f / 2][3]);
        acc2[f / 2 + 1][0] = __ffma2_rn(w23, vx, acc2[f / 2 + 1][0]);
        acc2[f / 2 + 1][1] = __ffma2_rn(w23, vy, acc2[f / 2 + 1][1]);
        acc2[f / 2 + 1][2] = __ffma2_rn(w23, vz, acc2[f / 2 + 1][2]);
        acc2[f / 2 + 1][3] = __ffma2_rn(w23, vw, acc2[f / 2 + 1][3]);
      }
    }
  }
#pragma unroll
  for (int f = 0; f < KT; ++f) {
    if (f < k) {
      const float2* a = acc2[f / 2];
      const float4 t = (f & 1) ? make_float4(a[0].y, a[1].y, a[2].y, a[3].y)
                               : make_float4(a[0].x, a[1].x, a[2].x, a[3].x);
      float* o = partial + (((int64_t)split * C + c) * k + f) * D + col;
      if (vec) {
        *reinterpret_cast<float4*>(o) = t;
      } else {
        o[0] = t.x;
        if (col + 1 < D) o[1] = t.y;
        if (col + 2 < D) o[2] = t.z;
        if (col + 3 < D) o[3] = t.w;
      }
    }
  }
}

// Second stage of the projection, one block per (class, chunk of 128 columns), one warp per filter f:
//   T[c][f][cols]         = sum over the row splits of the partial products   (fixed order)
//   PsiPart[c][chunk][f][g] = T[c][f][cols] . F[g][cols]      (this chunk's share of Psi = T F^T)
//   MuPart[c][chunk][f]     = F[f][cols] . m[c][cols]         (this chunk's share of mu' = F m)
// The chunk partials are summed per class, in chunk order, by psi_reduce_kernel (stand-alone
// projection) or by class_prepare_kernel (closure): deterministic, and parallel over C * D / 128
// blocks instead of one block per row of T.
constexpr int PF_COLS = 128;

__global__ void __launch_bounds__(1024)
project_finish_kernel(const float* __restrict__ partial, const float* __restrict__ F, const float* __restrict__ M,
                      int C, int D, int k, int nsplit, int vec16, float* __restrict__ T,
                      float* __restrict__ PsiPart, float* __restrict__ MuPart) {
  const int c = blockIdx.y, chunk = blockIdx.x, nchunk = gridDim.x;
  const int f = threadIdx.x >> 5, lane = threadIdx.x & 31;  // blockDim.x = 32 k
  const int col = chunk * PF_COLS + 4 * lane;
  const int64_t sstride = (int64_t)C * k * D;
  const int64_t row = ((int64_t)c * k + f) * D;
  float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
  const int nv = col >= D ? 0 : (D - col >= 4 ? 4 : D - col);  // valid columns of this thread
  if (vec16) {
    if (nv == 4) {
      const float* pj = partial + row + col;
      int s = 0;
      for (; s + 4 <= nsplit; s += 4) {  // four independent loads in flight, added in order
        const float4 a0 = *reinterpret_cast<const float4*>(pj + (int64_t)s * sstride);
        const float4 a1 = *reinterpret_cast<const float4*>(pj + (int64_t)(s + 1) * sstride);
        const float4 a2 = *reinterpret_cast<const float4*>(pj + (int64_t)(s + 2) * sstride);
        const float4 a3 = *reinterpret_cast<const float4*>(pj + (int64_t)(s + 3) * sstride);
        t.x += a0.x; t.y += a0.y; t.z += a0.z; t.w += a0.w;
        t.x += a1.x; t.y += a1.y; t.z += a1.z; t.w += a1.w;
        t.x += a2.x; t.y += a2.y; t.z += a2.z; t.w += a2.w;
        t.x += a3.x; t.y += a3.y; t.z += a3.z; t.w += a3.w;
      }
      for (; s < nsplit; ++s) {
        const float4 a0 = *reinterpret_cast<const float4*>(pj + (int64_t)s * sstride);
        t.x += a0.x; t.y += a0.y; t.z += a0.z; t.w += a0.w;
      }
      *reinterpret_cast<float4*>(T + row + col) = t;
    }
  } else {
    float tv[4] = {0.f, 0.f, 0.f, 0.f};
    for (int q = 0; q < nv; ++q) {
      for (int s = 0; s < nsplit; ++s) tv[q] += partial[(int64_t)s * sstride + row + col + q];
      T[row + col + q] = tv[q];
    }
    t = make_float4(tv[0], tv[1], tv[2], tv[3]);
  }
  auto load4 = [&](const float* p) {  // 4 columns of a row of F or M, zero beyond D
    float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
    if (vec16 && nv == 4) {
      w = __ldg(reinterpret_cast<const float4*>(p));
    } else {
      if (nv > 0) w.x = __ldg(p);
      if (nv > 1) w.y = __ldg(p + 1);
      if (nv > 2) w.z = __ldg(p + 2);
      if (nv > 3) w.w = __ldg(p + 3);
    }
    return w;
  };
  float* pp = PsiPart + (((int64_t)c * nchunk + chunk) * k + f) * k;
  for (int g = 0; g < k; ++g) {
    const float4 w = load4(F + (int64_t)g * D + col);
    float a = (t.x * w.x + t.y * w.y) + (t.z * w.z + t.w * w.w);
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) pp[g] = a;
  }
  if (M != nullptr) {
    const float4 w = load4(F + (int64_t)f * D + col);
    const float4 mm = load4(M + (int64_t)c * D + col);
    float a = (w.x * mm.x + w.y * mm.y) + (w.z * mm.z + w.w * mm.w);
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) MuPart[((int64_t)c * nchunk + chunk) * k + f] = a;
  }
}

// Psi[c] / Mu[c] = sum over the column chunks, in chunk order (stand-alone projection)
__global__ void psi_reduce_kernel(const float* __restrict__ PsiPart, const float* __restrict__ MuPart, int C, int k,
                                  int nchunk, float* __restrict__ Psi, float* __restrict__ Mu) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int per = k * k + k;
  if (idx >= (int64_t)C * per) return;
  const int c = (int)(idx / per), e = (int)(idx % per);
  float a = 0.f;
  if (e < k * k) {
    for (int ch = 0; ch < nchunk; ++ch) a += PsiPart[((int64_t)c * nchunk + ch) * k * k + e];
    Psi[(int64_t)c * k * k + e] = a;
  } else if (MuPart != nullptr) {
    for (int ch = 0; ch < nchunk; ++ch) a += MuPart[((int64_t)c * nchunk + ch) * k + (e - k * k)];
    Mu[(int64_t)c * k + (e - k * k)] = a;
  }
}

// Sphere constraint (reference constraints.py:37): F[f] = W[f] / |W[f]|, inv_norm[f] = 1 / |W[f]|.
// One block per filter, fixed reduction tree. T = float or double (the float64 closure).
template <typename T>
__global__ void __launch_bounds__(256)
constraint_fwd_kernel(const T* __restrict__ Wraw, int D, T* __restrict__ F, T* __restrict__ inv_norm) {
  __shared__ T red[256];
  const int f = blockIdx.x;
  const T* w = Wraw + (int64_t)f * D;
  T a = T(0);
  for (int j = threadIdx.x; j < D; j += 256) a = fma(w[j], w[j], a);
  red[threadIdx.x] = a;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  const T nrm = sqrt(red[0]);
  for (int j = threadIdx.x; j < D; j += 256) F[(int64_t)f * D + j] = w[j] / nrm;
  if (threadIdx.x == 0) inv_norm[f] = T(1) / nrm;
}

// Last kernel of a closure evaluation, one block per filter f:
//   dF[f] = sum of the class-split partials of the projection adjoint (fixed order),
//   the constraint's adjoint: sphere  grad[f] = (dF[f] - (dF[f] . F[f]) F[f]) / |W[f]|
//                             (autograd through constraints.py:37), none: grad[f] = dF[f];
//   rows f < n_fixed get a zero gradient (FixedFilters detaches them, constraints.py:95-141),
//   out[2] = max |grad| over all filters (atomicMax on the bits of the non-negative value: non-negative
//   IEEE numbers order like their bit patterns, so the result does not depend on the order of the blocks).
constexpr int CF_THREADS = 1024;

template <typename T>
__device__ __forceinline__ T block_reduce_1024(T v, T* red, bool take_max) {
  red[threadIdx.x] = v;
  __syncthreads();
  for (int o = CF_THREADS / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o)
      red[threadIdx.x] = take_max ? fmax(red[threadIdx.x], red[threadIdx.x + o]) : red[threadIdx.x] + red[threadIdx.x + o];
    __syncthreads();
  }
  const T r = red[0];
  __syncthreads();
  return r;
}

__device__ __forceinline__ void atomic_max_nonneg(float* p, float v) {
  atomicMax(reinterpret_cast<unsigned int*>(p), __float_as_uint(v));
}
__device__ __forceinline__ void atomic_max_nonneg(double* p, double v) {
  atomicMax(reinterpret_cast<unsigned long long*>(p), (unsigned long long)__double_as_longlong(v));
}

template <typename T>
__global__ void __launch_bounds__(CF_THREADS)
closure_finish_kernel(const T* __restrict__ partial, int D, int k, int csplit, const T* __restrict__ F,
                      const T* __restrict__ inv_norm, int sphere, int n_fixed, T* __restrict__ grad,
                      T* out, T* out_host, unsigned int* ticket) {
  __shared__ T red[CF_THREADS];
  const int f = blockIdx.x;
  T* g = grad + (int64_t)f * D;
  const int64_t sstride = (int64_t)k * D;
  T dot = T(0);
  for (int j = threadIdx.x; j < D; j += CF_THREADS) {
    const T* p = partial + (int64_t)f * D + j;
    T a = T(0);
    int s = 0;
    for (; s + 8 <= csplit; s += 8) {  // eight loads in flight, added in split order
      T u[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) u[q] = p[(int64_t)(s + q) * sstride];
#pragma unroll
      for (int q = 0; q < 8; ++q) a += u[q];
    }
    for (; s < csplit; ++s) a += p[(int64_t)s * sstride];
    g[j] = a;  // re-read below by the same thread
    if (sphere) dot = fma(a, F[(int64_t)f * D + j], dot);
  }
  if (sphere) dot = block_reduce_1024(dot, red, false);
  const T inv = sphere ? inv_norm[f] : T(1);
  T amax = T(0);
  for (int j = threadIdx.x; j < D; j += CF_THREADS) {
    T v = g[j];
    if (f < n_fixed) v = T(0);
    else if (sphere) v = (v - dot * F[(int64_t)f * D + j]) * inv;
    g[j] = v;
    amax = fmax(amax, fabs(v));
  }
  amax = block_reduce_1024(amax, red, true);
  // NaN gradients: fmax drops NaN, the loss / non-finite counter carry that information
  if (threadIdx.x == 0 && out != nullptr) {
    atomic_max_nonneg(out + 2, amax);
    if (out_host != nullptr) {
      // the last block to arrive publishes {loss, #non-finite, max |grad|} in the caller's mapped host
      // memory: the host then needs an event wait and no copy (`ticket` is zeroed by the closure's memset)
      __threadfence();
      if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
        __threadfence();
        volatile T* o = out;
        volatile T* h = out_host;
        h[0] = o[0];
        h[1] = o[1];
        h[2] = o[2];
        __threadfence_system();
      }
    }
  }
}

// dF[f][j] = sum_c ( sum_g (gPsi[c][f][g] + gPsi[c][g][f]) T[c][g][j] + gMu[c][f] M[c][j] )
// grid: (ceil(D/128), class splits); partial results reduced by project_bwd_finalize_kernel or
// closure_finish_kernel. k <= 32.
template <typename Real>
__global__ void __launch_bounds__(128)
project_bwd_kernel(const Real* __restrict__ gPsi, const Real* __restrict__ gMu, const Real* __restrict__ T,
                   const Real* __restrict__ M, int C, int D, int k, int csplit, Real* __restrict__ partial) {
  extern __shared__ __align__(16) unsigned char pb_smem[];
  Real* Gs = reinterpret_cast<Real*>(pb_smem);  // Gs[k][k] symmetrised, gm[k]
  Real* gm = Gs + k * k;
  const int j = blockIdx.x * 128 + threadIdx.x;
  const int c0 = (int)(((int64_t)C * blockIdx.y) / csplit), c1 = (int)(((int64_t)C * (blockIdx.y + 1)) / csplit);
  Real acc[32];
#pragma unroll
  for (int f = 0; f < 32; ++f) acc[f] = Real(0);
  for (int c = c0; c < c1; ++c) {
    __syncthreads();
    for (int idx = threadIdx.x; idx < k * k; idx += 128) {
      const int f = idx / k, g = idx % k;
      Gs[idx] = gPsi[(int64_t)c * k * k + f * k + g] + gPsi[(int64_t)c * k * k + g * k + f];
    }
    if (gMu != nullptr)
      for (int f = threadIdx.x; f < k; f += 128) gm[f] = gMu[(int64_t)c * k + f];
    __syncthreads();
    if (j < D) {
      const Real mj = (gMu != nullptr) ? M[(int64_t)c * D + j] : Real(0);
      for (int g = 0; g < k; ++g) {
        const Real t = T[((int64_t)c * k + g) * D + j];
#pragma unroll
        for (int f = 0; f < 32; ++f)
          if (f < k) acc[f] = fma(Gs[f * k + g], t, acc[f]);
      }
      if (gMu != nullptr) {
#pragma unroll
        for (int f = 0; f < 32; ++f)
          if (f < k) acc[f] = fma(gm[f], mj, acc[f]);
      }
    }
  }
  if (j < D) {
#pragma unroll
    for (int f = 0; f < 32; ++f)
      if (f < k) partial[((int64_t)blockIdx.y * k + f) * D + j] = acc[f];
  }
}

__global__ void project_bwd_finalize_kernel(const float* __restrict__ partial, int D, int k, int csplit,
                                            float* __restrict__ dF) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= (int64_t)k * D) return;
  float a = 0.f;
  for (int s = 0; s < csplit; ++s) a += partial[(int64_t)s * k * D + idx];
  dF[idx] = a;
}

// Z[n][f] = sum_j X[n][j] F[f][j]; one warp per row, F chunk in shared memory. T = float, __nv_bfloat16
// or __half (widened as it is loaded).
template <int KT, typename T>
__global__ void __launch_bounds__(256)
transform_kernel(const T* __restrict__ X, int64_t ldx, const float* __restrict__ F, int64_t n, int D, int k,
                 int f0, float* __restrict__ Z) {
  extern __shared__ float Fs[];  // [KT][512]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int64_t rows_per_block = 64;
  const int64_t r0 = blockIdx.x * rows_per_block;
  float acc[8][KT];  // 8 rows per warp
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int f = 0; f < KT; ++f) acc[r][f] = 0.f;
  for (int j0 = 0; j0 < D; j0 += 512) {
    __syncthreads();
    for (int idx = tid; idx < KT * 512; idx += 256) {
      const int f = idx / 512, jj = idx % 512;
      Fs[idx] = (f0 + f < k && j0 + jj < D) ? F[(int64_t)(f0 + f) * D + j0 + jj] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int64_t row = r0 + warp * 8 + r;
      if (row >= n) break;
      const T* xr = X + row * ldx + j0;
      for (int jj = lane; jj < 512 && j0 + jj < D; jj += 32) {
        const float x = ldg_widen(xr + jj);
#pragma unroll
        for (int f = 0; f < KT; ++f) acc[r][f] += x * Fs[f * 512 + jj];
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int64_t row = r0 + warp * 8 + r;
    if (row >= n) break;
#pragma unroll
    for (int f = 0; f < KT; ++f) {
      float v = acc[r][f];
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0 && f0 + f < k) Z[row * k + f0 + f] = v;
    }
  }
}

// Z = X F^T for 16-byte aligned rows: a persistent mini-GEMM. A block walks row tiles of 128 rows;
// per 64-column chunk the X tile (128 x 64, padded rows: conflict-free LDS.128) and the F^T tile
// ([column][filter], so four filters of one column are one LDS.128 broadcast) arrive with cp.async
// while the previous chunk is being multiplied (two buffers). Thread (row pair, g) owns KF = KT/4
// filters of TWO rows (every F value loaded from shared memory feeds two FMAs), accumulated as
// packed pairs: one fma.rn.f32x2 per two filters, row and column.
// HBM-bound for k <= 16 (one read of X), about FMA-bound at k = 32.
// bf16 / fp16 X is staged in shared memory as it is (16-byte cp.async of 8 elements, rows padded to 72
// elements: LDS.128 of 8 elements, conflict-free per quarter warp) and widened after the LDS: half the
// HBM and half the shared-memory bytes of a float32 row; the columns are multiplied in the same order.
constexpr int TT_ROWS = 128, TT_COLS = 64, TT_LDX = TT_COLS + 4, TT_THREADS = 256;
constexpr int TT_LDX_H = TT_COLS + 8;  // row pitch (elements) of a bf16 / fp16 X tile
template <typename T>
constexpr int tt_x_bytes() {  // both X buffers
  return sizeof(T) == 4 ? 2 * TT_ROWS * TT_LDX * 4 : 2 * TT_ROWS * TT_LDX_H * 2;
}

__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_4(uint32_t dst, const void* src, int src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

template <int KF, typename T>
__global__ void __launch_bounds__(TT_THREADS)
transform_tile_kernel(const T* __restrict__ X, int64_t ldx, const float* __restrict__ F, int64_t n, int D, int k,
                      float* __restrict__ Z) {
  constexpr int KT = 4 * KF;
  constexpr bool F32 = sizeof(T) == 4;
  constexpr int LDX = F32 ? TT_LDX : TT_LDX_H;  // row pitch of the X tile (elements)
  constexpr int XV = 16 / sizeof(T);            // elements per 16-byte cp.async
  extern __shared__ __align__(16) float tsm[];
  T* Xs = reinterpret_cast<T*>(tsm);                                    // [2][TT_ROWS][LDX]
  float* Fs = tsm + tt_x_bytes<T>() / 4;                                // [2][TT_COLS][KT]
  const int tid = threadIdx.x;
  const int rp = tid & 63, fg = tid >> 6;  // rows rp and rp + 64; a warp: 32 consecutive rows, one filter group
  const int nchunks = (D + TT_COLS - 1) / TT_COLS;
  const int64_t ntiles = (n + TT_ROWS - 1) / TT_ROWS;
  const uint32_t xs_u = (uint32_t)__cvta_generic_to_shared(Xs), fs_u = (uint32_t)__cvta_generic_to_shared(Fs);

  auto load_chunk = [&](int64_t r0, int c0, int buf) {
    // X tile: 128 rows x 16-byte pieces; rows past n and columns past D are zero-filled (src_bytes = 0).
    // D % 4 == 0 on this path: a piece is inside, outside, or (bf16 / fp16, 8 elements) half inside.
    constexpr int PIECES = TT_COLS / XV;
    for (int idx = tid; idx < TT_ROWS * PIECES; idx += TT_THREADS) {
      const int r = idx / PIECES, cv = idx % PIECES;
      const int64_t gr = r0 + r;
      const int gc = c0 + XV * cv;
      const bool ok = gr < n && gc < D;
      const int bytes = !ok ? 0 : (D - gc >= XV ? 16 : (D - gc) * (int)sizeof(T));
      const T* src = ok ? X + gr * ldx + gc : X;
      cp_async_16(xs_u + (uint32_t)(((buf * TT_ROWS + r) * LDX + XV * cv) * (int)sizeof(T)), src, bytes);
    }
    // F^T tile: Fs[c][f] = F[f][c0 + c]
    for (int idx = tid; idx < TT_COLS * KT; idx += TT_THREADS) {
      const int f = idx / TT_COLS, c = idx % TT_COLS;  // consecutive threads read consecutive columns
      const bool ok = f < k && c0 + c < D;
      const float* src = ok ? F + (int64_t)f * D + c0 + c : F;
      cp_async_4(fs_u + (uint32_t)(((buf * TT_COLS + c) * KT + f) * 4), src, ok ? 4 : 0);
    }
    cp_async_commit();
  };

  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t r0 = tile * TT_ROWS;
    float2 acc0[KF / 2], acc1[KF / 2];
#pragma unroll
    for (int i = 0; i < KF / 2; ++i) acc0[i] = acc1[i] = make_float2(0.f, 0.f);
    load_chunk(r0, 0, 0);
    for (int ch = 0; ch < nchunks; ++ch) {
      const int buf = ch & 1;
      if (ch + 1 < nchunks) {
        load_chunk(r0, (ch + 1) * TT_COLS, buf ^ 1);
        cp_async_wait<1>();
      } else {
        cp_async_wait<0>();
      }
      __syncthreads();
      const T* xr0 = Xs + (buf * TT_ROWS + rp) * LDX;
      const T* xr1 = xr0 + 64 * LDX;
      const float* fb = Fs + buf * TT_COLS * KT + fg * KF;
      // one LDS.128 per row and step: 4 float32 or 8 bf16 / fp16 columns, multiplied in column order
#pragma unroll(F32 ? 4 : 2)
      for (int cv = 0; cv < TT_COLS / XV; ++cv) {
        float va[XV], vb[XV];
        if constexpr (F32) {
          const float4 xa = *reinterpret_cast<const float4*>(xr0 + 4 * cv);
          const float4 xb = *reinterpret_cast<const float4*>(xr1 + 4 * cv);
          va[0] = xa.x; va[1] = xa.y; va[2] = xa.z; va[3] = xa.w;
          vb[0] = xb.x; vb[1] = xb.y; vb[2] = xb.z; vb[3] = xb.w;
        } else {
          const uint4 xa = *reinterpret_cast<const uint4*>(xr0 + 8 * cv);
          const uint4 xb = *reinterpret_cast<const uint4*>(xr1 + 8 * cv);
          const float4 a0 = widen4<T>(make_uint2(xa.x, xa.y)), a1 = widen4<T>(make_uint2(xa.z, xa.w));
          const float4 b0 = widen4<T>(make_uint2(xb.x, xb.y)), b1 = widen4<T>(make_uint2(xb.z, xb.w));
          va[0] = a0.x; va[1] = a0.y; va[2] = a0.z; va[3] = a0.w; va[4] = a1.x; va[5] = a1.y; va[6] = a1.z; va[7] = a1.w;
          vb[0] = b0.x; vb[1] = b0.y; vb[2] = b0.z; vb[3] = b0.w; vb[4] = b1.x; vb[5] = b1.y; vb[6] = b1.z; vb[7] = b1.w;
        }
#pragma unroll
        for (int u = 0; u < XV; ++u) {
          const float2 a2 = make_float2(va[u], va[u]), b2 = make_float2(vb[u], vb[u]);
          const float* fr = fb + (XV * cv + u) * KT;
          if constexpr (KF >= 4) {
#pragma unroll
            for (int g = 0; g < KF / 4; ++g) {
              const float4 w = *reinterpret_cast<const float4*>(fr + 4 * g);
              const float2 w01 = make_float2(w.x, w.y), w23 = make_float2(w.z, w.w);
              acc0[2 * g] = __ffma2_rn(a2, w01, acc0[2 * g]);
              acc0[2 * g + 1] = __ffma2_rn(a2, w23, acc0[2 * g + 1]);
              acc1[2 * g] = __ffma2_rn(b2, w01, acc1[2 * g]);
              acc1[2 * g + 1] = __ffma2_rn(b2, w23, acc1[2 * g + 1]);
            }
          } else {
            const float2 w = *reinterpret_cast<const float2*>(fr);
            acc0[0] = __ffma2_rn(a2, w, acc0[0]);
            acc1[0] = __ffma2_rn(b2, w, acc1[0]);
          }
        }
      }
      __syncthreads();  // the buffer is refilled two chunks later
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int64_t gr = r0 + rp + 64 * h;
      if (gr < n) {
#pragma unroll
        for (int i = 0; i < KF / 2; ++i) {
          const int f = fg * KF + 2 * i;
          const float2 a = h ? acc1[i] : acc0[i];
          if (f < k) Z[gr * k + f] = a.x;
          if (f + 1 < k) Z[gr * k + f + 1] = a.y;
        }
      }
    }
  }
}

__global__ void embed_fwd_kernel(const float* __restrict__ Psi, const float* __restrict__ Mu, float noise, int C,
                                 int k, int fr, float* __restrict__ E) {
  const int m = fr ? k + 1 : k;
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= (int64_t)C * m * m) return;
  const int c = (int)(idx / (m * m));
  const int r = (int)((idx / m) % m), s = (int)(idx % m);
  float v;
  if (r < k && s < k) {
    v = Psi[(int64_t)c * k * k + r * k + s] + (r == s ? noise : 0.f);
    if (fr) v += Mu[(int64_t)c * k + r] * Mu[(int64_t)c * k + s];
  } else if (r == k && s == k) {
    v = 1.f;
  } else {
    v = Mu[(int64_t)c * k + (r < k ? r : s)];
  }
  E[idx] = v;
}

// gPsi = gE[:k,:k];  gMu[r] = sum_s (gE[r][s] + gE[s][r]) mu[s] + gE[r][k] + gE[k][r]
__global__ void embed_bwd_kernel(const float* __restrict__ gE, const float* __restrict__ Mu, int C, int k, int fr,
                                 float* __restrict__ gPsi, float* __restrict__ gMu) {
  const int m = fr ? k + 1 : k;
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= (int64_t)C * k * (k + 1)) return;
  const int c = (int)(idx / (k * (k + 1)));
  const int r = (int)((idx / (k + 1)) % k), s = (int)(idx % (k + 1));
  const float* g = gE + (int64_t)c * m * m;
  if (s < k) {
    gPsi[(int64_t)c * k * k + r * k + s] = g[r * m + s];
  } else if (fr) {
    float a = g[r * m + k] + g[k * m + r];
    for (int t = 0; t < k; ++t) a += (g[r * m + t] + g[t * m + r]) * Mu[(int64_t)c * k + t];
    gMu[(int64_t)c * k + r] = a;
  }
}

template <int KT>
cudaError_t run_project_stream(const float* S, const float* F, int C, int D, int k, int rows, int nsplit,
                               float* partial, cudaStream_t st) {
  dim3 grid((D + PS_COLS - 1) / PS_COLS, nsplit, C);
  const int vec16 =
      (D % 4 == 0 && ((reinterpret_cast<uintptr_t>(S) | reinterpret_cast<uintptr_t>(partial)) & 15) == 0) ? 1 : 0;
  project_stream_kernel<KT><<<grid, PS_THREADS, 0, st>>>(S, F, C, D, k, rows, vec16, partial);
  return cudaGetLastError();
}

template <int KT, typename T>
cudaError_t run_transform(const T* X, int64_t ldx, const float* F, int64_t n, int D, int k, float* Z,
                          cudaStream_t st) {
  const int smem = KT * 512 * (int)sizeof(float);
  static int smem_set[kMaxDevices] = {0};
  {
    cudaError_t e = ensure_dynamic_smem(transform_kernel<KT, T>, smem, smem_set);
    if (e != cudaSuccess) return e;
  }
  const int64_t blocks = (n + 63) / 64;
  for (int f0 = 0; f0 < k; f0 += KT)
    transform_kernel<KT, T><<<(unsigned)blocks, 256, smem, st>>>(X, ldx, F, n, D, k, f0, Z);
  return cudaGetLastError();
}

}  // namespace

// Resident blocks of project_stream_kernel<KT> per device (occupancy query, cached per device)
template <int KT>
static int project_stream_capacity() {
  static int cap[kMaxDevices] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return 148 * 6;
  if (cap[dev] == 0) {
    int per_sm = 0, sms = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, project_stream_kernel<KT>, PS_THREADS, 0) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || per_sm <= 0 || sms <= 0)
      return 148 * 6;
    cap[dev] = per_sm * sms;
  }
  return cap[dev];
}

static int project_capacity(int k) {
  if (k <= 4) return project_stream_capacity<4>();
  if (k <= 8) return project_stream_capacity<8>();
  if (k <= 16) return project_stream_capacity<16>();
  return project_stream_capacity<32>();
}

// Row splits of the streaming pass. The grid is (column blocks x splits x classes); what costs time is
// a last wave of blocks that fills a fraction of the GPU (c4 with one split: 1000 blocks on 888 resident
// slots = 1.13 waves, 56 % wave efficiency) and, against it, the partial products every split writes and
// the finish kernel reads back (2 nsplit k / D of the bytes of S). Choose the split count that maximises
// wave efficiency / (1 + partial traffic), with at least 64 rows per split and at most PS_MAXROWS.
int project_nsplit(int C, int D, int k) {
  const int64_t colblocks = (D + PS_COLS - 1) / PS_COLS;
  const int64_t per_split = colblocks * (C > 0 ? C : 1);
  const int64_t cap = project_capacity(k);
  const int min_split = (D + PS_MAXROWS - 1) / PS_MAXROWS;
  int max_split = D / 64 > min_split ? D / 64 : min_split;
  if (max_split > 256) max_split = 256;
  int best = min_split;
  double best_score = -1.0;
  for (int n = min_split; n <= max_split; ++n) {
    const int64_t blocks = per_split * n;
    const int64_t waves = (blocks + cap - 1) / cap;
    const double eff = (double)blocks / (double)(waves * cap);
    const double score = eff / (1.0 + 2.0 * n * k / (double)D);
    if (score > best_score * 1.001) { best_score = score; best = n; }  // ties: fewer splits
  }
  return best;
}
int project_rows_per_split(int C, int D, int k) {
  const int n = project_nsplit(C, D, k);
  int rows = (D + n - 1) / n;
  rows = (rows + 7) & ~7;
  if (rows > PS_MAXROWS) rows = PS_MAXROWS;
  return rows;
}
static int project_nsplit_actual(int C, int D, int k) {
  const int rows = project_rows_per_split(C, D, k);
  return (D + rows - 1) / rows;
}

static size_t project_partial_floats(int C, int D, int k) {
  return (size_t)project_nsplit_actual(C, D, k) * C * k * D;
}

int project_nchunk(int D) { return (D + PF_COLS - 1) / PF_COLS; }
size_t project_psipart_floats(int C, int D, int k) { return al<float>((size_t)C * project_nchunk(D) * k * k); }
size_t project_mupart_floats(int C, int D, int k) { return al<float>((size_t)C * project_nchunk(D) * k); }
// most class splits of the projection adjoint (the float64 closure's workspace is sized for 128)
template <typename T> constexpr int PB_MAX_CSPLIT = 256;
template <> constexpr int PB_MAX_CSPLIT<double> = 128;
template <typename T>
int project_bwd_csplit(int C, int D) {
  // enough (column block, class split) blocks to fill the GPU about 8 times over: every block walks its
  // classes serially (one dependent round of loads per class), so short class lists hide latency
  const int colblocks = (D + 127) / 128;
  int csplit = (8 * 148 + colblocks - 1) / colblocks;
  if (csplit > PB_MAX_CSPLIT<T>) csplit = PB_MAX_CSPLIT<T>;
  if (csplit > C) csplit = C > 0 ? C : 1;
  return csplit < 1 ? 1 : csplit;
}
template int project_bwd_csplit<float>(int, int);
template int project_bwd_csplit<double>(int, int);

// workspace (floats): [ row-split partials | PsiPart | MuPart ] for the forward, [ class-split partials ] for
// the adjoint (they alias: the two are never live together)
size_t project_workspace_bytes(int C, int D, int k) {
  const size_t fwd = al<float>(project_partial_floats(C, D, k)) + project_psipart_floats(C, D, k) +
                     project_mupart_floats(C, D, k);
  const size_t bwd = (size_t)PB_MAX_CSPLIT<float> * k * D;
  return (fwd > bwd ? fwd : bwd) * sizeof(float);
}

// T and the per-chunk partials of Psi / Mu (the closure reduces them inside class_prepare_kernel)
cudaError_t launch_project_partials(const float* S, const float* M, const float* F, int C, int D, int k, float* T,
                                    float* partial, float* PsiPart, float* MuPart, cudaStream_t st) {
  if (C <= 0) return cudaSuccess;
  const int rows = project_rows_per_split(C, D, k);
  int nsplit = project_nsplit_actual(C, D, k);
  cudaError_t e;
  if (project_tc_applicable(S, F, D, k)) {  // k > 8: tensor cores (the SIMT pass is FP32-FMA bound there)
    e = launch_project_tc(S, F, C, D, k, partial, st);
    nsplit = 1;  // the finish kernel finds T itself in the first "row split"
  } else if (k <= 4) e = run_project_stream<4>(S, F, C, D, k, rows, nsplit, partial, st);
  else if (k <= 8) e = run_project_stream<8>(S, F, C, D, k, rows, nsplit, partial, st);
  else if (k <= 16) e = run_project_stream<16>(S, F, C, D, k, rows, nsplit, partial, st);
  else e = run_project_stream<32>(S, F, C, D, k, rows, nsplit, partial, st);
  if (e != cudaSuccess) return e;
  const int vec16 = (D % 4 == 0 && ((reinterpret_cast<uintptr_t>(partial) | reinterpret_cast<uintptr_t>(T) |
                                     reinterpret_cast<uintptr_t>(F) | reinterpret_cast<uintptr_t>(M)) & 15) == 0)
                        ? 1 : 0;
  project_finish_kernel<<<dim3(project_nchunk(D), C), 32 * k, 0, st>>>(partial, F, M, C, D, k, nsplit, vec16, T,
                                                                        PsiPart, MuPart);
  return cudaGetLastError();
}

cudaError_t launch_project_fwd(const float* S, const float* M, const float* F, int C, int D, int k, float* T,
                               float* Psi, float* Mu, float* ws, cudaStream_t st) {
  if (C <= 0) return cudaSuccess;
  float* PsiPart = ws + al<float>(project_partial_floats(C, D, k));
  float* MuPart = PsiPart + project_psipart_floats(C, D, k);
  cudaError_t e = launch_project_partials(S, M, F, C, D, k, T, ws, PsiPart, M != nullptr ? MuPart : nullptr, st);
  if (e != cudaSuccess) return e;
  const int64_t total = (int64_t)C * (k * k + k);
  psi_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(PsiPart, M != nullptr ? MuPart : nullptr, C, k,
                                                                     project_nchunk(D), Psi, Mu);
  return cudaGetLastError();
}

template <typename Real>
static cudaError_t launch_project_bwd_partials(const Real* gPsi, const Real* gMu, const Real* T, const Real* M, int C,
                                               int D, int k, Real* ws, int csplit, cudaStream_t st) {
  const int colblocks = (D + 127) / 128;
  const int smem = (k * k + k) * (int)sizeof(Real);
  project_bwd_kernel<Real><<<dim3(colblocks, csplit), 128, smem, st>>>(gPsi, gMu, T, M, C, D, k, csplit, ws);
  return cudaGetLastError();
}

cudaError_t launch_project_bwd(const float* gPsi, const float* gMu, const float* T, const float* M, int C, int D,
                               int k, float* dF, float* ws, cudaStream_t st) {
  const int csplit = project_bwd_csplit<float>(C, D);
  cudaError_t e = launch_project_bwd_partials(gPsi, gMu, T, M, C, D, k, ws, csplit, st);
  if (e != cudaSuccess) return e;
  const int64_t total = (int64_t)k * D;
  project_bwd_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(ws, D, k, csplit, dF);
  return cudaGetLastError();
}

// adjoint of the projection followed by the adjoint of the filter constraint (closure tail)
template <typename Real>
cudaError_t launch_project_bwd_constrained(const Real* gPsi, const Real* gMu, const Real* T, const Real* M, int C,
                                           int D, int k, const Real* F, const Real* inv_norm, int sphere, int n_fixed,
                                           Real* grad, Real* out, Real* out_host, unsigned int* ticket, Real* ws,
                                           cudaStream_t st) {
  const int csplit = project_bwd_csplit<Real>(C, D);
  cudaError_t e = launch_project_bwd_partials(gPsi, gMu, T, M, C, D, k, ws, csplit, st);
  if (e != cudaSuccess) return e;
  closure_finish_kernel<Real><<<k, CF_THREADS, 0, st>>>(ws, D, k, csplit, F, inv_norm, sphere, n_fixed, grad, out,
                                                     out_host, ticket);
  return cudaGetLastError();
}
template cudaError_t launch_project_bwd_constrained<float>(const float*, const float*, const float*, const float*, int,
                                                           int, int, const float*, const float*, int, int, float*,
                                                           float*, float*, unsigned int*, float*, cudaStream_t);
template cudaError_t launch_project_bwd_constrained<double>(const double*, const double*, const double*,
                                                            const double*, int, int, int, const double*,
                                                            const double*, int, int, double*, double*, double*,
                                                            unsigned int*, double*, cudaStream_t);

template <typename T>
cudaError_t launch_constraint_fwd(const T* Wraw, int D, int k, T* F, T* inv_norm, cudaStream_t st) {
  constraint_fwd_kernel<T><<<k, 256, 0, st>>>(Wraw, D, F, inv_norm);
  return cudaGetLastError();
}
template cudaError_t launch_constraint_fwd<float>(const float*, int, int, float*, float*, cudaStream_t);
template cudaError_t launch_constraint_fwd<double>(const double*, int, int, double*, double*, cudaStream_t);

template <int KF, typename T>
static cudaError_t run_transform_tile(const T* X, int64_t ldx, const float* F, int64_t n, int D, int k, float* Z,
                                      cudaStream_t st) {
  const int smem = tt_x_bytes<T>() + 2 * TT_COLS * 4 * KF * (int)sizeof(float);
  static int smem_set[kMaxDevices] = {0};
  {
    cudaError_t e = ensure_dynamic_smem(transform_tile_kernel<KF, T>, smem, smem_set);
    if (e != cudaSuccess) return e;
  }
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int64_t ntiles = (n + TT_ROWS - 1) / TT_ROWS;
  const int64_t grid = ntiles < 2 * (int64_t)sms ? ntiles : 2 * (int64_t)sms;
  transform_tile_kernel<KF, T><<<(unsigned)grid, TT_THREADS, smem, st>>>(X, ldx, F, n, D, k, Z);
  return cudaGetLastError();
}

template <typename T>
static cudaError_t launch_transform_t(const T* X, int64_t ldx, const float* F, int64_t n, int D, int k, float* Z,
                                      cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  // the tile kernel's 16-byte cp.async: every row starts 16-byte aligned (4 float32 / 8 bf16 / fp16 elements)
  constexpr int64_t XV = 16 / sizeof(T);
  if (D % 4 == 0 && ldx % XV == 0 && (reinterpret_cast<uintptr_t>(X) & 15) == 0 && k <= 32) {
    if (k <= 8) return run_transform_tile<2>(X, ldx, F, n, D, k, Z, st);
    if (k <= 16) return run_transform_tile<4>(X, ldx, F, n, D, k, Z, st);
    return run_transform_tile<8>(X, ldx, F, n, D, k, Z, st);
  }
  if (k <= 4) return run_transform<4>(X, ldx, F, n, D, k, Z, st);
  if (k <= 8) return run_transform<8>(X, ldx, F, n, D, k, Z, st);
  return run_transform<16>(X, ldx, F, n, D, k, Z, st);
}

cudaError_t launch_transform(const void* X, int elem, int64_t ldx, const float* F, int64_t n, int D, int k, float* Z,
                             cudaStream_t st) {
  if (elem == ELEM_BF16) return launch_transform_t(static_cast<const __nv_bfloat16*>(X), ldx, F, n, D, k, Z, st);
  if (elem == ELEM_F16) return launch_transform_t(static_cast<const __half*>(X), ldx, F, n, D, k, Z, st);
  return launch_transform_t(static_cast<const float*>(X), ldx, F, n, D, k, Z, st);
}

cudaError_t launch_embed_fwd(const float* Psi, const float* Mu, float noise, int C, int k, int fr, float* E,
                             cudaStream_t st) {
  const int m = fr ? k + 1 : k;
  const int64_t total = (int64_t)C * m * m;
  if (total <= 0) return cudaSuccess;
  embed_fwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(Psi, Mu, noise, C, k, fr, E);
  return cudaGetLastError();
}

cudaError_t launch_embed_bwd(const float* gE, const float* Mu, int C, int k, int fr, float* gPsi, float* gMu,
                             cudaStream_t st) {
  const int64_t total = (int64_t)C * k * (k + 1);
  if (total <= 0) return cudaSuccess;
  embed_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(gE, Mu, C, k, fr, gPsi, gMu);
  return cudaGetLastError();
}

}  // namespace sqfa
