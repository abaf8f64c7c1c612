// K2a: segmented per-class column sums (-> class means) and the pilot shift of the one-pass path,
// K3: statistics epilogue
// (mean, unbiased covariance, covariance + mu mu^T, optional OAS shrinkage).
//
// Reference semantics: /root/reference/src/sqfa/statistics.py
//   means[i]          = mean(class_points)                       :40
//   covariances[i]    = (Xc^T Xc) / (n_i - 1), Xc centred        :113-122
//   second_moments[i] = covariances[i] + outer(mean, mean)       :47
//   oas_covariance                                               :78-94
// Empty class -> mean NaN, covariance -0 (0 / -1), second moment NaN; singleton -> covariance NaN.
// The same values fall out of the arithmetic below (0/0, 0/-1) without special cases.
#include <cstdint>
#include <cuda_runtime.h>

#include "elem.cuh"
#include "sqfa_internal.h"

namespace sqfa {

namespace {

constexpr int SUM_THREADS = 256;
constexpr int SUM_BLOCK_ROWS = 512;  // inner block of the two-level (blocked) fp32 summation

__device__ __forceinline__ float4 f4add(float4 a, float4 b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}

// threads of a block that share one row (each owns 4 columns): 256 for D >= 1024, fewer for small D so
// that the remaining threads of the block form ROW LANES (D = 104: 32 threads per row, 8 row lanes --
// with one row lane, 230 of 256 threads had no column and the kernel ran at 1.6 TB/s)
__host__ __device__ inline int sums_threads_per_row(int D) {
  int tpr = 32;
  while (tpr < SUM_THREADS && tpr * 4 < D) tpr <<= 1;
  return tpr;
}

// partial[c][split][D] = sum over the split's rows of (x - shift_c)
// T = float, __nv_bfloat16 or __half: elements are widened to float32 as they are loaded. `blk_ok` selects
// the summation order (rows in groups of four into four accumulators), `vec_ok` the 4-element vector loads;
// for float32 they are the same flag. A bf16 / fp16 X keeps the order of a float32 copy of it (contiguous,
// so blocked whenever D % 4 == 0) even where its rows only allow element loads: the sums are bit-identical.
template <typename T>
__global__ void __launch_bounds__(SUM_THREADS)
class_sums_kernel(const T* __restrict__ X, int64_t ldx, const int32_t* __restrict__ perm,
                  const int64_t* __restrict__ offsets, const float* __restrict__ shift, int D, int nsplit,
                  float* __restrict__ partial, int vec_ok, int blk_ok) {
  __shared__ float4 red[SUM_THREADS];
  const int tpr = sums_threads_per_row(D), nlanes = SUM_THREADS / tpr;
  const int rlane = threadIdx.x / tpr, tcol = threadIdx.x % tpr;
  const int c = blockIdx.z;
  const int split = blockIdx.y;
  const int64_t begin = offsets[c];
  const int64_t n_c = offsets[c + 1] - begin;
  const int64_t s0 = (n_c * split) / nsplit, s1 = (n_c * (split + 1)) / nsplit;
  // the split's rows are cut into one contiguous piece per row lane
  const int64_t k0 = s0 + ((s1 - s0) * rlane) / nlanes, k1 = s0 + ((s1 - s0) * (rlane + 1)) / nlanes;
  const int col = (blockIdx.x * tpr + tcol) * 4;
  const bool live = col < D;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  const bool full = blk_ok && (col + 4 <= D);
  const bool vec = vec_ok != 0;
  if (shift != nullptr && live) {
    const float* sh = shift + (int64_t)c * D + col;
    s.x = sh[0];
    if (col + 1 < D) s.y = sh[1];
    if (col + 2 < D) s.z = sh[2];
    if (col + 3 < D) s.w = sh[3];
  }
  float4 outer = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t kb = k0; kb < k1 && live; kb += SUM_BLOCK_ROWS) {
    const int64_t ke = kb + SUM_BLOCK_ROWS < k1 ? kb + SUM_BLOCK_ROWS : k1;
    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
    int64_t k = kb;
    if (full) {
      for (; k + 4 <= ke; k += 4) {  // 4 independent 16-byte loads in flight per thread
        const T* r0 = X + (int64_t)perm[begin + k + 0] * ldx + col;
        const T* r1 = X + (int64_t)perm[begin + k + 1] * ldx + col;
        const T* r2 = X + (int64_t)perm[begin + k + 2] * ldx + col;
        const T* r3 = X + (int64_t)perm[begin + k + 3] * ldx + col;
        float4 v0, v1, v2, v3;
        if (sizeof(T) == 4 || vec) {  // float32: vec_ok == blk_ok
          v0 = ldg_widen4(r0); v1 = ldg_widen4(r1); v2 = ldg_widen4(r2); v3 = ldg_widen4(r3);
        } else {
          v0 = make_float4(ldg_widen(r0), ldg_widen(r0 + 1), ldg_widen(r0 + 2), ldg_widen(r0 + 3));
          v1 = make_float4(ldg_widen(r1), ldg_widen(r1 + 1), ldg_widen(r1 + 2), ldg_widen(r1 + 3));
          v2 = make_float4(ldg_widen(r2), ldg_widen(r2 + 1), ldg_widen(r2 + 2), ldg_widen(r2 + 3));
          v3 = make_float4(ldg_widen(r3), ldg_widen(r3 + 1), ldg_widen(r3 + 2), ldg_widen(r3 + 3));
        }
        a0 = f4add(a0, make_float4(v0.x - s.x, v0.y - s.y, v0.z - s.z, v0.w - s.w));
        a1 = f4add(a1, make_float4(v1.x - s.x, v1.y - s.y, v1.z - s.z, v1.w - s.w));
        a2 = f4add(a2, make_float4(v2.x - s.x, v2.y - s.y, v2.z - s.z, v2.w - s.w));
        a3 = f4add(a3, make_float4(v3.x - s.x, v3.y - s.y, v3.z - s.z, v3.w - s.w));
      }
    }
    for (; k < ke; ++k) {
      const T* r = X + (int64_t)perm[begin + k] * ldx + col;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      v.x = ldg_widen(r) - s.x;
      if (col + 1 < D) v.y = ldg_widen(r + 1) - s.y;
      if (col + 2 < D) v.z = ldg_widen(r + 2) - s.z;
      if (col + 3 < D) v.w = ldg_widen(r + 3) - s.w;
      a0 = f4add(a0, v);
    }
    outer = f4add(outer, f4add(f4add(a0, a1), f4add(a2, a3)));
  }
  if (nlanes > 1) {  // row lanes of a column group are added in lane order: deterministic
    red[threadIdx.x] = outer;
    __syncthreads();
    if (rlane != 0) return;
    for (int r = 1; r < nlanes; ++r) outer = f4add(outer, red[r * tpr + tcol]);
  }
  if (!live) return;
  float* out = partial + ((int64_t)c * nsplit + split) * D + col;
  out[0] = outer.x;
  if (col + 1 < D) out[1] = outer.y;
  if (col + 2 < D) out[2] = outer.z;
  if (col + 3 < D) out[3] = outer.w;
}

// sums[c][j] = sum_split partial ;  accumulate != 0 adds to the existing sums (streaming / chunks)
__global__ void class_sums_finalize_kernel(const float* __restrict__ partial, int nsplit, int D, int C,
                                           float* __restrict__ sums, int accumulate) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= (int64_t)C * D) return;
  const int c = (int)(idx / D), j = (int)(idx % D);
  double acc = 0.0;
  for (int s = 0; s < nsplit; ++s) acc += (double)partial[((int64_t)c * nsplit + s) * D + j];
  if (accumulate) acc += (double)sums[idx];
  sums[idx] = (float)acc;
}

// Pilot shift of the one-pass class_statistics: shift[c][j] = mean of the first min(n_c, PILOT_ROWS) rows of
// class c in bucket order (0 for an empty class). The Gram centres on it and writes sum (x - shift) on the
// way; the epilogue corrects the Gram by n d d^T, d = mean - shift. |d| ~ sigma / sqrt(32) makes the centred
// values (1 + 1/32) times larger in square than with the exact mean, i.e. 3 % more 3xTF32 and truncation
// error. One thread per column, the rows added in order: a bf16 / fp16 X gives the bits of its float32 copy.
constexpr int PILOT_ROWS = 32;
constexpr int PILOT_THREADS = 128;

template <typename T>
__global__ void __launch_bounds__(PILOT_THREADS)
class_pilot_shift_kernel(const T* __restrict__ X, int64_t ldx, const int32_t* __restrict__ perm,
                         const int64_t* __restrict__ offsets, int D, float* __restrict__ shift) {
  const int c = blockIdx.y;
  const int col = blockIdx.x * PILOT_THREADS + threadIdx.x;
  if (col >= D) return;
  const int64_t begin = offsets[c];
  const int64_t n_c = offsets[c + 1] - begin;
  const int p = n_c < PILOT_ROWS ? (int)(n_c > 0 ? n_c : 0) : PILOT_ROWS;
  float v[PILOT_ROWS];
#pragma unroll
  for (int r = 0; r < PILOT_ROWS; ++r)  // all loads in flight, then the sum
    v[r] = r < p ? ldg_widen(X + (int64_t)__ldg(perm + begin + r) * ldx + col) : 0.f;
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < PILOT_ROWS; ++r) s += v[r];
  shift[(int64_t)c * D + col] = p > 0 ? s / (float)p : 0.f;
}

// means[c][j] = sums[c][j] / n_c (+ shift[c][j]);  0/0 -> NaN for an empty class, as torch.mean does.
__global__ void class_means_kernel(const float* __restrict__ sums, const int64_t* __restrict__ counts,
                                   const float* __restrict__ shift, int D, int C, float* __restrict__ means) {
  const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (idx >= (int64_t)C * D) return;
  const int c = (int)(idx / D);
  const float n = (float)counts[c];
  float m = sums[idx] / n;
  if (shift != nullptr) m += shift[idx];
  means[idx] = m;
}

// ------------------------------------------------------------------------------------------------
// K3 epilogue. One block per (class, 32x32 tile pair ti <= tj) of the upper triangle of gram.
//   cov[r][q] = (G[r][q] - n * d_r d_q) / (n - 1)   with d = mean - shift (nullptr -> 0)
//   sm [r][q] = cov[r][q] + mu_r mu_q
// and the mirrored entries, through a shared-memory transpose so both writes are coalesced.
// `cov` may alias `gram` (a block reads only its own upper tile before it writes that tile and its
// mirror, and no other block touches either). `sm` may be NULL. ddof = 1 (unbiased) or 0.
// ------------------------------------------------------------------------------------------------
// Address of Gram element (r, q), r <= q tile-wise, in the full (C, D, D) layout or in the packed
// list of 256 x 256 upper tiles written by the Gram kernel for multi-device callers.
__device__ __forceinline__ const float* gram_elem(const float* gram, int packed, int c, int D, int r, int q) {
  if (!packed) return gram + ((int64_t)c * D + r) * D + q;
  const int TT = (D + 255) / 256, T = TT * (TT + 1) / 2;
  const int tm = r >> 8, tn = q >> 8;
  const int64_t t = (int64_t)tm * TT - (int64_t)tm * (tm - 1) / 2 + (tn - tm);
  return gram + (((int64_t)c * T + t) * 256 + (r & 255)) * 256 + (q & 255);
}

// d = mean - shift. With centred_sums, `shift` holds the class sums of (x - s) the Gram was centred for and
// d = sums / n: exact to float32 rounding of d itself, where mean - s would lose the bits of |mean| >> |d|
// (data far from the origin).
__device__ __forceinline__ float centring_offset(const float* mu, const float* shift, int c, int D, int r, float n,
                                                 int centred_sums) {
  const float v = shift[(int64_t)c * D + r];
  return centred_sums ? v / n : mu[r] - v;
}

__global__ void __launch_bounds__(256)
stats_epilogue_kernel(const float* gram, int packed, const float* __restrict__ means,
                      const float* __restrict__ shift, const int64_t* __restrict__ counts, int D, int NT, int ddof,
                      float* cov, float* sm, const GramSources src, int centred_sums) {
  __shared__ float s_cov[32][33];
  __shared__ float s_mu_i[32], s_mu_j[32], s_d_i[32], s_d_j[32];
  const int c = blockIdx.y;
  // decode linear upper-triangular tile index -> (ti, tj), ti <= tj
  int t = blockIdx.x, ti = 0;
  for (;; ++ti) {
    const int cnt = NT - ti;
    if (t < cnt) break;
    t -= cnt;
  }
  const int tj = ti + t;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  const float* mu = means + (int64_t)c * D;
  const float n = (float)counts[c];
  if (threadIdx.x < 32) {
    const int r = ti * 32 + threadIdx.x, q = tj * 32 + threadIdx.x;
    s_mu_i[threadIdx.x] = r < D ? mu[r] : 0.f;
    s_mu_j[threadIdx.x] = q < D ? mu[q] : 0.f;
    s_d_i[threadIdx.x] = (shift != nullptr && r < D) ? centring_offset(mu, shift, c, D, r, n, centred_sums) : 0.f;
    s_d_j[threadIdx.x] = (shift != nullptr && q < D) ? centring_offset(mu, shift, c, D, q, n, centred_sums) : 0.f;
  }
  __syncthreads();
  const float nm1 = n - (float)ddof;
  for (int rr = ty; rr < 32; rr += 8) {
    const int r = ti * 32 + rr, q = tj * 32 + tx;
    float v = 0.f;
    if (r < D && q < D) {
      float g;
      if (src.n_src <= 1) {
        g = *gram_elem(gram, packed, c, D, r, q);
      } else {  // fixed order over the source ranks: the result does not depend on arrival order
        g = 0.f;
        for (int s = 0; s < src.n_src; ++s)
          g += *gram_elem(s == src.self ? gram : src.peers + s * src.stride, packed, c, D, r, q);
      }
      if (shift != nullptr && n > 0.f) g -= n * s_d_i[rr] * s_d_j[tx];  // empty class: d is NaN, n d d^T is 0
      v = g / nm1;
    }
    s_cov[rr][tx] = v;
  }
  __syncthreads();
  float* covc = cov + (int64_t)c * D * D;
  float* smc = sm != nullptr ? sm + (int64_t)c * D * D : nullptr;
  const bool diag = (ti == tj);
  for (int rr = ty; rr < 32; rr += 8) {
    const int r = ti * 32 + rr, q = tj * 32 + tx;
    if (r < D && q < D) {
      // on diagonal tiles only the upper part of gram is defined: take the mirrored value below it
      const float v = (diag && tx < rr) ? s_cov[tx][rr] : s_cov[rr][tx];
      covc[(int64_t)r * D + q] = v;
      if (smc != nullptr) smc[(int64_t)r * D + q] = v + s_mu_i[rr] * s_mu_j[tx];
    }
  }
  if (!diag) {
    for (int rr = ty; rr < 32; rr += 8) {  // transposed tile: rows from tj, cols from ti
      const int r = tj * 32 + rr, q = ti * 32 + tx;
      if (r < D && q < D) {
        const float v = s_cov[tx][rr];
        covc[(int64_t)r * D + q] = v;
        if (smc != nullptr) smc[(int64_t)r * D + q] = v + s_mu_j[rr] * s_mu_i[tx];
      }
    }
  }
}

// Same epilogue for D % 4 == 0 (16-byte aligned rows): 64 x 64 tiles, every global access is a
// float4 of a 256-byte row segment (the 32 x 32 scalar version moves 128-byte segments and reaches
// about half of the HBM bandwidth). Reads 1/2 C D^2 floats, writes 2 C D^2: HBM-bound.
__global__ void __launch_bounds__(256)
stats_epilogue_v4_kernel(const float* gram, int packed, const float* __restrict__ means,
                         const float* __restrict__ shift, const int64_t* __restrict__ counts, int D, int NT, int ddof,
                         float* cov, float* sm, const GramSources src, int centred_sums) {
  __shared__ float s_cov[64][65];
  __shared__ float s_mu_i[64], s_mu_j[64], s_d_i[64], s_d_j[64];
  const int c = blockIdx.y;
  int t = blockIdx.x, ti = 0;
  for (;; ++ti) {
    const int cnt = NT - ti;
    if (t < cnt) break;
    t -= cnt;
  }
  const int tj = ti + t;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;  // 16 float4 columns x 16 rows per pass
  const float* mu = means + (int64_t)c * D;
  const float n = (float)counts[c];
  if (threadIdx.x < 64) {
    const int r = ti * 64 + threadIdx.x, q = tj * 64 + threadIdx.x;
    s_mu_i[threadIdx.x] = r < D ? mu[r] : 0.f;
    s_mu_j[threadIdx.x] = q < D ? mu[q] : 0.f;
    s_d_i[threadIdx.x] = (shift != nullptr && r < D) ? centring_offset(mu, shift, c, D, r, n, centred_sums) : 0.f;
    s_d_j[threadIdx.x] = (shift != nullptr && q < D) ? centring_offset(mu, shift, c, D, q, n, centred_sums) : 0.f;
  }
  __syncthreads();
  const float nm1 = n - (float)ddof;
  const int q0 = tj * 64 + 4 * tx;  // D % 4 == 0: a float4 is entirely inside or outside the matrix
#pragma unroll
  for (int rr = ty; rr < 64; rr += 16) {
    const int r = ti * 64 + rr;
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < D && q0 < D) {
      if (src.n_src <= 1) {
        g = *reinterpret_cast<const float4*>(gram_elem(gram, packed, c, D, r, q0));
      } else {  // all sources' loads in flight, then one fixed-order sum
        for (int s = 0; s < src.n_src; ++s) {
          const float4 v = *reinterpret_cast<const float4*>(
              gram_elem(s == src.self ? gram : src.peers + s * src.stride, packed, c, D, r, q0));
          g.x += v.x; g.y += v.y; g.z += v.z; g.w += v.w;
        }
      }
      if (shift != nullptr && n > 0.f) {  // empty class: d is NaN, n d d^T is 0
        const float a = n * s_d_i[rr];
        g.x -= a * s_d_j[4 * tx]; g.y -= a * s_d_j[4 * tx + 1];
        g.z -= a * s_d_j[4 * tx + 2]; g.w -= a * s_d_j[4 * tx + 3];
      }
      g.x /= nm1; g.y /= nm1; g.z /= nm1; g.w /= nm1;
    }
    s_cov[rr][4 * tx] = g.x; s_cov[rr][4 * tx + 1] = g.y;
    s_cov[rr][4 * tx + 2] = g.z; s_cov[rr][4 * tx + 3] = g.w;
  }
  __syncthreads();
  float* covc = cov + (int64_t)c * D * D;
  float* smc = sm != nullptr ? sm + (int64_t)c * D * D : nullptr;
  const bool diag = (ti == tj);
#pragma unroll
  for (int rr = ty; rr < 64; rr += 16) {
    const int r = ti * 64 + rr;
    if (r < D && q0 < D) {
      float v[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int cc = 4 * tx + i;
        // on diagonal tiles only the upper part of gram is defined: take the mirrored value below it
        v[i] = (diag && cc < rr) ? s_cov[cc][rr] : s_cov[rr][cc];
      }
      *reinterpret_cast<float4*>(covc + (int64_t)r * D + q0) = make_float4(v[0], v[1], v[2], v[3]);
      if (smc != nullptr) {
        const float m = s_mu_i[rr];
        *reinterpret_cast<float4*>(smc + (int64_t)r * D + q0) =
            make_float4(v[0] + m * s_mu_j[4 * tx], v[1] + m * s_mu_j[4 * tx + 1], v[2] + m * s_mu_j[4 * tx + 2],
                        v[3] + m * s_mu_j[4 * tx + 3]);
      }
    }
  }
  if (!diag) {
    const int p0 = ti * 64 + 4 * tx;  // transposed tile: rows from tj, cols from ti
#pragma unroll
    for (int rr = ty; rr < 64; rr += 16) {
      const int r = tj * 64 + rr;
      if (r < D && p0 < D) {
        const float v0 = s_cov[4 * tx][rr], v1 = s_cov[4 * tx + 1][rr], v2 = s_cov[4 * tx + 2][rr],
                    v3 = s_cov[4 * tx + 3][rr];
        *reinterpret_cast<float4*>(covc + (int64_t)r * D + p0) = make_float4(v0, v1, v2, v3);
        if (smc != nullptr) {
          const float m = s_mu_j[rr];
          *reinterpret_cast<float4*>(smc + (int64_t)r * D + p0) =
              make_float4(v0 + m * s_mu_i[4 * tx], v1 + m * s_mu_i[4 * tx + 1], v2 + m * s_mu_i[4 * tx + 2],
                          v3 + m * s_mu_i[4 * tx + 3]);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// OAS shrinkage (reference statistics.py:84-93): trace and sum of squares of the sample covariance
// per class, then (1-rho) S + rho tr(S)/D I and the second moment rebuilt from it.
// ------------------------------------------------------------------------------------------------
constexpr int OAS_BLOCKS = 64;

__global__ void __launch_bounds__(256)
oas_reduce_kernel(const float* __restrict__ cov, int D, double* __restrict__ partial /*C x OAS_BLOCKS x 2*/) {
  __shared__ double s_tr[256], s_sq[256];
  const int c = blockIdx.y;
  const float* S = cov + (int64_t)c * D * D;
  const int64_t total = (int64_t)D * D;
  double tr = 0.0, sq = 0.0;
  for (int64_t i = blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)OAS_BLOCKS * 256) {
    const float v = S[i];
    sq += (double)v * (double)v;
    if (i / D == i % D) tr += (double)v;
  }
  s_tr[threadIdx.x] = tr;
  s_sq[threadIdx.x] = sq;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) {
      s_tr[threadIdx.x] += s_tr[threadIdx.x + o];
      s_sq[threadIdx.x] += s_sq[threadIdx.x + o];
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    partial[((int64_t)c * OAS_BLOCKS + blockIdx.x) * 2 + 0] = s_tr[0];
    partial[((int64_t)c * OAS_BLOCKS + blockIdx.x) * 2 + 1] = s_sq[0];
  }
}

__global__ void __launch_bounds__(256)
oas_apply_kernel(const double* __restrict__ partial, const float* __restrict__ means,
                 const int64_t* __restrict__ counts, int D, float* __restrict__ cov, float* __restrict__ sm) {
  __shared__ float s_rho, s_target;
  const int c = blockIdx.y;
  if (threadIdx.x == 0) {
    double tr = 0.0, sq = 0.0;
    for (int b = 0; b < OAS_BLOCKS; ++b) {
      tr += partial[((int64_t)c * OAS_BLOCKS + b) * 2 + 0];
      sq += partial[((int64_t)c * OAS_BLOCKS + b) * 2 + 1];
    }
    const float trf = (float)tr, sqf = (float)sq;
    const float n = (float)counts[c];
    const float two_over_d = (float)(2.0 / (double)D);
    const float num = (1.0f - two_over_d) * sqf + trf * trf;
    const float den = (n + 1.0f - two_over_d) * (sqf - trf * trf / (float)D);
    const float s = num / den;
    s_rho = (s < 1.0f) ? s : 1.0f;  // python min(1.0, s): NaN -> 1.0
    s_target = trf / (float)D;
  }
  __syncthreads();
  const float rho = s_rho, target = s_target;
  float* S = cov + (int64_t)c * D * D;
  float* M = sm != nullptr ? sm + (int64_t)c * D * D : nullptr;
  const float* mu = means + (int64_t)c * D;
  const int64_t total = (int64_t)D * D;
  for (int64_t i = blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)gridDim.x * 256) {
    const int r = (int)(i / D), q = (int)(i % D);
    const float v = (1.0f - rho) * S[i] + rho * (r == q ? target : 0.0f);
    S[i] = v;
    if (sm != nullptr) M[i] = v + mu[r] * mu[q];
  }
}

// Class counts as two exact float32 words (count / 2^20, count mod 2^20) behind the class sums: ONE small
// all-reduce carries both (a multi-device caller), and back to int64 afterwards. Exact below 2^44 rows.
__global__ void counts_pack_kernel(const int64_t* __restrict__ counts, int C, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const int64_t n = counts[c];
  out[c] = (float)(n >> 20);
  out[C + c] = (float)(n & ((1 << 20) - 1));
}
__global__ void counts_unpack_kernel(const float* __restrict__ in, int C, int64_t* __restrict__ counts) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  counts[c] = ((int64_t)llrintf(in[c]) << 20) + (int64_t)llrintf(in[C + c]);
}

}  // namespace

cudaError_t launch_counts_pack(const int64_t* counts, int C, float* out, cudaStream_t stream) {
  if (C <= 0) return cudaSuccess;
  counts_pack_kernel<<<(C + 255) / 256, 256, 0, stream>>>(counts, C, out);
  return cudaGetLastError();
}
cudaError_t launch_counts_unpack(const float* in, int C, int64_t* counts, cudaStream_t stream) {
  if (C <= 0) return cudaSuccess;
  counts_unpack_kernel<<<(C + 255) / 256, 256, 0, stream>>>(in, C, counts);
  return cudaGetLastError();
}

int class_sums_splits(int64_t n, int C, int D, int num_sms) {
  const int tpr = sums_threads_per_row(D);
  const int colblocks = (D + tpr * 4 - 1) / (tpr * 4);
  int64_t want = (8ll * num_sms + (int64_t)colblocks * C - 1) / ((int64_t)colblocks * (C > 0 ? C : 1));
  const int64_t avg = C > 0 ? n / C : n;
  int64_t cap = avg / (64 * (SUM_THREADS / tpr));  // keep >= 64 rows per row lane
  if (want > cap) want = cap;
  if (want < 1) want = 1;
  if (want > 4096) want = 4096;
  return (int)want;
}

cudaError_t launch_class_sums(const void* X, int elem, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                              const float* shift, int64_t n, int D, int C, float* sums, int accumulate,
                              float* partial_ws, int nsplit, cudaStream_t stream) {
  (void)n;
  if (C <= 0 || D <= 0) return cudaSuccess;
  // 4-element loads: rows aligned to 4 elements (16 bytes for float32, 8 for bf16 / fp16)
  const uintptr_t al = 4u * (uintptr_t)elem_bytes(elem) - 1u;
  const int vec_ok = (D % 4 == 0) && (ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & al) == 0);
  const int blk_ok = elem == ELEM_F32 ? vec_ok : (D % 4 == 0);
  const int tpr = sums_threads_per_row(D);
  dim3 grid((D + tpr * 4 - 1) / (tpr * 4), nsplit, C);
  if (elem == ELEM_BF16)
    class_sums_kernel<<<grid, SUM_THREADS, 0, stream>>>(static_cast<const __nv_bfloat16*>(X), ldx, perm, offsets,
                                                        shift, D, nsplit, partial_ws, vec_ok, blk_ok);
  else if (elem == ELEM_F16)
    class_sums_kernel<<<grid, SUM_THREADS, 0, stream>>>(static_cast<const __half*>(X), ldx, perm, offsets, shift, D,
                                                        nsplit, partial_ws, vec_ok, blk_ok);
  else
    class_sums_kernel<<<grid, SUM_THREADS, 0, stream>>>(static_cast<const float*>(X), ldx, perm, offsets, shift, D,
                                                        nsplit, partial_ws, vec_ok, blk_ok);
  const int64_t total = (int64_t)C * D;
  class_sums_finalize_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(partial_ws, nsplit, D, C, sums,
                                                                               accumulate);
  return cudaGetLastError();
}

cudaError_t launch_class_pilot_shift(const void* X, int elem, int64_t ldx, const int32_t* perm,
                                    const int64_t* offsets, int D, int C, float* shift, cudaStream_t stream) {
  if (C <= 0 || D <= 0) return cudaSuccess;
  const dim3 grid((D + PILOT_THREADS - 1) / PILOT_THREADS, C);
  if (elem == ELEM_BF16)
    class_pilot_shift_kernel<<<grid, PILOT_THREADS, 0, stream>>>(static_cast<const __nv_bfloat16*>(X), ldx, perm,
                                                                 offsets, D, shift);
  else if (elem == ELEM_F16)
    class_pilot_shift_kernel<<<grid, PILOT_THREADS, 0, stream>>>(static_cast<const __half*>(X), ldx, perm, offsets, D,
                                                                 shift);
  else
    class_pilot_shift_kernel<<<grid, PILOT_THREADS, 0, stream>>>(static_cast<const float*>(X), ldx, perm, offsets, D,
                                                                 shift);
  return cudaGetLastError();
}

cudaError_t launch_class_sums_finalize(const float* partial, int nsplit, int D, int C, float* sums,
                                       cudaStream_t stream) {
  const int64_t total = (int64_t)C * D;
  if (total <= 0) return cudaSuccess;
  class_sums_finalize_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(partial, nsplit, D, C, sums, 0);
  return cudaGetLastError();
}

cudaError_t launch_class_means(const float* sums, const int64_t* counts, const float* shift, int D, int C,
                               float* means, cudaStream_t stream) {
  const int64_t total = (int64_t)C * D;
  if (total <= 0) return cudaSuccess;
  class_means_kernel<<<(int)((total + 255) / 256), 256, 0, stream>>>(sums, counts, shift, D, C, means);
  return cudaGetLastError();
}

size_t stats_epilogue_workspace_bytes(int C) { return (size_t)(C > 0 ? C : 1) * OAS_BLOCKS * 2 * sizeof(double); }

cudaError_t launch_stats_epilogue(const float* gram, int packed, const float* means, const float* shift,
                                  const int64_t* counts, int D, int C, int estimator, int ddof, float* cov, float* sm,
                                  void* ws, cudaStream_t stream, GramSources src, int centred_sums) {
  if (C <= 0 || D <= 0) return cudaSuccess;
  const bool al16 = ((reinterpret_cast<uintptr_t>(gram) | reinterpret_cast<uintptr_t>(cov) |
                      reinterpret_cast<uintptr_t>(sm) | reinterpret_cast<uintptr_t>(src.peers) |
                      (uintptr_t)((src.stride & 3) * 4)) & 15) == 0;
  if (D % 4 == 0 && al16) {
    const int NT = (D + 63) / 64;
    stats_epilogue_v4_kernel<<<dim3(NT * (NT + 1) / 2, C), 256, 0, stream>>>(gram, packed, means, shift, counts, D, NT,
                                                                             ddof, cov, sm, src, centred_sums);
  } else {
    const int NT = (D + 31) / 32;
    stats_epilogue_kernel<<<dim3(NT * (NT + 1) / 2, C), 256, 0, stream>>>(gram, packed, means, shift, counts, D, NT, ddof,
                                                                          cov, sm, src, centred_sums);
  }
  if (estimator == 1) {
    double* partial = static_cast<double*>(ws);
    oas_reduce_kernel<<<dim3(OAS_BLOCKS, C), 256, 0, stream>>>(cov, D, partial);
    int nb = (int)(((int64_t)D * D + 256 * 8 - 1) / (256 * 8));
    if (nb > 1024) nb = 1024;
    if (nb < 1) nb = 1;
    oas_apply_kernel<<<dim3(nb, C), 256, 0, stream>>>(partial, means, counts, D, cov, sm);
  }
  return cudaGetLastError();
}

}  // namespace sqfa
