// K5: per-class factorisation and the pairwise SPD distances with their analytic gradient.
//
// Reference path replaced (/root/reference/src/sqfa/):
//   spd_inv_sqrt            linalg.py:144-162   eigh-based whitening of every class matrix
//   generalized_eigenvalues linalg.py:48-70     C x C conjugations + C*C LAPACK eigvalsh calls
//   affine_invariant(_sq)   distances.py:46-89  sum log^2(lambda), sqrt(. + 1e-6)
//   fisher_rao_lower_bound(_sq) distances.py:177-237  AI^2 of the embedded matrices / 2
//   log_euclidean(_sq), spd_log  distances.py:92-138, linalg.py:165-183
//   closure loss + NaN/inf guard + autograd backward   _optim.py:16-30, 90-96
//
// Formulation. For a pair (i, j) the generalized eigenvalues of (E_i, E_j) are the squared singular
// values of B = L_j^-1 L_i (E = L L^T Cholesky). A one-sided (Hestenes) Jacobi orthogonalises the
// columns of A = B^T: A_f = A V, |a_q|^2 = lambda_q. m <= 34: columns in registers, two per lane, several
// problems per warp (pair_cp_kernel); 34 < m <= 64: columns in shared memory (pair_ai_kernel).
// The generalized eigenvectors come for free as Y = L_i^-T A_f (y_q^T E_j y_q = 1), so
//   d(d^2)/dE_i =  sum_q (2 log(lambda_q) / lambda_q) y_q y_q^T
//   d(d^2)/dE_j = -sum_q (2 log(lambda_q))            y_q y_q^T
// -- no 1/(lambda_a - lambda_b) terms (the eigh backward of the reference has them and NaNs on
// repeated eigenvalues). Only the strict lower triangle (i > j) is evaluated: the reference
// computes all C*C pairs and then reads the lower triangle (_optim.py:94).
//
// Bures-Wasserstein (m <= 34, column-pair kernel): the same Jacobi on A = L_i^T L_j instead. Its singular
// values sigma_q = |a_q| sum to the fidelity tr((E_j^1/2 E_i E_j^1/2)^1/2), so
//   d^2 = |L_i|_F^2 + |L_j|_F^2 - 2 sum_q sigma_q                         (clamped at 0)
//   d(d^2)/dE_i = I - sum_q sigma_q^-1 y_q y_q^T,   y_q = L_i^-T a_q
//   d(d^2)/dE_j = I - sum_q sigma_q^-3 z_q z_q^T,   z_q = L_i a_q
// -- again no 1/(sigma_a - sigma_b) terms. The Gaussian form adds |mu_i - mu_j|^2 (closure only).
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cuda_runtime.h>

#include "../../include/sqfa_b200.h"
#include "sqfa_internal.h"
#include "pair_tiles.cuh"
#include "spd_factor.cuh"

namespace sqfa {

// Deterministic accumulation. A warp owns a TILE of R x R pairs, (rows i = bi R + ii, columns
// j = bj R + jj); it walks the tile row by row (the pairs of a row side by side in the column-pair
// kernel), sums dLoss/dE_i over the row and keeps dLoss/dE_j of its R columns in shared memory, then
// stores both as per-tile PARTIALS (plain stores, every slot written). A second kernel sums, for every
// class, the partials of the tiles in its block row and block column in a fixed order. No floating-point
// atomics anywhere: loss and gradient are bit-reproducible from run to run (L-BFGS amplifies noise).
PairTiles make_pair_tiles(int nA, int nB, int tri, int64_t pair_begin, int64_t pair_end, int R) {
  PairTiles T;
  T.R = R < 1 ? 1 : R;
  T.tri = tri;
  T.nbj = (nB + T.R - 1) / T.R;
  T.bi0 = 0; T.bi1 = -1; T.tile0 = 0; T.ntiles = 0;
  if (pair_end <= pair_begin) return T;
  int64_t i_first, i_last;
  if (tri) {
    auto row_of = [](int64_t p) {
      int64_t ii = (int64_t)((1.0 + std::sqrt(1.0 + 8.0 * (double)p)) * 0.5);
      while (ii * (ii - 1) / 2 > p) --ii;
      while ((ii + 1) * ii / 2 <= p) ++ii;
      return ii;
    };
    i_first = row_of(pair_begin);
    i_last = row_of(pair_end - 1);
  } else {
    i_first = pair_begin / (nB > 0 ? nB : 1);
    i_last = (pair_end - 1) / (nB > 0 ? nB : 1);
  }
  T.bi0 = (int)(i_first / T.R);
  T.bi1 = (int)(i_last / T.R);
  if (tri) {
    T.tile0 = (int64_t)T.bi0 * (T.bi0 + 1) / 2;
    T.ntiles = (int64_t)(T.bi1 + 1) * (T.bi1 + 2) / 2 - T.tile0;
  } else {
    T.tile0 = (int64_t)T.bi0 * T.nbj;
    T.ntiles = (int64_t)(T.bi1 - T.bi0 + 1) * T.nbj;
  }
  return T;
}

namespace {

constexpr int PAIR_WARPS = 4;
constexpr float JACOBI_TOL = 1e-6f;  // |a_p . a_q| <= tol |a_p||a_q| counts as orthogonal
constexpr int JACOBI_MAX_SWEEPS = 24;
constexpr float JACOBI_LAST = 3e-4f;  // a sweep of rotations all below this is the last (they leave ~1e-7)
constexpr float DIST_EPS = 1e-6f;    // distances.py:29 EPSILON

__device__ __forceinline__ float rcp_approx(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// round-robin (circle method) partner of player p in round r, mp players (mp even)
__device__ __forceinline__ int rr_partner(int p, int r, int mp) {
  const int n1 = mp - 1;
  // players i, j < n1 meet in the round with i + j == 2 r (mod n1); the one left over (2 i == 2 r,
  // i.e. i == r because n1 is odd) meets the fixed player n1
  if (p == n1) return r;
  int q = 2 * r - p;  // in (-n1, 2 n1): one conditional correction replaces the modulo
  if (q < 0) q += n1;
  else if (q >= n1) q -= n1;
  return q == p ? n1 : q;
}

// One-sided Jacobi on the columns of the m x mp matrix in `cur` (row stride ld, column q of slot
// t = lane + 32 t). Double-buffered between cur and nxt; returns the buffer holding the result.
__device__ float* warp_jacobi(float* cur, float* nxt, int m, int mp, int ld, int lane) {
  const int nslot = (mp + 31) >> 5;
  for (int sweep = 0; sweep < JACOBI_MAX_SWEEPS; ++sweep) {
    bool rotated = false;
    for (int r = 0; r < mp - 1; ++r) {
      for (int t = 0; t < nslot; ++t) {
        const int p = lane + 32 * t;
        if (p < mp) {
          const int q = rr_partner(p, r, mp);
          float aa = 0.f, bb = 0.f, ab = 0.f;
          for (int s = 0; s < m; ++s) {
            const float x = cur[s * ld + p], y = cur[s * ld + q];
            aa += x * x; bb += y * y; ab += x * y;
          }
          // rotation for the ordered pair (lo, hi): x_lo' = c x_lo - s x_hi, x_hi' = s x_lo + c x_hi
          const bool is_lo = p < q;
          const float alpha = is_lo ? aa : bb, beta = is_lo ? bb : aa;
          float cs = 1.f, sn = 0.f;
          const float ab_sq = ab * ab, scale = alpha * beta;
          if (ab_sq > (JACOBI_TOL * JACOBI_TOL) * scale && alpha > 0.f && beta > 0.f) {
            // same rules as the register kernel: approximate reciprocal / square root for the angle,
            // and a sweep whose rotations were all below JACOBI_LAST is the last one
            const float zeta = (beta - alpha) * rcp_approx(2.f * ab);
            const float tt = copysignf(rcp_approx(fabsf(zeta) + sqrt_approx(fmaf(zeta, zeta, 1.f))), zeta);
            cs = rsqrtf(fmaf(tt, tt, 1.f));
            sn = cs * tt;
            rotated = rotated || ab_sq > (JACOBI_LAST * JACOBI_LAST) * scale;
          }
          const float mine = cs, other = is_lo ? -sn : sn;
          for (int s = 0; s < m; ++s) nxt[s * ld + p] = mine * cur[s * ld + p] + other * cur[s * ld + q];
        }
      }
      __syncwarp();
      float* tmp = cur; cur = nxt; nxt = tmp;
    }
    if (!__any_sync(0xffffffffu, rotated)) break;
  }
  return cur;
}

__device__ __forceinline__ float finish_distance(float d2, int dist, float* dd_dd2) {
  const int base = dist & 15;
  const float cfac = (base == SQFA_DIST_FISHER_RAO_LB) ? 0.5f : 1.f;
  if (dist & SQFA_DIST_SQUARED) {
    *dd_dd2 = cfac;
    return cfac * d2;
  }
  const float d = sqrtf(cfac * d2 + DIST_EPS);
  *dd_dd2 = cfac / (2.f * d);
  return d;
}

// ------------------------------------------------------------------------------------------------
// per-class factorisation
//   AI / FR: W[c] = [L (m*m) | L^-1 (m*m)]
//   LE     : W[c] = [V (m*m) | lambda (m) | log lambda (m) | logE (m*m)]
// ------------------------------------------------------------------------------------------------
// floats of per-warp scratch of the factorisation
__host__ __device__ inline int factor_scratch_floats(int m) {
  const int mp = (m + 1) & ~1;
  const int ld = (mp > 32 ? 64 : 32) + 1;
  return 4 * m * ld + 2 * m;
}

// One warp factorises one SPD matrix Esrc (m x m, global or shared memory) into W (layout above).
__device__ void warp_factor_class(const float* Esrc, int m, int dist, float* __restrict__ Wc, int32_t* __restrict__ flag,
                                  float* scratch, int lane) {
  const int mp = (m + 1) & ~1;
  const int ld = (mp > 32 ? 64 : 32) + 1;
  float* La = scratch;
  float* Li = La + m * ld;
  float* bufA = Li + m * ld;
  float* bufB = bufA + m * ld;
  float* lam = bufB + m * ld;
  float* loglam = lam + m;
  const bool ok = warp_cholesky_inverse(Esrc, La, Li, m, ld, lane);
  if (!ok && lane == 0) atomicOr(flag, 1);
  const bool le = (dist & 15) == SQFA_DIST_LOG_EUCLIDEAN;
  if (!le) {
    for (int idx = lane; idx < m * m; idx += 32) {
      const int r = idx / m, q = idx % m;
      Wc[idx] = (q <= r) ? La[r * ld + q] : 0.f;
      Wc[m * m + idx] = Li[r * ld + q];
    }
    return;
  }
  // LE: eigendecomposition of E = L L^T through Jacobi on the columns of A0 = L^T
  for (int s = 0; s < m; ++s)
    for (int q = lane; q < (ld - 1); q += 32) bufA[s * ld + q] = (q < m && s <= q) ? La[q * ld + s] : 0.f;
  __syncwarp();
  float* Af = warp_jacobi(bufA, bufB, m, mp, ld, lane);
  float* Vb = (Af == bufA) ? bufB : bufA;
  for (int q = lane; q < m; q += 32) {
    float n2 = 0.f;
    for (int s = 0; s < m; ++s) n2 += Af[s * ld + q] * Af[s * ld + q];
    lam[q] = n2;
    loglam[q] = logf(n2);
    // V[:, q] = L^-T a_q : A_f = L^T V with V orthogonal, so this is already a unit eigenvector
    for (int r = 0; r < m; ++r) {
      float v = 0.f;
      for (int s = r; s < m; ++s) v += Li[s * ld + r] * Af[s * ld + q];
      Vb[r * ld + q] = v;
    }
  }
  __syncwarp();
  for (int idx = lane; idx < m * m; idx += 32) {
    const int r = idx / m, s = idx % m;
    Wc[idx] = Vb[r * ld + s];
    float a = 0.f;
    for (int q = 0; q < m; ++q) a += loglam[q] * Vb[r * ld + q] * Vb[s * ld + q];
    Wc[m * m + 2 * m + idx] = a;
  }
  for (int q = lane; q < m; q += 32) {
    Wc[m * m + q] = lam[q];
    Wc[m * m + m + q] = loglam[q];
  }
}

__global__ void __launch_bounds__(PAIR_WARPS * 32)
class_factor_kernel(const float* __restrict__ E, int C, int m, int dist, float* __restrict__ W,
                    int32_t* __restrict__ flag) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + warp;
  if (c >= C) return;
  const int64_t wfl = ((dist & 15) == SQFA_DIST_LOG_EUCLIDEAN) ? 2 * m * m + 2 * m : 2 * m * m;
  warp_factor_class(E + (int64_t)c * m * m, m, dist, W + c * wfl, flag, smem + (size_t)warp * factor_scratch_floats(m),
                    lane);
}

// Closure: everything between the projection and the pair kernel for one class, one warp:
//   E_c from the chunk partials of Psi_c and mu'_c (assemble_class_matrix, spd_factor.cuh),
//   W_c = factorisation of E_c (above).  E is also written out (m x m per class).
// mu'_c is formed whenever MuPart is given (Fisher-Rao, Gaussian Wasserstein); only Fisher-Rao embeds it.
__global__ void __launch_bounds__(PAIR_WARPS * 32)
class_prepare_kernel(const float* __restrict__ PsiPart, const float* __restrict__ MuPart, int nchunk, float noise,
                     int C, int k, int dist, float* __restrict__ Mu, float* __restrict__ E, float* __restrict__ W,
                     int32_t* __restrict__ flag) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + warp;
  if (c >= C) return;
  const bool fr = (dist & 15) == SQFA_DIST_FISHER_RAO_LB;
  const int m = fr ? k + 1 : k;
  const int per_warp = factor_scratch_floats(m) + m * m + k;
  float* scratch = smem + (size_t)warp * per_warp;
  float* Es = scratch + factor_scratch_floats(m);
  float* mus = Es + m * m;
  assemble_class_matrix(PsiPart, MuPart, nchunk, noise, c, k, fr, Mu, mus, Es, E, lane);
  __syncwarp();
  const int64_t wfl = ((dist & 15) == SQFA_DIST_LOG_EUCLIDEAN) ? 2 * m * m + 2 * m : 2 * m * m;
  warp_factor_class(Es, m, dist, W + c * wfl, flag, scratch, lane);
}

// ------------------------------------------------------------------------------------------------
// pair kernel, affine-invariant family (AI, FR lower bound): one warp per pair
// ------------------------------------------------------------------------------------------------
// Column stride (floats) of the column-contiguous matrices of the shared-memory variant: a multiple
// of 4 whose quarter is odd, so that 16-byte accesses of 8 lanes to 8 different columns hit 8 different
// bank groups (conflict-free LDS.128 / STS.128).
__host__ __device__ inline int pair_col_stride(int m) {
  int m4 = (m + 3) >> 2;
  if ((m4 & 1) == 0) ++m4;
  return 4 * m4;
}

// One-sided Jacobi on the mp (even) columns of a matrix stored column-contiguous (column p at
// A + p * ldc, entries >= m are zero). Lane t < mp / 2 owns ONE COLUMN PAIR per round of the round-robin
// schedule: it loads both columns into registers (16-byte loads), forms the three dot products and the
// rotation, and writes both columns back in place -- no other lane touches them in that round, so there
// is no double buffer, no shuffle and no redundant dot product. M4 = float4s per column the registers
// are sized for.
template <int M4>
__device__ void warp_jacobi_cols(float* A, int m, int mp, int ldc, int lane) {
  const int n1 = mp - 1, np = mp >> 1;
  const int m4 = (m + 3) >> 2;
  for (int sweep = 0; sweep < JACOBI_MAX_SWEEPS; ++sweep) {
    bool rotated = false;
    for (int r = 0; r < n1; ++r) {
      if (lane < np) {
        // circle method: the fixed player n1 meets r; the others meet their mirror image around r
        int p, q;
        if (lane == 0) {
          p = n1; q = r;
        } else {
          p = r + lane; if (p >= n1) p -= n1;
          q = r - lane; if (q < 0) q += n1;
        }
        const int lo = p < q ? p : q, hi = p < q ? q : p;
        float4* xp = reinterpret_cast<float4*>(A + lo * ldc);
        float4* yp = reinterpret_cast<float4*>(A + hi * ldc);
        float4 x[M4], y[M4];
        float2 aa = make_float2(0.f, 0.f), bb = aa, ab = aa;
#pragma unroll
        for (int i = 0; i < M4; ++i) {
          if (i < m4) {
            x[i] = xp[i];
            y[i] = yp[i];
            const float2 x0 = make_float2(x[i].x, x[i].y), x1 = make_float2(x[i].z, x[i].w);
            const float2 y0 = make_float2(y[i].x, y[i].y), y1 = make_float2(y[i].z, y[i].w);
            aa = __ffma2_rn(x0, x0, aa); aa = __ffma2_rn(x1, x1, aa);
            bb = __ffma2_rn(y0, y0, bb); bb = __ffma2_rn(y1, y1, bb);
            ab = __ffma2_rn(x0, y0, ab); ab = __ffma2_rn(x1, y1, ab);
          }
        }
        const float alpha = aa.x + aa.y, beta = bb.x + bb.y, gamma = ab.x + ab.y;
        const float g2 = gamma * gamma, scale = alpha * beta;
        if (g2 > (JACOBI_TOL * JACOBI_TOL) * scale && alpha > 0.f && beta > 0.f) {
          // same rules as the register kernel: approximate reciprocal / square root for the angle, and
          // a sweep whose rotations were all below JACOBI_LAST is the last one
          const float zeta = (beta - alpha) * rcp_approx(2.f * gamma);
          const float tt = copysignf(rcp_approx(fabsf(zeta) + sqrt_approx(fmaf(zeta, zeta, 1.f))), zeta);
          const float cs = rsqrtf(fmaf(tt, tt, 1.f)), sn = cs * tt;
          rotated = rotated || g2 > (JACOBI_LAST * JACOBI_LAST) * scale;
          const float2 c2 = make_float2(cs, cs), s2 = make_float2(sn, sn), ns2 = make_float2(-sn, -sn);
#pragma unroll
          for (int i = 0; i < M4; ++i) {
            if (i < m4) {  // x' = c x - s y, y' = s x + c y
              const float2 x0 = make_float2(x[i].x, x[i].y), x1 = make_float2(x[i].z, x[i].w);
              const float2 y0 = make_float2(y[i].x, y[i].y), y1 = make_float2(y[i].z, y[i].w);
              const float2 nx0 = __ffma2_rn(c2, x0, __fmul2_rn(ns2, y0)), nx1 = __ffma2_rn(c2, x1, __fmul2_rn(ns2, y1));
              const float2 ny0 = __ffma2_rn(c2, y0, __fmul2_rn(s2, x0)), ny1 = __ffma2_rn(c2, y1, __fmul2_rn(s2, x1));
              xp[i] = make_float4(nx0.x, nx0.y, nx1.x, nx1.y);
              yp[i] = make_float4(ny0.x, ny0.y, ny1.x, ny1.y);
            }
          }
        }
      }
      __syncwarp();
    }
    if (!__any_sync(0xffffffffu, rotated)) break;
  }
}

// floats of per-warp scratch of the shared-memory pair kernel
__host__ __device__ inline int pair_smem_floats(int m) {
  const int mp = (m + 1) & ~1, ldc = pair_col_stride(m);
  return mp * ldc + m * ldc + ((m * m + 3) & ~3) + 4 * ((m + 3) & ~3);
}

template <int M4>
__global__ void __launch_bounds__(PAIR_WARPS * 32)
pair_ai_kernel(const PairArgs A) {
  // shared-memory variant (32 < m <= 64): tiles are single pairs (R = 1), tile (bi, bj) = pair (i, j).
  // Matrices are column-contiguous: column q of A = (L_j^-1 L_i)^T at bufA + q * ldc.
  extern __shared__ __align__(16) float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (t >= A.T.ntiles) return;
  const int m = A.m, nB = A.nB, tri = A.tri, dist = A.dist;
  int i, j;
  decode_tile(A.T, t, i, j);
  const bool active = pair_in_launch(i, j, A.nA, nB, tri, A.pair_begin, A.pair_end);
  const bool want_grad = A.rowpart != nullptr;
  const int mp = (m + 1) & ~1;
  const int ldc = pair_col_stride(m);
  const int nslot = (m + 31) >> 5;
  const int mpad = (m + 3) & ~3;
  float* bufA = smem + (size_t)warp * pair_smem_floats(m);  // [mp][ldc]  columns of A, then of A_f
  float* bufY = bufA + mp * ldc;                            // [m][ldc]   Linv_j^T (staging), later columns of Y
  float* Ls = bufY + m * ldc;                               // [m][m]     L_i, later L_i^-1
  float* ci = Ls + ((m * m + 3) & ~3);                      // per-eigenvalue coefficients
  float* cj = ci + mpad;
  float* lamv = cj + mpad;
  float dval = 0.f, bad = 0.f;
  float* gi = want_grad ? A.rowpart + t * m * m : nullptr;
  float* gj = want_grad ? A.colpart + t * m * m : nullptr;
  if (!active && want_grad) {  // every partial slot is written: the reduction reads all of them
    for (int idx = lane; idx < m * m; idx += 32) { gi[idx] = 0.f; gj[idx] = 0.f; }
  }
  if (active) {
    const float* Wi = A.Wa + (int64_t)i * 2 * m * m;
    const float* Wj = A.Wb + (int64_t)j * 2 * m * m;
    // stage L_i (row-major) and L_j^-1 transposed (bufY[r][q] = Linv_j[q][r], row stride ldc); zero A
    for (int idx = lane; idx < mp * ldc; idx += 32) bufA[idx] = 0.f;
    for (int idx = lane; idx < m * m; idx += 32) {
      Ls[idx] = Wi[idx];
      const int q = idx / m, r = idx % m;
      bufY[r * ldc + q] = Wj[m * m + idx];
    }
    __syncwarp();
    // column q of A: A[s][q] = sum_{r >= s} Linv_j[q][r] L_i[r][s]   (column mp - 1 > m - 1 stays zero)
    for (int tt = 0; tt < nslot; ++tt) {
      const int q = lane + 32 * tt;
      if (q < m) {
        for (int s = 0; s < m; ++s) {
          float a = 0.f;
          for (int r = s; r < m; ++r) a += bufY[r * ldc + q] * Ls[r * m + s];
          bufA[q * ldc + s] = a;
        }
      }
    }
    __syncwarp();
    warp_jacobi_cols<M4>(bufA, m, mp, ldc, lane);
    // eigenvalues and the distance
    float d2 = 0.f;
    for (int tt = 0; tt < nslot; ++tt) {
      const int q = lane + 32 * tt;
      if (q < m) {
        float n2 = 0.f;
        for (int s = 0; s < m; ++s) n2 += bufA[q * ldc + s] * bufA[q * ldc + s];
        const float ll = logf(n2);
        d2 += ll * ll;
        ci[q] = 2.f * ll / n2;
        cj[q] = -2.f * ll;
        lamv[q] = n2;
      }
    }
    d2 = warp_sum(d2);
    if (A.eig_out != nullptr) {  // generalized eigenvalues, descending (linalg.py:69-70)
      __syncwarp();
      float* eo = A.eig_out + ((int64_t)i * nB + j) * m;
      for (int tt = 0; tt < nslot; ++tt) {
        const int q = lane + 32 * tt;
        if (q < m) {
          const float v = lamv[q];
          int rank = 0;
          for (int u = 0; u < m; ++u) rank += (lamv[u] > v || (lamv[u] == v && u < q)) ? 1 : 0;
          eo[rank] = v;
        }
      }
    }
    float dd_dd2;
    dval = finish_distance(d2, dist, &dd_dd2);
    if (!isfinite(dval)) bad = 1.f;
    if (A.dist_out != nullptr && lane == 0) {
      A.dist_out[(int64_t)i * nB + j] = dval;
      if (tri) A.dist_out[(int64_t)j * nB + i] = dval;
    }
    if (want_grad) {
      float w = A.weight * dd_dd2;
      if (A.gD != nullptr)
        w *= tri ? (A.gD[(int64_t)i * nB + j] + A.gD[(int64_t)j * nB + i]) : A.gD[(int64_t)i * nB + j];
      __syncwarp();
      // column q of Y = L_i^-T A_f : Y[r][q] = sum_{s >= r} Linv_i[s][r] A_f[s][q]
      for (int idx = lane; idx < m * m; idx += 32) Ls[idx] = Wi[m * m + idx];
      __syncwarp();
      for (int tt = 0; tt < nslot; ++tt) {
        const int q = lane + 32 * tt;
        if (q < m) {
          for (int r = 0; r < m; ++r) {
            float v = 0.f;
            for (int s = r; s < m; ++s) v += Ls[s * m + r] * bufA[q * ldc + s];
            bufY[q * ldc + r] = v;
          }
        }
      }
      __syncwarp();
      // G_i[r][s] = sum_q (w ci_q) Y[r][q] Y[s][q],  G_j[r][s] = sum_q (w cj_q) Y[r][q] Y[s][q];
      // lane <-> column s; stored as this pair's partials (plain stores)
      for (int tt = 0; tt < nslot; ++tt) {
        const int s = lane + 32 * tt;
        if (s < m) {
          for (int r = 0; r < m; ++r) {
            float a = 0.f, b = 0.f;
            for (int q = 0; q < m; ++q) {
              const float yy = bufY[q * ldc + r] * bufY[q * ldc + s];
              a += ci[q] * yy;
              b += cj[q] * yy;
            }
            gi[r * m + s] = w * a;
            gj[r * m + s] = w * b;
          }
        }
      }
    }
  }
  if (A.losspart != nullptr && lane == 0) {
    A.losspart[2 * t] = dval;
    A.losspart[2 * t + 1] = bad;
  }
}

// ------------------------------------------------------------------------------------------------
// pair kernel, affine-invariant family, COLUMN-PAIR variant for m <= 34 (MJ = m rounded up to even).
//
// A lane owns TWO adjacent columns of A = (L_j^-1 L_i)^T in registers (positions 2 lg and 2 lg + 1),
// so a problem occupies LP = MJ / 2 lanes and a warp works on NP = 32 / LP problems side by side
// (m = 17: 3, m = 9: 6, m = 4: 16, m = 33: 1) -- the pairs of one ROW of its R x R tile, which share L_i.
// The Jacobi pairing is the odd-even transposition ordering: in an odd step a lane rotates its own two
// columns (no data movement at all: one dot product, one set of rotation parameters, both columns
// updated -- nothing is computed twice), in an even step the pairs (2 lg + 1, 2 lg + 2) straddle
// neighbouring lanes: the left lane fetches the neighbour's column with MJ shuffles, rotates, and sends
// the neighbour's half back. Every rotation also swaps the two columns, which is what makes MJ steps
// meet every pair of columns exactly once (and reverses the column order: the zero padding column of an
// odd m is at position MJ - 1 after an even number of sweeps, at 0 after an odd number).
// Against one column per lane (round-robin pairing, partner's column by shuffle, dot product and
// rotation parameters computed by both lanes, 18 of 32 lanes busy at m = 17) this executes about a
// third of the warp instructions per pair.
// ------------------------------------------------------------------------------------------------
template <int MJ>
struct CpGeom {
  static constexpr int LP = MJ / 2;          // lanes per problem
  static constexpr int NP = 32 / LP;         // problems per warp
  static constexpr int MP4 = (MJ + 3) & ~3;  // row length in shared memory (16-byte loads)
  static constexpr int MH = MP4 / 2;         // packed register pairs per column
  static constexpr int LDJ = MP4 + 1;        // odd row stride of Linv_j (lane-varying scalar reads)
};

// floats of shared memory per warp: [L_i rows | per problem: Linv_j rows (later Y rows), coefficients, column
// accumulator]. Linv_j is dead once the columns of a pair are formed and Y takes its place (Linv_j is staged
// again for the next row of the tile): 11 KB per warp at m = 17, which is what lets 20 warps share an SM.
__host__ __device__ inline int cp_group_floats(int MJ, int m) {
  const int MP4 = (MJ + 3) & ~3;
  return ((MJ * (MP4 + 1) + 3) & ~3) + 2 * MP4 + ((m * m + 3) & ~3);
}
__host__ __device__ inline int cp_warp_floats(int MJ, int m) {
  const int MP4 = (MJ + 3) & ~3;
  return m * MP4 + (32 / (MJ / 2)) * cp_group_floats(MJ, m);
}

__device__ __forceinline__ float rsqrt_approx(float x) {
  float r;
  asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Rotation of the column pair (x at position p, y at position p + 1) with squared norms alpha, beta and
// x . y = ab, FOLLOWED BY THE SWAP: position p receives c (y + t x) (squared norm n0), position p + 1 receives
// c (x - t y) (n1). No rotation (converged pair, or has_pair false): t = 0, c = 1 -- the swap alone.
__device__ __forceinline__ void cp_rotation(float alpha, float beta, float ab, bool has_pair, float& t, float& c,
                                            float& n0, float& n1, bool& rotated) {
  t = 0.f; c = 1.f; n0 = beta; n1 = alpha;
  const float ab_sq = ab * ab, scale = alpha * beta;
  if (has_pair && ab_sq > (JACOBI_TOL * JACOBI_TOL) * scale) {
    // t = sign(zeta) / (|zeta| + sqrt(zeta^2 + 1)) with zeta = d / h, d = beta - alpha, h = 2 ab, written as
    // sign(d) h / (|d| + sqrt(d^2 + h^2)): one reciprocal less on the dependent chain, no division by a tiny ab.
    // Approximate reciprocal / square roots: a rotation only has to be orthogonal to fp32 precision
    // (an angle off by 1e-7 leaves an off-diagonal of that size, far below the tolerance).
    const float d = beta - alpha, h = ab + ab;
    const float hs = __uint_as_float(__float_as_uint(h) ^ (__float_as_uint(d) & 0x80000000u));  // sign(d) h
    t = hs * rcp_approx(fabsf(d) + sqrt_approx(fmaf(d, d, h * h)));
    c = rsqrt_approx(fmaf(t, t, 1.f));
    n0 = fmaf(t, ab, beta);
    n1 = fmaf(-t, ab, alpha);
    rotated = rotated || ab_sq > (JACOBI_LAST * JACOBI_LAST) * scale;
  }
}

// BW = true: Bures-Wasserstein (A = L_i^T L_j; L_j^T is staged where Linv_j is) -- see the file header.
template <int MJ, bool BW>
__global__ void __launch_bounds__(PAIR_WARPS * 32, (MJ <= 12 ? 6 : (MJ <= 20 ? 5 : 3)))
pair_cp_kernel(const PairArgs A) {
  using G = CpGeom<MJ>;
  constexpr int LP = G::LP, NP = G::NP, MP4 = G::MP4, MH = G::MH, LDJ = G::LDJ;
  constexpr unsigned FULL = 0xffffffffu;
  extern __shared__ __align__(16) float smem[];
  const int m = A.m, m2 = m * m, nB = A.nB, tri = A.tri, dist = A.dist, R = A.T.R;
  const bool m_odd = m != MJ;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (t >= A.T.ntiles) return;  // no block-wide synchronisation below
  const int szLi = m * MP4, szJ = (MJ * LDJ + 3) & ~3, szCo = 2 * MP4;
  const int per_group = cp_group_floats(MJ, m);
  float* sLi = smem + (size_t)warp * cp_warp_floats(MJ, m);  // [m][MP4]: L_i, later Linv_i (shared by the problems)
  const int g = lane / LP, lg = lane - g * LP;
  const bool alive = g < NP;                // lanes beyond NP * LP only follow the instruction stream
  float* sJ = sLi + szLi + (alive ? g : NP - 1) * per_group;  // [MJ][LDJ]: Linv_j of this problem's column class
  float* sY = sJ;                           // [m][MP4]: generalized eigenvectors (over Linv_j), row = component, column = position
  float* sCo = sJ + szJ;                        // [2][MP4]: coefficients ci | cj per position
  float* sC = sCo + szCo;                   // [m][m]: dLoss/dE_j of this problem's column class
  const bool want_grad = A.rowpart != nullptr;
  auto div_m = [&](int idx) { return m_odd ? idx / (MJ - 1) : idx / MJ; };  // division by a compile-time constant

  int bi, bj;
  decode_tile(A.T, t, bi, bj);
  for (int idx = lane; idx < NP * per_group; idx += 32) sLi[szLi + idx] = 0.f;  // padding rows / columns, accumulators
  __syncwarp();
  const int j = bj * R + g;
  const bool jvalid = alive && g < R && j < nB;
  float dsum = 0.f, badsum = 0.f;
  for (int ii = 0; ii < R; ++ii) {
    const int i = bi * R + ii;
    const bool active = jvalid && pair_in_launch(i, j, A.nA, nB, tri, A.pair_begin, A.pair_end);
    if (__ballot_sync(FULL, active) == 0u) {  // no pair of this row belongs to the launch: the slot is still written
      if (want_grad) {
        float* rp = A.rowpart + ((int64_t)t * R + ii) * m2;
        for (int idx = lane; idx < m2; idx += 32) rp[idx] = 0.f;
      }
      if constexpr (BW) {
        if (A.pwpart != nullptr)
          for (int idx = lane; idx < R; idx += 32) A.pwpart[((int64_t)t * R + ii) * R + idx] = 0.f;
      }
      continue;
    }
    const float* Wi = A.Wa + (int64_t)i * 2 * m2;
    __syncwarp();
    for (int idx = lane; idx < m * MP4; idx += 32) {
      const int r = idx / MP4, c = idx - r * MP4;
      sLi[idx] = c < m ? Wi[r * m + c] : 0.f;
    }
    if (active) {  // Linv_j of this problem's column class (row MJ - 1 of sJ stays zero: Y never reaches it)
      if constexpr (BW) {  // L_j^T: sJ[q][r] = L_j[r][q]
        const float* Wj = A.Wb + (int64_t)j * 2 * m2;
        for (int idx = lg; idx < m2; idx += LP) {
          const int r = div_m(idx);
          sJ[(idx - r * m) * LDJ + r] = Wj[idx];
        }
      } else {
        const float* Wj = A.Wb + (int64_t)j * 2 * m2 + m2;
        for (int idx = lg; idx < m2; idx += LP) {
          const int q = div_m(idx);
          sJ[q * LDJ + (idx - q * m)] = Wj[idx];
        }
      }
    }
    __syncwarp();
    // ---- columns 2 lg and 2 lg + 1 of A: a[s] = sum_r Linv_j[q][r] L_i[r][s]  (row MJ - 1 of sJ is zero for odd m;
    // BW: L_j^T[q][r] in place of Linv_j[q][r])
    float2 a[MH], b[MH];
#pragma unroll
    for (int s = 0; s < MH; ++s) { a[s] = make_float2(0.f, 0.f); b[s] = make_float2(0.f, 0.f); }
    if (active) {
      const float* ja = sJ + (2 * lg) * LDJ;
      const float* jb = ja + LDJ;
#pragma unroll
      for (int r = 0; r < MJ; ++r) {
        if (r < m) {
          const float la = ja[r], lb = jb[r];
          const float2 la2 = make_float2(la, la), lb2 = make_float2(lb, lb);
#pragma unroll
          for (int s4 = 0; s4 <= r / 4; ++s4) {  // L_i is lower triangular: row r ends at column r
            const float4 w = *reinterpret_cast<const float4*>(sLi + r * MP4 + 4 * s4);
            const float2 w0 = make_float2(w.x, w.y), w1 = make_float2(w.z, w.w);
            a[2 * s4] = __ffma2_rn(la2, w0, a[2 * s4]);
            a[2 * s4 + 1] = __ffma2_rn(la2, w1, a[2 * s4 + 1]);
            b[2 * s4] = __ffma2_rn(lb2, w0, b[2 * s4]);
            b[2 * s4 + 1] = __ffma2_rn(lb2, w1, b[2 * s4 + 1]);
          }
        }
      }
    }
    // ---- one-sided Jacobi, odd-even transposition ordering, scaled ("fast") rotations: a column is kept as
    // scale * vector, a rotation c [[1, t], [-t, 1]] updates the vectors with ONE packed FMA per element pair
    // and column (y + tau1 x, x - tau2 y; tau1 = t s_x / s_y, tau2 = t s_y / s_x) and multiplies the two
    // scales by c, instead of two multiplies and two FMAs. The scales are folded back once per sweep (they
    // shrink by at most 2^-1/2 per rotation).
    const int up = (lane + 1) & 31, dn = (lane + 31) & 31;
    const bool has_right = alive && lg < LP - 1;
    float sA = 1.f, sB = 1.f;
    int sweeps = 0;
    for (int sweep = 0; sweep < JACOBI_MAX_SWEEPS; ++sweep) {
      float2 na2 = make_float2(0.f, 0.f), nb2 = make_float2(0.f, 0.f);
      {
        const float2 sa2 = make_float2(sA, sA), sb2 = make_float2(sB, sB);
#pragma unroll
        for (int s = 0; s < MJ / 2; ++s) {
          a[s] = __fmul2_rn(sa2, a[s]);
          b[s] = __fmul2_rn(sb2, b[s]);
          na2 = __ffma2_rn(a[s], a[s], na2);
          nb2 = __ffma2_rn(b[s], b[s], nb2);
        }
        sA = 1.f; sB = 1.f;
      }
      float nA = na2.x + na2.y, nBq = nb2.x + nb2.y;  // squared norms of the columns, carried incrementally
      bool rotated = false;
#pragma unroll 1
      for (int st = 0; st < LP; ++st) {
        {  // odd step: this lane's own two columns
          float2 ab2 = make_float2(0.f, 0.f);
#pragma unroll
          for (int s = 0; s < MJ / 2; ++s) ab2 = __ffma2_rn(a[s], b[s], ab2);
          const float sab = sA * sB;
          float t, c, n0, n1;
          cp_rotation(nA, nBq, sab * (ab2.x + ab2.y), true, t, c, n0, n1, rotated);
          const float tq = t * rcp_approx(sab);
          const float tau1 = tq * sA * sA, tau2 = -tq * sB * sB;
          const float2 t1 = make_float2(tau1, tau1), t2 = make_float2(tau2, tau2);
#pragma unroll
          for (int s = 0; s < MJ / 2; ++s) {
            const float2 x = a[s], y = b[s];
            a[s] = __ffma2_rn(t1, x, y);
            b[s] = __ffma2_rn(t2, y, x);
          }
          const float sa_old = sA;
          sA = c * sB; sB = c * sa_old;
          nA = n0; nBq = n1;
        }
        {  // even step: (this lane's second column, the right neighbour's first column)
          float2 x2[MJ / 2];
          float2 ab2 = make_float2(0.f, 0.f);
#pragma unroll
          for (int s = 0; s < MJ / 2; ++s) {
            x2[s].x = __shfl_sync(FULL, a[s].x, up);
            x2[s].y = __shfl_sync(FULL, a[s].y, up);
            ab2 = __ffma2_rn(b[s], x2[s], ab2);
          }
          const float nX = __shfl_sync(FULL, nA, up), sX = __shfl_sync(FULL, sA, up);
          const float sbx = sB * sX;
          float t, c, n0, n1;
          cp_rotation(nBq, nX, sbx * (ab2.x + ab2.y), has_right, t, c, n0, n1, rotated);
          const float tq = t * rcp_approx(sbx);
          // the end of the line has no partner: its column stays (1 * b + 0 * x)
          const float keep = has_right ? tq * sB * sB : 1.f, take = has_right ? 1.f : 0.f, tau2 = -tq * sX * sX;
          const float2 k2 = make_float2(keep, keep), m2v = make_float2(take, take), t2 = make_float2(tau2, tau2);
#pragma unroll
          for (int s = 0; s < MJ / 2; ++s) {
            const float2 x = b[s], y = x2[s];
            b[s] = __ffma2_rn(k2, x, __fmul2_rn(m2v, y));
            x2[s] = __ffma2_rn(t2, y, x);  // the neighbour's new first column
          }
          const float sT = c * sB;  // scale of the column that goes back
          if (has_right) { sB = c * sX; nBq = n0; }
#pragma unroll
          for (int s = 0; s < MJ / 2; ++s) {
            const float rx = __shfl_sync(FULL, x2[s].x, dn), ry = __shfl_sync(FULL, x2[s].y, dn);
            if (lg > 0) a[s] = make_float2(rx, ry);
          }
          const float nr = __shfl_sync(FULL, n1, dn), sr = __shfl_sync(FULL, sT, dn);
          if (lg > 0) { nA = nr; sA = sr; }
        }
      }
      ++sweeps;
      // a sweep whose largest rotation was below JACOBI_LAST leaves off-diagonals of that size squared
      if (!__any_sync(FULL, rotated)) break;
    }
    {
      const float2 sa2 = make_float2(sA, sA), sb2 = make_float2(sB, sB);
#pragma unroll
      for (int s = 0; s < MJ / 2; ++s) {
        a[s] = __fmul2_rn(sa2, a[s]);
        b[s] = __fmul2_rn(sb2, b[s]);
      }
    }
    // ---- eigenvalues, distance. The padding column of an odd m sits at one end of the line.
    float2 na2 = make_float2(0.f, 0.f), nb2 = make_float2(0.f, 0.f);
#pragma unroll
    for (int s = 0; s < MJ / 2; ++s) {
      na2 = __ffma2_rn(a[s], a[s], na2);
      nb2 = __ffma2_rn(b[s], b[s], nb2);
    }
    const float n2a = na2.x + na2.y, n2b = nb2.x + nb2.y;
    const bool pad_first = m_odd && (sweeps & 1);
    const bool real_a = active && !(pad_first && lg == 0);
    const bool real_b = active && !(m_odd && !pad_first && lg == LP - 1);
    // AI: log lambda; BW: sigma
    const float lla = BW ? (real_a ? sqrtf(n2a) : 0.f) : (real_a ? logf(n2a) : 0.f);
    const float llb = BW ? (real_b ? sqrtf(n2b) : 0.f) : (real_b ? logf(n2b) : 0.f);
    const int g0 = (g * LP) & 31;
    float d2 = 0.f;
    bool bw_live = true;  // BW: d^2 of the matrices was not clamped (its gradient is live)
    if constexpr (BW) {
      // |L_i|_F^2 + |L_j|_F^2 - 2 (sigma_a + sigma_b) over this lane's rows 2 lg, 2 lg + 1 of L_i and L_j^T;
      // Gaussian form: the lane's share of |mu_i - mu_j|^2 (components lg, lg + LP, ...)
      float part = -2.f * (lla + llb), pmu = 0.f;
      if (active) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int row = 2 * lg + h;
          if (row < m) {
            for (int c = 0; c <= row; ++c) part = fmaf(sLi[row * MP4 + c], sLi[row * MP4 + c], part);
            for (int c = row; c < m; ++c) part = fmaf(sJ[row * LDJ + c], sJ[row * LDJ + c], part);
          }
        }
        if (A.Mu != nullptr) {
          const float* mui = A.Mu + (int64_t)i * A.k;
          const float* muj = A.Mu + (int64_t)j * A.k;
          for (int e = lg; e < A.k; e += LP) {
            const float df = mui[e] - muj[e];
            pmu = fmaf(df, df, pmu);
          }
        }
      }
      float dmu = 0.f;
#pragma unroll
      for (int u = 0; u < LP; ++u) {  // fixed order, same in every lane
        d2 += __shfl_sync(FULL, part, (g0 + u) & 31);
        dmu += __shfl_sync(FULL, pmu, (g0 + u) & 31);
      }
      bw_live = d2 > 0.f;
      d2 = (d2 < 0.f ? 0.f : d2) + dmu;  // not fmaxf: a NaN (failed Cholesky) must reach the non-finite count
    } else {
      const float part = lla * lla + llb * llb;
#pragma unroll
      for (int u = 0; u < LP; ++u) d2 += __shfl_sync(FULL, part, (g0 + u) & 31);  // fixed order, same in every lane
    }
    if (!BW && A.eig_out != nullptr) {  // descending order (linalg.py:69-70); the padding column has norm 0 and ranks last
      int ra = 0, rb = 0;
#pragma unroll
      for (int u = 0; u < LP; ++u) {
        const float va = __shfl_sync(FULL, n2a, (g0 + u) & 31), vb = __shfl_sync(FULL, n2b, (g0 + u) & 31);
        ra += (va > n2a || (va == n2a && 2 * u < 2 * lg)) ? 1 : 0;
        ra += (vb > n2a || (vb == n2a && 2 * u + 1 < 2 * lg)) ? 1 : 0;
        rb += (va > n2b || (va == n2b && 2 * u < 2 * lg + 1)) ? 1 : 0;
        rb += (vb > n2b || (vb == n2b && 2 * u + 1 < 2 * lg + 1)) ? 1 : 0;
      }
      float* eo = A.eig_out + ((int64_t)i * nB + j) * m;
      if (real_a) eo[ra] = n2a;
      if (real_b) eo[rb] = n2b;
    }
    float dd_dd2;
    const float dval = finish_distance(d2, dist, &dd_dd2);
    if (active && lg == 0) {
      dsum += dval;
      if (!isfinite(dval)) badsum += 1.f;
      if (A.dist_out != nullptr) {
        A.dist_out[(int64_t)i * nB + j] = dval;
        if (tri) A.dist_out[(int64_t)j * nB + i] = dval;
      }
    }
    if (want_grad) {
      float w = 0.f;
      if (active) {
        w = A.weight * dd_dd2;
        if (A.gD != nullptr)
          w *= tri ? (A.gD[(int64_t)i * nB + j] + A.gD[(int64_t)j * nB + i]) : A.gD[(int64_t)i * nB + j];
      }
      if constexpr (BW) {
        if (A.pwpart != nullptr && alive && lg == 0 && g < R) A.pwpart[((int64_t)t * R + ii) * R + g] = 2.f * w;
        if (!bw_live) w = 0.f;
        // G of the positions' vectors V (rows of sY = component, columns = position) with one coefficient per
        // position (sCo), plus w I: a lane owns the rows s0 = lg and s1 = lg + LP, packed in the two halves.
        // toRow: G_i, summed over the problems of the row in a fixed order and stored by the first one;
        // else G_j, added to the problem's column accumulator.
        float* rp = A.rowpart + ((int64_t)t * R + ii) * m2;
        auto gram_pass = [&](bool toRow) {
          const int s0 = lg, s1 = lg + LP;
          const bool mine0 = alive && s0 < m, mine1 = alive && s1 < m;
          float2 cij[MP4];
          {
            const float* v0 = sY + (mine0 ? s0 : 0) * MP4;
            const float* v1 = sY + (mine1 ? s1 : 0) * MP4;
#pragma unroll
            for (int q4 = 0; q4 < MP4 / 4; ++q4) {
              const float4 y0 = *reinterpret_cast<const float4*>(v0 + 4 * q4);
              const float4 y1 = *reinterpret_cast<const float4*>(v1 + 4 * q4);
              const float4 c = *reinterpret_cast<const float4*>(sCo + 4 * q4);
              cij[4 * q4] = make_float2(y0.x * c.x, y1.x * c.x);
              cij[4 * q4 + 1] = make_float2(y0.y * c.y, y1.y * c.y);
              cij[4 * q4 + 2] = make_float2(y0.z * c.z, y1.z * c.z);
              cij[4 * q4 + 3] = make_float2(y0.w * c.w, y1.w * c.w);
            }
          }
#pragma unroll 1
          for (int r = 0; r < m; ++r) {
            float2 gab = make_float2(r == s0 ? w : 0.f, r == s1 ? w : 0.f);
#pragma unroll
            for (int q4 = 0; q4 < MP4 / 4; ++q4) {
              const float4 yr = *reinterpret_cast<const float4*>(sY + r * MP4 + 4 * q4);
              gab = __ffma2_rn(make_float2(yr.x, yr.x), cij[4 * q4], gab);
              gab = __ffma2_rn(make_float2(yr.y, yr.y), cij[4 * q4 + 1], gab);
              gab = __ffma2_rn(make_float2(yr.z, yr.z), cij[4 * q4 + 2], gab);
              gab = __ffma2_rn(make_float2(yr.w, yr.w), cij[4 * q4 + 3], gab);
            }
            if (toRow) {
              const float g0v = (active && mine0) ? gab.x : 0.f, g1v = (active && mine1) ? gab.y : 0.f;
              float t0 = 0.f, t1 = 0.f;
#pragma unroll
              for (int gg = 0; gg < NP; ++gg) {
                t0 += __shfl_sync(FULL, g0v, (gg * LP + lg) & 31);
                t1 += __shfl_sync(FULL, g1v, (gg * LP + lg) & 31);
              }
              if (g == 0 && mine0) rp[r * m + s0] = t0;
              if (g == 0 && mine1) rp[r * m + s1] = t1;
            } else if (active) {
              if (mine0) sC[r * m + s0] += gab.x;
              if (mine1) sC[r * m + s1] += gab.y;
            }
          }
        };
        // ---- pass 1: Z = L_i A_f (sLi still holds L_i; L_j^T in sJ is dead) -> G_j with -w sigma^-3
        __syncwarp();
        if constexpr (MP4 > MJ) {  // the two padding columns of sY lie on what was L_j^T: zero them
          for (int idx = lg; idx < 2 * m; idx += LP) sY[(idx >> 1) * MP4 + MJ + (idx & 1)] = 0.f;
        }
        if (alive) {
#pragma unroll
          for (int r = 0; r < MJ; ++r) {
            if (r < m) {
              float2 za = make_float2(0.f, 0.f), zb = za;
#pragma unroll
              for (int s4 = 0; s4 <= r / 4; ++s4) {  // L_i is lower triangular: row r ends at column r
                const float4 wv = *reinterpret_cast<const float4*>(sLi + r * MP4 + 4 * s4);
                const float2 w0 = make_float2(wv.x, wv.y), w1 = make_float2(wv.z, wv.w);
                za = __ffma2_rn(w0, a[2 * s4], za);
                za = __ffma2_rn(w1, a[2 * s4 + 1], za);
                zb = __ffma2_rn(w0, b[2 * s4], zb);
                zb = __ffma2_rn(w1, b[2 * s4 + 1], zb);
              }
              *reinterpret_cast<float2*>(sY + r * MP4 + 2 * lg) = make_float2(za.x + za.y, zb.x + zb.y);
            }
          }
          *reinterpret_cast<float2*>(sCo + 2 * lg) =
              make_float2(real_a ? -w / (lla * n2a) : 0.f, real_b ? -w / (llb * n2b) : 0.f);
        }
        __syncwarp();
        gram_pass(false);
        // ---- pass 2: Y = L_i^-T A_f -> G_i with -w sigma^-1
        __syncwarp();
        for (int idx = lane; idx < m * MP4; idx += 32) {
          const int r = idx / MP4, c = idx - r * MP4;
          sLi[idx] = c < m ? Wi[m2 + r * m + c] : 0.f;
        }
        __syncwarp();
        float2 ya[MH], yb[MH];
#pragma unroll
        for (int s = 0; s < MH; ++s) { ya[s] = make_float2(0.f, 0.f); yb[s] = make_float2(0.f, 0.f); }
#pragma unroll
        for (int s = 0; s < MJ; ++s) {
          if (s < m) {
            const float as = (s & 1) ? a[s / 2].y : a[s / 2].x, bs = (s & 1) ? b[s / 2].y : b[s / 2].x;
            const float2 as2 = make_float2(as, as), bs2 = make_float2(bs, bs);
#pragma unroll
            for (int r4 = 0; r4 <= s / 4; ++r4) {  // Linv_i is lower triangular
              const float4 wv = *reinterpret_cast<const float4*>(sLi + s * MP4 + 4 * r4);
              const float2 w0 = make_float2(wv.x, wv.y), w1 = make_float2(wv.z, wv.w);
              ya[2 * r4] = __ffma2_rn(as2, w0, ya[2 * r4]);
              ya[2 * r4 + 1] = __ffma2_rn(as2, w1, ya[2 * r4 + 1]);
              yb[2 * r4] = __ffma2_rn(bs2, w0, yb[2 * r4]);
              yb[2 * r4 + 1] = __ffma2_rn(bs2, w1, yb[2 * r4 + 1]);
            }
          }
        }
        __syncwarp();  // every lane has read Z
        if (alive) {
#pragma unroll
          for (int r = 0; r < MJ; ++r) {
            if (r < m) {
              const float y0 = (r & 1) ? ya[r / 2].y : ya[r / 2].x, y1 = (r & 1) ? yb[r / 2].y : yb[r / 2].x;
              *reinterpret_cast<float2*>(sY + r * MP4 + 2 * lg) = make_float2(y0, y1);
            }
          }
          *reinterpret_cast<float2*>(sCo + 2 * lg) = make_float2(real_a ? -w / lla : 0.f, real_b ? -w / llb : 0.f);
        }
        __syncwarp();
        gram_pass(true);
        continue;
      }
      // ---- Y = L_i^-T A_f for this lane's two columns: y[r] = sum_s Linv_i[s][r] a[s]
      __syncwarp();
      for (int idx = lane; idx < m * MP4; idx += 32) {
        const int r = idx / MP4, c = idx - r * MP4;
        sLi[idx] = c < m ? Wi[m2 + r * m + c] : 0.f;
      }
      __syncwarp();
      float2 ya[MH], yb[MH];
#pragma unroll
      for (int s = 0; s < MH; ++s) { ya[s] = make_float2(0.f, 0.f); yb[s] = make_float2(0.f, 0.f); }
#pragma unroll
      for (int s = 0; s < MJ; ++s) {
        if (s < m) {
          const float as = (s & 1) ? a[s / 2].y : a[s / 2].x, bs = (s & 1) ? b[s / 2].y : b[s / 2].x;
          const float2 as2 = make_float2(as, as), bs2 = make_float2(bs, bs);
#pragma unroll
          for (int r4 = 0; r4 <= s / 4; ++r4) {  // Linv_i is lower triangular
            const float4 wv = *reinterpret_cast<const float4*>(sLi + s * MP4 + 4 * r4);
            const float2 w0 = make_float2(wv.x, wv.y), w1 = make_float2(wv.z, wv.w);
            ya[2 * r4] = __ffma2_rn(as2, w0, ya[2 * r4]);
            ya[2 * r4 + 1] = __ffma2_rn(as2, w1, ya[2 * r4 + 1]);
            yb[2 * r4] = __ffma2_rn(bs2, w0, yb[2 * r4]);
            yb[2 * r4 + 1] = __ffma2_rn(bs2, w1, yb[2 * r4 + 1]);
          }
        }
      }
      // ---- Y -> shared memory (row = component r, column = position), coefficients of both matrices
      if constexpr (MP4 > MJ) {  // the two padding columns of Y lie on what was Linv_j: zero them
        for (int idx = lg; idx < 2 * m; idx += LP) sY[(idx >> 1) * MP4 + MJ + (idx & 1)] = 0.f;
      }
      if (alive) {
#pragma unroll
        for (int r = 0; r < MJ; ++r) {
          if (r < m) {
            const float y0 = (r & 1) ? ya[r / 2].y : ya[r / 2].x, y1 = (r & 1) ? yb[r / 2].y : yb[r / 2].x;
            *reinterpret_cast<float2*>(sY + r * MP4 + 2 * lg) = make_float2(y0, y1);
          }
        }
        const float cia = real_a ? w * 2.f * lla / n2a : 0.f, cib = real_b ? w * 2.f * llb / n2b : 0.f;
        *reinterpret_cast<float2*>(sCo + 2 * lg) = make_float2(cia, cib);
        *reinterpret_cast<float2*>(sCo + MP4 + 2 * lg) = make_float2(real_a ? -w * 2.f * lla : 0.f,
                                                                     real_b ? -w * 2.f * llb : 0.f);
      }
      __syncwarp();
      // ---- G_i[r][s'] = sum_q ci_q Y[r][q] Y[s'][q] and G_j with cj; a lane owns rows s' = lg and lg + LP.
      // G_j goes to the problem's column accumulator (only its own lanes touch it); G_i of the NP problems
      // of the row is summed across the problems in a fixed order (shuffles) and stored by the first one.
      float* rp = A.rowpart + ((int64_t)t * R + ii) * m2;
#pragma unroll 1
      for (int u = 0; u < 2; ++u) {
        const int sp = lg + LP * u;
        const bool mine = alive && sp < m;
        float2 cij[MP4];
        {
          const float* yrow = sY + (mine ? sp : 0) * MP4;
#pragma unroll
          for (int q4 = 0; q4 < MP4 / 4; ++q4) {
            const float4 yy = *reinterpret_cast<const float4*>(yrow + 4 * q4);
            const float4 c1 = *reinterpret_cast<const float4*>(sCo + 4 * q4);
            const float4 c2 = *reinterpret_cast<const float4*>(sCo + MP4 + 4 * q4);
            cij[4 * q4] = make_float2(yy.x * c1.x, yy.x * c2.x);
            cij[4 * q4 + 1] = make_float2(yy.y * c1.y, yy.y * c2.y);
            cij[4 * q4 + 2] = make_float2(yy.z * c1.z, yy.z * c2.z);
            cij[4 * q4 + 3] = make_float2(yy.w * c1.w, yy.w * c2.w);
          }
        }
#pragma unroll 1
        for (int r = 0; r < m; ++r) {
          float2 gab = make_float2(0.f, 0.f);
#pragma unroll
          for (int q4 = 0; q4 < MP4 / 4; ++q4) {
            const float4 yr = *reinterpret_cast<const float4*>(sY + r * MP4 + 4 * q4);
            gab = __ffma2_rn(make_float2(yr.x, yr.x), cij[4 * q4], gab);
            gab = __ffma2_rn(make_float2(yr.y, yr.y), cij[4 * q4 + 1], gab);
            gab = __ffma2_rn(make_float2(yr.z, yr.z), cij[4 * q4 + 2], gab);
            gab = __ffma2_rn(make_float2(yr.w, yr.w), cij[4 * q4 + 3], gab);
          }
          const float gi = (active && mine) ? gab.x : 0.f;
          float tot = 0.f;
#pragma unroll
          for (int gg = 0; gg < NP; ++gg) tot += __shfl_sync(FULL, gi, (gg * LP + lg) & 31);
          if (g == 0 && mine) rp[r * m + sp] = tot;
          if (active && mine) sC[r * m + sp] += gab.y;
        }
      }
    }
  }
  if (want_grad) {  // column partials of the tile: every slot is written (zeros where a column had no pair)
    __syncwarp();
    float* cp = A.colpart + (int64_t)t * R * m2;
    const float* sC0 = sLi + szLi + (per_group - ((m2 + 3) & ~3));
    for (int gg = 0; gg < R; ++gg)
      for (int idx = lane; idx < m2; idx += 32) cp[gg * m2 + idx] = sC0[gg * per_group + idx];
  }
  if (A.losspart != nullptr) {
    float ds = 0.f, bs = 0.f;
#pragma unroll
    for (int gg = 0; gg < NP; ++gg) {
      ds += __shfl_sync(FULL, dsum, (gg * LP) & 31);
      bs += __shfl_sync(FULL, badsum, (gg * LP) & 31);
    }
    if (lane == 0) {
      A.losspart[2 * t] = ds;
      A.losspart[2 * t + 1] = bs;
    }
  }
}

template <int MJ, bool BW>
static cudaError_t launch_pair_cp_t(const PairArgs& A, cudaStream_t st) {
  const int smem = PAIR_WARPS * cp_warp_floats(MJ, A.m) * (int)sizeof(float);
  static int smem_set[kMaxDevices] = {0};
  {
    cudaError_t e = ensure_dynamic_smem(pair_cp_kernel<MJ, BW>, smem, smem_set);
    if (e != cudaSuccess) return e;
  }
  const unsigned blocks = (unsigned)((A.T.ntiles + PAIR_WARPS - 1) / PAIR_WARPS);
  pair_cp_kernel<MJ, BW><<<blocks, PAIR_WARPS * 32, smem, st>>>(A);
  return cudaGetLastError();
}

__host__ __device__ inline bool is_bw_family(int dist) {
  return (dist & 15) == SQFA_DIST_BURES_WASSERSTEIN || (dist & 15) == SQFA_DIST_WASSERSTEIN_GAUSSIAN;
}

template <int MJ>
static cudaError_t launch_pair_cp(const PairArgs& A, cudaStream_t st) {
  return is_bw_family(A.dist) ? launch_pair_cp_t<MJ, true>(A, st) : launch_pair_cp_t<MJ, false>(A, st);
}

// ------------------------------------------------------------------------------------------------
// pair kernel, log-Euclidean: d^2 = |logE_i - logE_j|_F^2. Tiles are single pairs. The gradient
// w.r.t. the matrix logarithms is sum_o pw(c, o) (logE_c - logE_o): this kernel stores the per-pair
// factor pw = 2 w dd/d(d^2) and le_grad_kernel forms the sums class by class in a fixed order.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(PAIR_WARPS * 32)
pair_le_kernel(const PairArgs A) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (t >= A.T.ntiles) return;
  const int m = A.m, nB = A.nB, tri = A.tri;
  int i, j;
  decode_tile(A.T, t, i, j);
  const int stride = 2 * m * m + 2 * m;
  float dval = 0.f, bad = 0.f, pw = 0.f;
  if (pair_in_launch(i, j, A.nA, nB, tri, A.pair_begin, A.pair_end)) {
    const float* Li = A.Wa + (int64_t)i * stride + m * m + 2 * m;
    const float* Lj = A.Wb + (int64_t)j * stride + m * m + 2 * m;
    float d2 = 0.f;
    for (int idx = lane; idx < m * m; idx += 32) {
      const float df = Li[idx] - Lj[idx];
      d2 += df * df;
    }
    d2 = warp_sum(d2);
    float dd_dd2;
    dval = finish_distance(d2, A.dist, &dd_dd2);
    if (!isfinite(dval)) bad = 1.f;
    if (A.dist_out != nullptr && lane == 0) {
      A.dist_out[(int64_t)i * nB + j] = dval;
      if (tri) A.dist_out[(int64_t)j * nB + i] = dval;
    }
    pw = 2.f * A.weight * dd_dd2;
    if (A.gD != nullptr)
      pw *= tri ? (A.gD[(int64_t)i * nB + j] + A.gD[(int64_t)j * nB + i]) : A.gD[(int64_t)i * nB + j];
  }
  if (lane == 0) {
    if (A.rowpart != nullptr) A.rowpart[t] = pw;  // LE: rowpart holds one factor per pair
    if (A.losspart != nullptr) {
      A.losspart[2 * t] = dval;
      A.losspart[2 * t + 1] = bad;
    }
  }
}

// gLa[c] += sum_b pw(c, b) (xA_c - xB_b)   and   gLb[c] -= sum_a pw(a, c) (xA_a - xB_c),
// pairs in launch order; block = class, thread = element. x = the ne floats at Wa / Wb + class * stride + off
// (log-Euclidean: the matrix logs; Gaussian Wasserstein: the means), pw = one factor per pair in the R x R
// tiles of T. Self distances (tri): one sum over all other classes.
__global__ void __launch_bounds__(256)
le_grad_kernel(const PairTiles T, const float* __restrict__ Wa, const float* __restrict__ Wb, int nA, int nB, int ne,
               int stride, int off, const float* __restrict__ pw, float* gLa, float* gLb) {
  const int c = blockIdx.x;
  const int R = T.R, R2 = R * R;
  // factor of pair (i, j): tile (i / R, j / R), slot (i % R, j % R)
  auto pw_at = [&](int i, int j) {
    const int64_t bi = i / R;
    const int64_t tt = (T.tri ? bi * (bi + 1) / 2 : bi * T.nbj) + j / R - T.tile0;
    return pw[tt * R2 + (i % R) * R + j % R];
  };
  for (int e = threadIdx.x; e < ne; e += blockDim.x) {
    float ga = 0.f, gb = 0.f;
    if (c < nA && c / R >= T.bi0 && c / R <= T.bi1) {  // row side: pairs (c, j)
      const float lc = Wa[(int64_t)c * stride + off + e];
      const int nj = T.tri ? c : nB;
      for (int j = 0; j < nj; ++j) ga += pw_at(c, j) * (lc - Wb[(int64_t)j * stride + off + e]);
    }
    if (c < nB) {  // column side: pairs (i, c)
      const float lc = Wb[(int64_t)c * stride + off + e];
      const int i0 = T.tri ? max(T.bi0 * R, c + 1) : T.bi0 * R;
      const int i1 = min((T.bi1 + 1) * R, nA);
      for (int i = i0; i < i1; ++i) gb -= pw_at(i, c) * (Wa[(int64_t)i * stride + off + e] - lc);
    }
    if (gLa == gLb) {
      if (c < nA) gLa[(int64_t)c * ne + e] += ga + gb;
    } else {
      if (c < nA) gLa[(int64_t)c * ne + e] += ga;
      if (c < nB) gLb[(int64_t)c * ne + e] += gb;
    }
  }
}

// dLoss/dE of class c = its row partials (tiles of block row c / R, ascending block column) + its
// column partials (tiles of block column c / R, ascending block row): blocks 0 .. max(nA, nB) - 1.
// The last block reduces the loss partials. Block size: pair_reduce_threads(m) (one matrix element per thread
// and pass; m = 17 has 289 elements: 256 threads would run a second, almost empty pass of the same latency).
//   CLOSURE = false: gEa[c] += rows, gEb[c] += columns (gEa == gEb: one sum); loss[0..1] += {sum d, #bad}
//   CLOSURE = true : the closure's tail fused in: (gPsi, gMu) = adjoint of the embedding applied to the
//                    reduced dLoss/dE (reference model.py:216-217 / 537-538, distances.py:162-174) and
//                    loss = {weight * sum d, #bad, 0}
template <typename Real, bool CLOSURE>
__global__ void __launch_bounds__(1024)
pair_reduce_kernel(const PairTiles T, int nA, int nB, int m, const Real* __restrict__ rowpart,
                   const Real* __restrict__ colpart, const Real* __restrict__ losspart, Real* gEa, Real* gEb, Real* loss,
                   Real weight, const Real* __restrict__ Mu, int k, int fr, Real* __restrict__ gPsi,
                   Real* __restrict__ gMu) {
  extern __shared__ __align__(16) unsigned char pr_smem[];
  Real* sg = reinterpret_cast<Real*>(pr_smem);  // CLOSURE: the reduced m x m gradient of this class
  const int nC = max(nA, nB);
  const int c = blockIdx.x;
  if (c == nC) {
    if (loss == nullptr || losspart == nullptr) return;
    Real sum, bad;
    reduce_loss_partials(losspart, T.ntiles, sum, bad);
    if (threadIdx.x == 0) {
      if (CLOSURE) {
        loss[0] = weight * sum;
        loss[1] = bad;
        loss[2] = Real(0);  // max |grad|, filled by closure_finish_kernel with atomicMax on the bits
      } else {
        loss[0] += sum;
        loss[1] += bad;
      }
    }
    return;
  }
  if (rowpart == nullptr) return;
  const int R = T.R, m2 = m * m;
  const int slot = c % R, bc = c / R;
  const int64_t pstride = (int64_t)R * m2;
  for (int e = threadIdx.x; e < m2; e += blockDim.x) {
    Real a = Real(0), b = Real(0);
    if (c < nA && bc >= T.bi0 && bc <= T.bi1) {
      const int nb = T.tri ? bc + 1 : T.nbj;
      const Real* p = rowpart + ((T.tri ? (int64_t)bc * (bc + 1) / 2 : (int64_t)bc * T.nbj) - T.tile0) * pstride +
                       (int64_t)slot * m2 + e;
      int bj = 0;
      for (; bj + 8 <= nb; bj += 8) {  // eight loads in flight, added in order
        Real v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = p[u * pstride];
#pragma unroll
        for (int u = 0; u < 8; ++u) a += v[u];
        p += 8 * pstride;
      }
      for (; bj < nb; ++bj, p += pstride) a += *p;
    }
    if (c < nB) {
      const int i0 = T.tri ? max(T.bi0, bc) : T.bi0;
      int bi = i0;
      auto cp = [&](int bi_) {
        const int64_t tt = (T.tri ? (int64_t)bi_ * (bi_ + 1) / 2 + bc : (int64_t)bi_ * T.nbj + bc) - T.tile0;
        return colpart[tt * pstride + (int64_t)slot * m2 + e];
      };
      for (; bi + 8 <= T.bi1 + 1; bi += 8) {
        Real v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = cp(bi + u);
#pragma unroll
        for (int u = 0; u < 8; ++u) b += v[u];
      }
      for (; bi <= T.bi1; ++bi) b += cp(bi);
    }
    if (CLOSURE) {
      sg[e] = a + b;
    } else if (gEa == gEb) {
      gEa[(int64_t)c * m2 + e] += a + b;
    } else {
      if (c < nA) gEa[(int64_t)c * m2 + e] += a;
      if (c < nB) gEb[(int64_t)c * m2 + e] += b;
    }
  }
  if (CLOSURE) {
    __syncthreads();
    // gPsi = gE[:k,:k];  gMu[r] = sum_s (gE[r][s] + gE[s][r]) mu[s] + gE[r][k] + gE[k][r]   (Fisher-Rao)
    for (int idx = threadIdx.x; idx < k * (k + 1); idx += blockDim.x) {
      const int r = idx / (k + 1), s = idx % (k + 1);
      if (s < k) {
        gPsi[(int64_t)c * k * k + r * k + s] = sg[r * m + s];
      } else if (fr) {
        Real v = sg[r * m + k] + sg[k * m + r];
        for (int u = 0; u < k; ++u) v = fma(sg[r * m + u] + sg[u * m + r], Mu[(int64_t)c * k + u], v);
        gMu[(int64_t)c * k + r] = v;
      }
    }
  }
}

// Daleckii-Krein adjoint of logE = V log(Lambda) V^T:  gE += V [ (V^T gLog V) o Gamma ] V^T,
// Gamma_ab = (log l_a - log l_b) / (l_a - l_b), Gamma_aa = 1 / l_a. One warp per class.
__global__ void __launch_bounds__(PAIR_WARPS * 32)
le_factor_bwd_kernel(const float* __restrict__ W, const float* __restrict__ gLog, int C, int m,
                     float* __restrict__ gE) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + warp;
  if (c >= C) return;
  const int per_warp = 3 * m * m;
  float* V = smem + (size_t)warp * per_warp;
  float* G = V + m * m;
  float* H = G + m * m;
  const float* Wc = W + (int64_t)c * (2 * m * m + 2 * m);
  const float* lam = Wc + m * m;
  const float* ll = Wc + m * m + m;
  for (int idx = lane; idx < m * m; idx += 32) {
    V[idx] = Wc[idx];
    const int r = idx / m, s = idx % m;  // symmetrise the incoming gradient
    G[idx] = 0.5f * (gLog[(int64_t)c * m * m + idx] + gLog[(int64_t)c * m * m + s * m + r]);
  }
  __syncwarp();
  // H = G V
  for (int idx = lane; idx < m * m; idx += 32) {
    const int r = idx / m, b = idx % m;
    float a = 0.f;
    for (int s = 0; s < m; ++s) a += G[r * m + s] * V[s * m + b];
    H[idx] = a;
  }
  __syncwarp();
  // G = (V^T H) o Gamma
  for (int idx = lane; idx < m * m; idx += 32) {
    const int a_ = idx / m, b = idx % m;
    float a = 0.f;
    for (int r = 0; r < m; ++r) a += V[r * m + a_] * H[r * m + b];
    const float la = lam[a_], lb = lam[b];
    const float dl = la - lb;
    float gam;
    if (fabsf(dl) > 1e-4f * fmaxf(la, lb)) gam = (ll[a_] - ll[b]) / dl;
    else gam = 2.f / (la + lb);  // limit of the divided difference of log
    G[idx] = a * gam;
  }
  __syncwarp();
  // H = V G ; gE = H V^T
  for (int idx = lane; idx < m * m; idx += 32) {
    const int r = idx / m, b = idx % m;
    float a = 0.f;
    for (int a_ = 0; a_ < m; ++a_) a += V[r * m + a_] * G[a_ * m + b];
    H[idx] = a;
  }
  __syncwarp();
  for (int idx = lane; idx < m * m; idx += 32) {
    const int r = idx / m, s = idx % m;
    float a = 0.f;
    for (int b = 0; b < m; ++b) a += H[r * m + b] * V[s * m + b];
    gE[(int64_t)c * m * m + idx] += a;
  }
}

__global__ void fill_diagonal_kernel(float* dist_out, int C, float v) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) dist_out[(int64_t)c * C + c] = v;
}

}  // namespace

size_t class_factor_floats(int m, int dist) {
  return ((dist & 15) == SQFA_DIST_LOG_EUCLIDEAN) ? (size_t)(2 * m * m + 2 * m) : (size_t)(2 * m * m);
}

cudaError_t launch_class_factor(const float* E, int C, int m, int dist, float* W, int32_t* flag, cudaStream_t st) {
  if (C <= 0) return cudaSuccess;
  const int per_warp = factor_scratch_floats(m) * (int)sizeof(float);
  const int nw = warps_for(per_warp, PAIR_WARPS);
  const int smem = nw * per_warp;
  static int smem_set[kMaxDevices] = {0};
  {
    cudaError_t e = ensure_dynamic_smem(class_factor_kernel, smem, smem_set);
    if (e != cudaSuccess) return e;
  }
  cudaError_t e = cudaMemsetAsync(flag, 0, sizeof(int32_t), st);
  if (e != cudaSuccess) return e;
  class_factor_kernel<<<(C + nw - 1) / nw, nw * 32, smem, st>>>(E, C, m, dist, W, flag);
  return cudaGetLastError();
}

cudaError_t launch_class_prepare(const float* PsiPart, const float* MuPart, int nchunk, float noise, int C, int k,
                                 int dist, float* Mu, float* E, float* W, int32_t* flag, cudaStream_t st) {
  if (C <= 0) return cudaSuccess;
  const int m = ((dist & 15) == SQFA_DIST_FISHER_RAO_LB) ? k + 1 : k;
  const int per_warp = (factor_scratch_floats(m) + m * m + k) * (int)sizeof(float);
  const int nw = warps_for(per_warp, PAIR_WARPS);
  const int smem = nw * per_warp;
  static int smem_set[kMaxDevices] = {0};
  {
    cudaError_t e = ensure_dynamic_smem(class_prepare_kernel, smem, smem_set);
    if (e != cudaSuccess) return e;
  }
  cudaError_t e = cudaMemsetAsync(flag, 0, 2 * sizeof(int32_t), st);  // flag[1]: closure_finish's arrival ticket
  if (e != cudaSuccess) return e;
  class_prepare_kernel<<<(C + nw - 1) / nw, nw * 32, smem, st>>>(PsiPart, MuPart, nchunk, noise, C, k, dist, Mu, E, W,
                                                                  flag);
  return cudaGetLastError();
}

// AI family up to m = 34: the column-pair kernel; 34 < m <= 64: the shared-memory kernel
static bool pair_use_cp(int m, int dist) { return (dist & 15) != SQFA_DIST_LOG_EUCLIDEAN && m <= 34; }

// Tile edge R (a warp owns R x R pairs). Column-pair kernel: the NP = 32 / (lanes per problem) pairs of a tile
// row run side by side, so R goes up to NP as soon as there are enough tiles to fill the GPU a few times
// over (R = 1 for short pair lists: every pair its own warp, latency). The shared-memory variant (m > 34)
// and log-Euclidean always use single pairs.
static int pair_tile_edge(int m, int dist, int64_t npairs) {
  if ((dist & 15) == SQFA_DIST_LOG_EUCLIDEAN || m > 34) return 1;
  if (pair_use_cp(m, dist)) {
    const int np = 32 / (((m + 1) & ~1) / 2);
    int R = 1;
    while (R < np && R < 8 && npairs / ((int64_t)(R + 1) * (R + 1)) >= 4096) ++R;
    return R;
  }
  return 1;
}

// threads of pair_reduce_kernel: the m^2 elements in as few, evenly filled passes as possible
static int pair_reduce_threads(int m) {
  const int m2 = m * m, passes = (m2 + 1023) / 1024;
  int nt = (((m2 + passes - 1) / passes) + 31) & ~31;
  return nt < 128 ? 128 : nt;
}

PairWorkspace pair_workspace(int nA, int nB, int m, int dist, int tri, int64_t pair_begin, int64_t pair_end) {
  PairWorkspace w;
  const int64_t npairs = pair_end > pair_begin ? pair_end - pair_begin : 0;
  w.T = make_pair_tiles(nA, nB, tri, pair_begin, pair_end, pair_tile_edge(m, dist, npairs));
  const bool le = (dist & 15) == SQFA_DIST_LOG_EUCLIDEAN;
  const bool w2 = (dist & 15) == SQFA_DIST_WASSERSTEIN_GAUSSIAN;
  const size_t part = le ? (size_t)w.T.ntiles : (size_t)w.T.ntiles * w.T.R * m * m;
  w.rowpart = 0;
  w.colpart = al<float>(part);
  w.losspart = w.colpart + (le ? 0 : al<float>(part));
  w.pwpart = w.losspart + al<float>((size_t)2 * w.T.ntiles);
  w.total_floats = w.pwpart + (w2 ? al<float>((size_t)w.T.ntiles * w.T.R * w.T.R) : 0) + 64;
  return w;
}

static cudaError_t launch_pair_kernel(const PairArgs& A, cudaStream_t st) {
  const int m = A.m;
  if (A.T.ntiles <= 0) return cudaSuccess;
  if ((A.dist & 15) == SQFA_DIST_LOG_EUCLIDEAN) {
    const unsigned blocks = (unsigned)((A.T.ntiles + PAIR_WARPS - 1) / PAIR_WARPS);
    pair_le_kernel<<<blocks, PAIR_WARPS * 32, 0, st>>>(A);
    return cudaGetLastError();
  }
  if (is_bw_family(A.dist) && m > 34) return cudaErrorNotSupported;
  if (pair_use_cp(m, A.dist)) {  // two columns per lane, several problems per warp
    switch ((m + 1) / 2) {
      case 1: return launch_pair_cp<2>(A, st);
      case 2: return launch_pair_cp<4>(A, st);
      case 3: return launch_pair_cp<6>(A, st);
      case 4: return launch_pair_cp<8>(A, st);
      case 5: return launch_pair_cp<10>(A, st);
      case 6: return launch_pair_cp<12>(A, st);
      case 7: return launch_pair_cp<14>(A, st);
      case 8: return launch_pair_cp<16>(A, st);
      case 9: return launch_pair_cp<18>(A, st);
      case 10: return launch_pair_cp<20>(A, st);
      case 11: return launch_pair_cp<22>(A, st);
      case 12: return launch_pair_cp<24>(A, st);
      case 13: return launch_pair_cp<26>(A, st);
      case 14: return launch_pair_cp<28>(A, st);
      case 15: return launch_pair_cp<30>(A, st);
      case 16: return launch_pair_cp<32>(A, st);
      default: return launch_pair_cp<34>(A, st);
    }
  }
  const int per_warp = pair_smem_floats(m) * (int)sizeof(float);
  const int nw = warps_for(per_warp, PAIR_WARPS);
  const int smem = nw * per_warp;
  const unsigned blocks = (unsigned)((A.T.ntiles + nw - 1) / nw);
  static int smem_set12[kMaxDevices] = {0}, smem_set17[kMaxDevices] = {0};
  if (m <= 48) {
    cudaError_t e = ensure_dynamic_smem(pair_ai_kernel<12>, smem, smem_set12);
    if (e != cudaSuccess) return e;
    pair_ai_kernel<12><<<blocks, nw * 32, smem, st>>>(A);
  } else {
    cudaError_t e = ensure_dynamic_smem(pair_ai_kernel<17>, smem, smem_set17);
    if (e != cudaSuccess) return e;
    pair_ai_kernel<17><<<blocks, nw * 32, smem, st>>>(A);
  }
  return cudaGetLastError();
}

static PairArgs make_pair_args(const float* Wa, const float* Wb, int nA, int nB, int m, int dist, int tri,
                               int64_t pair_begin, int64_t pair_end, float weight, const float* gD, float* dist_out,
                               float* eig_out, bool want_grad, bool want_loss, float* ws, const PairWorkspace& L) {
  PairArgs A;
  A.Wa = Wa; A.Wb = Wb; A.nA = nA; A.nB = nB; A.m = m; A.dist = dist; A.tri = tri;
  A.pair_begin = pair_begin; A.pair_end = pair_end; A.weight = weight; A.gD = gD;
  A.dist_out = dist_out; A.eig_out = eig_out;
  A.rowpart = want_grad ? ws + L.rowpart : nullptr;
  A.colpart = want_grad ? ws + L.colpart : nullptr;
  A.losspart = want_loss ? ws + L.losspart : nullptr;
  A.Mu = nullptr;
  A.k = 0;
  A.pwpart = nullptr;
  A.T = L.T;
  return A;
}

cudaError_t launch_pair_distances(const float* Wa, const float* Wb, int nA, int nB, int m, int dist, int tri,
                                  int64_t pair_begin, int64_t pair_end, float weight, const float* gD,
                                  float* dist_out, float* loss, float* gEa, float* gEb, float* eig_out, float* ws,
                                  cudaStream_t st) {
  if (tri && dist_out != nullptr && nA > 0) {
    const float dv = (dist & SQFA_DIST_SQUARED) ? 0.f : sqrtf(DIST_EPS);  // d(i,i): lambda = 1 exactly
    fill_diagonal_kernel<<<(nA + 255) / 256, 256, 0, st>>>(dist_out, nA, dv);
  }
  if (pair_end <= pair_begin) return cudaGetLastError();
  const PairWorkspace L = pair_workspace(nA, nB, m, dist, tri, pair_begin, pair_end);
  const bool want_grad = gEa != nullptr, want_loss = loss != nullptr;
  const PairArgs A = make_pair_args(Wa, Wb, nA, nB, m, dist, tri, pair_begin, pair_end, weight, gD, dist_out, eig_out,
                                    want_grad, want_loss, ws, L);
  cudaError_t e = launch_pair_kernel(A, st);
  if (e != cudaSuccess) return e;
  if (!want_grad && !want_loss) return cudaSuccess;
  const int nC = nA > nB ? nA : nB;
  const bool le = (dist & 15) == SQFA_DIST_LOG_EUCLIDEAN;
  if (le && want_grad)
    le_grad_kernel<<<nC, 256, 0, st>>>(L.T, Wa, Wb, nA, nB, m * m, 2 * m * m + 2 * m, m * m + 2 * m, A.rowpart, gEa, gEb);
  pair_reduce_kernel<float, false><<<nC + 1, pair_reduce_threads(m), 0, st>>>(L.T, nA, nB, m, le ? nullptr : A.rowpart, A.colpart, A.losspart,
                                                    gEa, gEb, loss, 1.f, nullptr, 0, 0, nullptr, nullptr);
  return cudaGetLastError();
}

// The pair stage of the closure: distances of the pairs [pair_begin, pair_end) of the C classes, then
// per class the reduced dLoss/dE pushed through the adjoint of the embedding -> (gPsi, gMu), and
// out = {weight * sum d, #non-finite, 0}. Log-Euclidean: the gradient w.r.t. the matrix logarithms is
// accumulated in gLog (zeroed here) and the caller applies the factorisation's adjoint.
cudaError_t launch_pair_closure(const float* W, int C, int m, int dist, int64_t pair_begin, int64_t pair_end,
                                float weight, const float* Mu, int k, float* out, float* gPsi, float* gMu, float* gLog,
                                float* ws, cudaStream_t st) {
  const bool le = (dist & 15) == SQFA_DIST_LOG_EUCLIDEAN;
  const bool fr = (dist & 15) == SQFA_DIST_FISHER_RAO_LB;
  const bool w2 = (dist & 15) == SQFA_DIST_WASSERSTEIN_GAUSSIAN;
  const PairWorkspace L = pair_workspace(C, C, m, dist, 1, pair_begin, pair_end);
  PairArgs A = make_pair_args(W, W, C, C, m, dist, 1, pair_begin, pair_end, weight, nullptr, nullptr, nullptr,
                              true, true, ws, L);
  if (w2) {  // |mu'_i - mu'_j|^2 joins d^2; the pair factors give gMu below
    A.Mu = Mu;
    A.k = k;
    A.pwpart = ws + L.pwpart;
  }
  cudaError_t e = launch_pair_kernel(A, st);
  if (e != cudaSuccess) return e;
  if (w2) {  // gMu[c] = sum_o pw(c, o) (mu'_c - mu'_o), fixed order
    if ((e = cudaMemsetAsync(gMu, 0, (size_t)C * k * sizeof(float), st)) != cudaSuccess) return e;
    if (L.T.ntiles > 0) le_grad_kernel<<<C, 256, 0, st>>>(L.T, Mu, Mu, C, C, k, k, 0, A.pwpart, gMu, gMu);
  }
  if (le) {
    if ((e = cudaMemsetAsync(gLog, 0, (size_t)C * m * m * sizeof(float), st)) != cudaSuccess) return e;
    if (L.T.ntiles > 0)
      le_grad_kernel<<<C, 256, 0, st>>>(L.T, W, W, C, C, m * m, 2 * m * m + 2 * m, m * m + 2 * m, A.rowpart, gLog,
                                        gLog);
    pair_reduce_kernel<float, true><<<C + 1, pair_reduce_threads(m), 0, st>>>(L.T, C, C, m, nullptr, nullptr, A.losspart, nullptr, nullptr, out,
                                                    weight, nullptr, k, 0, nullptr, nullptr);
    return cudaGetLastError();
  }
  return launch_pair_reduce_closure(L.T, C, m, k, fr ? 1 : 0, A.rowpart, A.colpart, A.losspart, weight, Mu, out, gPsi,
                                    gMu, st);
}

template <typename T>
cudaError_t launch_pair_reduce_closure(const PairTiles& tiles, int C, int m, int k, int fr, const T* rowpart,
                                       const T* colpart, const T* losspart, T weight, const T* Mu, T* out, T* gPsi,
                                       T* gMu, cudaStream_t st) {
  pair_reduce_kernel<T, true><<<C + 1, pair_reduce_threads(m), m * m * sizeof(T), st>>>(
      tiles, C, C, m, rowpart, colpart, losspart, nullptr, nullptr, out, weight, Mu, k, fr, gPsi, gMu);
  return cudaGetLastError();
}
template cudaError_t launch_pair_reduce_closure<float>(const PairTiles&, int, int, int, int, const float*, const float*,
                                                       const float*, float, const float*, float*, float*, float*,
                                                       cudaStream_t);
template cudaError_t launch_pair_reduce_closure<double>(const PairTiles&, int, int, int, int, const double*,
                                                        const double*, const double*, double, const double*, double*,
                                                        double*, double*, cudaStream_t);

cudaError_t launch_class_factor_bwd(const float* W, const float* gLog, int C, int m, int dist, float* gE,
                                    cudaStream_t st) {
  if ((dist & 15) != SQFA_DIST_LOG_EUCLIDEAN || C <= 0) return cudaSuccess;
  const int per_warp = 3 * m * m * (int)sizeof(float);
  const int nw = warps_for(per_warp, PAIR_WARPS);
  const int smem = nw * per_warp;
  static int smem_set[kMaxDevices] = {0};
  {
    cudaError_t e = ensure_dynamic_smem(le_factor_bwd_kernel, smem, smem_set);
    if (e != cudaSuccess) return e;
  }
  le_factor_bwd_kernel<<<(C + nw - 1) / nw, nw * 32, smem, st>>>(W, gLog, C, m, gE);
  return cudaGetLastError();
}

}  // namespace sqfa
