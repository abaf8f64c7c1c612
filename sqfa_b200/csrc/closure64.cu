// The fitting closure of closure.cu in float64, for the affine-invariant and Fisher-Rao lower-bound distances
// (plain and squared), k <= 32 filters (m = k or k + 1 <= 33), constraint none or sphere, the first n_fixed
// filters frozen. It is what a model converted with `.double()` evaluates: the reference's remedy for NaN / inf
// distances (_optim.py:28-30). Same formulation as the float32 closure (pairs.cu header), every operation in
// double, with exact division, square root and logarithm. Eight launches and one 4-byte memset, no
// floating-point atomics (loss and gradient are bit-reproducible). The kernels marked * are the float32
// closure's, instantiated for double (project.cu, pairs.cu); this file holds what differs in float64:
//   constraint_fwd_kernel*    F = W / |W| row-wise                              (sphere only)
//   project64_stream_kernel   row-split partials of T_c = F S_c                 (the one pass over C D^2 doubles)
//   project64_finish_kernel   T_c; per-chunk partials of Psi_c = T_c F^T and mu'_c = F m_c
//   class64_kernel            E_c (assemble_class_matrix*, spd_factor.cuh), L_c and L_c^-1 (one warp per class)
//   pair64_kernel             one-sided Jacobi per pair, distances, per-tile partial dLoss/dE (one warp per tile)
//   pair_reduce_kernel*       dLoss/dE_c in a fixed order -> embedding adjoint (gPsi, gMu); loss, #non-finite
//   project_bwd_kernel*       class-split partials of dLoss/dF
//   closure_finish_kernel*    dLoss/dF, constraint adjoint -> grad, max |grad|; the last block publishes out
// The mean-covariance distances (Mahalanobis, Bhattacharyya, Hellinger; launch_gauss_closure_f64) share the
// constraint, the projection and its adjoint, and replace class64 / pair64 / pair_reduce with the class, pair and
// reduce stages of gauss.cu instantiated for double (DESIGN.md section 19).
//
// Pair stage. A = (L_j^-1 L_i)^T; the one-sided Jacobi orthogonalises its columns, A_f = A V, and
// lambda_q = |a_q|^2 are the generalized eigenvalues of (E_i, E_j). d^2 = sum_q log^2 lambda_q (FR: / 2).
// Y = L_i^-T A_f (a back substitution with L_i) holds the generalized eigenvectors, y_q^T E_j y_q = 1:
//   d(d^2)/dE_i =  sum_q (2 log(lambda_q) / lambda_q) y_q y_q^T,   d(d^2)/dE_j = -sum_q 2 log(lambda_q) y_q y_q^T.
// Stopping rule of the Jacobi (DESIGN.md section 18): a column pair is rotated while
// |a_p . a_q| > J64_TOL |a_p| |a_q|; a sweep whose rotations all had |a_p . a_q| <= J64_LAST |a_p| |a_q| is the
// last one (what it leaves is of order J64_LAST^2 relative); at most J64_MAX_SWEEPS sweeps.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/sqfa_b200.h"
#include "sqfa_internal.h"
#include "pair_tiles.cuh"
#include "spd_factor.cuh"

namespace sqfa {

namespace {

constexpr double J64_TOL = 1e-14;
constexpr double J64_LAST = 1e-8;
constexpr int J64_MAX_SWEEPS = 30;
constexpr double DIST_EPS64 = 1e-6;  // distances.py:29 EPSILON
constexpr int W64 = 4;               // warps per block of the per-class and pair kernels
constexpr int PS64_THREADS = 128;    // projection stream: threads per block
constexpr int PS64_FROWS = 64;       // rows of F^T staged in shared memory at a time
constexpr int PF64_COLS = 64;        // columns per chunk of the Psi / mu' partials

// ---------------------------------------------------------------------------------------------------------------
// projection
// ---------------------------------------------------------------------------------------------------------------
// part[split][c][f][j] = sum_{i in the rows of split} F[f][i] S[c][i][j]. A thread owns VEC adjacent columns
// (VEC = 2: one 16-byte load per row) and all KT filters; F^T arrives in shared memory PS64_FROWS rows at a
// time and is read as double2 broadcasts (two filters per load, four DFMAs per load when VEC = 2).
template <int KT, int VEC>
__global__ void __launch_bounds__(PS64_THREADS)
project64_stream_kernel(const double* __restrict__ S, const double* __restrict__ F, int C, int D, int k, int rows,
                        double* __restrict__ part) {
  __shared__ __align__(16) double Fs[PS64_FROWS][KT];
  const int c = blockIdx.z, split = blockIdx.y;
  const int j0 = (blockIdx.x * PS64_THREADS + threadIdx.x) * VEC;
  const int i0 = split * rows, i1 = min(D, i0 + rows);
  double acc[VEC][KT];
#pragma unroll
  for (int v = 0; v < VEC; ++v)
#pragma unroll
    for (int f = 0; f < KT; ++f) acc[v][f] = 0.0;
  const double* Sc = S + (int64_t)c * D * D;
  for (int ib = i0; ib < i1; ib += PS64_FROWS) {
    const int nr = min(PS64_FROWS, i1 - ib);
    __syncthreads();
    for (int idx = threadIdx.x; idx < PS64_FROWS * KT; idx += PS64_THREADS) {
      const int r = idx / KT, f = idx % KT;
      Fs[r][f] = (r < nr && f < k) ? F[(int64_t)f * D + ib + r] : 0.0;
    }
    __syncthreads();
    if (j0 < D) {
      const double* srow = Sc + (int64_t)ib * D + j0;
#pragma unroll 4
      for (int r = 0; r < nr; ++r, srow += D) {
        double s[VEC];
        if (VEC == 2) {
          const double2 t = *reinterpret_cast<const double2*>(srow);
          s[0] = t.x;
          s[VEC - 1] = t.y;
        } else {
          s[0] = *srow;
        }
#pragma unroll
        for (int f = 0; f < KT; f += 2) {
          const double2 fv = *reinterpret_cast<const double2*>(&Fs[r][f]);
#pragma unroll
          for (int v = 0; v < VEC; ++v) {
            acc[v][f] = fma(fv.x, s[v], acc[v][f]);
            acc[v][f + 1] = fma(fv.y, s[v], acc[v][f + 1]);
          }
        }
      }
    }
  }
  if (j0 < D) {
    double* out = part + ((int64_t)split * C + c) * k * D + j0;
#pragma unroll
    for (int f = 0; f < KT; ++f) {
      if (f < k) {
        if (VEC == 2) *reinterpret_cast<double2*>(out + (int64_t)f * D) = make_double2(acc[0][f], acc[VEC - 1][f]);
        else out[(int64_t)f * D] = acc[0][f];
      }
    }
  }
}

// One block per (chunk of PF64_COLS columns, class), one thread per column:
//   T[c][f][j]               = sum over the row splits (in split order)
//   PsiPart[c][chunk][f][g]  = sum_{j in chunk} T[c][f][j] F[g][j]
//   MuPart[c][chunk][f]      = sum_{j in chunk} F[f][j] m[c][j]          (M given: Fisher-Rao)
// Psi[f][g] and Psi[g][f] are different products and agree only up to rounding; the class stage reads the lower
// triangle only.
__global__ void __launch_bounds__(PF64_COLS)
project64_finish_kernel(const double* __restrict__ part, const double* __restrict__ F, const double* __restrict__ M,
                        int C, int D, int k, int nsplit, double* __restrict__ T, double* __restrict__ PsiPart,
                        double* __restrict__ MuPart) {
  __shared__ double Ts[32][PF64_COLS + 1];
  __shared__ double Fs[32][PF64_COLS + 1];
  __shared__ double ms[PF64_COLS];
  const int c = blockIdx.y, chunk = blockIdx.x, nchunk = gridDim.x;
  const int tx = threadIdx.x, j = chunk * PF64_COLS + tx;
  const bool in = j < D;
  for (int f = 0; f < k; ++f) {
    double a = 0.0;
    if (in) {
      for (int s = 0; s < nsplit; ++s) a += part[(((int64_t)s * C + c) * k + f) * D + j];
      T[((int64_t)c * k + f) * D + j] = a;
    }
    Ts[f][tx] = a;
    Fs[f][tx] = in ? F[(int64_t)f * D + j] : 0.0;
  }
  ms[tx] = (M != nullptr && in) ? M[(int64_t)c * D + j] : 0.0;
  __syncthreads();
  const int ncol = min(PF64_COLS, D - chunk * PF64_COLS);
  double* pp = PsiPart + ((int64_t)c * nchunk + chunk) * k * k;
  for (int e = tx; e < k * k; e += PF64_COLS) {
    const int f = e / k, g = e % k;
    double a = 0.0;
    for (int u = 0; u < ncol; ++u) a = fma(Ts[f][u], Fs[g][u], a);
    pp[e] = a;
  }
  if (M != nullptr) {
    for (int f = tx; f < k; f += PF64_COLS) {
      double a = 0.0;
      for (int u = 0; u < ncol; ++u) a = fma(Fs[f][u], ms[u], a);
      MuPart[((int64_t)c * nchunk + chunk) * k + f] = a;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// class stage: E_c, L_c, L_c^-1 (one warp per class)
// ---------------------------------------------------------------------------------------------------------------
__host__ __device__ inline int class64_smem_doubles(int m, int k) { return 2 * m * (m + 1) + m * m + k; }

// W[c] = [L (m*m) | L^-1 (m*m)], row-major. A pivot that is not positive / finite fills W[c]
// with NaN, so every distance of the class is NaN and the fit raises the reference's NaN message.
__global__ void __launch_bounds__(W64 * 32)
class64_kernel(const double* __restrict__ PsiPart, const double* __restrict__ MuPart, int nchunk,
               const double* __restrict__ noise_p, int C, int k, int fr, double* __restrict__ Mu, double* __restrict__ W) {
  extern __shared__ double smem64[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + warp;
  if (c >= C) return;
  const int m = fr ? k + 1 : k, ld = m + 1;
  double* La = smem64 + (size_t)warp * class64_smem_doubles(m, k);
  double* Li = La + m * ld;
  double* Es = Li + m * ld;
  double* mus = Es + m * m;
  assemble_class_matrix(PsiPart, fr ? MuPart : nullptr, nchunk, *noise_p, c, k, fr != 0, Mu, mus, Es, nullptr, lane);
  __syncwarp();
  const bool ok = warp_cholesky_inverse<double>(Es, La, Li, m, ld, lane);
  double* Wc = W + (int64_t)c * 2 * m * m;
  for (int idx = lane; idx < m * m; idx += 32) {
    const int r = idx / m, q = idx % m;
    Wc[idx] = ok ? ((q <= r) ? La[r * ld + q] : 0.0) : NAN;
    Wc[m * m + idx] = ok ? Li[r * ld + q] : NAN;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// pair stage
// ---------------------------------------------------------------------------------------------------------------
struct Pair64Args {
  const double* W;
  int C, m, dist;
  int64_t pair_begin, pair_end;
  double weight;
  double* rowpart;   // [ntiles][R][m*m]
  double* colpart;   // [ntiles][R][m*m]
  double* losspart;  // [ntiles][2] {sum of distances, non-finite count}
  PairTiles T;
};

// column stride (doubles) of the column-contiguous matrices: odd, so the columns of different lanes spread over
// the banks
__host__ __device__ inline int p64_ldc(int m) { return m | 1; }
// doubles of shared memory per warp: [A columns (mp) | staging of L_j^-T, later Y columns (m) | L_i | ci | cj]
__host__ __device__ inline int p64_smem_doubles(int m) {
  const int mp = (m + 1) & ~1;
  return (mp + m) * p64_ldc(m) + m * m + 2 * mp;
}

// One-sided Jacobi on the mp (even) columns of A (column p at A + p * ldc, m rows; a padding column is zero).
// Round-robin (circle method) ordering: in each of the mp - 1 rounds of a sweep lane t < mp / 2 owns one
// column pair, forms the three dot products and rotates both columns in place.
__device__ void jacobi64(double* A, int m, int mp, int ldc, int lane) {
  const int n1 = mp - 1, np = mp >> 1;
  for (int sweep = 0; sweep < J64_MAX_SWEEPS; ++sweep) {
    bool big = false;
    for (int r = 0; r < n1; ++r) {
      if (lane < np) {
        int p, q;
        if (lane == 0) {
          p = n1; q = r;
        } else {
          p = r + lane; if (p >= n1) p -= n1;
          q = r - lane; if (q < 0) q += n1;
        }
        double* x = A + (p < q ? p : q) * ldc;
        double* y = A + (p < q ? q : p) * ldc;
        double al = 0.0, be = 0.0, ga = 0.0;
        for (int s = 0; s < m; ++s) {
          const double xv = x[s], yv = y[s];
          al = fma(xv, xv, al);
          be = fma(yv, yv, be);
          ga = fma(xv, yv, ga);
        }
        const double g2 = ga * ga, sc = al * be;
        if (al > 0.0 && be > 0.0 && g2 > (J64_TOL * J64_TOL) * sc) {
          // x' = c x - s y, y' = s x + c y with t = tan of the angle that zeroes x' . y'
          const double zeta = (be - al) / (2.0 * ga);
          const double t = copysign(1.0 / (fabs(zeta) + sqrt(fma(zeta, zeta, 1.0))), zeta);
          const double cs = 1.0 / sqrt(fma(t, t, 1.0)), sn = cs * t;
          big = big || g2 > (J64_LAST * J64_LAST) * sc;
          for (int s = 0; s < m; ++s) {
            const double xv = x[s], yv = y[s];
            x[s] = fma(cs, xv, -sn * yv);
            y[s] = fma(sn, xv, cs * yv);
          }
        }
      }
      __syncwarp();
    }
    if (!__any_sync(0xffffffffu, big)) break;
  }
}

__device__ __forceinline__ double finish_distance64(double d2, int dist, double* dd_dd2) {
  const double cfac = ((dist & 15) == SQFA_DIST_FISHER_RAO_LB) ? 0.5 : 1.0;
  if (dist & SQFA_DIST_SQUARED) {
    *dd_dd2 = cfac;
    return cfac * d2;
  }
  const double d = sqrt(cfac * d2 + DIST_EPS64);
  *dd_dd2 = cfac / (2.0 * d);
  return d;
}

// One warp per R x R tile of the strict lower triangle, walked row by row. The warp owns its tile's partial slots:
// it zeroes them, then adds every pair's dLoss/dE_i to the slot of row i and dLoss/dE_j to the slot of column j
// (the lane that owns matrix column s reads and writes element (r, s) every time: no hazard, fixed order).
__global__ void __launch_bounds__(W64 * 32)
pair64_kernel(const Pair64Args A) {
  extern __shared__ double smem64[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (t >= A.T.ntiles) return;
  const int m = A.m, m2 = m * m, R = A.T.R;
  const int mp = (m + 1) & ~1, ldc = p64_ldc(m), nslot = (m + 31) >> 5;
  int bi, bj;
  decode_tile(A.T, t, bi, bj);
  double* bufA = smem64 + (size_t)warp * p64_smem_doubles(m);
  double* bufY = bufA + mp * ldc;
  double* Ls = bufY + m * ldc;
  double* ci = Ls + m2;
  double* cj = ci + mp;
  double* rp = A.rowpart + t * R * m2;
  double* cp = A.colpart + t * R * m2;
  for (int u = 0; u < R; ++u)
    for (int tt = 0; tt < nslot; ++tt) {
      const int s = lane + 32 * tt;
      if (s < m)
        for (int r = 0; r < m; ++r) {
          rp[u * m2 + r * m + s] = 0.0;
          cp[u * m2 + r * m + s] = 0.0;
        }
    }
  double dsum = 0.0, bad = 0.0;
  for (int ii = 0; ii < R; ++ii) {
    const int i = bi * R + ii;
    bool have_i = false;
    for (int jj = 0; jj < R; ++jj) {
      const int j = bj * R + jj;
      if (!pair_in_launch(i, j, A.C, A.C, 1, A.pair_begin, A.pair_end)) continue;
      const double* Wi = A.W + (int64_t)i * 2 * m2;
      const double* Wj = A.W + (int64_t)j * 2 * m2;
      __syncwarp();
      if (!have_i) {
        for (int idx = lane; idx < m2; idx += 32) Ls[idx] = Wi[idx];
        have_i = true;
      }
      // stage L_j^-1 transposed: bufY[r][q] = Linv_j[q][r]
      for (int idx = lane; idx < m2; idx += 32) {
        const int q = idx / m, r = idx % m;
        bufY[r * ldc + q] = Wj[m2 + idx];
      }
      if (mp != m)
        for (int s = lane; s < m; s += 32) bufA[(mp - 1) * ldc + s] = 0.0;
      __syncwarp();
      // column q of A: A[s][q] = sum_{s <= r <= q} Linv_j[q][r] L_i[r][s]
      for (int tt = 0; tt < nslot; ++tt) {
        const int q = lane + 32 * tt;
        if (q < m)
          for (int s = 0; s < m; ++s) {
            double a = 0.0;
            for (int r = s; r <= q; ++r) a = fma(bufY[r * ldc + q], Ls[r * m + s], a);
            bufA[q * ldc + s] = a;
          }
      }
      __syncwarp();
      jacobi64(bufA, m, mp, ldc, lane);
      double d2 = 0.0;
      for (int tt = 0; tt < nslot; ++tt) {
        const int q = lane + 32 * tt;
        if (q < m) {
          double n2 = 0.0;
          for (int s = 0; s < m; ++s) n2 = fma(bufA[q * ldc + s], bufA[q * ldc + s], n2);
          const double ll = log(n2);
          d2 = fma(ll, ll, d2);
          ci[q] = 2.0 * ll / n2;
          cj[q] = -2.0 * ll;
        }
      }
      d2 = warp_sum(d2);
      double dd_dd2;
      const double dval = finish_distance64(d2, A.dist, &dd_dd2);
      dsum += dval;
      if (!isfinite(dval)) bad += 1.0;
      const double w = A.weight * dd_dd2;
      __syncwarp();
      // column q of Y = L_i^-T A_f: back substitution L_i^T y_q = a_q, over the (dead) staging buffer
      for (int tt = 0; tt < nslot; ++tt) {
        const int q = lane + 32 * tt;
        if (q < m)
          for (int r = m - 1; r >= 0; --r) {
            double v = bufA[q * ldc + r];
            for (int s = r + 1; s < m; ++s) v = fma(-Ls[s * m + r], bufY[q * ldc + s], v);
            bufY[q * ldc + r] = v / Ls[r * m + r];
          }
      }
      __syncwarp();
      // G_i[r][s] += w sum_q ci_q Y[r][q] Y[s][q],  G_j[r][s] += w sum_q cj_q Y[r][q] Y[s][q]; lane <-> column s
      for (int tt = 0; tt < nslot; ++tt) {
        const int s = lane + 32 * tt;
        if (s < m)
          for (int r = 0; r < m; ++r) {
            double a = 0.0, b = 0.0;
            for (int q = 0; q < m; ++q) {
              const double yy = bufY[q * ldc + r] * bufY[q * ldc + s];
              a = fma(ci[q], yy, a);
              b = fma(cj[q], yy, b);
            }
            rp[ii * m2 + r * m + s] += w * a;
            cp[jj * m2 + r * m + s] += w * b;
          }
      }
    }
  }
  if (lane == 0) {
    A.losspart[2 * t] = dsum;
    A.losspart[2 * t + 1] = bad;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
// row splits of the streaming pass: enough (column block, split, class) blocks for about eight per SM, at least
// 64 rows per split
int p64_nsplit(int C, int D) {
  const int64_t colblocks = (D + 2 * PS64_THREADS - 1) / (2 * PS64_THREADS);
  const int64_t per_split = colblocks * (C > 0 ? C : 1);
  int n = (int)((8 * 148 + per_split - 1) / per_split);
  const int max_split = D / 64 > 1 ? D / 64 : 1;
  if (n > max_split) n = max_split;
  return n < 1 ? 1 : n;
}

// Tile edge: single pairs for short pair lists (every pair its own warp), up to 4 x 4 once there are enough tiles
// to fill the GPU several times over (the per-tile partials shrink with R: 2 R m^2 doubles per R^2 pairs).
int p64_tile_edge(int64_t npairs) {
  int R = 1;
  while (R < 4 && npairs / ((int64_t)(R + 1) * (R + 1)) >= 4096) ++R;
  return R;
}

struct Closure64Layout {
  size_t F, inv_norm, T, Mu, W, logdet, sinv, gPsi, gMu, red_out, ticket, proj, psipart, mupart, rowpart, colpart,
      losspart, pair, total;
  int rows, nsplit, nchunk, csplit;
  PairTiles tiles;
};

// One layout for both float64 closures. The mean-covariance distances (gauss) keep Psi_c in W, logdet Psi_c and
// Psi_c^-1 for Bhattacharyya / Hellinger, and the pair stage's workspace of gauss.cu in `pair`; the
// affine-invariant / Fisher-Rao closure keeps [L_c | L_c^-1] in W and its tile partials.
Closure64Layout closure64_layout(int C, int D, int k, int dist, int64_t pair_begin, int64_t pair_end) {
  const bool fr = (dist & 15) == SQFA_DIST_FISHER_RAO_LB;
  const bool gauss = is_gauss_closure(dist);
  const bool ld = gauss_closure_needs_logdet(dist);
  const int m = fr ? k + 1 : k;
  Closure64Layout L;
  L.nsplit = p64_nsplit(C, D);
  L.rows = (D + L.nsplit - 1) / L.nsplit;
  L.nsplit = (D + L.rows - 1) / L.rows;
  L.nchunk = (D + PF64_COLS - 1) / PF64_COLS;
  L.csplit = project_bwd_csplit<double>(C, D);
  const int64_t npairs = pair_end > pair_begin ? pair_end - pair_begin : 0;
  L.tiles = make_pair_tiles(C, C, 1, pair_begin, pair_end, gauss ? 1 : p64_tile_edge(npairs));
  const size_t part = gauss ? 0 : (size_t)L.tiles.ntiles * L.tiles.R * m * m;
  const size_t fwd = (size_t)L.nsplit * C * k * D, bwd = (size_t)L.csplit * k * D;
  size_t o = 0;
  L.F = o;        o += al<double>((size_t)k * D);
  L.inv_norm = o; o += al<double>(k);
  L.T = o;        o += al<double>((size_t)C * k * D);
  L.Mu = o;       o += al<double>((size_t)C * k);
  L.W = o;        o += al<double>(gauss ? (size_t)C * k * k : (size_t)C * 2 * m * m);
  L.logdet = o;   o += ld ? al<double>(C) : 0;
  L.sinv = o;     o += ld ? al<double>((size_t)C * k * k) : 0;
  L.gPsi = o;     o += al<double>((size_t)C * k * k);
  L.gMu = o;      o += al<double>((size_t)C * k);
  L.red_out = o;  o += al<double>(64);  // {loss, #non-finite} of a rank's pairs: [gPsi | gMu | red_out] is one exchange span
  L.ticket = o;   o += al<double>(1);  // uint32 arrival ticket of closure_finish_kernel; int32 [2, 4): gauss class flag
  L.proj = o;     o += al<double>(fwd > bwd ? fwd : bwd);  // row-split partials of T, later the class-split partials of dF
  L.psipart = o;  o += al<double>((size_t)C * L.nchunk * k * k);
  L.mupart = o;   o += al<double>((size_t)C * L.nchunk * k);
  L.rowpart = o;  o += al<double>(part);
  L.colpart = o;  o += al<double>(part);
  L.losspart = o; o += gauss ? 0 : al<double>((size_t)2 * L.tiles.ntiles);
  L.pair = o;     o += gauss ? al<double>(gauss_closure_workspace_elems(C, k, pair_begin, pair_end)) : 0;
  L.total = o;
  return L;
}

template <int KT, int VEC>
cudaError_t run_project64(const double* S, const double* F, int C, int D, int k, int rows, int nsplit, double* part,
                          cudaStream_t st) {
  const dim3 grid((D + PS64_THREADS * VEC - 1) / (PS64_THREADS * VEC), nsplit, C);
  project64_stream_kernel<KT, VEC><<<grid, PS64_THREADS, 0, st>>>(S, F, C, D, k, rows, part);
  return cudaGetLastError();
}

template <int VEC>
cudaError_t run_project64_k(const double* S, const double* F, int C, int D, int k, int rows, int nsplit, double* part,
                            cudaStream_t st) {
  if (k <= 4) return run_project64<4, VEC>(S, F, C, D, k, rows, nsplit, part, st);
  if (k <= 8) return run_project64<8, VEC>(S, F, C, D, k, rows, nsplit, part, st);
  if (k <= 16) return run_project64<16, VEC>(S, F, C, D, k, rows, nsplit, part, st);
  return run_project64<32, VEC>(S, F, C, D, k, rows, nsplit, part, st);
}

// The streaming pass over the n classes that S, M, T, PsiPart and MuPart start at (nsplit splits of `rows` rows,
// partials in `part`), then T and the per-chunk partials of Psi_c and, with M, mu'_c.
cudaError_t project64_partials(const double* S, const double* M, const double* F, int n, int D, int k, int rows,
                               int nsplit, int nchunk, double* part, double* T, double* PsiPart, double* MuPart,
                               cudaStream_t st) {
  // 16-byte loads of S when every row starts 16-byte aligned
  const bool vec2 = (D % 2 == 0) && (reinterpret_cast<uintptr_t>(S) & 15) == 0;
  cudaError_t e = vec2 ? run_project64_k<2>(S, F, n, D, k, rows, nsplit, part, st)
                       : run_project64_k<1>(S, F, n, D, k, rows, nsplit, part, st);
  if (e != cudaSuccess) return e;
  project64_finish_kernel<<<dim3(nchunk, n), PF64_COLS, 0, st>>>(part, F, M, n, D, k, nsplit, T, PsiPart, MuPart);
  return cudaGetLastError();
}

// The front of both float64 closures: the sphere constraint (F = W / |W| into the workspace; *F_out is the
// filters the rest reads), the ticket memset, the streaming pass over S and the per-chunk partials of Psi_c and,
// with M, mu'_c.
cudaError_t closure64_front(const double* S, const double* M, const double* raw_filters, int C, int D, int k,
                            int sphere, const Closure64Layout& L, double* ws, const double** F_out, cudaStream_t st) {
  cudaError_t e;
  const double* F = raw_filters;
  if (sphere) {
    if ((e = launch_constraint_fwd(raw_filters, D, k, ws + L.F, ws + L.inv_norm, st)) != cudaSuccess) return e;
    F = ws + L.F;
  }
  *F_out = F;
  if ((e = cudaMemsetAsync(ws + L.ticket, 0, sizeof(unsigned int), st)) != cudaSuccess) return e;
  return project64_partials(S, M, F, C, D, k, L.rows, L.nsplit, L.nchunk, ws + L.proj, ws + L.T, ws + L.psipart,
                            ws + L.mupart, st);
}

// The middle of both float64 closures, from the per-chunk partials of all C classes: the class stage, the pair stage
// on [pair_begin, pair_end) and the per-class reduce into (gPsi, gMu) of every class and out = {weight * sum d,
// #non-finite, 0}. Affine-invariant / Fisher-Rao: class64, pair64, pair_reduce; the mean-covariance distances: the
// class, pair and reduce stages of gauss.cu.
cudaError_t closure64_middle(const double* noise, int C, int k, int dist, int64_t pair_begin, int64_t pair_end,
                             double weight, const Closure64Layout& L, double* out, double* ws, cudaStream_t st) {
  cudaError_t e;
  if (is_gauss_closure(dist)) {
    int32_t* flag = reinterpret_cast<int32_t*>(ws + L.ticket) + 2;
    if ((e = launch_gauss_closure_class(ws + L.psipart, ws + L.mupart, L.nchunk, noise, C, k, dist, ws + L.W,
                                        ws + L.Mu, ws + L.logdet, ws + L.sinv, flag, st)) != cudaSuccess)
      return e;
    return launch_gauss_closure_pairs(ws + L.W, ws + L.Mu, ws + L.logdet, ws + L.sinv, C, k, dist, pair_begin,
                                      pair_end, weight, out, ws + L.gPsi, ws + L.gMu, ws + L.pair, st);
  }
  const int fr = (dist & 15) == SQFA_DIST_FISHER_RAO_LB ? 1 : 0;
  const int m = fr ? k + 1 : k;
  {
    const int per_warp = class64_smem_doubles(m, k) * (int)sizeof(double);
    const int nw = warps_for(per_warp, W64);
    static int smem_set[kMaxDevices] = {0};
    if ((e = ensure_dynamic_smem(class64_kernel, nw * per_warp, smem_set)) != cudaSuccess) return e;
    class64_kernel<<<(C + nw - 1) / nw, nw * 32, nw * per_warp, st>>>(ws + L.psipart, ws + L.mupart, L.nchunk, noise,
                                                                       C, k, fr, ws + L.Mu, ws + L.W);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  if (L.tiles.ntiles > 0) {
    Pair64Args A;
    A.W = ws + L.W;
    A.C = C; A.m = m; A.dist = dist;
    A.pair_begin = pair_begin; A.pair_end = pair_end;
    A.weight = weight;
    A.rowpart = ws + L.rowpart;
    A.colpart = ws + L.colpart;
    A.losspart = ws + L.losspart;
    A.T = L.tiles;
    const int per_warp = p64_smem_doubles(m) * (int)sizeof(double);
    const int nw = warps_for(per_warp, W64);
    static int smem_set[kMaxDevices] = {0};
    if ((e = ensure_dynamic_smem(pair64_kernel, nw * per_warp, smem_set)) != cudaSuccess) return e;
    pair64_kernel<<<(unsigned)((L.tiles.ntiles + nw - 1) / nw), nw * 32, nw * per_warp, st>>>(A);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  return launch_pair_reduce_closure(L.tiles, C, m, k, fr, ws + L.rowpart, ws + L.colpart, ws + L.losspart, weight,
                                    ws + L.Mu, out, ws + L.gPsi, fr ? ws + L.gMu : nullptr, st);
}

// The back of both float64 closures: the projection adjoint with gMu when M is given, the constraint's adjoint,
// the frozen rows, max |grad| and the published out.
cudaError_t closure64_back(const double* M, int C, int D, int k, const double* F, int sphere, int n_fixed,
                           const Closure64Layout& L, double* out, double* out_host, double* grad, double* ws,
                           cudaStream_t st) {
  return launch_project_bwd_constrained(ws + L.gPsi, M != nullptr ? ws + L.gMu : nullptr, ws + L.T, M, C, D, k, F,
                                        ws + L.inv_norm, sphere, n_fixed, grad, out, out_host,
                                        reinterpret_cast<unsigned int*>(ws + L.ticket), ws + L.proj, st);
}

}  // namespace

size_t fused_loss_workspace_bytes_f64(int C, int D, int k, int dist, int64_t pair_begin, int64_t pair_end) {
  return closure64_layout(C, D, k, dist, pair_begin, pair_end).total * sizeof(double);
}

cudaError_t launch_closure_f64(const double* S, const double* M, const double* raw_filters, int C, int D, int k,
                               const double* noise, int dist, int constraint, int n_fixed, int64_t pair_begin,
                               int64_t pair_end, double* out, double* out_host, double* grad, double* ws,
                               cudaStream_t st) {
  const Closure64Layout L = closure64_layout(C, D, k, dist, pair_begin, pair_end);
  const int sphere = constraint == 1 ? 1 : 0;
  const double* Mfr = (dist & 15) == SQFA_DIST_FISHER_RAO_LB ? M : nullptr;
  const int64_t P = (int64_t)C * (C - 1) / 2;
  const double weight = -1.0 / (double)(P > 0 ? P : 1);
  const double* F;
  cudaError_t e;
  if ((e = closure64_front(S, Mfr, raw_filters, C, D, k, sphere, L, ws, &F, st)) != cudaSuccess) return e;
  if ((e = closure64_middle(noise, C, k, dist, pair_begin, pair_end, weight, L, out, ws, st)) != cudaSuccess) return e;
  return closure64_back(Mfr, C, D, k, F, sphere, n_fixed, L, out, out_host, grad, ws, st);
}

// The mean-covariance distances (Mahalanobis, Bhattacharyya, Hellinger) in float64: the front above, the class,
// pair and reduce stages of gauss.cu instantiated for double, and the back with gMu.
cudaError_t launch_gauss_closure_f64(const double* S, const double* M, const double* raw_filters, int C, int D, int k,
                                     const double* noise, int dist, int constraint, int n_fixed, int64_t pair_begin,
                                     int64_t pair_end, double* out, double* out_host, double* grad, double* ws,
                                     cudaStream_t st) {
  const Closure64Layout L = closure64_layout(C, D, k, dist, pair_begin, pair_end);
  const int sphere = constraint == 1 ? 1 : 0;
  const int64_t P = (int64_t)C * (C - 1) / 2;
  const double weight = -1.0 / (double)(P > 0 ? P : 1);
  const double* F;
  cudaError_t e;
  if ((e = closure64_front(S, M, raw_filters, C, D, k, sphere, L, ws, &F, st)) != cudaSuccess) return e;
  if ((e = closure64_middle(noise, C, k, dist, pair_begin, pair_end, weight, L, out, ws, st)) != cudaSuccess) return e;
  return closure64_back(M, C, D, k, F, sphere, n_fixed, L, out, out_host, grad, ws, st);
}

// ---------------------------------------------------------------------------------------------------------------
// The float64 closure with the CLASSES and the PAIRS sharded over ranks: the three phases of
// launch_fused_loss_sharded (closure.cu) on the float64 layout, for every code of the two closures above. F is the
// constrained filters; the caller all-reduces exchange span 0 after phase 0 and span 1 after phase 1.
//   phase 0  zero span 0 = [PsiPart | MuPart]; the streaming projection of classes [c0, c1) only, its row split
//            chosen for c1 - c0 classes (bounded by the proj region, which the layout sizes for C classes)
//   phase 1  class stage of all C classes from the summed partials, pair stage on [pair_begin, pair_end), reduce
//            into span 1 = [gPsi | gMu | red_out] (every class's gPsi is written, red_out[0..1] = {weight * sum d,
//            #non-finite}, the rest of red_out zero)
//   phase 2  the projection adjoint over classes [c0, c1) into dF: the closure's tail with no constraint, no
//            frozen rows and no published out
void fused_loss_exchange_span_f64(int C, int D, int k, int dist, int64_t pair_begin, int64_t pair_end, int which,
                                  size_t* offset_bytes, size_t* bytes) {
  const Closure64Layout L = closure64_layout(C, D, k, dist, pair_begin, pair_end);
  if (which == 0) {
    *offset_bytes = L.psipart * sizeof(double);
    *bytes = (L.rowpart - L.psipart) * sizeof(double);  // psipart and mupart are adjacent
  } else {
    *offset_bytes = L.gPsi * sizeof(double);
    *bytes = (L.ticket - L.gPsi) * sizeof(double);  // gPsi | gMu | red_out
  }
}

cudaError_t launch_fused_loss_sharded_f64(int phase, const double* S, const double* M, const double* F, int C, int D,
                                          int k, const double* noise, int dist, int c0, int c1, int64_t pair_begin,
                                          int64_t pair_end, double* dF, double* ws, cudaStream_t st) {
  const Closure64Layout L = closure64_layout(C, D, k, dist, pair_begin, pair_end);
  const bool means = (dist & 15) == SQFA_DIST_FISHER_RAO_LB || is_gauss_closure(dist);
  const double* Mm = means ? M : nullptr;
  const int n_own = c1 > c0 ? c1 - c0 : 0;
  cudaError_t e;
  if (phase == 0) {
    if ((e = cudaMemsetAsync(ws + L.psipart, 0, (L.rowpart - L.psipart) * sizeof(double), st)) != cudaSuccess)
      return e;
    if (n_own == 0) return cudaSuccess;
    const size_t per_split = (size_t)n_own * k * D;
    const int cap = (int)std::min<size_t>((L.psipart - L.proj) / per_split, (size_t)D);
    const int nsplit = std::max(1, std::min(p64_nsplit(n_own, D), cap));
    const int rows = (D + nsplit - 1) / nsplit;
    return project64_partials(S + (size_t)c0 * D * D, Mm != nullptr ? Mm + (size_t)c0 * D : nullptr, F, n_own, D, k,
                              rows, (D + rows - 1) / rows, L.nchunk, ws + L.proj, ws + L.T + (size_t)c0 * k * D,
                              ws + L.psipart + (size_t)c0 * L.nchunk * k * k,
                              ws + L.mupart + (size_t)c0 * L.nchunk * k, st);
  }
  if (phase == 1) {
    const int64_t P = (int64_t)C * (C - 1) / 2;
    const double weight = -1.0 / (double)(P > 0 ? P : 1);
    if ((e = cudaMemsetAsync(ws + L.red_out, 0, 64 * sizeof(double), st)) != cudaSuccess) return e;
    return closure64_middle(noise, C, k, dist, pair_begin, pair_end, weight, L, ws + L.red_out, ws, st);
  }
  // phase 2: (gPsi, gMu) are now the sums over all pairs
  return launch_project_bwd_constrained<double>(
      ws + L.gPsi + (size_t)c0 * k * k, Mm != nullptr ? ws + L.gMu + (size_t)c0 * k : nullptr,
      ws + L.T + (size_t)c0 * k * D, Mm != nullptr ? Mm + (size_t)c0 * D : nullptr, n_own, D, k, F, nullptr, 0, 0, dF,
      nullptr, nullptr, nullptr, ws + L.proj, st);
}

}  // namespace sqfa
