// One L-BFGS direction update on the device, in one launch.
//
// The reference optimises the filters with torch.optim.LBFGS (/root/reference/src/sqfa/_optim.py:78-79,
// default arguments: history 100, no line search). On a GPU that optimiser spends its time in the
// two-loop recursion: 4 tiny kernels and 2 implicit host synchronisations (`alpha=-al[i]` converts a
// device scalar) per history entry and iteration -- about 1 ms per iteration at half-full history,
// three times the loss + gradient evaluation it drives (SURVEY.md section 8(f), rank 1).
//
// This kernel does the whole "update memory + two-loop recursion" step of one iteration with the
// same arithmetic, in the same order:
//   y = g - prev_g, s = t_prev d, ys = y.s;  if ys > 1e-10: push (y, s, 1/ys), H = ys / y.y
//   q = -g;  for newest..oldest: al_i = ro_i s_i.q, q -= al_i y_i;  r = H q;
//   for oldest..newest: r += (al_i - ro_i y_i.r) s_i;  d = r;  prev_g = g
// and reports the scalars the host needs for the optimiser's stopping rules.
//
// The vector (k D <= 131072 floats) lives in the registers of one cluster of 8 CTAs x 1024 threads;
// every dot product is a warp-shuffle / shared-memory / distributed-shared-memory reduction with one
// cluster barrier, so a history entry costs about a microsecond instead of four launches and two
// host round trips. All CTAs add the 8 partial sums in the same order: the result is identical
// everywhere and deterministic.
//
// The kernel is a template on the scalar type. The float64 instantiation (a `.double()` model) does the
// same operations in the same order in double, with the cluster's partial sums exchanged as 64-bit
// values; a double vector takes twice the registers, so it is capped at 8 elements per thread
// (n <= 65536, every benchmark shape's k D).
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cuda_runtime.h>

#include "ptx.cuh"
#include "sqfa_internal.h"

namespace sqfa {

namespace {

constexpr int LB_CTAS = 8, LB_THREADS = 1024, LB_STRIDE = LB_CTAS * LB_THREADS;
constexpr int LB_MAX_HISTORY = 127;

// one partial sum into CTA `rank`'s slot, through distributed shared memory
__device__ __forceinline__ void st_cluster(uint32_t cluster_addr, float v) {
  st_cluster_u32(cluster_addr, __float_as_uint(v));
}
__device__ __forceinline__ void st_cluster(uint32_t cluster_addr, double v) {
  st_cluster_u64(cluster_addr, (uint64_t)__double_as_longlong(v));
}

template <typename T>
struct Red3 {
  T a, b, c;  // a, b: sums; c: maximum
};

// cluster-wide reduction of two sums and one maximum; every thread of every CTA gets the result
template <typename T>
__device__ __forceinline__ Red3<T> cluster_reduce3(Red3<T> v, T (*s_part)[32], T (*s_slots)[LB_CTAS][4], int& parity,
                                                   uint32_t rank) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    v.a += __shfl_xor_sync(0xffffffffu, v.a, o);
    v.b += __shfl_xor_sync(0xffffffffu, v.b, o);
    v.c = fmax(v.c, __shfl_xor_sync(0xffffffffu, v.c, o));
  }
  if (lane == 0) { s_part[0][warp] = v.a; s_part[1][warp] = v.b; s_part[2][warp] = v.c; }
  __syncthreads();
  if (warp == 0) {
    Red3<T> w = {s_part[0][lane], s_part[1][lane], s_part[2][lane]};
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      w.a += __shfl_xor_sync(0xffffffffu, w.a, o);
      w.b += __shfl_xor_sync(0xffffffffu, w.b, o);
      w.c = fmax(w.c, __shfl_xor_sync(0xffffffffu, w.c, o));
    }
    if (lane < LB_CTAS) {  // lane r hands this CTA's partials to CTA r
      const uint32_t base = mapa_u32(smem_u32(&s_slots[parity][rank][0]), (uint32_t)lane);
      st_cluster(base, w.a);
      st_cluster(base + sizeof(T), w.b);
      st_cluster(base + 2 * sizeof(T), w.c);
    }
  }
  cluster_sync_all();  // release / acquire: the remote stores are visible, s_part may be reused
  Red3<T> r = {T(0), T(0), T(-INFINITY)};
#pragma unroll
  for (int k = 0; k < LB_CTAS; ++k) {
    r.a += s_slots[parity][k][0];
    r.b += s_slots[parity][k][1];
    r.c = fmax(r.c, s_slots[parity][k][2]);
  }
  parity ^= 1;
  return r;
}

template <typename T, int EPT>
__global__ void __cluster_dims__(LB_CTAS, 1, 1) __launch_bounds__(LB_THREADS, 1)
lbfgs_direction_kernel(const T* __restrict__ g, T* __restrict__ prev_g, T* __restrict__ d, T* __restrict__ S,
                       T* __restrict__ Y, T* __restrict__ ro, T* hdiag, int32_t* meta, int n, int rows, T t_prev,
                       int first, T* param, T lr, T tol_change, T* out) {
  __shared__ T s_part[3][32];
  __shared__ T s_slots[2][LB_CTAS][4];
  __shared__ T s_al[LB_MAX_HISTORY + 1];
  const uint32_t rank = cluster_ctarank();
  const int j0 = (int)rank * LB_THREADS + (int)threadIdx.x;
  int parity = 0;

  // Register budget: 1024 threads leave 64 registers per thread, so only the running vector r
  // stays in registers; g, and the pair written speculatively below, are re-read from L2.
  T r[EPT];
  T l1 = T(0);
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int j = j0 + e * LB_STRIDE;
    const T gj = j < n ? g[j] : T(0);
    r[e] = -gj;  // q of the two-loop recursion (and d itself on the first iteration)
    l1 += fabs(gj);
  }
  int head = 0, count = 0;
  T hd = T(1), ys = T(0);
  if (!first) {
    head = meta[0];
    count = meta[1];
    hd = hdiag[0];
    const int slot = (head + count) % rows;  // the ring has one spare row: the write below is speculative
    Red3<T> v = {T(0), T(0), T(0)};
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int j = j0 + e * LB_STRIDE;
      if (j < n) {
        const T yv = -r[e] - prev_g[j];
        const T sv = t_prev * d[j];
        v.a = fma(yv, sv, v.a);
        v.b = fma(yv, yv, v.b);
        Y[(int64_t)slot * n + j] = yv;
        S[(int64_t)slot * n + j] = sv;
      }
    }
    v = cluster_reduce3(v, s_part, s_slots, parity, rank);  // also orders the meta reads above before the update below
    ys = v.a;
    T ro_new = T(0);
    const bool pushed = ys > T(1e-10);  // identical in every thread of the cluster
    if (pushed) {
      if (count == rows - 1) head = (head + 1) % rows;  // history full: drop the oldest pair
      else ++count;
      ro_new = T(1) / ys;
      hd = ys / v.b;
      if (rank == 0 && threadIdx.x == 0) {
        ro[slot] = ro_new;
        hdiag[0] = hd;
        meta[0] = head;
        meta[1] = count;
      }
    }
    // ---- two-loop recursion (torch/optim/lbfgs.py: "iteration in L-BFGS loop collapsed")
    for (int i = count - 1; i >= 0; --i) {
      const int idx = (head + i) % rows;
      T yr[EPT];
      Red3<T> w = {T(0), T(0), T(0)};
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const int j = j0 + e * LB_STRIDE;
        const T sr = j < n ? S[(int64_t)idx * n + j] : T(0);
        yr[e] = j < n ? Y[(int64_t)idx * n + j] : T(0);  // in flight during the reduction
        w.a = fma(sr, r[e], w.a);
      }
      w = cluster_reduce3(w, s_part, s_slots, parity, rank);
      const T al = w.a * ((pushed && idx == slot) ? ro_new : ro[idx]);
      if (threadIdx.x == 0) s_al[i] = al;
#pragma unroll
      for (int e = 0; e < EPT; ++e) r[e] = fma(-al, yr[e], r[e]);
    }
#pragma unroll
    for (int e = 0; e < EPT; ++e) r[e] *= hd;
    for (int i = 0; i < count; ++i) {
      const int idx = (head + i) % rows;
      T sr[EPT];
      Red3<T> w = {T(0), T(0), T(0)};
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const int j = j0 + e * LB_STRIDE;
        const T yr = j < n ? Y[(int64_t)idx * n + j] : T(0);
        sr[e] = j < n ? S[(int64_t)idx * n + j] : T(0);
        w.a = fma(yr, r[e], w.a);
      }
      w = cluster_reduce3(w, s_part, s_slots, parity, rank);  // its barriers also publish s_al
      const T be = w.a * ((pushed && idx == slot) ? ro_new : ro[idx]);
      const T c = s_al[i] - be;
#pragma unroll
      for (int e = 0; e < EPT; ++e) r[e] = fma(c, sr[e], r[e]);
    }
  }
  Red3<T> v = {T(0), l1, T(0)};
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int j = j0 + e * LB_STRIDE;
    if (j < n) {
      const T gj = g[j];
      d[j] = r[e];
      prev_g[j] = gj;
      v.a = fma(gj, r[e], v.a);
      v.c = fmax(v.c, fabs(r[e]));
    }
  }
  v = cluster_reduce3(v, s_part, s_slots, parity, rank);
  // The fixed step of the optimiser (no line search), applied here when the caller passes the parameter:
  // x += t d with t = min(1, 1 / |g|_1) lr on the first iteration, lr afterwards -- unless the directional
  // derivative is above -tolerance_change, the test on which the optimiser stops BEFORE stepping. Every
  // thread holds the same reduced scalars, so the decision is uniform.
  const T t_step = first ? fmin(T(1), T(1) / v.b) * lr : lr;
  const bool apply = param != nullptr && !(v.a > -tol_change);
  if (apply) {
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int j = j0 + e * LB_STRIDE;
      if (j < n) param[j] = fma(t_step, r[e], param[j]);
    }
  }
  if (rank == 0 && threadIdx.x == 0) {
    if (first) {
      hdiag[0] = T(1);
      meta[0] = 0;
      meta[1] = 0;
    }
    volatile T* o = out;
    o[0] = ys;           // y.s of this update (0 on the first iteration)
    o[1] = v.a;          // g.d
    o[2] = v.c;          // max |d|
    o[3] = v.b;          // sum |g|
    o[4] = (T)count;      // pairs in the history
    o[5] = t_step;        // the step length of this iteration
    o[6] = apply ? T(1) : T(0);  // whether the step was applied to `param`
    __threadfence_system();
  }
}

// the instantiation with the fewest elements per thread that covers n; MAX_EPT bounds the register budget
template <typename T, int MAX_EPT>
cudaError_t launch_direction(const T* g, T* prev_g, T* d, T* S, T* Y, T* ro, T* hdiag, int32_t* meta, int64_t n,
                             int history, T t_prev, int first, T* param, T lr, T tol_change, T* out,
                             cudaStream_t stream) {
  if (n <= 0 || n > (int64_t)LB_STRIDE * MAX_EPT || history < 1 || history > LB_MAX_HISTORY)
    return cudaErrorInvalidValue;
  const int rows = history + 1;
  const int ept = (int)((n + LB_STRIDE - 1) / LB_STRIDE);
#define SQFA_LBFGS(E)                                                                                        \
  lbfgs_direction_kernel<T, E><<<LB_CTAS, LB_THREADS, 0, stream>>>(g, prev_g, d, S, Y, ro, hdiag, meta, (int)n, \
                                                                   rows, t_prev, first, param, lr, tol_change, out)
  if (ept <= 1) SQFA_LBFGS(1);
  else if (ept <= 2) SQFA_LBFGS(2);
  else if (ept <= 4) SQFA_LBFGS(4);
  else if (ept <= 8 || MAX_EPT == 8) SQFA_LBFGS(8);
  else if constexpr (MAX_EPT == 16) SQFA_LBFGS(16);
#undef SQFA_LBFGS
  return cudaGetLastError();
}

constexpr int LB_MAX_EPT_F32 = 16;
constexpr int LB_MAX_EPT_F64 = 8;  // double r[] takes twice the registers: 8 elements are 16 of the 64

}  // namespace

int lbfgs_max_n() { return LB_STRIDE * LB_MAX_EPT_F32; }
int lbfgs_max_n_f64() { return LB_STRIDE * LB_MAX_EPT_F64; }
int lbfgs_max_history() { return LB_MAX_HISTORY; }

cudaError_t launch_lbfgs_direction(const float* g, float* prev_g, float* d, float* S, float* Y, float* ro, float* hdiag,
                                   int32_t* meta, int64_t n, int history, float t_prev, int first, float* param,
                                   float lr, float tol_change, float* out, cudaStream_t stream) {
  return launch_direction<float, LB_MAX_EPT_F32>(g, prev_g, d, S, Y, ro, hdiag, meta, n, history, t_prev, first,
                                                 param, lr, tol_change, out, stream);
}

cudaError_t launch_lbfgs_direction_f64(const double* g, double* prev_g, double* d, double* S, double* Y, double* ro,
                                       double* hdiag, int32_t* meta, int64_t n, int history, double t_prev, int first,
                                       double* param, double lr, double tol_change, double* out, cudaStream_t stream) {
  return launch_direction<double, LB_MAX_EPT_F64>(g, prev_g, d, S, Y, ro, hdiag, meta, n, history, t_prev, first,
                                                  param, lr, tol_change, out, stream);
}

}  // namespace sqfa
