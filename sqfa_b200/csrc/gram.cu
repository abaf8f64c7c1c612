// K2: segmented per-class Gram accumulation  G_c = sum_{i in class c} (x_i - s_c)(x_i - s_c)^T
// on the sm_100a tensor cores (tcgen05.mma kind::tf32, fp32 accumulators in TMEM) as 3xTF32
// split precision:  x = hi + lo,  G ~= hi^T hi + hi^T lo + lo^T hi   (fp32-level accuracy).
//
// Replaces the per-class loop of the reference (gather `points[indices]`, centre, einsum
// "ij,ik->jk"):  /root/reference/src/sqfa/statistics.py:36-47 and :113-122.
// Only the 256 x 256 tiles that intersect the upper triangle are computed; K3 mirrors them.
//
// Two CTAs of a cluster (one SM each) share one tcgen05.mma.cta_group::2 with M = 256, N = 256:
// CTA r supplies the 128 operand columns m0 + 128 r .. of A and HALF of B (n0 + (N/2) r ..) from its
// own shared memory, the tensor cores of both SMs compute 128 x 256 accumulators each (TMEM of
// each SM). Relative to one CTA per 128 x 256 tile this cuts, per SM and per MMA cycle, the operand
// bytes read from shared memory and the transform work (gather + centre + hi/lo split + store) by
// 1/3 -- shared-memory bandwidth and instruction issue are what bound 3xTF32 (DESIGN.md).
//
// Warp roles per CTA (13 warps):
//   0-7   producers : a thread owns a block of 4 samples x 4 adjacent columns of a stage: four
//                     16-byte loads (512 B per warp and sample row, gathered through the bucket
//                     permutation) straight into registers; it centres, splits hi/lo and stores four
//                     K-major 16-byte chunks per half. The four columns of a thread go to operand
//                     SLOTS l, 32+l, 64+l, 96+l (slot s holds column 4 (s % 32) + s / 32 of the
//                     tile), which keeps every STS.128 conflict-free; the epilogue undoes the
//                     permutation. The loads run as a register pipeline in batches of GB stages
//                     with ONE wait per batch (ptxas tracks all of them on one scoreboard), the
//                     next batch's loads issued right behind that wait; registers for it come from
//                     setmaxnreg (producers 144, the other warps 96).
//   8     MMA       : leader CTA only; per K=8 step 3 tcgen05.mma.cta_group::2 (cross terms into
//                     their own TMEM accumulator, hi*hi into the main one), multicast commits
//   9-12  epilogue  : the tensor core truncates when it adds into its fp32 accumulator (bias
//                     ~ -2^-25 per MMA, measured), so the main accumulator only ever holds a CHAIN
//                     of <= chain_rows samples: at every chain end these warps add it (fp32,
//                     round-to-nearest, pipelined tcgen05.ld + LDS.128/STS.128) to a 128 x 256
//                     running sum in shared memory and hand the accumulator back; at the end of
//                     the tile they add the cross-term accumulator and store the tile
//                     (red.global.add only when a tile is split along K or the caller accumulates).
// Jobs (class, tile, K part) are listed by a device-side plan (largest classes first) and dealt
// round-robin to the CTA pairs: no atomics, no host sync, no cluster barrier per job.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cuda_runtime.h>
#include <type_traits>

#include "elem.cuh"
#include "ptx.cuh"
#include "sqfa_internal.h"

namespace sqfa {

namespace {

constexpr int TM2 = 256;  // tile rows    (UMMA M over the CTA pair)
constexpr int TN2 = 256;  // tile columns (UMMA N)
constexpr int BK = 16;    // samples per stage
constexpr int STAGES2 = 3;
constexpr int PROD_WARPS2 = 8;   // warp = (operand A/B, quad of 4 samples); a thread owns a 4 x 4 block
constexpr int PROD_REGS = 144, OTHER_REGS = 96;
constexpr int GB = 3;            // stages per producer register batch (two batches of registers)
constexpr int EPI_WARPS2 = 4;   // one per TMEM lane quarter
static_assert(PROD_WARPS2 * PROD_REGS + (1 + EPI_WARPS2) * OTHER_REGS <= (PROD_WARPS2 + 1 + EPI_WARPS2) * 128, "register pool");
constexpr int MMA_WARP2 = PROD_WARPS2;
constexpr int GRAM2_THREADS = (PROD_WARPS2 + 1 + EPI_WARPS2) * 32;
constexpr int OP_BYTES = 128 * BK * 4;                    // 8 KB: 128 columns x 16 samples
constexpr int STAGE2_BYTES = 4 * OP_BYTES;                // A_hi, A_lo, B_hi, B_lo = 32 KB
constexpr int RUN_BYTES = 128 * TN2 * 4;                  // 128 KB running sum [col][row]
constexpr int GRAM2_SMEM = STAGES2 * STAGE2_BYTES + RUN_BYTES + 1024;
// Operand layout in shared memory: K-major, no swizzle ("interleaved" core matrices), pinned on
// hardware by tools/umma_probe.py: element (column c, sample k) of a 128-column operand lives at
//   (k/4) * 2048 + (c/8) * 128 + (c%8) * 16 + (k%4) * 4   bytes,
// i.e. 8 x (4 samples) core matrices of 128 contiguous bytes; LBO = 2048 (next 4 samples),
// SBO = 128 (next 8 columns). One tcgen05.mma (K = 8 tf32) consumes two k-chunks.
constexpr uint32_t OP_LBO = 128 * 16, OP_SBO2 = 128;
constexpr uint32_t TMEM_COLS2 = 512, TMEM_SMALL2 = 256;

__device__ __align__(16) float g_zero[4] = {0.f, 0.f, 0.f, 0.f};  // read with 16-byte loads

struct GramParams {
  const void* X;     // float, __nv_bfloat16 or __half (the kernel's template argument)
  int64_t ldx;
  int64_t n;         // rows of X (= entries of perm)
  const int32_t* perm;
  const int64_t* offsets;
  const float* shift;
  float* gram;
  float* sums;       // optional class-sum partials [C][KS][4][D]: sum of (x - shift) over the samples of one
                     //   K part that one sample quad of a diagonal tile saw (see produce)
  int32_t* done;     // optional completion counters: done[c G / C] += 1 per (job, CTA, epilogue warp) once the
  int n_groups;      //   job's tile is stored -- a collective on another stream can be gated on a class group
  int class_order;   // jobs in class order (so class groups finish in order) instead of largest class first
  int first_class;   // class order starts here and wraps around (a rank's own classes can be made to run last)
  const int4* jobs;  // (class, tile row, tile col, K part)
  int njobs;
  int D, C, KS;
  int chain_kb;      // stages per accumulation chain
  int atomic_out;    // KS > 1 or accumulate: red.add into gram, else plain store
  int packed;        // gram = packed list of upper tiles [class][tile][256][256] instead of (C, D, D)
  int T, TT;         // tiles per class, tiles per side
  int vec_ok;
  int vecx;          // rows of X are aligned to 4 elements: LDG.128 (float32) / LDG.64 (bf16, fp16)
  int flags;         // tuning switches (env SQFA_GRAM_FLAGS): 1 = no A-as-B reuse on diagonal tiles,
                     // 2 = A / B producer warps share the A operand of diagonal tiles, 4 = scalar loads,
                     // 8 = no early cross-term MMAs during a chain drain (1 and 2 are off with `sums`)
};

__device__ __forceinline__ uint32_t ldg_nc_u16(const void* p) {  // zero-extended
  uint32_t v;
  asm volatile("ld.global.nc.u16 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}

// How a producer thread's 4 adjacent columns of one sample arrive in registers: ONE aligned unit per
// sample (16 bytes of float32 or 8 bytes of bf16 / fp16), or element loads where the rows are not
// aligned to 4 elements or the last column tile ends inside the four. The element type changes nothing
// else: widen() gives the float32 values the float32 path would have loaded.
template <typename T>
struct GramLoad {  // bf16 / fp16
  using raw = uint64_t;
  static __device__ __forceinline__ raw vec(const T* p) {
    uint64_t v;
    asm volatile("ld.global.nc.b64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
  }
  static __device__ __forceinline__ raw scalar(const T* p, int ncol) {
    uint32_t e0 = 0u, e1 = 0u, e2 = 0u, e3 = 0u;  // past D: zero bits, which widen to 0.f like the float32 zeros
    if (ncol > 0) e0 = ldg_nc_u16(p);
    if (ncol > 1) e1 = ldg_nc_u16(p + 1);
    if (ncol > 2) e2 = ldg_nc_u16(p + 2);
    if (ncol > 3) e3 = ldg_nc_u16(p + 3);
    uint64_t v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "r"(e0 | (e1 << 16)), "r"(e2 | (e3 << 16)));
    return v;
  }
  static __device__ __forceinline__ float4 widen(raw q) {
    uint2 w;  // volatile like unpack_b128: the split stays where it is written, after the batch's wait
    asm volatile("mov.b64 {%0, %1}, %2;" : "=r"(w.x), "=r"(w.y) : "l"(q));
    return widen4<T>(w);
  }
};
template <>
struct GramLoad<float> {
  using raw = b128_t;
  static __device__ __forceinline__ raw vec(const float* p) { return ldg_nc_b128(p); }
  static __device__ __forceinline__ raw scalar(const float* p, int ncol) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ncol > 0) v.x = ldg_nc_f32(p);
    if (ncol > 1) v.y = ldg_nc_f32(p + 1);
    if (ncol > 2) v.z = ldg_nc_f32(p + 2);
    if (ncol > 3) v.w = ldg_nc_f32(p + 3);
    return pack_b128(v);
  }
  static __device__ __forceinline__ float4 widen(raw q) { return unpack_b128(q); }
};

// Job list: classes in descending size; within a class the K parts, and within a K part its tiles:
// the CTA pairs that run concurrently work on the tiles of the SAME rows, which they share in L2.
// job = ((rank * KS) + ks) * T + t
__global__ void __launch_bounds__(256) gram_plan_kernel(const int64_t* __restrict__ offsets, int C, int TT, int KS,
                                                         int class_order, int first_class, int4* __restrict__ jobs) {
  // one warp per class: its rank among the classes by descending size (lanes stride over the other classes),
  // then its (K part, tile) jobs
  const int T = TT * (TT + 1) / 2;
  const int lane = threadIdx.x & 31;
  for (int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); c < C; c += gridDim.x * (blockDim.x >> 5)) {
    int rank = 0;
    if (class_order) {
      rank = (c - first_class + C) % C;
    } else {
      const int64_t n_c = offsets[c + 1] - offsets[c];
      for (int o = lane; o < C; o += 32) {
        const int64_t n_o = offsets[o + 1] - offsets[o];
        rank += (n_o > n_c || (n_o == n_c && o < c)) ? 1 : 0;
      }
      for (int sh = 16; sh > 0; sh >>= 1) rank += __shfl_xor_sync(0xffffffffu, rank, sh);
    }
    for (int e = lane; e < T * KS; e += 32) {
      const int t = e / KS, ks = e - t * KS;
      int tm = 0, rem = t;  // t -> (tm, tn), tm <= tn, row-major over the upper triangle
      while (rem >= TT - tm) { rem -= TT - tm; ++tm; }
      jobs[((int64_t)rank * KS + ks) * T + t] = make_int4(c, tm, tm + rem, ks);
    }
  }
}

struct JobGeom {
  int c, m0, n0, n_eff, nh;
  bool diag;  // full diagonal tile: each CTA's B half is the same data as its A operand
  int64_t row_begin, n_c;
  int ks, kb0, kb1;
};

template <int TM, int TN>
__device__ __forceinline__ JobGeom decode_job(const GramParams& P, int j) {
  const int4 jb = __ldg(P.jobs + j);
  JobGeom g;
  g.c = jb.x;
  g.m0 = jb.y * TM;
  g.n0 = jb.z * TN;
  g.n_eff = TN;  // full N: the slot permutation spreads a tile's columns over all 128 slots of a CTA
  g.nh = TN / 2;
  g.diag = (jb.y == jb.z) && !(P.flags & 1);
  g.row_begin = P.offsets[g.c];
  g.n_c = P.offsets[g.c + 1] - g.row_begin;
  const int nkb_total = (int)((g.n_c + BK - 1) / BK);
  g.ks = jb.w;
  g.kb0 = (int)(((int64_t)jb.w * nkb_total) / P.KS);
  g.kb1 = (int)(((int64_t)(jb.w + 1) * nkb_total) / P.KS);
  return g;
}

// PAIR = true : tcgen05.mma.cta_group::2, a 256 x 256 tile over a cluster of two CTAs (the general kernel)
// PAIR = false: tcgen05.mma.cta_group::1, ONE CTA computes a 128 x TN tile (TN = 128): the variant for
//               n_dim <= 128, where a class has a single (diagonal) tile and a 256 x 256 tile would execute
//               (256 / D)^2 times the useful MMA work. A launch without cluster dimensions is a cluster of
//               one CTA, so the cluster-window barrier addressing below is valid in both variants.
template <typename T, bool PAIR, int TN>
__device__ __forceinline__ void gram_body(const GramParams& P) {
  using Load = GramLoad<T>;
  using raw_t = typename Load::raw;
  constexpr int TM = PAIR ? 256 : 128;
  constexpr int NCTA = PAIR ? 2 : 1;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* run = reinterpret_cast<float*>(smem + STAGES2 * STAGE2_BYTES);  // [256 cols][128 rows]

  __shared__ __align__(8) uint64_t full_bar[STAGES2];   // leader: 16 producer-warp arrivals (both CTAs)
  __shared__ __align__(8) uint64_t empty_bar[STAGES2];  // per CTA: multicast tcgen05.commit
  __shared__ __align__(8) uint64_t acc_full_bar;        // per CTA: chain finished (multicast commit)
  __shared__ __align__(8) uint64_t acc_empty_bar;       // leader: 8 epilogue-warp arrivals (both CTAs)
  __shared__ uint32_t s_tmem_base;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;

  if (tid == 0) {
    for (int s = 0; s < STAGES2; ++s) {
      mbar_init(&full_bar[s], NCTA * PROD_WARPS2);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&acc_full_bar, 1);
    mbar_init(&acc_empty_bar, NCTA * EPI_WARPS2);
    mbar_fence_init();
  }
  if (warp == MMA_WARP2) {
    if constexpr (PAIR) tmem_alloc_2cta<TMEM_COLS2>(&s_tmem_base);
    else tmem_alloc<TMEM_COLS2>(&s_tmem_base);
  }
  tc_fence_before_sync();
  __syncthreads();
  cluster_sync_all();  // barriers of both CTAs initialised before anyone arrives remotely
  tc_fence_after_sync();
  const uint32_t tmem_base = s_tmem_base;

  const int D = P.D;
  const int pair = PAIR ? (blockIdx.x >> 1) : blockIdx.x, npairs = PAIR ? (gridDim.x >> 1) : gridDim.x;

  // Registers: 13 warps put 4 warps on one SM sub-partition, so the launch gets 128 per thread.
  // The MMA and epilogue warps (warpgroups 2, 3) give some back and the producers (warpgroups 0, 1)
  // take them for their load pipeline. The pool is per CTA: 8 x 144 + 5 x 96 <= 13 x 128 (a
  // request beyond the pool never completes), and per sub-partition 2 x 144 + 2 x 96 <= 512.
  if (warp < PROD_WARPS2) setmaxnreg_inc<PROD_REGS>(); else setmaxnreg_dec<OTHER_REGS>();

  if (warp < PROD_WARPS2) {
    // =========================== producers (both CTAs) ===========================
    uint32_t stage = 0, phase = 0;
    const bool isA = (warp & 1) == 0;
    const int quad = warp >> 1;  // samples 4 quad .. 4 quad + 3 of a stage = K-major chunk `quad`
    // chunk of slot 32 j + lane in k-chunk `quad`:  quad * 2048 + j * 512 + (lane / 8) * 128 + (lane % 8) * 16
    const uint32_t hi_A = smem_u32(smem) + quad * OP_LBO + (lane >> 3) * 128 + (lane & 7) * 16;  // A operand buffers
    const uint32_t hi_B = hi_A + 2 * OP_BYTES;                                                    // B operand buffers
    const uint32_t full0 = mapa_u32(smem_u32(&full_bar[0]), 0);  // the leader's barriers, cluster window
    const bool vecx = P.vecx != 0;
    for (int j = pair; j < P.njobs; j += npairs) {
      const JobGeom g = decode_job<TM, TN>(P, j);
      const int kb0 = g.kb0, kb1 = g.kb1;
      const int64_t n_c = g.n_c;
      // Diagonal tile: the MMA reads this CTA's A buffers as its B half, so there is no B operand to
      // produce and the B warps only keep the barrier protocol going. Experiment (SQFA_GRAM_FLAGS & 2):
      // the A and the B warp of a sample quad SHARE the A operand, the A warp producing the even stages
      // of the job and the B warp the odd ones -- twice the global loads in flight on diagonal tiles.
      // Measured: c5 shard 77.0 -> 73.0 ms, c4 2.20 -> 2.43 ms, c2 / c3 unchanged; off by default.
      const bool share = g.diag && (P.flags & 2);
      // Class sums: every column of a class lies in exactly one diagonal tile (tm == tn) per K part, where
      // the B warps have no operand to produce. There they load the A warp's samples and columns again (L2
      // hits) and add up x - s (fixed order) while keeping the barrier protocol going; each stores its
      // float4 at the end of the job, one slot per (class, K part, quad, column): no atomics, and an empty
      // K part stores zeros. The A producers and the off-diagonal jobs run exactly as without sums.
      const bool sum_job = P.sums != nullptr && g.diag && !isA;
      if (g.diag && !isA && !share && !sum_job) {
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(full0 + stage * 8);
          if (++stage == STAGES2) { stage = 0; phase ^= 1; }
        }
        continue;
      }
      const bool asA = isA || share || sum_job;
      const uint32_t hi_base = asA ? hi_A : hi_B;
      const uint32_t lo_base = hi_base + OP_BYTES;  // 32-bit shared addresses: no 64-bit math in the loop
      const int col = (asA ? g.m0 : g.n0) + 128 * (int)rank + 4 * lane;  // first of this thread's 4 columns
      const int ncol = col >= D ? 0 : (D - col >= 4 ? 4 : D - col);      // how many of them exist
      float4 sh = make_float4(0.f, 0.f, 0.f, 0.f);
      if (P.shift != nullptr && ncol > 0) {
        const float* sp = P.shift + (int64_t)g.c * D + col;
        sh.x = __ldg(sp);
        if (ncol > 1) sh.y = __ldg(sp + 1);
        if (ncol > 2) sh.z = __ldg(sp + 2);
        if (ncol > 3) sh.w = __ldg(sp + 3);
      }
      // a thread without columns (past D) reads a fixed zero vector with row stride 0
      const T* const xcol = ncol > 0 ? static_cast<const T*>(P.X) + col : reinterpret_cast<const T*>(g_zero);
      const uint32_t stride = ncol > 0 ? (uint32_t)P.ldx * (uint32_t)sizeof(T) : 0u;
      // warp-uniform choice of the load path: one vector load when rows are 4-element aligned and every
      // thread of the warp owns all four of its columns or none (straight-line code, no
      // per-load branches); scalar loads only in the last column tile of a D not divisible by 4
      const bool fastw = __all_sync(0xffffffffu, vecx && (ncol == 4 || ncol == 0));

      auto produce = [&](auto fast_tag, auto share_tag, auto sum_tag) {
        constexpr bool FAST = decltype(fast_tag)::value;
        constexpr bool SHARE = decltype(share_tag)::value;
        constexpr bool SUM = decltype(sum_tag)::value;  // sums only: nothing is stored to shared memory
        float4 psum = make_float4(0.f, 0.f, 0.f, 0.f);
        constexpr int S = SHARE ? 2 : 1;          // stride between the stages this warp produces
        const int off = (SHARE && !isA) ? 1 : 0;  // its first stage, relative to kb0
        // Register pipeline. ptxas tracks every global load of this loop on ONE scoreboard, so the
        // first use of any loaded value waits for ALL loads in flight (ncu: the per-slot prefetch
        // of the previous version waited for the refill issued one stage earlier). The loop is
        // therefore organised in batches of GB stages and two register sets: the loads of batch
        // j + 1 are issued right after the single wait of batch j and have the whole time batch j
        // is being written to shared memory (GB stage periods) to land. All loads are volatile
        // asm so they stay where they are written relative to the barrier waits and stores.
        raw_t bufA[GB][4], bufB[GB][4];
        // lane r < 4 holds the row id of sample (4 quad + r) of a stage; refilled one batch ahead,
        // unconditional and clamped (a predicated load needs a select that waits on it)
        auto load_row = [&](int kb) -> uint32_t {
          const int64_t k = (int64_t)kb * BK + 4 * quad + (lane & 3);
          const int64_t idx = g.row_begin + min(k, n_c - 1);  // an empty class may sit at either end
          return ldg_nc_u32(P.perm + max(min(idx, P.n - 1), (int64_t)0));
        };
        uint32_t rowreg[GB];
        int ring_kb = kb0;  // stage index the shared-memory ring position (stage, phase) stands for
        auto skip_stage = [&]() {  // a stage some other warp produces: keep the arrival counts going
          mbar_wait(&empty_bar[stage], phase ^ 1);
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(full0 + stage * 8);
          if (++stage == STAGES2) { stage = 0; phase ^= 1; }
          ++ring_kb;
        };
        auto issue = [&](int kb, raw_t(&b)[GB][4]) {  // loads of stages kb, kb + S, .. kb + (GB - 1) S
#pragma unroll
          for (int u = 0; u < GB; ++u) {
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              const uint32_t row = __shfl_sync(0xffffffffu, rowreg[u], r);
              uint64_t addr;  // xcol + row * ldx elements
              asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(addr) : "r"(row), "r"(stride), "l"(xcol));
              const T* ptr = reinterpret_cast<const T*>(addr);
              if constexpr (FAST) {
                b[u][r] = Load::vec(ptr);
              } else {
                b[u][r] = Load::scalar(ptr, ncol);
              }
            }
          }
#pragma unroll
          for (int u = 0; u < GB; ++u) rowreg[u] = load_row(kb + S * (GB + u));  // ids of the NEXT batch
        };
        auto put = [&](uint32_t hp, uint32_t lp, float x0, float x1, float x2, float x3) {
          float4 h, l;
          h.x = to_tf32(x0); l.x = x0 - h.x;
          h.y = to_tf32(x1); l.y = x1 - h.y;
          h.z = to_tf32(x2); l.z = x2 - h.z;
          h.w = to_tf32(x3); l.w = x3 - h.w;
          st_shared_v4(hp, h);
          st_shared_v4(lp, l);
        };
        auto consume = [&](int kb, const raw_t(&bq)[4]) {
          if constexpr (SHARE) {
            while (ring_kb < kb) skip_stage();
            ++ring_kb;
          }
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if constexpr (SUM) {  // the stage's arrival does not wait for this warp's loads
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(full0 + stage * 8);
            if (++stage == STAGES2) { stage = 0; phase ^= 1; }
          }
          float4 b[4];
#pragma unroll
          for (int r = 0; r < 4; ++r) b[r] = Load::widen(bq[r]);
          const int64_t nv = n_c - (int64_t)kb * BK - 4 * quad;  // valid samples among this thread's four
          if (nv < 4) {  // ragged last stage of the class: padded samples must be exact zeros
            const float4 z = make_float4(sh.x, sh.y, sh.z, sh.w);
#pragma unroll
            for (int r = 0; r < 4; ++r)
              if (r >= (int)nv) b[r] = z;
          }
          if constexpr (SUM) {  // padded samples are exactly zero after centring
            psum.x += ((b[0].x - sh.x) + (b[1].x - sh.x)) + ((b[2].x - sh.x) + (b[3].x - sh.x));
            psum.y += ((b[0].y - sh.y) + (b[1].y - sh.y)) + ((b[2].y - sh.y) + (b[3].y - sh.y));
            psum.z += ((b[0].z - sh.z) + (b[1].z - sh.z)) + ((b[2].z - sh.z) + (b[3].z - sh.z));
            psum.w += ((b[0].w - sh.w) + (b[1].w - sh.w)) + ((b[2].w - sh.w) + (b[3].w - sh.w));
            return;
          }
          const uint32_t hp = hi_base + stage * STAGE2_BYTES;
          const uint32_t lp = lo_base + stage * STAGE2_BYTES;
          // column j of the thread -> slot 32 j + lane -> + j * 512 bytes; the 4 samples are one chunk
          put(hp, lp, b[0].x - sh.x, b[1].x - sh.x, b[2].x - sh.x, b[3].x - sh.x);
          put(hp + 512, lp + 512, b[0].y - sh.y, b[1].y - sh.y, b[2].y - sh.y, b[3].y - sh.y);
          put(hp + 1024, lp + 1024, b[0].z - sh.z, b[1].z - sh.z, b[2].z - sh.z, b[3].z - sh.z);
          put(hp + 1536, lp + 1536, b[0].w - sh.w, b[1].w - sh.w, b[2].w - sh.w, b[3].w - sh.w);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive_cluster(full0 + stage * 8);
          if (++stage == STAGES2) { stage = 0; phase ^= 1; }
        };
        // one batch: the first stage's write (which contains the one wait for the batch's loads),
        // then the loads of the next batch into the other register set, then the remaining stages
        auto batch = [&](int kb, raw_t(&cur)[GB][4], raw_t(&nxt)[GB][4]) {
          if (kb < kb1) consume(kb, cur[0]);
          issue(kb + S * GB, nxt);  // unconditional: stages past the end re-read valid rows, never consumed
#pragma unroll
          for (int u = 1; u < GB; ++u)
            if (kb + S * u < kb1) consume(kb + S * u, cur[u]);
        };
#pragma unroll
        for (int u = 0; u < GB; ++u) rowreg[u] = load_row(kb0 + off + S * u);
        issue(kb0 + off, bufA);
        for (int kb = kb0 + off; kb < kb1; kb += 2 * GB * S) {
          batch(kb, bufA, bufB);
          batch(kb + GB * S, bufB, bufA);
        }
        if constexpr (SHARE) {
          while (ring_kb < kb1) skip_stage();  // trailing stages of the other warp
        }
        if constexpr (SUM) {
          float* const out = P.sums + (((int64_t)g.c * P.KS + g.ks) * 4 + quad) * D + col;
          if (ncol > 0) out[0] = psum.x;
          if (ncol > 1) out[1] = psum.y;
          if (ncol > 2) out[2] = psum.z;
          if (ncol > 3) out[3] = psum.w;
        }
      };
      using T_ = std::true_type;
      using F_ = std::false_type;
      if (share) {
        if (fastw) produce(T_{}, T_{}, F_{}); else produce(F_{}, T_{}, F_{});
      } else if (sum_job) {
        if (fastw) produce(T_{}, F_{}, T_{}); else produce(F_{}, F_{}, T_{});
      } else {
        if (fastw) produce(T_{}, F_{}, F_{}); else produce(F_{}, F_{}, F_{});
      }
    }
  } else if (warp == MMA_WARP2) {
    // =========================== MMA issuer (leader CTA only) ===========================
    if (leader) {
      uint32_t stage = 0, phase = 0, chain_phase = 0;
      for (int j = pair; j < P.njobs; j += npairs) {
        const JobGeom g = decode_job<TM, TN>(P, j);
        const uint32_t idesc = make_idesc_tf32(TM, (uint32_t)g.n_eff, 0, 0);
        auto mma = [&](uint32_t d, uint64_t da, uint64_t db, uint32_t acc) {
          if constexpr (PAIR) umma_tf32_ss_2cta(d, da, db, idesc, acc);
          else umma_tf32_ss(d, da, db, idesc, acc);
        };
        auto commit = [&](uint64_t* bar) {
          if constexpr (PAIR) umma_commit_2cta(bar, 3);
          else umma_commit(bar);
        };
        // cross terms (small accumulator) / hi*hi (main accumulator) of one stage
        auto issue_stage = [&](uint32_t stg, bool cross, bool mainp, int kb, int cb) {
          const uint32_t st = smem_u32(smem + stg * STAGE2_BYTES);
          const uint32_t a_hi = st, a_lo = st + OP_BYTES;
          const uint32_t b_hi = g.diag ? a_hi : st + 2 * OP_BYTES, b_lo = g.diag ? a_lo : st + 3 * OP_BYTES;
#pragma unroll
          for (int k8 = 0; k8 < BK / 8; ++k8) {
            const uint32_t ko = k8 * 2 * OP_LBO;
            const uint64_t dA_hi = make_smem_desc(a_hi + ko, OP_LBO, OP_SBO2, 0);
            const uint64_t dA_lo = make_smem_desc(a_lo + ko, OP_LBO, OP_SBO2, 0);
            const uint64_t dB_hi = make_smem_desc(b_hi + ko, OP_LBO, OP_SBO2, 0);
            const uint64_t dB_lo = make_smem_desc(b_lo + ko, OP_LBO, OP_SBO2, 0);
            if (cross) {
              const uint32_t acc_small = (kb > g.kb0 || k8 > 0) ? 1u : 0u;  // zeroed once per job
              mma(tmem_base + TMEM_SMALL2, dA_lo, dB_hi, acc_small);
              mma(tmem_base + TMEM_SMALL2, dA_hi, dB_lo, 1u);
            }
            if (mainp) {
              const uint32_t acc_main = (kb > cb || k8 > 0) ? 1u : 0u;  // zeroed at every chain start
              mma(tmem_base, dA_hi, dB_hi, acc_main);
            }
          }
        };
        for (int cb = g.kb0; cb < g.kb1; cb += P.chain_kb) {
          const int ce = min(g.kb1, cb + P.chain_kb);
          // While the epilogue warps drain the previous chain's main accumulator, the cross terms
          // of the first stages of this chain (they go to the OTHER accumulator, which is only read
          // at the end of the job) keep the tensor pipe busy.
          const int early = (cb > g.kb0 && !(P.flags & 8)) ? min(STAGES2, ce - cb) : 0;
          {
            uint32_t st = stage, ph = phase;
            for (int e = 0; e < early; ++e) {
              mbar_wait_cluster(&full_bar[st], ph);
              tc_fence_after_sync();
              if (elect_one()) issue_stage(st, true, false, cb + e, cb);
              __syncwarp();
              if (++st == STAGES2) { st = 0; ph ^= 1; }
            }
          }
          // the epilogue warps of both CTAs must have drained the previous chain
          mbar_wait_cluster(&acc_empty_bar, chain_phase ^ 1);
          chain_phase ^= 1;
          tc_fence_after_sync();
          for (int kb = cb; kb < ce; ++kb) {
            const bool crossed = kb - cb < early;
            if (!crossed) {
              mbar_wait_cluster(&full_bar[stage], phase);
              tc_fence_after_sync();
            }
            if (elect_one()) {
              issue_stage(stage, !crossed, true, kb, cb);
              commit(&empty_bar[stage]);
              if (kb == ce - 1) commit(&acc_full_bar);
            }
            __syncwarp();
            if (++stage == STAGES2) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else {
    // =========================== epilogue warps (both CTAs) ===========================
    const int q = warp & 3;  // TMEM lane quarter this warp may access
    const int lrow = 32 * q + lane;
    const uint32_t tq = tmem_base + ((uint32_t)(32 * q) << 16);
    const uint32_t acc_empty0 = mapa_u32(smem_u32(&acc_empty_bar), 0);
    uint32_t acc_phase = 0;
    // job finished as far as this warp is concerned: its stores are visible device-wide before the
    // group's counter moves (a collective on another stream waits for the counter with a stream
    // memory operation and then reads the tiles)
    auto signal_done = [&](int c) {
      if (P.done != nullptr) {
        __threadfence();
        __syncwarp();
        if (lane == 0) atomicAdd(P.done + (int)(((int64_t)c * P.n_groups) / P.C), 1);
      }
    };
    for (int j = pair; j < P.njobs; j += npairs) {
      const JobGeom g = decode_job<TM, TN>(P, j);
      // TMEM lane i = 32 q + lane is operand slot i of this CTA -> tile row 4 (i % 32) + i / 32
      const int row = g.m0 + 128 * (int)rank + 4 * lane + q;
      // output row pointer, indexed by the GLOBAL column: full (C, D, D) layout, or the packed
      // tile list (what a multi-device caller all-reduces: upper tiles only)
      float* grow;
      if (P.packed) {
        const int tm = g.m0 / TM, tn = g.n0 / TN;
        const int64_t t = (int64_t)tm * P.TT - (int64_t)tm * (tm - 1) / 2 + (tn - tm);
        grow = P.gram + (((int64_t)g.c * P.T + t) * TM + (row - g.m0)) * TN - g.n0;
      } else {
        grow = P.gram + ((int64_t)g.c * D + row) * D;
      }
      if (g.kb1 <= g.kb0) {  // empty class / empty K part: the tile contribution is exactly zero
        if (!P.atomic_out && row < D)
          for (int cc = 0; cc < TN; ++cc)
            if (g.n0 + cc < D) grow[g.n0 + cc] = 0.f;
        signal_done(g.c);
        continue;
      }
      bool first = true;
      for (int cb = g.kb0; cb < g.kb1; cb += P.chain_kb) {
        const bool last = cb + P.chain_kb >= g.kb1;
        mbar_wait(&acc_full_bar, acc_phase);
        acc_phase ^= 1;
        tc_fence_after_sync();
        // running sum layout: float4 (columns 4 t .. 4 t + 3 of TMEM lane r) at run4[t * 128 + r]:
        // every warp access is 512 contiguous bytes (LDS.128 / STS.128, conflict-free)
        float4* const run4 = reinterpret_cast<float4*>(run) + lrow;
        if (!last) {
          // Drain the chain's main accumulator in 32-column chunks, the TMEM load of chunk c + 1 in
          // flight while chunk c is added to the running sum; the accumulator goes back to the MMA
          // warp as soon as the last load has landed.
          uint32_t va[32], vb[32];
          tmem_ld_32x32b_x32(tq, va);
          auto add_chunk = [&](int c, const uint32_t(&v)[32]) {
#pragma unroll
            for (int t = 0; t < 8; ++t) {
              float4* rp = run4 + (8 * c + t) * 128;
              float4 a = make_float4(__uint_as_float(v[4 * t]), __uint_as_float(v[4 * t + 1]),
                                     __uint_as_float(v[4 * t + 2]), __uint_as_float(v[4 * t + 3]));
              if (!first) {
                const float4 o = *rp;
                a.x += o.x; a.y += o.y; a.z += o.z; a.w += o.w;
              }
              *rp = a;
            }
          };
#pragma unroll
          for (int c = 0; c < TN / 32; c += 2) {
            tmem_ld_wait();
            tmem_ld_32x32b_x32(tq + (uint32_t)(32 * (c + 1)), vb);
            add_chunk(c, va);
            tmem_ld_wait();
            if (c + 2 < TN / 32) {
              tmem_ld_32x32b_x32(tq + (uint32_t)(32 * (c + 2)), va);
            } else {  // main accumulator fully read: hand it back to the MMA warp
              tc_fence_before_sync();
              __syncwarp();
              if (lane == 0) mbar_arrive_cluster(acc_empty0);
            }
            add_chunk(c + 1, vb);
          }
        } else if (P.vec_ok) {
          // Last chain of the tile: main + running sum + cross terms -> output, 16 bytes at a time.
          // Tile columns 4 s .. 4 s + 3 are accumulator columns s, 32 + s, 64 + s, 96 + s of a
          // 128-column half (the slot permutation), so one chunk reads 4 slots from each quarter.
#pragma unroll 1
          for (int ch = 0; ch < TN / 16; ++ch) {  // 4 slots from each quarter per chunk (register budget of this role)
            const int half = ch >> 3, s0 = 4 * (ch & 7);
            uint32_t m[4][4], w[4][4];
#pragma unroll
            for (int qd = 0; qd < 4; ++qd) {
              const uint32_t col = (uint32_t)(128 * half + 32 * qd + s0);
              tmem_ld_32x32b_x4(tq + col, m[qd]);
              tmem_ld_32x32b_x4(tq + TMEM_SMALL2 + col, w[qd]);
            }
            tmem_ld_wait();
            if (ch == TN / 16 - 1) {  // both accumulators read: the next job may start
              tc_fence_before_sync();
              __syncwarp();
              if (lane == 0) mbar_arrive_cluster(acc_empty0);
            }
#pragma unroll
            for (int qd = 0; qd < 4; ++qd) {
              float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
              if (!first) o = run4[((128 * half + 32 * qd + s0) / 4) * 128];
              m[qd][0] = __float_as_uint(__uint_as_float(m[qd][0]) + o.x + __uint_as_float(w[qd][0]));
              m[qd][1] = __float_as_uint(__uint_as_float(m[qd][1]) + o.y + __uint_as_float(w[qd][1]));
              m[qd][2] = __float_as_uint(__uint_as_float(m[qd][2]) + o.z + __uint_as_float(w[qd][2]));
              m[qd][3] = __float_as_uint(__uint_as_float(m[qd][3]) + o.w + __uint_as_float(w[qd][3]));
            }
            if (row < D) {
#pragma unroll
              for (int jj = 0; jj < 4; ++jj) {
                const int cidx = g.n0 + 128 * half + 4 * (s0 + jj);
                if (cidx < D) {  // D % 4 == 0: the four columns are all inside
                  const float4 v = make_float4(__uint_as_float(m[0][jj]), __uint_as_float(m[1][jj]),
                                               __uint_as_float(m[2][jj]), __uint_as_float(m[3][jj]));
                  if (P.atomic_out) red_add_v4(grow + cidx, v);
                  else *reinterpret_cast<float4*>(grow + cidx) = v;
                }
              }
            }
          }
        } else {
#pragma unroll 1
          for (int col0 = 0; col0 < TN; col0 += 16) {
            uint32_t v[16], w[16];
            tmem_ld_32x32b_x16(tq + (uint32_t)col0, v);
            tmem_ld_32x32b_x16(tq + TMEM_SMALL2 + (uint32_t)col0, w);
            tmem_ld_wait();
            if (col0 + 16 >= TN) {  // both accumulators read: the next job may start
              tc_fence_before_sync();
              __syncwarp();
              if (lane == 0) mbar_arrive_cluster(acc_empty0);
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
              if (!first) o = run4[(col0 / 4 + t) * 128];
              v[4 * t] = __float_as_uint(__uint_as_float(v[4 * t]) + o.x + __uint_as_float(w[4 * t]));
              v[4 * t + 1] = __float_as_uint(__uint_as_float(v[4 * t + 1]) + o.y + __uint_as_float(w[4 * t + 1]));
              v[4 * t + 2] = __float_as_uint(__uint_as_float(v[4 * t + 2]) + o.z + __uint_as_float(w[4 * t + 2]));
              v[4 * t + 3] = __float_as_uint(__uint_as_float(v[4 * t + 3]) + o.w + __uint_as_float(w[4 * t + 3]));
            }
            if (row < D) {
              // accumulator column n = 128 (n / 128) + slot  ->  tile column 128 (n / 128) + 4 (slot % 32) + slot / 32:
              // the 16 columns of this chunk are 16 bytes apart in the output row
              const int gc = g.n0 + (col0 & 128) + 4 * (col0 & 31) + ((col0 & 127) >> 5);
#pragma unroll
              for (int jj = 0; jj < 16; ++jj) {
                const int cidx = gc + 4 * jj;
                if (cidx < D) {
                  if (P.atomic_out) atomicAdd(grow + cidx, __uint_as_float(v[jj]));
                  else grow[cidx] = __uint_as_float(v[jj]);
                }
              }
            }
          }
        }
        first = false;
      }
      signal_done(g.c);
    }
  }

  tc_fence_before_sync();
  cluster_sync_all();
  if (warp == MMA_WARP2) {
    if constexpr (PAIR) tmem_dealloc_2cta<TMEM_COLS2>(tmem_base);
    else tmem_dealloc<TMEM_COLS2>(tmem_base);
  }
}

template <typename T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GRAM2_THREADS, 1)
gram_tf32x3_kernel(const GramParams P) { gram_body<T, true, TN2>(P); }

constexpr int TN1 = 128;  // tile edge of the single-CTA variant
constexpr int GRAM1_SMEM = STAGES2 * STAGE2_BYTES + 128 * TN1 * 4 + 1024;
template <typename T>
__global__ void __launch_bounds__(GRAM2_THREADS, 1)
gram_tf32x3_small_kernel(const GramParams P) { gram_body<T, false, TN1>(P); }

}  // namespace

size_t gram_packed_floats(int D, int C) {
  return (size_t)(C > 0 ? C : 0) * gram_tiles_per_class(D, nullptr) * TM2 * TN2;
}

int gram_tiles_per_class(int D, int* TT_out) {
  const int TT = (D + TM2 - 1) / TM2;
  if (TT_out) *TT_out = TT;
  return TT * (TT + 1) / 2;
}

// n_dim <= 128: the single-CTA variant (one 128 x 128 tile per class) unless the packed layout is asked for
static bool gram_use_small(int D, int packed) { return D <= TN1 && !packed; }

// Accumulator area (rows x columns) the tensor cores execute per sample for one class: every tile that
// intersects the upper triangle is a full MMA tile, whatever part of it lies beyond D.
int64_t gram_executed_tile_area(int D) {
  if (gram_use_small(D, 0)) return (int64_t)128 * TN1;
  return (int64_t)gram_tiles_per_class(D, nullptr) * TM2 * TN2;
}

// K parts per class for the single-CTA variant: ONE round of jobs (a job's fixed cost -- cold load
// pipeline, accumulator drain, 64 KB of red.add -- is as long as 500 samples of MMA work; measured on c3:
// 380 jobs of 526 samples ran at 24 % tensor-pipe activity), at least 256 samples per part
int gram_ksplit_small(int64_t n, int C, int num_sms) {
  if (C <= 0) return 1;
  int64_t ks = num_sms / C;
  const int64_t avg = n / C;
  const int64_t cap = avg / 256 > 1 ? avg / 256 : 1;
  if (ks > cap) ks = cap;
  if (ks > 64) ks = 64;
  return (int)(ks < 1 ? 1 : ks);
}

// K parts per tile so that small problems still fill the CTA pairs. elem_size: bytes per element of X
// (the L2-residency rule below counts the bytes of a class's rows, so bf16 / fp16 rows split half as often)
int gram_ksplit(int64_t n, int C, int D, int num_sms, int elem_size) {
  const int T = gram_tiles_per_class(D, nullptr);
  const int64_t tiles = (int64_t)C * T;
  const int pairs = num_sms / 2 > 0 ? num_sms / 2 : 1;
  if (tiles <= 0) return 1;
  if (tiles >= 6 * (int64_t)pairs) {
    // Enough tiles to fill the GPU. A tile reads the rows of its class once per column slab, and the
    // tiles of a class re-read them: free while the concurrently running (class, K part) groups fit in
    // the 126 MB L2, HBM-bound otherwise (measured on the c5 shard, 125 000 rows x 4 KB per class:
    // 5x the algorithmic traffic, 3.3 TB/s). Large classes are therefore cut into K parts whose rows
    // -- times the number of groups in flight -- stay L2-resident; parts are summed with red.add.
    const int64_t avg = C > 0 ? n / C : n;
    const double groups_in_flight = (double)pairs / T > 1.0 ? (double)pairs / T : 1.0;
    const double part_bytes = 96e6 / groups_in_flight;
    const double class_bytes = (double)avg * D * (double)elem_size;
    if (class_bytes <= part_bytes) return 1;
    int64_t ks = (int64_t)(class_bytes / part_bytes + 0.999);
    const int64_t cap = avg / 2048 > 1 ? avg / 2048 : 1;  // keep >= 2048 samples per part (epilogue amortised)
    if (ks > cap) ks = cap;
    if (ks > 64) ks = 64;
    return (int)(ks < 1 ? 1 : ks);
  }
  int64_t ks = (4 * (int64_t)pairs + tiles - 1) / tiles;
  const int64_t avg = C > 0 ? n / C : n;
  const int64_t cap = avg / 512 > 1 ? avg / 512 : 1;  // keep >= 512 samples per part
  if (ks > cap) ks = cap;
  if (ks > 64) ks = 64;
  return (int)(ks < 1 ? 1 : ks);
}

// K parts per class of a launch (either variant): the class-sum partials come in 4 per K part
int gram_ksplit_launch(int64_t n, int C, int D, int packed, int num_sms, int elem_size) {
  return gram_use_small(D, packed) ? gram_ksplit_small(n, C, num_sms) : gram_ksplit(n, C, D, num_sms, elem_size);
}

size_t gram_workspace_bytes(int C, int D, int ksplit_max) {
  // the job plan of either variant (the single-CTA variant splits K up to 64 ways)
  const size_t pair = (size_t)C * gram_tiles_per_class(D, nullptr) * (ksplit_max > 0 ? ksplit_max : 1);
  const size_t small = D <= TN1 ? (size_t)C * 64 : 0;
  return (pair > small ? pair : small) * sizeof(int4) + 256;
}

template <typename T>
static cudaError_t launch_class_gram_t(const T* X, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                                       const float* shift, int64_t n, int D, int C, float* gram, int accumulate,
                                       int packed, int chain_rows, int32_t* done, int n_groups, int first_class,
                                       int reserve_sms, void* ws, int num_sms, cudaStream_t stream, float* sums) {
  const bool small = gram_use_small(D, packed);
  static int smem_set[kMaxDevices] = {0}, smem_set1[kMaxDevices] = {0};  // per element type
  {
    cudaError_t e = small ? ensure_dynamic_smem(gram_tf32x3_small_kernel<T>, GRAM1_SMEM, smem_set1)
                          : ensure_dynamic_smem(gram_tf32x3_kernel<T>, GRAM2_SMEM, smem_set);
    if (e != cudaSuccess) return e;
  }
  if (C <= 0) return cudaSuccess;
  GramParams P;
  int TT = 0;
  int T_ = gram_tiles_per_class(D, &TT);
  if (small) { TT = 1; T_ = 1; }
  P.X = X; P.ldx = ldx; P.n = n; P.perm = perm; P.offsets = offsets; P.shift = shift; P.gram = gram; P.sums = sums;
  P.done = done; P.n_groups = n_groups > 0 ? n_groups : 1; P.class_order = done != nullptr ? 1 : 0;
  P.first_class = (P.class_order && first_class > 0 && first_class < C) ? first_class : 0;
  P.jobs = reinterpret_cast<const int4*>(ws);
  P.D = D; P.C = C;
  P.KS = gram_ksplit_launch(n, C, D, packed, num_sms, (int)sizeof(T));
  P.njobs = C * T_ * P.KS;
  const int cr = chain_rows > 0 ? chain_rows : 512;
  P.chain_kb = (cr + BK - 1) / BK;
  P.atomic_out = (accumulate || P.KS > 1) ? 1 : 0;
  P.packed = packed ? 1 : 0; P.T = T_; P.TT = TT;
  P.vec_ok = (D % 4 == 0) && ((reinterpret_cast<uintptr_t>(gram) & 15) == 0);
  static const int env_flags = [] { const char* e = getenv("SQFA_GRAM_FLAGS"); return e ? atoi(e) : 0; }();
  P.flags = sums != nullptr ? env_flags & ~3 : env_flags;  // class sums need the B warps of diagonal tiles idle
  P.vecx = ((ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & (4 * sizeof(T) - 1)) == 0) && !(env_flags & 4)) ? 1 : 0;
  if ((uint64_t)ldx * sizeof(T) >= (1ull << 32)) return cudaErrorInvalidValue;
  if (P.atomic_out && !accumulate) {  // K parts are summed with red.add -> start from zero
    const size_t floats = packed ? (size_t)C * T_ * TM2 * TN2 : (size_t)C * D * D;
    cudaError_t e = cudaMemsetAsync(gram, 0, floats * sizeof(float), stream);
    if (e != cudaSuccess) return e;
  }
  gram_plan_kernel<<<(C + 7) / 8, 256, 0, stream>>>(offsets, C, TT, P.KS, P.class_order, P.first_class,
                                                        reinterpret_cast<int4*>(ws));
  // reserve_sms SMs are left to other streams (the collective that runs while this kernel still computes)
  const int usable = num_sms - (reserve_sms > 0 ? reserve_sms : 0);
  if (small) {
    int grid = usable > 1 ? usable : 1;
    if (grid > P.njobs) grid = P.njobs;
    gram_tf32x3_small_kernel<T><<<grid, GRAM2_THREADS, GRAM1_SMEM, stream>>>(P);
    return cudaGetLastError();
  }
  int grid = ((usable > 2 ? usable : 2) / 2) * 2;
  if (grid > 2 * P.njobs) grid = 2 * P.njobs;
  gram_tf32x3_kernel<T><<<grid, GRAM2_THREADS, GRAM2_SMEM, stream>>>(P);
  return cudaGetLastError();
}

cudaError_t launch_class_gram(const void* X, int elem, int64_t ldx, const int32_t* perm, const int64_t* offsets,
                              const float* shift, int64_t n, int D, int C, float* gram, int accumulate, int packed,
                              int chain_rows, int32_t* done, int n_groups, int first_class, int reserve_sms, void* ws,
                              int num_sms, cudaStream_t stream, float* sums) {
  if (elem == ELEM_BF16)
    return launch_class_gram_t(static_cast<const __nv_bfloat16*>(X), ldx, perm, offsets, shift, n, D, C, gram,
                               accumulate, packed, chain_rows, done, n_groups, first_class, reserve_sms, ws, num_sms,
                               stream, sums);
  if (elem == ELEM_F16)
    return launch_class_gram_t(static_cast<const __half*>(X), ldx, perm, offsets, shift, n, D, C, gram, accumulate,
                               packed, chain_rows, done, n_groups, first_class, reserve_sms, ws, num_sms, stream, sums);
  return launch_class_gram_t(static_cast<const float*>(X), ldx, perm, offsets, shift, n, D, C, gram, accumulate,
                             packed, chain_rows, done, n_groups, first_class, reserve_sms, ws, num_sms, stream, sums);
}

}  // namespace sqfa
