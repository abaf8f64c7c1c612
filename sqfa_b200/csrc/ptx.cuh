// Thin inline-PTX wrappers for the sm_100a features the SQFA kernels use:
// mbarrier, tcgen05 (alloc / mma / commit / ld / fences), proxy fences.
// Everything here is hand-written PTX; no CUTLASS/CuTe dependency.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace sqfa {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_fence_init() {
  // make barrier inits visible to the async proxy / other threads
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .b64 st;\n\t"
      "mbarrier.arrive.shared::cta.b64 st, [%0];\n\t}"
      ::"r"(smem_u32(bar))
      : "memory");
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  // (an explicit suspend-time hint was measured to make the pipeline 18% slower: wake-ups lag)
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

// Bounded wait: a broken pipeline traps (-> CUDA error) instead of hanging the GPU box.
// (Measured alternatives on the Gram pipeline: a suspend-time hint, a bare spin and a
// __nanosleep back-off were all ~18% slower than this clock-paced loop.)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {  // ~2 s at 2 GHz
      printf("sqfa: mbarrier wait timeout (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}

// ----------------------------------------------------------------------------------------------
// bulk asynchronous copies (the copy unit behind TMA, non-tensor form): global -> shared, completion
// reported to an mbarrier as transferred bytes
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile(
      "{\n\t.reg .b64 st;\n\t"
      "mbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}"
      ::"r"(smem_u32(bar)), "r"(bytes)
      : "memory");
}
// 16-byte aligned source, destination and size
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ float4 ld_shared_v4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

// ----------------------------------------------------------------------------------------------
// proxy / tcgen05 fences
// ----------------------------------------------------------------------------------------------
// generic-proxy smem writes -> visible to the async proxy (tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// TMEM allocation (one full warp executes these)
// ----------------------------------------------------------------------------------------------
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst) {
  static_assert(kCols >= 32 && kCols <= 512 && (kCols & (kCols - 1)) == 0, "TMEM columns: pow2 in [32,512]");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05.mma kind::tf32, operands from shared memory descriptors, accumulator in TMEM.
// Issued by ONE thread.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void umma_tf32_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// A operand from TMEM (lane = m, column = k), B from shared memory.
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

// All previously issued tcgen05.mma of this thread arrive (count 1) on `bar` when complete.
// Implies tcgen05.fence::before_thread_sync.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ----------------------------------------------------------------------------------------------
// UMMA descriptors
// ----------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor (sm_100 format, version 1).
//   layout_type: 0 none/interleave, 2 = 128B swizzle, 4 = 64B, 6 = 32B
__host__ __device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes,
                                                            uint32_t sbo_bytes, uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)(layout_type & 7u) << 61;
  return d;
}

// Instruction descriptor for kind::tf32, fp32 accumulate.
__host__ __device__ __forceinline__ uint32_t make_idesc_tf32(uint32_t m, uint32_t n, uint32_t a_mn_major,
                                                             uint32_t b_mn_major) {
  uint32_t d = 0;
  d |= 1u << 4;                    // D format: F32
  d |= 2u << 7;                    // A format: TF32
  d |= 2u << 10;                   // B format: TF32
  d |= (a_mn_major & 1u) << 15;    // A major-ness (1 = MN-major)
  d |= (b_mn_major & 1u) << 16;    // B major-ness
  d |= ((n >> 3) & 0x3Fu) << 17;   // N / 8
  d |= ((m >> 4) & 0x1Fu) << 24;   // M / 16
  return d;
}

// ----------------------------------------------------------------------------------------------
// TMEM -> registers. Each warp may touch only lanes [32*(warp%4), +32). 32 consecutive columns.
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x4(uint32_t taddr, uint32_t (&r)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// registers -> TMEM, 8 consecutive columns of this thread's lane
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
               "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// fp32 -> tf32 (round to nearest, ties away from zero): the low 13 mantissa bits are cleared after
// adding half an ulp to the magnitude. Two integer instructions; `cvt.rna.tf32.f32` is emulated
// by ptxas with ~7 (measured: it was a third of the Gram producers' instructions).
__device__ __forceinline__ float to_tf32(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}

// 16-byte global reductions: into local memory, or through an NVSwitch multicast address into the
// same offset of every device of the multicast group (each copy receives the add).
__device__ __forceinline__ void red_add_v4(float* p, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() {
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N));
}
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N));
}
// Read-only global loads as volatile asm: they keep their place relative to other volatile asm
// (barrier waits, shared stores), which a register software pipeline relies on.
// 16-byte load into ONE 128-bit register: the four words stay an aligned unit until unpack_b128,
// so the register allocator can never put a (load-waiting) MOV behind the load itself.
typedef unsigned __int128 b128_t;
__device__ __forceinline__ b128_t ldg_nc_b128(const float* p) {
  b128_t v;
  asm volatile("ld.global.nc.b128 %0, [%1];" : "=q"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ float4 unpack_b128(b128_t q) {
  float4 v;
  asm volatile("mov.b128 {%0, %1, %2, %3}, %4;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "q"(q));
  return v;
}
__device__ __forceinline__ b128_t pack_b128(float4 v) {
  b128_t q;
  asm volatile("mov.b128 %0, {%1, %2, %3, %4};" : "=q"(q) : "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
  return q;
}
__device__ __forceinline__ float ldg_nc_f32(const float* p) {
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ uint32_t ldg_nc_u32(const int32_t* p) {
  uint32_t v;
  asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

}  // namespace sqfa

// ------------------------------------------------------------------------------------------------
// Thread-block clusters and the 2-CTA (cta_group::2) flavour of tcgen05
// ------------------------------------------------------------------------------------------------
namespace sqfa {

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() { cluster_arrive(); cluster_wait(); }

// shared::cta address -> shared::cluster address of the same variable in CTA `rank`
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // default .release.cta semantics: the operand bytes were already handed to the async proxy by
  // fence.proxy.async in the writing CTA; a cluster-scope release would compile to MEMBAR.ALL.GPU
  // on every stage (measured: 13% of all stall samples)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void st_cluster_u32(uint32_t cluster_addr, uint32_t v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(cluster_addr), "r"(v) : "memory");
}
__device__ __forceinline__ void st_cluster_u64(uint32_t cluster_addr, uint64_t v) {
  asm volatile("st.shared::cluster.u64 [%0], %1;" ::"r"(cluster_addr), "l"(v) : "memory");
}

// wait on a barrier that also receives arrivals from the peer CTA (cta-scope acquire: a
// cluster-scope acquire would invalidate L1 (CCTL.IVALL) on every wake-up)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); }

template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}

// D[tmem, both CTAs] (+)= A[smem of each CTA: its 128 rows] * B[smem of each CTA: its N/2 columns]
__device__ __forceinline__ void umma_tf32_ss_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (count 1) on the barrier at the same shared-memory offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t mask) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(mask)
      : "memory");
}

}  // namespace sqfa
