// vb_ptx.cuh — thin inline-PTX layer for sm_100a: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (alloc / mma / commit / ld / st / fences) and UMMA descriptor builders.
// Everything here is hand-written for Blackwell; nothing is dispatched per architecture.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace vb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase completes or the hint expires, so
// a waiting warp does not burn issue slots of its scheduler (the softmax warps of the other tile share it)
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(1000000u)
      : "memory");
  return ok != 0;
}
// Wait for a phase.  With -DVB_WATCHDOG (bring-up builds) a protocol bug becomes a trap instead of a hang.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
#ifdef VB_WATCHDOG
  uint32_t spins = 0;
#endif
  while (!mbar_try_wait(bar, parity)) {
#ifdef VB_WATCHDOG
    if (++spins > (1u << 16)) {
      printf("vb: mbarrier watchdog block(%d,%d,%d) thread %d bar@%u parity %u\n", blockIdx.x, blockIdx.y,
             blockIdx.z, threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
#endif
  }
}

// Non-blocking phase test for a warp-converged poller (the MMA issuer's event loop); lane 0's view is broadcast so
// that every lane takes the same branch.
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred P;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return __shfl_sync(0xffffffffu, ok, 0) != 0;
}

// named barrier among a subset of warps (id 1..15; id 0 is __syncthreads)
__device__ __forceinline__ void named_bar_sync(int id, int n_threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n_threads) : "memory");
}

// generic-proxy writes to shared memory -> visible to the async proxy (TMA / UMMA operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// TMA
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 4-D tiled load: coordinates are (c0 = innermost element, c1, c2, c3)
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];"
      :
      : "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1),
        "r"(c2), "r"(c3)
      : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05: TMEM allocation
// ----------------------------------------------------------------------------------------------
// Whole warp must call. Writes the TMEM base address (lane<<16 | column) to *smem_slot.
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05: UMMA descriptors
// ----------------------------------------------------------------------------------------------
// Shared-memory matrix descriptor (64-bit):
//   [0,14)  start address >> 4      [16,30) leading-dim byte offset >> 4
//   [32,46) stride-dim byte offset >> 4   [46,48) version (1 on sm_100)
//   [49,52) base offset             [61,64) layout type (2 = SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= static_cast<uint64_t>(1) << 46;   // descriptor version for Blackwell
  d |= static_cast<uint64_t>(2) << 61;   // SWIZZLE_128B
  return d;
}
// Instruction descriptor for kind::f16 with bf16 A/B, fp32 accumulate.
//   [4,6) c format (1 = f32)  [7,10) a format (1 = bf16)  [10,13) b format (1 = bf16)
//   [15] a major (0 = K)      [16] b major (0 = K, 1 = MN) [17,23) N >> 3   [24,29) M >> 4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N, int a_mn_major, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]; single thread issues.
__device__ __forceinline__ void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]; A is 128 lanes x (K/2) 32-bit columns of packed bf16 pairs.
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once every tcgen05 op issued so far by this thread has completed.
// (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ----------------------------------------------------------------------------------------------
// tcgen05: TMEM <-> registers (32 lanes x 32-bit, N consecutive columns per thread)
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]),
        "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]),
        "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
        "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
        "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
// 16-column variants (correction path: fewer live registers)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ----------------------------------------------------------------------------------------------
// misc math
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// Blackwell packed fp32x2 arithmetic: one issue slot and one FMA-pipe pass for two lanes of work
__device__ __forceinline__ void ffma2(float& d0, float& d1, float a0, float a1, float b0, float b1, float c0, float c1) {
  asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d0), "=f"(d1)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1), "f"(c0), "f"(c1));
}
__device__ __forceinline__ void fadd2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
  asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "add.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d0), "=f"(d1)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
// exp2 of two values on the FMA / ALU pipes (no MUFU): round-to-nearest split x = n + f, |f| <= 0.5, degree-3
// minimax polynomial for 2^f (max relative error 7.5e-5, far below the bf16 rounding P receives anyway), exponent
// added as an integer.  The MUFU ex2 unit (16 / clk / SM) is co-critical with the tensor pipe at head_dim 128
// (512 MMA flops per exp), so a fraction of the exps is computed here instead.
// Below -126 the result is exactly 0, as ex2.approx.ftz gives: the integer exponent add needs x >= -126, and the clamp
// alone turned a masked key (x = -inf) into a weight of 2^-126 * p(0) that the PV MMA multiplies by a real V row.
__device__ __forceinline__ void exp2_poly2(float x0, float x1, float& e0, float& e1) {
  constexpr float kMagic = 12582912.f;   // 1.5 * 2^23: adding it rounds to an integer held in the low mantissa bits
  const bool z0 = x0 < -126.f, z1 = x1 < -126.f;
  x0 = fmaxf(x0, -126.f);
  x1 = fmaxf(x1, -126.f);
  float t0, t1, r0, r1, f0, f1, p0, p1;
  fadd2(t0, t1, x0, x1, kMagic, kMagic);
  fadd2(r0, r1, t0, t1, -kMagic, -kMagic);
  ffma2(f0, f1, r0, r1, -1.f, -1.f, x0, x1);
  ffma2(p0, p1, f0, f1, 0.055171020f, 0.055171020f, 0.24260981f, 0.24260981f);
  ffma2(p0, p1, p0, p1, f0, f1, 0.69326097f, 0.69326097f);
  ffma2(p0, p1, p0, p1, f0, f1, 0.99992818f, 0.99992818f);
  e0 = z0 ? 0.f : __int_as_float(__float_as_int(p0) + (__float_as_int(t0) << 23));
  e1 = z1 ? 0.f : __int_as_float(__float_as_int(p1) + (__float_as_int(t1) << 23));
}

// pack two fp32 -> bf16x2 (lo in bits [0,16), hi in bits [16,32)), round-to-nearest-even
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

}  // namespace vb
