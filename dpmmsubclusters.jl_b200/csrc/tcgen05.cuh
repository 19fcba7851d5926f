// What every tensor-core kernel shares: the tc:: PTX wrappers (mbarrier, TMA, tcgen05.mma / ld / commit, TMEM
// allocation), the shared-memory and instruction descriptors, and gauss_tc_screen_q, the squared norm of one
// cluster's 32 accumulator columns used by the Gaussian label and sub-label screens.
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Wait for the phase with the given parity.  try_wait suspends the thread in hardware until the phase completes or a
// time limit passes; without a hint that limit is short and the loop around it spins -- in the warp-specialised
// kernels here a quarter of all issued instructions were such polls, competing with the working warps of the same
// scheduler.  Yet an explicit suspend-time hint measured slower (see the header of kernels_substats_tc.cuh).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "LAB_WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra LAB_DONE_%=;\n\t"
      "bra LAB_WAIT_%=;\n\t"
      "LAB_DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] . B[smem]^T, both operands K-major, TF32 inputs, FP32 accumulate.
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the same with the accumulate flag fixed at compile time (no predicate set-up in the issuing thread)
__device__ __forceinline__ void umma_tf32_first(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, 0, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_acc(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.eq.b32 p, 0, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc)
      : "memory");
}
// Warp-collective forms: EVERY lane of the (converged) issuing warp executes the call and one elected
// lane issues the instruction.  With warp-uniform control flow and operands the compiler keeps the
// descriptors in uniform registers; issuing from an `if (lane == 0)` branch instead costs four R2UR
// moves and an ELECT/R2UR.BROADCAST waterfall loop per MMA (~100 cycles of issue latency each).
__device__ __forceinline__ void umma_tf32_first_w(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, 0, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_acc_w(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.eq.b32 p, 0, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ void umma_commit_w(uint64_t* bar) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}" ::"r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread (thread = lane).
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor, K-major operand stored as rows of 128 bytes with the 128B swizzle
// (8-row groups 1024 B apart): start address, LBO = 1 (ignored), SBO = 1024 B, version 1, SWIZZLE_128B.
__device__ __forceinline__ uint64_t smem_desc_k128(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | ((uint64_t)1 << 46) |
         ((uint64_t)2 << 61);
}
// K-major operand of one 8-element k-step without swizzle: 8-row x 16-byte core matrices, the two core
// matrices of the k-step LBO = 128 B apart, 8-row groups SBO = 256 B apart.
__device__ __forceinline__ uint64_t smem_desc_k_noswz(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | ((uint64_t)1 << 46);
}
// the same with explicit strides: LBO between the two k halves, SBO between 8-row groups
__device__ __forceinline__ uint64_t smem_desc_k_noswz2(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | ((uint64_t)1 << 46);
}
// Instruction descriptor: FP32 accumulator, TF32 A and B, both K-major, M = 128, N = n.
__device__ __forceinline__ uint32_t idesc_tf32(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

}  // namespace tc

// q~ = sum_i y_i^2 over the 32 accumulator columns of one cluster (y = U x - U mu from the MMA)
__device__ __forceinline__ float gauss_tc_screen_q(const uint32_t (&v)[32]) {
  f32x2_t acc0 = 0ull, acc1 = 0ull;
#pragma unroll
  for (int j = 0; j < 32 / 4; ++j) {
    const f32x2_t p0 = f2_pack(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]));
    const f32x2_t p1 = f2_pack(__uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
    acc0 = f2_fma(p0, p0, acc0);
    acc1 = f2_fma(p1, p1, acc1);
  }
  float a0, a1, b0, b1;
  f2_unpack(acc0, a0, a1);
  f2_unpack(acc1, b0, b1);
  return (a0 + a1) + (b0 + b1);
}
