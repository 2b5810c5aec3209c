// sm_100a primitives of the tcgen05 kernels (gemm_tc.cu, conv_tc.cu): mbarriers, TMA tensor loads, tensor-memory
// allocation, UMMA issue and tcgen05.ld.  Thin forceinline PTX wrappers: a kernel built on them compiles to the same
// instructions as one that spells the PTX out.
#pragma once
#include <cuda.h>
#include <cstdint>

namespace tacorl {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarriers (shared::cta, 64-bit)
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// makes the mbarrier.init of this thread visible to the other threads and to the async proxy (TMA, tcgen05.commit)
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  } while (!done);
}

// ---- TMA tensor loads: box at coordinates (c0 = innermost, ...) -> shared memory at dst, completion bytes on bar
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3,
                                            uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, int c4,
                                            uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
      ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(bar) : "memory");
}

// ---- tensor memory.  One whole warp allocates `cols` columns (a power of two >= 32) and writes their base address to
// the shared-memory slot; it gives up the allocation permit so that other CTAs on the SM can allocate.  The same warp
// frees them at the end (after the other warps' last TMEM access, ordered by tc_fence_before / sync / tc_fence_after).
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}

// ---- tcgen05 ordering, MMA issue and accumulator loads
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// arrives once on bar when every MMA this thread issued before it has completed
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem_d] (+)= A . B for the shapes in idesc; accumulate == 0 overwrites D
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// The same two for an issue loop run by a whole converged warp instead of one lane: the descriptors are then warp-uniform,
// so ptxas keeps them in uniform registers, and one elected lane issues.  From a single lane every tcgen05.mma compiles to
// descriptor moves into uniform registers inside an ELECT / BRA.U.ANY loop, which slows a loop of short MMAs.
__device__ __forceinline__ void tc_mma_bf16_warp(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_commit_warp(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar) : "memory");
}
// 16 consecutive fp32 columns of this thread's TMEM lane (taddr = lane << 16 | column); tc_ld16 also waits for them
__device__ __forceinline__ void tc_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  tc_ld16_nowait(taddr, r);
  tc_ld_wait();
}

// ---- UMMA shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 in bits [0,14), leading
// byte offset >> 4 in [16,30), stride byte offset >> 4 in [32,46), version 1 in [46,48), layout in [61,64).  The
// layout is the swizzle TMA wrote the tile with (CU_TENSOR_MAP_SWIZZLE_128B / _64B).
enum UmmaSwizzle : uint32_t { UMMA_SW128 = 2, UMMA_SW64 = 4 };
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              UmmaSwizzle layout = UMMA_SW128) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}

// ---- kind::f16 instruction descriptor for bf16 A and B with an fp32 accumulator: D format f32 = 1 in bits [4,6),
// A format bf16 = 1 in [7,10), B format bf16 = 1 in [10,13), A MN-major in bit 15, B MN-major in bit 16 (0 = K-major),
// N >> 3 in [17,23), M >> 4 in [24,29).
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N, bool a_mn = false, bool b_mn = false) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

}  // namespace tacorl
