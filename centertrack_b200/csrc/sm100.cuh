// Inline-PTX wrappers for the sm_100a asynchronous units: mbarriers, bulk / tensor (TMA) copies, tcgen05 (MMA, TMEM
// loads, allocation) and the UMMA descriptors.  Each wrapper is named after the PTX it emits.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace ctb {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ----
__device__ __forceinline__ void mbarrier_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void fence_mbarrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbarrier_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrives (counts as one of the barrier's arrivals) and adds `bytes` to the phase's expected transaction count
__device__ __forceinline__ void mbarrier_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// adds `bytes` to the expected transaction count WITHOUT arriving
__device__ __forceinline__ void mbarrier_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbarrier_try_wait_parity(uint32_t bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(done) : "r"(bar), "r"(parity) : "memory");
  return done != 0;
}
// Waits for the phase with `parity`; traps after 20 M polls so that a protocol bug cannot hang the GPU.
__device__ __forceinline__ void mbarrier_wait_parity(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbarrier_try_wait_parity(bar, parity))
    if (++spins > 20000000u) __trap();
}

// ---- bulk and tensor copies global -> shared, completing on an mbarrier ----
__device__ __forceinline__ void cp_async_bulk(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void cp_async_bulk_tensor_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2,
                                                        uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}
__device__ __forceinline__ void cp_async_bulk_tensor_4d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2,
                                                        int c3, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar) : "memory");
}
// generic-proxy shared-memory writes -> visible to the async proxy (tensor cores, TMA)
__device__ __forceinline__ void fence_proxy_async_shared_cta() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- tcgen05 ----
__device__ __forceinline__ void tcgen05_fence_before_thread_sync() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after_thread_sync() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// whole warp: allocates `cols` TMEM columns and writes their address to shared memory at `slot`
__device__ __forceinline__ void tcgen05_alloc(uint32_t slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(cols) : "memory");
}
__device__ __forceinline__ void tcgen05_relinquish_alloc_permit() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A x B, kind::f16; accumulates into D when `accumulate` != 0
__device__ __forceinline__ void tcgen05_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// Issued by ALL lanes of the (converged) warp: elect.sync picks one lane and predicates the instruction, so there is no
// divergent branch around the UTCHMMA and its operands stay warp-uniform (cute::elect_one_sync idiom).
__device__ __forceinline__ void tcgen05_mma_elect(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                  uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred pe, pa;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "setp.ne.b32 pa, %4, 0;\n\t"
      "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, pa;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// arrives on `bar` once every tcgen05 operation issued before it by this thread has completed
__device__ __forceinline__ void tcgen05_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tcgen05_commit_elect(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred pe;\n\t"
      "elect.sync _|pe, 0xffffffff;\n\t"
      "@pe tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
      ::"r"(bar) : "memory");
}
// 32 TMEM lanes x 8 / 16 columns into registers, followed by tcgen05.wait::ld
__device__ __forceinline__ void tcgen05_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// ---- UMMA descriptors (cute::UMMA::SmemDescriptor / InstrDescriptor) ----
// K-major SWIZZLE_NONE operand: [0,14) start>>4 | [16,30) LBO>>4 (next K core matrix) | [32,46) SBO>>4 (next 8-row
// group) | [46,48) version = 1 | [61,64) layout = 0
__device__ __forceinline__ uint64_t umma_sdesc_none(uint32_t addr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
// K-major 128B-swizzled operand of 128-byte rows: LBO = 1 (unused), SBO = 64 (8 rows x 128 B), layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t umma_sdesc_sw128(uint32_t addr) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, M = 128, N = n
__device__ __forceinline__ uint32_t umma_idesc_bf16_m128(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

}  // namespace ctb
