// tc.cuh — minimal hand-written tcgen05 / TMEM / mbarrier layer for sm_100a (no CUTLASS).
//
// Conventions (bit layouts cross-checked against cute/arch/mma_sm100_desc.hpp in the image):
//  * shared-memory matrix descriptor (64 bit): [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 |
//    [46,48) version=1 | [49,52) base_offset | [52] lbo_mode | [61,64) layout (0 none, 2 SW128, 4 SW64, 6 SW32)
//  * instruction descriptor (32 bit, kind::f16): [4,6) D fmt (1=f32) | [7,10) A fmt (0=f16) |
//    [10,13) B fmt | [15] A major (0=K) | [16] B major | [17,23) N>>3 | [24,29) M>>4
//  * K-major operand tiles are stored as rows of 32/64/128 bytes with the matching 32B/64B/128B
//    swizzle: 16-byte chunk c of row r lands at chunk c ^ f(r) (f = (r>>2)&1 / (r>>1)&3 / r&7); tiles
//    are 1024-byte aligned; 8-row groups are SBO bytes apart; advancing K by 16 elements = +32 bytes
//    on the start address (the hardware swizzles on address bits).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace f2b { namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

enum : uint64_t { kLayoutNone = 0, kLayoutSW128 = 2, kLayoutSW64 = 4, kLayoutSW32 = 6 };

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint64_t layout) {
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         (1ull << 46) | (layout << 61);
}
// K-major tile with `row_bytes` (32/64/128) per row and the matching swizzle
__device__ __forceinline__ uint64_t kmajor_desc(uint32_t saddr, int row_bytes) {
  const uint64_t layout = row_bytes == 128 ? kLayoutSW128 : (row_bytes == 64 ? kLayoutSW64 : kLayoutSW32);
  return make_desc(saddr, 16, 8 * row_bytes, layout);
}
__host__ __device__ constexpr uint32_t idesc_f16_f32(int M, int N, int a_mn_major = 0, int b_mn_major = 0) {
  return (1u << 4) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// byte offset of 16-byte chunk `c` of row `r` inside a swizzled K-major tile
__device__ __forceinline__ uint32_t sw128_off(int r, int c) { return r * 128 + ((c ^ (r & 7)) << 4); }
__device__ __forceinline__ uint32_t sw64_off(int r, int c) { return r * 64 + ((c ^ ((r >> 1) & 3)) << 4); }
__device__ __forceinline__ uint32_t sw32_off(int r, int c) { return r * 32 + ((c ^ ((r >> 2) & 1)) << 4); }

// ---- TMEM ---------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {   // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {     // same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// generic-proxy smem writes -> visible to the async proxy (UMMA operand reads)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread
__device__ __forceinline__ void mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once every previously issued MMA of this thread has completed
__device__ __forceinline__ void mma_commit(uint64_t* mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(mbar)) : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* mbar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(mbar)), "r"(count) : "memory");
}
// one arrival (release at CTA scope: the caller's earlier shared-memory writes are visible to the thread that waits)
__device__ __forceinline__ void mbar_arrive(uint64_t* mbar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(mbar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* mbar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred P1;\n\tLAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\tbra LAB_WAIT;\n\tDONE:\n\t}\n" ::"r"(smem_u32(mbar)),
      "r"(parity)
      : "memory");
}

// 32 lanes x 16 consecutive fp32 columns -> 16 registers per thread (lane = TMEM lane of taddr + laneid)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

}}  // namespace f2b::tc
