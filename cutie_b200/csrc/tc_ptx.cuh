// Inline-PTX helpers for the tcgen05 / mbarrier / bulk-copy kernels (sm_100a): shared by the affinity filter
// (affinity_f16.cu) and the object-transformer attention kernels (qt_tc.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cutie {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity), "r"(200000u)      // suspend-time hint (ns): sleep in hardware, do not spin
        : "memory");
  }
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ float to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t smem_slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_slot), "n"(COLS));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t tmem) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(COLS));
}
// 32 consecutive accumulator columns of this thread's TMEM lane (warp w of a warpgroup reads lanes 32 (w % 4) ..)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptors (SWIZZLE_128B, Blackwell descriptor version 1).
// K-major: a block is [rows x 128 B] (rows = M or N index, 128 B = 32 tf32 / 64 f16 along K), 8-row groups 1024 B
// apart (SBO); one MMA k-step = +32 B inside the swizzle atom.
__device__ __forceinline__ uint64_t desc_sw128_kmajor(uint32_t addr) {
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;                        // leading byte offset: unused for swizzled K-major
  d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset: 8 rows x 128 B
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
  return d;
}
// MN-major (storage [k][mn], mn contiguous) for 32-bit operands: SWIZZLE_128B_BASE32B (layout type 1) is the only
// MN-major layout tf32 has.  A group is [k rows x 128 B] holding 32 tf32 along MN per row; inside each 4-row atom
// (512 B) the four 32-BYTE chunks of row k are stored at chunk ^ (k & 3); atoms of 4 k-rows follow each other at SBO,
// groups of 32 MN elements at LBO.  One tf32 MMA k-step (K = 8) is two atoms per group: advance the start address by
// 1024 B.  (tests/cuda/umma_probe.cu checks this encoding on hardware.)
__device__ __forceinline__ uint64_t desc_sw128_mnmajor(uint32_t addr, uint32_t group_stride_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((addr >> 4) & 0x3FFF);
  d |= (uint64_t)((group_stride_bytes >> 4) & 0x3FFF) << 16;   // LBO: next 32 MN elements
  d |= (uint64_t)(512 >> 4) << 32;                             // SBO: next 4 k rows
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;                                      // SWIZZLE_128B_BASE32B
  return d;
}
// byte offset of the 16-byte piece c4 (0..7: four MN elements each) of k-row `k` inside an MN-major group
__device__ __forceinline__ int off_mn32(int k, int c4) {
  return k * 128 + ((((c4 >> 1) ^ (k & 3))) << 5) + ((c4 & 1) << 4);
}
// kind::tf32 instruction descriptor: D = F32, A = B = TF32, M x N, optional MN-major operands.
__device__ __forceinline__ uint32_t idesc_tf32(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

}  // namespace cutie
