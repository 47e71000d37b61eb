// PTX wrappers shared by the tcgen05 GEMMs (linear_tc.cu, linear_bwd.cu) and the bulk-copy edge kernel (edge.cu):
// mbarrier, TMA tile and bulk loads, tcgen05 alloc / mma / commit / ld, shared-memory matrix descriptors, the CTA-pair
// (cta_group::2) forms, and the host-side tensor-map encoder.  sm_100a only.
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace tcp {

__device__ __forceinline__ uint32_t s_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// ---- mbarrier ----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster.  Default (.cta-scope) semantics:
// the pair barriers carry no generic-proxy data (operands arrive through TMA complete_tx, accumulators are handed over
// with tcgen05.commit / tcgen05.fence), and the .release.cluster form compiles to MEMBAR.ALL.GPU + ERRBAR
// (profiles/r02_gemm_epilogue_ab.md).
__device__ __forceinline__ void mbar_arrive_cta(uint32_t bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
      "}"
      ::"r"(bar), "r"(cta)
      : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}

// ---- cluster -----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---- TMA / bulk copies -------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const CUtensorMap* map, int c0, int c1, int c2,
                                            uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// CTA-pair form: the copy lands in the issuing CTA's shared memory, its complete_tx goes to the barrier at `bar` in the
// leader CTA (peer bit cleared).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t smem_dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(map), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
// 1-D bulk copy of `bytes` (multiple of 16) contiguous bytes.
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src_gmem, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   dst_smem), "l"(src_gmem), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void prefetch_map(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// ---- tcgen05 -----------------------------------------------------------------------------------------------------------
// TMEM allocation by one warp, which then gives up the allocation permit; CG = 1 for a single CTA, 2 for a CTA pair.
template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  if constexpr (CG == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  if constexpr (CG == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_ss_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// Arrives on the barrier at `bar` in both CTAs of the pair.
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---- descriptors -------------------------------------------------------------------------------------------------------
// K-major SWIZZLE_128B operand tile (rows of 64 bf16 = 128 B, 8-row swizzle atoms 1024 B apart).
__device__ __forceinline__ uint64_t desc_k_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;                               // LBO: ignored for swizzled K-major
  d |= (uint64_t)(1024 >> 4) << 32;                     // SBO: next 8-row group
  d |= (uint64_t)1 << 46;                               // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                               // SWIZZLE_128B
  return d;
}
// MN-major SWIZZLE_128B operand tile as TMA leaves it when the box is {64 MN-elements (128 B), R k-rows}: k-row r of
// MN-atom j sits at j*lbo_bytes + r*128 (+ swizzle).  Canonical form (cute/atom/mma_traits_sm100.hpp, Major-MN B128,
// in 16-byte units): ((8,n),(8,k)):((1,LBO),(8,SBO)) => SBO = 8 rows * 128 B = 1024 B, LBO = distance between atoms.
__device__ __forceinline__ uint64_t desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor: D = f32, A = B = bf16, M x N tile; a_mn / b_mn select MN-major operands.
__device__ __forceinline__ uint32_t idesc_bf16(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

}  // namespace tcp

// Host: 2-D bf16 tensor map over [rows, cols] with a row stride of `ld` elements, box {64 columns, box_rows rows},
// SWIZZLE_128B, out-of-bounds reads filled with zeros.  A zero-row operand is mapped as one row (the encoder rejects
// empty extents; no tile of such an operand is ever loaded).  Returns 0, or 1 with the error message set.
int hgt_make_tma_map_bf16(CUtensorMap* map, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows);
