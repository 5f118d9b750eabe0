// PTX wrappers for the tcgen05 / TMA / mbarrier / cluster instructions used by the
// tensor-core kernels (sm_100a only).  Shared by tc_kernels.cu and tcb_kernels.cu.
#pragma once

#include <cuda.h>
#include <stdint.h>
#include <stdio.h>

namespace nnab {

// ---------------------------------------------------------------------------
// PTX wrappers (sm_100a)
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a descriptor / barrier bug must trap, never hang the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  unsigned long long t0 = 0;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0xFFFu) == 0) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000ull) {  // 4 s
        printf("nnab: mbarrier wait timeout (block %d thread %d bar %u parity %u)\n",
               (int)blockIdx.x, (int)threadIdx.x, bar, parity);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                            int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tcgen05_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols)
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
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

// K-major swizzled smem matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start>>4 | [16,30) LBO>>4 (unused when swizzled) | [32,46) SBO>>4 |
//   [46,48) version=1 | [61,64) layout (2 = SWIZZLE_128B, 4 = SWIZZLE_64B)
template <int BK>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  constexpr uint64_t SBO = (8u * BK * 2u) >> 4;  // 8 rows of one swizzle atom
  constexpr uint64_t LAYOUT = (BK == 64) ? 2 : 4;
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | (SBO << 32) | (1ull << 46) |
         (LAYOUT << 61);
}


__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive (optionally with expect_tx) on the barrier at the same offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t cta) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(bar), "r"(cta)
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_remote(uint32_t bar, uint32_t cta, uint32_t bytes) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.expect_tx.shared::cluster.b64 _, [ra], %2;\n\t}"
      ::"r"(bar), "r"(cta), "r"(bytes)
      : "memory");
}
// TMA load whose completion bytes are credited to the LEADER CTA's barrier (peer bit cleared)
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                                int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1),
        "r"(c2)
      : "memory");
}
// Cheap descriptor arithmetic for MMA issue loops whose MMAs are short (N <= 64: 8-32 clocks each, so
// the single issuing thread must not spend ~25 instructions per K16 step on descriptor construction).
// The high word of a K-major swizzled descriptor is a constant; the low word is (addr >> 4) | 1 << 16
// and moving along K (+32 B per K16 slice) or down rows (+128 B per row) is an add of the low word
// (no carry leaves the 14-bit address field for shared-memory addresses < 256 KB).
template <int BK>
__device__ __forceinline__ uint32_t smem_desc_lo(uint32_t saddr) {
  return ((saddr & 0x3FFFFu) >> 4) | (1u << 16);
}
template <int BK>
__device__ __forceinline__ uint32_t smem_desc_hi() {
  constexpr uint32_t SBO = (8u * BK * 2u) >> 4;
  constexpr uint32_t LAYOUT = (BK == 64) ? 2u : 4u;
  return SBO | (1u << 14) | (LAYOUT << 29);
}
__device__ __forceinline__ uint64_t desc64(uint32_t lo, uint32_t hi) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
  return d;
}
// D (+)= A * B with the accumulate flag as an immediate (no per-call setp on a register)
template <bool ACC>
__device__ __forceinline__ void umma_bf16_2sm_i(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                                uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.eq.u32 p, %4, 1;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "n"(ACC ? 1 : 0)
      : "memory");
}
// one K block (BK = 64: four K16 slices) of the 3-term bf16 split: A (hi, lo planes) x B (hi, lo planes)
__device__ __forceinline__ void umma_kblock_split3(uint32_t d_tmem, uint32_t a_hi_lo, uint32_t a_lo_lo,
                                                   uint32_t b_hi_lo, uint32_t b_lo_lo, uint32_t hi,
                                                   uint32_t idesc, bool first_accumulates) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint64_t a_hi = desc64(a_hi_lo + 2u * k, hi), a_lo = desc64(a_lo_lo + 2u * k, hi);
    const uint64_t b_hi = desc64(b_hi_lo + 2u * k, hi), b_lo = desc64(b_lo_lo + 2u * k, hi);
    if (k == 0 && !first_accumulates) umma_bf16_2sm_i<false>(d_tmem, a_lo, b_hi, idesc);
    else umma_bf16_2sm_i<true>(d_tmem, a_lo, b_hi, idesc);
    umma_bf16_2sm_i<true>(d_tmem, a_hi, b_lo, idesc);
    umma_bf16_2sm_i<true>(d_tmem, a_hi, b_hi, idesc);
  }
}

// the same K block for a bf16 A operand (zero lo plane): A_hi x (B_hi, B_lo) only
__device__ __forceinline__ void umma_kblock_split2(uint32_t d_tmem, uint32_t a_hi_lo, uint32_t b_hi_lo,
                                                   uint32_t b_lo_lo, uint32_t hi, uint32_t idesc,
                                                   bool first_accumulates) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint64_t a_hi = desc64(a_hi_lo + 2u * k, hi);
    const uint64_t b_hi = desc64(b_hi_lo + 2u * k, hi), b_lo = desc64(b_lo_lo + 2u * k, hi);
    if (k == 0 && !first_accumulates) umma_bf16_2sm_i<false>(d_tmem, a_hi, b_lo, idesc);
    else umma_bf16_2sm_i<true>(d_tmem, a_hi, b_lo, idesc);
    umma_bf16_2sm_i<true>(d_tmem, a_hi, b_hi, idesc);
  }
}

__device__ __forceinline__ void tma_load_4d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar,
                                                int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1),
        "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_2sm() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                              uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit -> arrive on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 "
      "[%0], %1;"
      ::"r"(bar), "h"((uint16_t)3)
      : "memory");
}

}  // namespace nnab
