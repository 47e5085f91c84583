// tcgen05 / TMA / mbarrier PTX wrappers shared by the tensor-core kernels (sm_100a).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace mtts {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// ---- CTA pair (cta_group::2): two SMs of a TPC run one 256-row MMA, each staging half of the operands ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// shared::cluster address of `addr` (a shared::cta address) in CTA `rank` of this cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_cluster) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_cluster) : "memory");
}
// the copy lands in THIS CTA's shared memory; its bytes are counted on the barrier at cluster address `bar_cluster`
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar_cluster, int c0, int c1,
                                                int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives (once the MMAs issued so far have retired) on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void tc_commit_2sm(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}

// K-major swizzled operand tile with SWB-byte rows (SWB = 128 or 64): 8-row atoms of 8*SWB bytes
template <int SWB>
__device__ __forceinline__ uint64_t umma_desc_kmajor(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)((8 * SWB) >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(SWB == 128 ? 2 : 4) << 61;          // SWIZZLE_128B : SWIZZLE_64B
  return d;
}

// ---- warp-uniform issue: every lane reaches the instruction with identical (uniform-register) operands and the one
// lane whose `leader` flag is set executes it
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_mma_l(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate,
                                         uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tc_mma_2sm_l(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate,
                                             uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "setp.ne.b32 q, %5, 0;\n\t"
      "@q tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tc_commit_l(uint32_t bar, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
      "}" ::"r"(bar), "r"(leader)
      : "memory");
}
__device__ __forceinline__ void tc_commit_2sm_l(uint32_t bar, uint32_t leader) {
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "@q tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %2;\n\t"
      "}" ::"r"(bar), "r"(leader), "h"((uint16_t)3)
      : "memory");
}

// descriptor of an operand whose start address is shifted by whole rows inside a swizzled tile: low word = address, base
// offset left at zero (the swizzle follows the address bits, conv_tc.cu)
__device__ __forceinline__ uint64_t umma_desc_shifted(uint64_t desc_base, uint32_t smem_addr) {
  return desc_base | (uint64_t)((smem_addr >> 4) & 0x3FFF);
}

// One tap of the f16x2 halo form: NKS k-steps x three MMAs (x1 w2' and x2' w1 into the correction accumulator, x1 w1 into
// the main one), issued from ONE asm block whose operand descriptors are derived inside it by 64-bit adds from the two
// base descriptors.  Written this way because, given one asm statement per MMA with four 64-bit operands each, ptxas
// re-materialises and re-pairs the (identical) high words and the instruction descriptor for every instruction: ~104
// uniform-datapath instructions per tap, which - not the tensor pipe - paced the C = 32 / 64 vocoder convolutions
// (ncu source page of the issuing warp, gpurun call P).
//   a1 / b1: descriptors of plane 0 at k-step 0; a_plane16 / b_plane16: plane stride >> 4; first: 0 to overwrite the
//   accumulators with the first k-step (the tile's first tap), else accumulate
template <int NKS, int PAIR>
__device__ __forceinline__ void tc_tap_f16x2(uint32_t d_main, uint32_t d_corr, uint64_t a1, uint64_t b1, uint32_t a_plane16,
                                             uint32_t b_plane16, uint32_t idesc, uint32_t first, uint32_t leader) {
  static_assert(NKS == 2 || NKS == 4, "k-steps per K-slab");
#define MTTS_MMA_CG1 "tcgen05.mma.cta_group::1.kind::f16"
#define MTTS_MMA_CG2 "tcgen05.mma.cta_group::2.kind::f16"
#define MTTS_TAP_BODY(MMA)                                                                     \
  "{\n\t"                                                                                      \
  ".reg .pred p, q, t;\n\t"                                                                    \
  ".reg .b64 a2, b2, ap, bp;\n\t"                                                              \
  "setp.ne.b32 p, %6, 0;\n\t"                                                                  \
  "setp.ne.b32 q, %7, 0;\n\t"                                                                  \
  "setp.eq.b32 t, 0, 0;\n\t"                                                                   \
  "cvt.u64.u32 ap, %4;\n\t"                                                                    \
  "cvt.u64.u32 bp, %5;\n\t"                                                                    \
  "add.s64 a2, %2, ap;\n\t"                                                                    \
  "add.s64 b2, %3, bp;\n\t"                                                                    \
  "@q " MMA " [%1], %2, b2, %8, p;\n\t"                                                        \
  "@q " MMA " [%1], a2, %3, %8, t;\n\t"                                                        \
  "@q " MMA " [%0], %2, %3, %8, p;\n\t"
#define MTTS_TAP_STEP(MMA, OFF)                                                                \
  "{\n\t"                                                                                      \
  ".reg .b64 a1k, b1k, a2k, b2k;\n\t"                                                          \
  "add.s64 a1k, %2, " #OFF ";\n\t"                                                             \
  "add.s64 b1k, %3, " #OFF ";\n\t"                                                             \
  "add.s64 a2k, a2, " #OFF ";\n\t"                                                             \
  "add.s64 b2k, b2, " #OFF ";\n\t"                                                             \
  "@q " MMA " [%1], a1k, b2k, %8, t;\n\t"                                                      \
  "@q " MMA " [%1], a2k, b1k, %8, t;\n\t"                                                      \
  "@q " MMA " [%0], a1k, b1k, %8, t;\n\t"                                                      \
  "}\n\t"
  if constexpr (NKS == 2) {
    if constexpr (PAIR)
      asm volatile(MTTS_TAP_BODY(MTTS_MMA_CG2) MTTS_TAP_STEP(MTTS_MMA_CG2, 2) "}"
                   ::"r"(d_main), "r"(d_corr), "l"(a1), "l"(b1), "r"(a_plane16), "r"(b_plane16), "r"(first), "r"(leader), "r"(idesc)
                   : "memory");
    else
      asm volatile(MTTS_TAP_BODY(MTTS_MMA_CG1) MTTS_TAP_STEP(MTTS_MMA_CG1, 2) "}"
                   ::"r"(d_main), "r"(d_corr), "l"(a1), "l"(b1), "r"(a_plane16), "r"(b_plane16), "r"(first), "r"(leader), "r"(idesc)
                   : "memory");
  } else {
    if constexpr (PAIR)
      asm volatile(MTTS_TAP_BODY(MTTS_MMA_CG2) MTTS_TAP_STEP(MTTS_MMA_CG2, 2) MTTS_TAP_STEP(MTTS_MMA_CG2, 4) MTTS_TAP_STEP(MTTS_MMA_CG2, 6) "}"
                   ::"r"(d_main), "r"(d_corr), "l"(a1), "l"(b1), "r"(a_plane16), "r"(b_plane16), "r"(first), "r"(leader), "r"(idesc)
                   : "memory");
    else
      asm volatile(MTTS_TAP_BODY(MTTS_MMA_CG1) MTTS_TAP_STEP(MTTS_MMA_CG1, 2) MTTS_TAP_STEP(MTTS_MMA_CG1, 4) MTTS_TAP_STEP(MTTS_MMA_CG1, 6) "}"
                   ::"r"(d_main), "r"(d_corr), "l"(a1), "l"(b1), "r"(a_plane16), "r"(b_plane16), "r"(first), "r"(leader), "r"(idesc)
                   : "memory");
  }
#undef MTTS_TAP_STEP
#undef MTTS_TAP_BODY
#undef MTTS_MMA_CG2
#undef MTTS_MMA_CG1
}

}  // namespace mtts
