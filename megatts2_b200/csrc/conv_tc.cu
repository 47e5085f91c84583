// Tensor-core tap-GEMM: every stride-1 Conv1d / ConvTranspose1d (2-tap form) / Linear (k = 1) on tcgen05 with fp32-grade
// accuracy from split operands and two TMEM accumulators (leading product | corrections):
//   NP = 3 (bf16x3): x = x1 + x2 + x3 in bf16 (to 2^-24); the six products whose weight is >= 2^-16 are issued.
//   NP = 2 (f16x2):  x = x1 + x2' * 2^-11 in fp16 (the residual is stored scaled by 2^11, so it stays a normal fp16 number
//                    whenever x is); three products x1*w1 | x1*w2' + x2'*w1, the correction accumulator is scaled by 2^-11
//                    in the epilogue.  22 significant bits per operand: the dropped x2*w2 term is 2^-22 relative, below
//                    the rounding noise of an fp32 dot product; half the MMAs and two thirds of the operand bytes.
// Eligible wherever Cin % 8 == 0, Cin >= 32, Cout in {32, 64, >= 128 and % 32 == 0} and B*T >= 128; everything else
// stays on the exact FFMA engine (tapconv.cu).  Reference layers: modules/convnet.py:13-18, modules/transformer.py:16-102,
// the speechbrain HiFi-GAN generator (ResBlock1 convs, ConvTranspose1d upsamplers).
//
// Data flow:  activation planes (B, T + halo, C) bf16 x 3 with the padding MATERIALISED (zero / reflect / replicate)
// and the pre-activation applied - written by the producing kernel (LayerNorm, attention, the previous tap-GEMM's
// epilogue) or, failing that, by split_pad_bf16x3_kernel - so that the conv is a "valid" conv over the planes and tap j
// of an output tile is simply the same 128-row tile shifted by j*dil rows: one 3-D TMA box load per (tap, channel
// slab, plane), no im2col, the k-fold re-reads are served by L2.  Weights are packed per tap as (k, Cout, Cin) bf16
// planes (K-major B).  Variants: tile width BN 128 / 64 / 32 by grid fill, CTA pairs (cta_group::2) for the dense
// layers, split-K with a fixed-order reduction kernel for under-filled dense layers.  DESIGN.md section 4 has the
// anatomy and the measured bounds.
#include <mutex>
#include <unordered_map>

#include "kernels.h"
#include "tc_ptx.cuh"

namespace mtts {

struct ConvTcMaps {
  CUtensorMap a[3];   // 3-D: (C, Tp, B)
  CUtensorMap b[3];   // 2-D: (Cin, k*Cout)
};

struct ConvTcArgs {
  int32_t B, T, Cin, Cout, k, dil;
  const float* bias;
  const float* res; int64_t res_sb; int32_t ldr;
  float* y; int64_t y_sb; int32_t ldy;
  int32_t post_act; float post_slope; float out_scale; int32_t accumulate;
  int64_t out_shift, ybe;      // transposed-conv form: element offset of the output and valid range per batch item
  // optional bf16x3 copy of the result for the next tensor-core layer
  __nv_bfloat16* op; int64_t op_stride; int32_t op_ld, op_tp, op_hl, op_act; float op_slope;
  // split-K (dense layers with too few tiles): work item = (tile, split); partial sums go to `partial`
  int32_t splits; float* partial;
  int32_t fmt; int32_t* ovf;   // operand format of the plane output (== the kernel's own NP) and the f16 range flag
  int32_t row0;                // first padded row of this conv inside a shared plane buffer (0 for its own planes)
};

// PAIR = 1: two CTAs of a cluster run one 256 x BN tile with cta_group::2 MMAs; each CTA stages its own 128 rows of
// the activations and HALF of the weight tile, so the L2 -> SM traffic per FLOP drops by a quarter
// HALO = 1 (convolutions whose input channels fit ONE K-slab, Cin <= SWB / 2): the activation tile of an output tile -
// its 128 rows plus the dil * (k - 1) halo rows - is loaded ONCE into a double-buffered region and every tap reads it
// through a row-shifted UMMA descriptor; only the (tiny) per-tap weight tiles stream through the stage ring.  The plain
// form re-reads the tile once per tap (k-fold L2 -> SM traffic), which is what bounds the C = 32 / 64 HiFi-GAN stages.
constexpr int CTC_HALO_ROWS = 192;     // rows of a halo tile buffer: 128 + dil * (k - 1) <= 192, a multiple of 8
template <int BN, int SWB, int PAIR = 0, int NP = 3, int HALO = 0>
struct ConvTcCfg {
  static constexpr int BK = SWB / 2;                       // bf16 elements per swizzled row
  static constexpr int A_PLANE = (HALO ? CTC_HALO_ROWS : 128) * SWB;
  static constexpr int B_ROWS = PAIR ? BN / 2 : BN;        // weight rows staged by one CTA
  static constexpr int B_PLANE = B_ROWS * SWB;
  static constexpr int STAGE = HALO ? NP * B_PLANE : NP * (A_PLANE + B_PLANE);
  // halo-tile buffers: a tile's rows are requested when the buffer of the tile A_BUFS back is released, i.e. A_BUFS - 1 tiles
  // of MMA time ahead; the k = 3 convolutions have ~1 us of MMA work per tile against ~1.3 us of HBM latency, so two
  // buffers left the tensor pipe waiting on every tile
  static constexpr int A_BUFS = HALO ? (SWB == 64 ? 4 : (NP == 2 ? 3 : 2)) : 0;
  static constexpr int A_REGION = A_BUFS * NP * A_PLANE;
  static constexpr int EPI_STAGE = 8 * 32 * 20 * 4;          // epilogue transpose buffers: 8 warps x [32 rows][20 floats]
  static constexpr int STAGES_RAW = (227 * 1024 - 1024 - 256 - EPI_STAGE - A_REGION) / STAGE;
  static constexpr int STAGES = STAGES_RAW > 6 ? 6 : (STAGES_RAW < 2 ? 2 : STAGES_RAW);
  static constexpr int SMEM = A_REGION + STAGES * STAGE + 1024 + 256 + EPI_STAGE;
  static constexpr int NACC = (4 * BN > 512) ? 1 : 2;            // accumulator buffers: BN = 256 fills TMEM with one
  static constexpr int TMEM_COLS = NACC * 2 * BN < 32 ? 32 : NACC * 2 * BN;   // NACC x (main + correction) x BN
  static_assert(SMEM <= 227 * 1024 && STAGES_RAW >= 2, "shared-memory budget");
};

template <int BN, int SWB, int PAIR, int NP, int HALO>
__global__ void __launch_bounds__(384, 1)
conv_tc_kernel(const __grid_constant__ ConvTcMaps maps, const ConvTcArgs g) {
  using Cfg = ConvTcCfg<BN, SWB, PAIR, NP, HALO>;
  pdl_trigger();                                           // the next kernel may be scheduled; it waits for this grid itself
  constexpr int BM = PAIR ? 256 : 128;                     // rows of one (pair) tile
  const uint32_t crank = PAIR ? cluster_ctarank() : 0u;
  const int worker = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;       // tile walker id (a CTA or a CTA pair)
  const int nworkers = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int NACC = Cfg::NACC;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_a = (smem_u32(smem_raw) + 1023u) & ~1023u;      // HALO: the two halo-tile buffers come first
  const uint32_t smem_base = smem_a + Cfg::A_REGION;                   // the stage ring
  const uint32_t bars = smem_base + STAGES * Cfg::STAGE;
  const uint32_t full_bar = bars, empty_bar = bars + 8 * STAGES;
  const uint32_t tfull_bar = bars + 16 * STAGES, tempty_bar = tfull_bar + 16;
  const uint32_t tmem_slot = tempty_bar + 16;
  const uint32_t afull_bar = tmem_slot + 16, aempty_bar = afull_bar + 32;   // HALO only (16 * STAGES + 48 + 64 <= 256)
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));
  float* epi_stage = reinterpret_cast<float*>(smem_raw + (bars + 256 - smem_u32(smem_raw)));   // 16-byte aligned

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // warp-uniform as far as the compiler can tell
  const int lane = threadIdx.x & 31;
  const int num_t = (g.T + BM - 1) / BM, num_n = (g.Cout + BN - 1) / BN;
  const int num_tiles = g.B * num_t * num_n * g.splits;      // work items: (tile, K split)
  const int ncb = (g.Cin + Cfg::BK - 1) / Cfg::BK;
  const int num_k = g.k * ncb;

  if (warp == 0 && lane == 0) {
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(&maps.a[i]) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(&maps.b[i]) : "memory");
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar + 8 * s, 1);
      mbar_init(empty_bar + 8 * s, 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar + 8 * s, 1);
      mbar_init(tempty_bar + 8 * s, PAIR ? 16 : 8);     // one arrive per epilogue warp (8 warps per CTA)
    }
    if constexpr (HALO) {
      for (int s = 0; s < Cfg::A_BUFS; ++s) {
        mbar_init(afull_bar + 8 * s, 1);
        mbar_init(aempty_bar + 8 * s, 1);
      }
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    if constexpr (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(Cfg::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(Cfg::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync_all();      // the peer's barriers are initialised before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);
  pdl_wait();        // everything above (barriers, TMEM, descriptor prefetch) overlapped the previous kernel's tail

  // The two issuing roles run WARP-UNIFORMLY: every lane walks the loops and computes the (identical) addresses and
  // descriptors, and one elected lane executes the TMA / MMA / commit instructions.  Those instructions take their
  // operands from uniform registers; issued from inside a single-lane branch (the round-1 form) ptxas wraps EACH of
  // them in ELECT + 5 x R2UR + a waterfall loop, about 100 cycles per tcgen05.mma - measured as the limiter of every
  // tile shape (ncu source page: the issuing warp never waits, profiles/r2e_mma_issue_bound.md).
  if (warp == 0) {
    // ================= TMA producer =================
    const bool leader = elect_one();
    int stage = 0, phase = 0;
    [[maybe_unused]] int ait = 0;
    for (int item = worker; item < num_tiles; item += nworkers) {
      const int sp = item % g.splits, tile = item / g.splits;
      const int kb0 = (int)((int64_t)sp * num_k / g.splits), kb1 = (int)((int64_t)(sp + 1) * num_k / g.splits);
      const int nb = tile % num_n, r = tile / num_n;
      const int tb = r % num_t, b = r / num_t;
      const int trow = tb * BM + (int)crank * 128 + g.row0;      // this CTA's first (padded) input row
      if constexpr (HALO) {
        // the tile's activation rows [trow, trow + 128 + dil * (k - 1)) once, then one weight tile per tap
        const int ab = ait % Cfg::A_BUFS, aph = (ait / Cfg::A_BUFS) & 1;
        ++ait;
        mbar_wait(aempty_bar + 8 * ab, aph ^ 1);
        const uint32_t a_bytes = (uint32_t)(NP * (128 + g.dil * (g.k - 1)) * SWB);
        if constexpr (PAIR) {
          // both CTAs' tiles are counted on the LEADER's barrier (the leader issues the MMAs for the pair)
          const uint32_t fa = mapa_u32(afull_bar + 8 * ab, 0);
          if (leader) {
            if (crank == 0) mbar_expect_tx(afull_bar + 8 * ab, 2 * a_bytes);
#pragma unroll
            for (int q = 0; q < NP; ++q)
              tma_load_3d_2sm(smem_a + (ab * NP + q) * Cfg::A_PLANE, &maps.a[q], fa, 0, trow, b);
          }
        } else if (leader) {
          mbar_expect_tx(afull_bar + 8 * ab, a_bytes);
#pragma unroll
          for (int q = 0; q < NP; ++q)
            tma_load_3d(smem_a + (ab * NP + q) * Cfg::A_PLANE, &maps.a[q], afull_bar + 8 * ab, 0, trow, b);
        }
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar + 8 * stage, phase ^ 1);
          const uint32_t sb = smem_base + stage * Cfg::STAGE;
          if constexpr (PAIR) {
            const uint32_t fb = mapa_u32(full_bar + 8 * stage, 0);
            if (leader) {
              if (crank == 0) mbar_expect_tx(full_bar + 8 * stage, 2 * Cfg::STAGE);
#pragma unroll
              for (int q = 0; q < NP; ++q)
                tma_load_2d_2sm(sb + q * Cfg::B_PLANE, &maps.b[q], fb, 0, kb * g.Cout + nb * BN + (int)crank * Cfg::B_ROWS);
            }
          } else {
            const uint32_t fb = full_bar + 8 * stage;
            if (leader) {
              mbar_expect_tx(fb, Cfg::STAGE);
#pragma unroll
              for (int q = 0; q < NP; ++q) tma_load_2d(sb + q * Cfg::B_PLANE, &maps.b[q], fb, 0, kb * g.Cout + nb * BN);
            }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        continue;
      }
      for (int kb = kb0; kb < kb1; ++kb) {
        const int j = kb / ncb, cb = kb - j * ncb;
        mbar_wait(empty_bar + 8 * stage, phase ^ 1);
        const uint32_t sa = smem_base + stage * Cfg::STAGE;
        const uint32_t sb = sa + NP * Cfg::A_PLANE;
        if constexpr (PAIR) {
          // both CTAs' bytes are counted on the LEADER's barrier (the leader issues the MMAs for the pair)
          const uint32_t fb = mapa_u32(full_bar + 8 * stage, 0);
          if (leader) {
            if (crank == 0) mbar_expect_tx(full_bar + 8 * stage, 2 * Cfg::STAGE);
#pragma unroll
            for (int q = 0; q < NP; ++q) tma_load_3d_2sm(sa + q * Cfg::A_PLANE, &maps.a[q], fb, cb * Cfg::BK, trow + j * g.dil, b);
#pragma unroll
            for (int q = 0; q < NP; ++q)
              tma_load_2d_2sm(sb + q * Cfg::B_PLANE, &maps.b[q], fb, cb * Cfg::BK, j * g.Cout + nb * BN + (int)crank * Cfg::B_ROWS);
          }
        } else {
          const uint32_t fb = full_bar + 8 * stage;
          if (leader) {
            mbar_expect_tx(fb, Cfg::STAGE);
#pragma unroll
            for (int q = 0; q < NP; ++q) tma_load_3d(sa + q * Cfg::A_PLANE, &maps.a[q], fb, cb * Cfg::BK, trow + j * g.dil, b);
#pragma unroll
            for (int q = 0; q < NP; ++q) tma_load_2d(sb + q * Cfg::B_PLANE, &maps.b[q], fb, cb * Cfg::BK, j * g.Cout + nb * BN);
          }
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (crank == 0) {   // ================= MMA issuer (the leader CTA issues for a pair) =================
      const uint32_t leader = elect_one() ? 1u : 0u;
      // instruction descriptor: D = f32, A / B = bf16 (1) or f16 (0), K-major, N >> 3, M >> 4
      const uint32_t ab_fmt = NP == 3 ? ((1u << 7) | (1u << 10)) : 0u;
      const uint32_t idesc = (1u << 4) | ab_fmt | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
      const uint64_t desc_base = umma_desc_kmajor<SWB>(0u);      // everything except the start address
      int stage = 0, phase = 0, it = 0;
      for (int item = worker; item < num_tiles; item += nworkers, ++it) {
        const int sp = item % g.splits;
        const int kb0 = (int)((int64_t)sp * num_k / g.splits), kb1 = (int)((int64_t)(sp + 1) * num_k / g.splits);
        const int as = it % NACC, aphase = (it / NACC) & 1;
        mbar_wait(tempty_bar + 8 * as, aphase ^ 1);        // the epilogue (of both CTAs) has drained this buffer
        tc_fence_after();
        const uint32_t d_main = tmem_base + as * (2 * BN);
        const uint32_t d_corr = d_main + BN;
        if constexpr (HALO && NP == 2) {
          // f16x2 halo form: per tap ONE asm block issues the k-steps' MMAs from two base descriptors (tc_tap_f16x2); the
          // A descriptor advances by dil rows per tap, the B descriptor follows the stage ring - a handful of uniform
          // instructions per tap instead of ~100
          const int ab = it % Cfg::A_BUFS, aph = (it / Cfg::A_BUFS) & 1;
          mbar_wait(afull_bar + 8 * ab, aph);
          uint64_t a_tap = desc_base | (uint64_t)((smem_a + ab * NP * Cfg::A_PLANE + (uint32_t)(kb0 * g.dil) * SWB) >> 4);
          const uint64_t a_step = (uint64_t)((uint32_t)(g.dil * SWB) >> 4);
          for (int kb = kb0; kb < kb1; ++kb) {          // kb == tap (one K-slab per tap)
            mbar_wait(full_bar + 8 * stage, phase);
            tc_fence_after();
            const uint64_t b_tap = desc_base | (uint64_t)((smem_base + stage * Cfg::STAGE) >> 4);
            tc_tap_f16x2<Cfg::BK / 16, PAIR>(d_main, d_corr, a_tap, b_tap, Cfg::A_PLANE >> 4, Cfg::B_PLANE >> 4, idesc,
                                             (kb == kb0) ? 0u : 1u, leader);
            a_tap += a_step;
            if constexpr (PAIR) {
              tc_commit_2sm_l(empty_bar + 8 * stage, leader);
              if (kb == kb1 - 1) {
                tc_commit_2sm_l(aempty_bar + 8 * ab, leader);       // the halo tiles of both CTAs are free once these MMAs retire
                tc_commit_2sm_l(tfull_bar + 8 * as, leader);
              }
            } else {
              tc_commit_l(empty_bar + 8 * stage, leader);
              if (kb == kb1 - 1) {
                tc_commit_l(aempty_bar + 8 * ab, leader);           // the halo tile is free once this tile's MMAs have retired
                tc_commit_l(tfull_bar + 8 * as, leader);
              }
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          continue;
        } else if constexpr (HALO) {
          const int ab = it % Cfg::A_BUFS, aph = (it / Cfg::A_BUFS) & 1;
          mbar_wait(afull_bar + 8 * ab, aph);
          for (int kb = kb0; kb < kb1; ++kb) {          // kb == tap (one K-slab per tap)
            mbar_wait(full_bar + 8 * stage, phase);
            tc_fence_after();
            // A: the halo tile shifted by kb * dil rows.  The swizzle is a function of the shared-memory ADDRESS bits (the
            // TMA wrote with them, the MMA reads with them), so a start address that is a whole number of rows into the
            // tile needs nothing else: measured on B200, every parity case passes with the descriptor's base-offset field
            // left at zero and fails with (addr >> 7) & 7 in it (gpurun call D, profiles/r2d_halo_form.md).
            const uint32_t a_addr = smem_a + ab * NP * Cfg::A_PLANE + (uint32_t)(kb * g.dil) * SWB;
            const uint32_t b_addr = smem_base + stage * Cfg::STAGE;
            const uint32_t first = (kb == kb0) ? 0u : 1u;
#pragma unroll
            for (int ks = 0; ks < Cfg::BK / 16; ++ks) {
              const uint32_t aa = a_addr + ks * 32, bb = b_addr + ks * 32;
              const uint64_t a1 = umma_desc_shifted(desc_base, aa), a2 = umma_desc_shifted(desc_base, aa + Cfg::A_PLANE);
              const uint64_t b1 = desc_base | (uint64_t)((bb >> 4) & 0x3FFF), b2 = desc_base | (uint64_t)(((bb + Cfg::B_PLANE) >> 4) & 0x3FFF);
              const uint32_t f = (ks == 0) ? first : 1u;
              if constexpr (NP == 2) {
                if constexpr (PAIR) {
                  tc_mma_2sm_l(d_corr, a1, b2, idesc, f, leader);
                  tc_mma_2sm_l(d_corr, a2, b1, idesc, 1u, leader);
                  tc_mma_2sm_l(d_main, a1, b1, idesc, f, leader);
                } else {
                  tc_mma_l(d_corr, a1, b2, idesc, f, leader);
                  tc_mma_l(d_corr, a2, b1, idesc, 1u, leader);
                  tc_mma_l(d_main, a1, b1, idesc, f, leader);
                }
              } else {
                const uint64_t a3 = umma_desc_shifted(desc_base, aa + 2 * Cfg::A_PLANE);
                const uint64_t b3 = desc_base | (uint64_t)(((bb + 2 * Cfg::B_PLANE) >> 4) & 0x3FFF);
                if constexpr (PAIR) {
                  tc_mma_2sm_l(d_corr, a2, b2, idesc, f, leader);
                  tc_mma_2sm_l(d_corr, a1, b3, idesc, 1u, leader);
                  tc_mma_2sm_l(d_corr, a3, b1, idesc, 1u, leader);
                  tc_mma_2sm_l(d_corr, a1, b2, idesc, 1u, leader);
                  tc_mma_2sm_l(d_corr, a2, b1, idesc, 1u, leader);
                  tc_mma_2sm_l(d_main, a1, b1, idesc, f, leader);
                } else {
                  tc_mma_l(d_corr, a2, b2, idesc, f, leader);
                  tc_mma_l(d_corr, a1, b3, idesc, 1u, leader);
                  tc_mma_l(d_corr, a3, b1, idesc, 1u, leader);
                  tc_mma_l(d_corr, a1, b2, idesc, 1u, leader);
                  tc_mma_l(d_corr, a2, b1, idesc, 1u, leader);
                  tc_mma_l(d_main, a1, b1, idesc, f, leader);
                }
              }
            }
            if constexpr (PAIR) {
              tc_commit_2sm_l(empty_bar + 8 * stage, leader);
              if (kb == kb1 - 1) {
                tc_commit_2sm_l(aempty_bar + 8 * ab, leader);       // the halo tiles of both CTAs are free once these MMAs retire
                tc_commit_2sm_l(tfull_bar + 8 * as, leader);
              }
            } else {
              tc_commit_l(empty_bar + 8 * stage, leader);
              if (kb == kb1 - 1) {
                tc_commit_l(aempty_bar + 8 * ab, leader);           // the halo tile is free once this tile's MMAs have retired
                tc_commit_l(tfull_bar + 8 * as, leader);
              }
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
          continue;
        }
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar + 8 * stage, phase);
          tc_fence_after();
          // descriptors: constant high word, low word = (smem address >> 4); planes / k-steps are plain adds
          const uint64_t a0 = desc_base | (uint64_t)(((smem_base + stage * Cfg::STAGE) >> 4) & 0x3FFF);
          const uint64_t b0 = a0 + (NP * Cfg::A_PLANE >> 4);
          const uint32_t first = (kb == kb0) ? 0u : 1u;
#pragma unroll
          for (int ks = 0; ks < Cfg::BK / 16; ++ks) {
            const uint64_t a1 = a0 + 2 * ks, a2 = a1 + (Cfg::A_PLANE >> 4), a3 = a2 + (Cfg::A_PLANE >> 4);
            const uint64_t b1 = b0 + 2 * ks, b2 = b1 + (Cfg::B_PLANE >> 4), b3 = b2 + (Cfg::B_PLANE >> 4);
            const uint32_t f = (ks == 0) ? first : 1u;
            if constexpr (NP == 2) {
              (void)a3; (void)b3;
              if constexpr (PAIR) {
                tc_mma_2sm_l(d_corr, a1, b2, idesc, f, leader);    // x1 w2'
                tc_mma_2sm_l(d_corr, a2, b1, idesc, 1u, leader);   // x2' w1
                tc_mma_2sm_l(d_main, a1, b1, idesc, f, leader);    // x1 w1
              } else {
                tc_mma_l(d_corr, a1, b2, idesc, f, leader);
                tc_mma_l(d_corr, a2, b1, idesc, 1u, leader);
                tc_mma_l(d_main, a1, b1, idesc, f, leader);
              }
            } else if constexpr (PAIR) {
              tc_mma_2sm_l(d_corr, a2, b2, idesc, f, leader);
              tc_mma_2sm_l(d_corr, a1, b3, idesc, 1u, leader);
              tc_mma_2sm_l(d_corr, a3, b1, idesc, 1u, leader);
              tc_mma_2sm_l(d_corr, a1, b2, idesc, 1u, leader);
              tc_mma_2sm_l(d_corr, a2, b1, idesc, 1u, leader);
              tc_mma_2sm_l(d_main, a1, b1, idesc, f, leader);
            } else {
              tc_mma_l(d_corr, a2, b2, idesc, f, leader);      // x2 w2   (smallest terms first)
              tc_mma_l(d_corr, a1, b3, idesc, 1u, leader);     // x1 w3
              tc_mma_l(d_corr, a3, b1, idesc, 1u, leader);     // x3 w1
              tc_mma_l(d_corr, a1, b2, idesc, 1u, leader);     // x1 w2
              tc_mma_l(d_corr, a2, b1, idesc, 1u, leader);     // x2 w1
              tc_mma_l(d_main, a1, b1, idesc, f, leader);      // x1 w1
            }
          }
          if constexpr (PAIR) {
            tc_commit_2sm_l(empty_bar + 8 * stage, leader);          // frees the stage in both CTAs
            if (kb == kb1 - 1) tc_commit_2sm_l(tfull_bar + 8 * as, leader);
          } else {
            tc_commit_l(empty_bar + 8 * stage, leader);
            if (kb == kb1 - 1) tc_commit_l(tfull_bar + 8 * as, leader);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue: 8 warps, two per TMEM lane quarter, 16-column units =================
    // (the small-channel convs are epilogue-bound: per output element there is more CUDA-core work than
    //  tensor-pipe work, so the epilogue gets as many warps as the register file allows - and its per-tile
    //  integer work is kept small: the tile index is advanced in mixed radix instead of being re-divided, every
    //  global address is a per-tile base plus unit / row steps, and the halo form (one K split, no
    //  transposed-conv shift) drops those paths at compile time)
    constexpr float CS = NP == 2 ? F16X2_INV_SCALE : 1.0f;   // weight of the correction accumulator (exact: a power of two)
    const int ew = warp - 4;                      // 0..7
    const int q = ew & 3;                         // == warp % 4: the TMEM lane quarter this warp may read
    const int half = ew >> 2;                     // which 16-column units of a tile this warp owns
    const int chunk = lane & 3, rsub = lane >> 2;
    const int splits = HALO ? 1 : g.splits;
    const int64_t out_shift = HALO ? (int64_t)0 : g.out_shift;
    const bool partial_out = splits > 1;          // raw partial sums; bias / activation / residual run in the reduction kernel
    const bool has_bias = g.bias != nullptr && !partial_out;
    const bool has_res = g.res != nullptr && out_shift == 0 && !partial_out;
    const bool has_acc = g.accumulate != 0 && out_shift == 0 && !partial_out;
    const bool has_y = g.y != nullptr, has_op = g.op != nullptr;
    const int64_t ystep = 8 * (int64_t)g.ldy, rstep = 8 * (int64_t)g.ldr, ostep = 8 * (int64_t)g.op_ld;
    const int64_t pstep = 8 * (int64_t)g.Cout;
    // work item -> (K split, column block, row block, batch item), walked with stride nworkers
    int sp, nb, tb, b, d_sp, d_nb, d_tb, d_b;
    {
      int c = worker / splits;
      sp = worker - c * splits;
      nb = c % num_n; c /= num_n;
      tb = c % num_t; b = c / num_t;
      c = nworkers / splits;
      d_sp = nworkers - c * splits;
      d_nb = c % num_n; c /= num_n;
      d_tb = c % num_t; d_b = c / num_t;
    }
    // Each unit = this warp's 32 rows x 16 columns.  The accumulators arrive row-per-lane (TMEM lane == row);
    // writing them out like that would make every global instruction touch 32 different lines, so the unit
    // is transposed through a padded shared buffer and ALL global traffic of the epilogue (y, residual,
    // accumulate, operand planes) is issued as 8 rows x 64 contiguous bytes per instruction.
    float* stg = epi_stage + ew * (32 * 20);
    int it = 0;
    for (int item = worker; item < num_tiles; item += nworkers, ++it) {
      const int as = it % NACC, aphase = (it / NACC) & 1;
      const int t0 = tb * BM + (int)crank * 128 + q * 32 + rsub;          // this lane's rows: t0 + 8 i
      const int nbase = nb * BN + chunk * 4;
      const int64_t yo = (int64_t)t0 * g.ldy + nbase;                      // within batch item b
      const int64_t yb = (int64_t)b * g.y_sb;
      const int64_t ro = (int64_t)b * g.res_sb + (int64_t)t0 * g.ldr + nbase;
      const int64_t oo = ((int64_t)b * g.op_tp + g.op_hl + t0) * g.op_ld + nbase;
      const int64_t po = (((int64_t)sp * g.B + b) * g.T + t0) * g.Cout + nbase;
      bool waited = false;      // the accumulator wait is deferred until the unit's global loads are in flight
#pragma unroll 1
      for (int u = half; u < BN / 16; u += 2) {
        const int n = nbase + u * 16;
        const bool ncol = n < g.Cout;                 // Cout % 4 == 0: a 4-wide chunk is all-in or all-out
        float4 bvec = make_float4(0.f, 0.f, 0.f, 0.f);
        if (has_bias && ncol) bvec = __ldg(reinterpret_cast<const float4*>(g.bias + n));
        float4 rv[4], ov[4];
        bool ok[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          ok[i] = ncol && (t0 + 8 * i) < g.T;
          rv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          ov[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (has_res && ok[i]) rv[i] = *reinterpret_cast<const float4*>(g.res + ro + i * rstep + u * 16);
          if (has_acc && ok[i]) ov[i] = *reinterpret_cast<const float4*>(g.y + yb + yo + i * ystep + u * 16);
        }
        if (!waited) {
          mbar_wait(tfull_bar + 8 * as, aphase);
          tc_fence_after();
          waited = true;
        }
        uint32_t r[16], rc[16];
        const uint32_t ta = tmem_base + as * (2 * BN) + u * 16 + ((uint32_t)(q * 32) << 16);
        tmem_ld16(ta, r);
        tmem_ld16(ta + BN, rc);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<float4*>(stg + lane * 20 + 4 * j) =
              make_float4(fmaf(__uint_as_float(rc[4 * j + 0]), CS, __uint_as_float(r[4 * j + 0])),
                          fmaf(__uint_as_float(rc[4 * j + 1]), CS, __uint_as_float(r[4 * j + 1])),
                          fmaf(__uint_as_float(rc[4 * j + 2]), CS, __uint_as_float(r[4 * j + 2])),
                          fmaf(__uint_as_float(rc[4 * j + 3]), CS, __uint_as_float(r[4 * j + 3])));
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (!ok[i]) continue;
          const float4 a4 = *reinterpret_cast<const float4*>(stg + (i * 8 + rsub) * 20 + chunk * 4);
          if (partial_out) {
            *reinterpret_cast<float4*>(g.partial + po + i * pstep + u * 16) = a4;
            continue;
          }
          float v[4] = {a4.x + bvec.x, a4.y + bvec.y, a4.z + bvec.z, a4.w + bvec.w};
          if (g.post_act != MTTS_ACT_NONE) {
#pragma unroll
            for (int e = 0; e < 4; ++e) v[e] = act_apply(v[e], g.post_act, g.post_slope);
          }
          v[0] = (v[0] + rv[i].x) * g.out_scale + ov[i].x;
          v[1] = (v[1] + rv[i].y) * g.out_scale + ov[i].y;
          v[2] = (v[2] + rv[i].z) * g.out_scale + ov[i].z;
          v[3] = (v[3] + rv[i].w) * g.out_scale + ov[i].w;
          if (has_y) {
            const int64_t flat = yo + i * ystep + u * 16 + out_shift;      // out_shift % 4 == 0: all-in or all-out
            if (HALO || (flat >= 0 && flat + 4 <= g.ybe))
              *reinterpret_cast<float4*>(g.y + yb + flat) = make_float4(v[0], v[1], v[2], v[3]);
          }
          if (has_op) {
            if (g.op_act != MTTS_ACT_NONE) {
#pragma unroll
              for (int e = 0; e < 4; ++e) v[e] = act_apply(v[e], g.op_act, g.op_slope);
            }
            store_planes4(g.op, g.op_stride, oo + i * ostep + u * 16, v, NP == 2 ? MTTS_TC_F16X2 : MTTS_TC_BF16X3, g.ovf);
          }
        }
        __syncwarp();   // the staging buffer is reused by the next unit
      }
      if (!waited) {
        mbar_wait(tfull_bar + 8 * as, aphase);
        tc_fence_after();
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (PAIR) mbar_arrive_cluster(mapa_u32(tempty_bar + 8 * as, 0));     // the leader's MMA issuer waits
        else mbar_arrive(tempty_bar + 8 * as);
      }
      // next work item: (sp, nb, tb, b) += the stride's digits, with carries
      sp += d_sp;
      int carry = sp >= splits;
      sp -= carry ? splits : 0;
      nb += d_nb + carry;
      carry = nb >= num_n;
      nb -= carry ? num_n : 0;
      tb += d_tb + carry;
      carry = tb >= num_t;
      tb -= carry ? num_t : 0;
      b += d_b + carry;
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync_all();      // no CTA exits (or frees TMEM) while its peer still reads its memory
  if (warp == 2) {
    tc_fence_after();
    if constexpr (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
  }
}

// split-K reduction: sums the partial tiles in a FIXED order (bit-reproducible) and applies the tap-GEMM epilogue
// (bias -> activation -> residual -> scale -> accumulate -> fp32 and/or bf16x3 plane store)
__global__ void __launch_bounds__(256)
tc_splitk_reduce_kernel(const ConvTcArgs g, int64_t total4) {
  pdl_entry();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int c4 = g.Cout / 4;
  const int n = (int)(i % c4) * 4;
  const int64_t row = i / c4;                 // b * T + t
  const int b = (int)(row / g.T), tt = (int)(row - (int64_t)b * g.T);
  const int64_t stride = (int64_t)g.B * g.T * g.Cout;
  float4 a = *reinterpret_cast<const float4*>(g.partial + row * g.Cout + n);
  for (int sp = 1; sp < g.splits; ++sp) {
    const float4 q = *reinterpret_cast<const float4*>(g.partial + sp * stride + row * g.Cout + n);
    a.x += q.x; a.y += q.y; a.z += q.z; a.w += q.w;
  }
  float v[4] = {a.x, a.y, a.z, a.w};
  if (g.bias) {
    const float4 bv = __ldg(reinterpret_cast<const float4*>(g.bias + n));
    v[0] += bv.x; v[1] += bv.y; v[2] += bv.z; v[3] += bv.w;
  }
  if (g.post_act != MTTS_ACT_NONE) {
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = act_apply(v[e], g.post_act, g.post_slope);
  }
  float4 rv = make_float4(0.f, 0.f, 0.f, 0.f), ov = rv;
  if (g.res) rv = *reinterpret_cast<const float4*>(g.res + (int64_t)b * g.res_sb + (int64_t)tt * g.ldr + n);
  if (g.accumulate) ov = *reinterpret_cast<const float4*>(g.y + (int64_t)b * g.y_sb + (int64_t)tt * g.ldy + n);
  v[0] = (v[0] + rv.x) * g.out_scale + ov.x;
  v[1] = (v[1] + rv.y) * g.out_scale + ov.y;
  v[2] = (v[2] + rv.z) * g.out_scale + ov.z;
  v[3] = (v[3] + rv.w) * g.out_scale + ov.w;
  if (g.y) *reinterpret_cast<float4*>(g.y + (int64_t)b * g.y_sb + (int64_t)tt * g.ldy + n) = make_float4(v[0], v[1], v[2], v[3]);
  if (g.op) {
    if (g.op_act != MTTS_ACT_NONE) {
#pragma unroll
      for (int e = 0; e < 4; ++e) v[e] = act_apply(v[e], g.op_act, g.op_slope);
    }
    store_planes4(g.op, g.op_stride, ((int64_t)b * g.op_tp + g.op_hl + tt) * g.op_ld + n, v, g.fmt, g.ovf);
  }
}

// split-K reduction + LayerNorm of the finished rows (one warp per row, Cout = 128 * NV): the row is reduced exactly like
// tc_splitk_reduce_kernel does (same order of the partial sums, bias -> activation -> residual -> scale -> accumulate), stored
// as fp32, and - still in registers - normalised exactly like layernorm_reg_kernel (ops.cu) and written as operand planes.
// Bit-identical to the two separate launches it replaces.
template <int NV>
__global__ void __launch_bounds__(256)
tc_splitk_reduce_ln_kernel(const ConvTcArgs g, const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                           const PlanesOut po) {
  pdl_entry();
  constexpr int C = 128 * NV;
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);      // b * T + t
  if (row >= (int64_t)g.B * g.T) return;
  const int b = (int)(row / g.T), tt = (int)(row - (int64_t)b * g.T);
  const int64_t stride = (int64_t)g.B * g.T * C;
  float4 v[NV];
  // partial sums: split 0, then + split 1, + split 2 ... per element (the order of tc_splitk_reduce_kernel); the NV loads of
  // one split are independent and in flight together
  const float* pr = g.partial + row * C + lane * 4;
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = *reinterpret_cast<const float4*>(pr + i * 128);
  for (int sp = 1; sp < g.splits; ++sp) {
    float4 q[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) q[i] = *reinterpret_cast<const float4*>(pr + sp * stride + i * 128);
#pragma unroll
    for (int i = 0; i < NV; ++i) { v[i].x += q[i].x; v[i].y += q[i].y; v[i].z += q[i].z; v[i].w += q[i].w; }
  }
  {
    float4 bvv[NV], rvv[NV], ovv[NV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int n = i * 128 + lane * 4;
      bvv[i] = g.bias ? __ldg(reinterpret_cast<const float4*>(g.bias + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
      rvv[i] = g.res ? *reinterpret_cast<const float4*>(g.res + (int64_t)b * g.res_sb + (int64_t)tt * g.ldr + n) : make_float4(0.f, 0.f, 0.f, 0.f);
      ovv[i] = g.accumulate ? *reinterpret_cast<const float4*>(g.y + (int64_t)b * g.y_sb + (int64_t)tt * g.ldy + n) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int n = i * 128 + lane * 4;
      float w[4] = {v[i].x, v[i].y, v[i].z, v[i].w};
      if (g.bias) { w[0] += bvv[i].x; w[1] += bvv[i].y; w[2] += bvv[i].z; w[3] += bvv[i].w; }
      if (g.post_act != MTTS_ACT_NONE) {
#pragma unroll
        for (int e = 0; e < 4; ++e) w[e] = act_apply(w[e], g.post_act, g.post_slope);
      }
      v[i] = make_float4((w[0] + rvv[i].x) * g.out_scale + ovv[i].x, (w[1] + rvv[i].y) * g.out_scale + ovv[i].y,
                         (w[2] + rvv[i].z) * g.out_scale + ovv[i].z, (w[3] + rvv[i].w) * g.out_scale + ovv[i].w);
      *reinterpret_cast<float4*>(g.y + (int64_t)b * g.y_sb + (int64_t)tt * g.ldy + n) = v[i];
    }
  }
  // ---- LayerNorm of the row (the arithmetic of layernorm_reg_kernel, operation for operation)
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float a = v[i].x - mean, bb = v[i].y - mean, d = v[i].z - mean, e = v[i].w - mean;
    q += (a * a + bb * bb) + (d * d + e * e);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)C + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 bt = __ldg(reinterpret_cast<const float4*>(beta + c));
    float o[4] = {(v[i].x - mean) * rstd * gm.x + bt.x, (v[i].y - mean) * rstd * gm.y + bt.y,
                  (v[i].z - mean) * rstd * gm.z + bt.z, (v[i].w - mean) * rstd * gm.w + bt.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) o[e] = act_apply(o[e], po.act, po.slope);
    store_planes4(po.p, po.stride, row * po.ld + c, o, po.fmt, po.ovf);
  }
}

// fp32 (B,T,C) -> operand planes (B, Tp = T + hl + hr, C): padding materialised, pre-activation applied
__global__ void __launch_bounds__(256)
split_pad_kernel(const float* __restrict__ x, int64_t x_sb, int ldx, int T, int C, int hl, int Tp, int pad_mode,
                 int pre_act, float slope, __nv_bfloat16* __restrict__ planes, int64_t plane_stride,
                 int64_t total4, int fmt, int32_t* ovf) {
  pdl_entry();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total4) return;
  const int cq = C >> 2;
  const int c = (int)(i % cq) * 4;
  const int64_t bu = i / cq;
  const int u = (int)(bu % Tp);
  const int b = (int)(bu / Tp);
  int ti = u - hl;
  if (ti < 0 || ti >= T) {
    if (pad_mode == MTTS_PAD_ZERO) ti = -1;
    else if (pad_mode == MTTS_PAD_REPLICATE) ti = ti < 0 ? 0 : T - 1;
    else {
      if (ti < 0) ti = -ti;
      if (ti >= T) ti = 2 * (T - 1) - ti;
      if (ti < 0 || ti >= T) ti = -1;
    }
  }
  float f[4] = {0.f, 0.f, 0.f, 0.f};
  if (ti >= 0) {
    const float4 v = *reinterpret_cast<const float4*>(x + (int64_t)b * x_sb + (int64_t)ti * ldx + c);
    f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) f[e] = act_apply(f[e], pre_act, slope);
  store_planes4(planes, plane_stride, ((int64_t)b * Tp + u) * C + c, f, fmt, ovf);
}

// Materialise the padding rows of plane buffers whose interior rows were written by a producer epilogue:
// planes (3, B, Tp, C) bf16 with hl leading halo rows; reflect / replicate / zero about the T interior rows.
__global__ void __launch_bounds__(256)
halo_fill_kernel(__nv_bfloat16* __restrict__ planes, int64_t plane_stride, int T, int C, int hl, int Tp, int pad_mode) {
  pdl_entry();
  const int b = blockIdx.y, q = blockIdx.z;
  const int nh = Tp - T;                     // halo rows in total (hl leading, the rest trailing)
  const int c8 = C / 8;                      // 16-byte chunks per row
  __nv_bfloat16* base = planes + q * plane_stride + (int64_t)b * Tp * C;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nh * c8; i += gridDim.x * blockDim.x) {
    const int hr = i / c8, ch = i - hr * c8;
    const int u = hr < hl ? hr : T + hr;     // padded row index of this halo row
    int ti = u - hl;
    if (pad_mode == MTTS_PAD_REPLICATE) ti = ti < 0 ? 0 : T - 1;
    else if (pad_mode == MTTS_PAD_REFLECT) {
      if (ti < 0) ti = -ti;
      if (ti >= T) ti = 2 * (T - 1) - ti;
      if (ti < 0 || ti >= T) ti = -1;
    } else ti = -1;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (ti >= 0) v = *reinterpret_cast<const uint4*>(base + (int64_t)(hl + ti) * C + ch * 8);
    *reinterpret_cast<uint4*>(base + (int64_t)u * C + ch * 8) = v;
  }
}

int halo_fill(void* planes_base, int B, int T, int C, int hl, int hr, int pad_mode, cudaStream_t st) {
  MTTS_REQUIRE(planes_base && C % 8 == 0 && hl >= 0 && hr >= 0, "bad arguments");
  if (hl + hr == 0 || B <= 0) return 0;
  __nv_bfloat16* planes = reinterpret_cast<__nv_bfloat16*>((((uintptr_t)planes_base) + 1023) & ~(uintptr_t)1023);
  const int Tp = T + hl + hr;
  const int64_t plane_stride = (int64_t)B * Tp * C;
  const int work = (hl + hr) * (C / 8);
  dim3 grid((unsigned)cdiv64(work, 256), (unsigned)B, 3);
  launch_k(halo_fill_kernel, grid, 256, 0, st, planes, plane_stride, T, C, hl, Tp, pad_mode);
  MTTS_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------ host
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_enc = nullptr;
static std::mutex g_ctc_mu;          // guards g_enc, the descriptor cache and the per-device table (not the launches)

// per-device state: SM count, which kernel instantiations have had their shared-memory attribute raised (the attribute
// is per device), and the caller-registered f16 range flag
constexpr int MAX_DEV = 64;
struct DevState { int sms = 0; uint32_t attr_done = 0; int32_t* ovf = nullptr; };
static DevState g_dev[MAX_DEV];

int cur_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev < 0 || dev >= MAX_DEV ? 0 : dev;
}
int cur_device_sms() {
  const int dev = cur_device();
  if (!g_dev[dev].sms) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    g_dev[dev].sms = n > 0 ? n : 1;
  }
  return g_dev[dev].sms;
}
int32_t* tc_ovf_ptr() { return g_dev[cur_device()].ovf; }
int tc_overflow_bind(int32_t* flag) {
  g_dev[cur_device()].ovf = flag;
  return 0;
}

struct CMapKey {
  const void* p; uint64_t d0, d1, d2, b0, b1; int swb, dt;
  bool operator==(const CMapKey& o) const {
    return p == o.p && d0 == o.d0 && d1 == o.d1 && d2 == o.d2 && b0 == o.b0 && b1 == o.b1 && swb == o.swb && dt == o.dt;
  }
};
struct CMapKeyHash {
  size_t operator()(const CMapKey& k) const {
    uint64_t h = (uint64_t)k.p;
    h = h * 0x9E3779B97F4A7C15ull + k.d0; h = h * 0x9E3779B97F4A7C15ull + k.d1; h = h * 0x9E3779B97F4A7C15ull + k.d2;
    h = h * 0x9E3779B97F4A7C15ull + k.b0 * 131 + k.b1 * 7 + k.swb + 1000 * k.dt;
    return (size_t)h;
  }
};
// Descriptor cache: keyed by (pointer, dims, box, swizzle, dtype); a descriptor holds nothing but those, so a stale entry
// for a freed-and-reused address is still correct.  Bounded: when full, the older half (by insertion order) is dropped.
static std::unordered_map<CMapKey, std::pair<CUtensorMap, uint64_t>, CMapKeyHash> g_cmaps;
static uint64_t g_cmap_tick = 0;
constexpr size_t CMAP_CAP = 16384;

static int ctc_init_locked() {
  if (g_enc) return 0;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn)
    return fail(MTTS_ERR_CUDA, "%s: cuTensorMapEncodeTiled not available", "conv_tc");
  g_enc = (EncodeTiledFn)fn;
  return 0;
}

// 2-byte-element tensor (d2, d1, d0) row-major, box (1, b1, b0), SWB-byte swizzle; rank 2 when d2 == 0
static int cmap_get(const void* p, uint64_t d0, uint64_t d1, uint64_t d2, uint32_t b0, uint32_t b1, int swb, int fmt,
                    CUtensorMap* out) {
  std::lock_guard<std::mutex> lk(g_ctc_mu);
  MTTS_TRY(ctc_init_locked());
  CMapKey key{p, d0, d1, d2, b0, b1, swb, fmt};
  auto itf = g_cmaps.find(key);
  if (itf != g_cmaps.end()) { *out = itf->second.first; return 0; }
  const int rank = d2 ? 3 : 2;
  cuuint64_t dims[3] = {d0, d1, d2 ? d2 : 1};
  cuuint64_t strides[2] = {d0 * 2, d0 * d1 * 2};
  cuuint32_t box[3] = {b0, b1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMap m;
  CUresult r = g_enc(&m, fmt == MTTS_TC_F16X2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank,
                     const_cast<void*>(p), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     swb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(MTTS_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed: %lld", "conv_tc", (long long)r);
  if (g_cmaps.size() >= CMAP_CAP) {
    const uint64_t cut = g_cmap_tick - CMAP_CAP / 2;
    for (auto it = g_cmaps.begin(); it != g_cmaps.end();) it = it->second.second < cut ? g_cmaps.erase(it) : ++it;
  }
  g_cmaps[key] = {m, g_cmap_tick++};
  *out = m;
  return 0;
}

template <int BN, int SWB, int PAIR, int NP, int HALO = 0>
static int conv_tc_launch(const ConvTcMaps& maps, const ConvTcArgs& a, cudaStream_t st) {
  using Cfg = ConvTcCfg<BN, SWB, PAIR, NP, HALO>;
  // one bit per instantiation in the per-device table (the max-dynamic-shared-memory attribute is per device)
  constexpr int slot = HALO ? 24 + (BN == 64 ? 0 : 1) + 2 * (NP == 3 ? 0 : 1) + 4 * PAIR
                            : (BN == 128 ? 0 : BN == 64 ? 1 : 2) + 3 * (SWB == 128 ? 0 : 1) + 6 * PAIR + 12 * (NP == 3 ? 0 : 1);
  static_assert(slot < 32, "attribute slots");
  const int dev = cur_device();
  const int sms = cur_device_sms();
  if (!(g_dev[dev].attr_done & (1u << slot))) {
    std::lock_guard<std::mutex> lk(g_ctc_mu);
    cudaError_t e =
        cudaFuncSetAttribute(conv_tc_kernel<BN, SWB, PAIR, NP, HALO>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
    if (e != cudaSuccess) return fail(MTTS_ERR_CUDA, "%s: cudaFuncSetAttribute failed: %lld", "conv_tc", (long long)e);
    g_dev[dev].attr_done |= (1u << slot);
  }
  const int64_t tiles = (int64_t)a.B * cdiv64(a.T, PAIR ? 256 : 128) * cdiv64(a.Cout, BN) * a.splits;
  if (PAIR) {
    const int64_t pairs = tiles < sms / 2 ? tiles : sms / 2;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(2 * pairs));
    cfg.blockDim = dim3(384);
    cfg.dynamicSmemBytes = Cfg::SMEM;
    cfg.stream = st;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl_enabled() ? 2 : 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, conv_tc_kernel<BN, SWB, PAIR, NP, HALO>, maps, a);
    if (e != cudaSuccess) return fail(MTTS_ERR_CUDA, "%s: cluster launch failed: %lld", "conv_tc", (long long)e);
  } else {
    const int grid = (int)(tiles < sms ? tiles : sms);
    launch_k(conv_tc_kernel<BN, SWB, PAIR, NP, HALO>, grid, 384, Cfg::SMEM, st, maps, a);
  }
  MTTS_CHECK_LAUNCH();
  return 0;
}

template <int NP>
static int conv_tc_dispatch(const ConvTcMaps& maps, const ConvTcArgs& a, int BN, int SWB, bool pair, cudaStream_t st) {
  if (pair) return conv_tc_launch<128, 128, 1, NP>(maps, a, st);
  if (SWB == 64) return conv_tc_launch<32, 64, 0, NP>(maps, a, st);
  if (BN == 128) return conv_tc_launch<128, 128, 0, NP>(maps, a, st);
  if (BN == 64) return conv_tc_launch<64, 128, 0, NP>(maps, a, st);
  return conv_tc_launch<32, 128, 0, NP>(maps, a, st);
}

bool conv_tc_eligible(const mtts_conv_params& p) {
  if (!p.w_tc || !p.tc_scratch) return false;
  if (p.tc_fmt != MTTS_TC_BF16X3 && p.tc_fmt != MTTS_TC_F16X2) return false;
  if (p.stride != 1 || p.in_lens) return false;
  if (p.out_shift != 0 && (p.out_shift % 4 != 0 || p.y_batch_elems % 4 != 0 || p.res || p.accumulate || p.tc_out_planes || !p.y))
    return false;
  if (p.Cin % 8 != 0 || p.Cin < 32) return false;
  if (!p.tc_presplit && (p.ldx % 4 != 0 || (p.x_batch_stride % 4) != 0 || (((uintptr_t)p.x) & 15) != 0)) return false;
  if (!(p.Cout == 32 || p.Cout == 64 || (p.Cout >= 128 && p.Cout % 32 == 0))) return false;
  if (p.Cin < 64 && p.Cout != 32) return false;          // the SWB=64 variant is instantiated for BN=32 only
  if (p.y && (p.ldy % 4 != 0 || p.y_batch_stride % 4 != 0 || (((uintptr_t)p.y) & 15) != 0)) return false;
  if (!p.y && (!p.tc_out_planes || p.accumulate)) return false;
  if (p.tc_out_planes && (p.Cout % 32 != 0 || p.tc_out_ld % 4 != 0 || p.tc_out_plane_stride % 4 != 0)) return false;
  if (p.res && (p.ldr % 4 != 0 || p.res_batch_stride % 4 != 0 || (((uintptr_t)p.res) & 15) != 0)) return false;
  if (p.Tout != p.Tin + 2 * p.pad - p.dil * (p.k - 1)) return false;
  // tiny problems stay on the exact FFMA engine - except rows that already sit in a plane buffer of >= 128 rows (the last
  // rows of an AR step: one half-filled tile, K split across the SMs)
  if ((int64_t)p.B * p.Tout < ((p.tc_presplit && p.tc_rows_cap >= 128) ? 32 : 128)) return false;
  int64_t Tp = p.Tout + p.dil * (p.k - 1);
  if (p.tc_in_tp > 0 || p.tc_in_row0 != 0) {      // shared plane buffer: this conv's rows must lie inside it
    if (!p.tc_presplit || p.tc_rows_cap > 0 || p.tc_in_row0 < 0 || p.tc_in_tp < p.tc_in_row0 + Tp) return false;
    Tp = p.tc_in_tp;
  }
  int64_t rows = (int64_t)p.B * Tp;
  if (p.tc_rows_cap > 0) {
    if (p.k != 1 || p.B != 1 || p.tc_rows_cap < rows) return false;
    rows = p.tc_rows_cap;
  }
  return 3 * rows * p.Cin * 2 + 2048 <= p.tc_scratch_bytes;
}

// Split-K cost model (cycles per CTA): at most CTC_SPLITK_MAX splits, taken when the split walk plus its reduction costs less
// than CTC_SPLITK_MARGIN of the unsplit walk.  A reduction that REPLACES the LayerNorm launch that would follow anyway
// (tc_splitk_reduce_ln_kernel) is modelled at 2000 cycles instead of the plain reduction's 9000: that makes the out-projection /
// FF2 layers split up to steps 18 (PLM) / 24 (ADM), and every affected step got faster, PLM -0.4 ms, ADM -1.0 ms per decode
// (profiles/r3c_splitk_constants.log, r3d_lncost_curves.log)
constexpr int CTC_SPLITK_MAX = 8;
constexpr double CTC_SPLITK_MARGIN = 0.85;
constexpr double CTC_REDUCE_CYCLES = 9000.0, CTC_REDUCE_LN_CYCLES = 2000.0;

// The launch plan of one tap-GEMM: K-slab width, N-tile width, K splits, CTA pairing, halo form.  A pure function of the shape
// and the SM count, so the policy can be queried and tested without a GPU (mtts_tc_plan_query, tests/test_abi_and_host.py).
struct TcPlan { int SWB, BN, splits; bool pair, halo_form, halo_pair; };
static TcPlan tc_plan(int sms, const mtts_conv_params& p, int np, bool ln_rides) {
  const int halo = p.dil * (p.k - 1);
  const int SWB = p.Cin >= 64 ? 128 : 64;
  int BN = 32;
  int splits = 1;
  bool pair = false;
  // N-tile width.  Dense layers (k = 1): a persistent CTA walks ceil(tiles / SMs) tiles of nk K-slabs; a slab's MMAs cost 65
  // cycles each at N = 128 and 55 (the per-instruction floor) at N <= 64, so the width with the cheapest walk wins and ties go
  // to the narrower tile (under-filled grids are latency-bound: more SMs stream the weights).  The earlier rule - the widest
  // tile that still gives 80 % of the SMs a tile - ran e.g. the PLM FF2 layer of steps 19 ... 28 as 160 tiles of N = 64 on
  // 148 SMs, two waves, where 80 tiles of N = 128 take one: -0.25 ms per step there, -0.03 ms on ADM steps 25 ... 38
  // (profiles/r2tm_ar_curves.log).  Convolutions (k > 1) keep that fill rule: their grids are hundreds of waves deep and the
  // halo form wants BN == Cout.
  if (SWB == 128) {
    const int64_t mt = (int64_t)p.B * cdiv64(p.Tout, 128);
    const int cands[3] = {128, 64, 32};
    if (p.k == 1) {
      int64_t best = INT64_MAX;
      for (int i = 0; i < 3; ++i) {
        if (cands[i] > p.Cout) continue;
        const int64_t c = cdiv64(mt * cdiv64(p.Cout, cands[i]), sms) * (cands[i] == 128 ? 65 : 55);
        if (c <= best) { best = c; BN = cands[i]; }
      }
    } else {
      for (int i = 0; i < 3; ++i) {
        if (cands[i] > p.Cout) continue;
        BN = cands[i];
        if (mt * cdiv64(p.Cout, cands[i]) >= (int64_t)(sms * 4) / 5) break;
      }
    }
  }
  // split-K for dense layers with too few output tiles to fill the GPU (the early steps of the AR loops, the N = 1024
  // layers up to ~30 steps): narrow tiles would pay the 55-cycle minimum per MMA (tools/microbench/mma_floor.cu) on
  // every k-step, so K is split across CTAs at full tile width instead and a second kernel reduces the partials
  {
    const int64_t rows = (int64_t)p.B * p.Tout;
    const int64_t t128 = (int64_t)p.B * cdiv64(p.Tout, 128) * cdiv64(p.Cout, 128);
    const int nk = (p.Cin + 63) / 64;
    if (SWB == 128 && p.k == 1 && p.out_shift == 0 && p.tc_partial && p.Cout >= 128 && t128 < (int64_t)(sms * 4) / 5) {
      int sk = (int)(sms / t128);
      if (sk > CTC_SPLITK_MAX) sk = CTC_SPLITK_MAX;
      if (sk > nk / 2) sk = nk / 2;
      if (sk >= 2 && (int64_t)sk * rows * p.Cout * 4 <= p.tc_partial_bytes) {
        const int64_t tiles_bn = (int64_t)p.B * cdiv64(p.Tout, 128) * cdiv64(p.Cout, BN);
        const double waves = (double)cdiv64(tiles_bn, sms);
        const double mmas = 4.0 * (2 * np);                                                 // MMAs per 64-wide K-slab
        const double cost_now = waves * nk * mmas * (BN == 128 ? 65.0 : 55.0);                // cycles per CTA
        const double cost_split = (double)cdiv64(nk, sk) * mmas * 65.0 + (ln_rides ? CTC_REDUCE_LN_CYCLES : CTC_REDUCE_CYCLES);
        if (cost_split < CTC_SPLITK_MARGIN * cost_now) { splits = sk; BN = 128; }
      }
    }
  }
  // CTA pairs (cta_group::2): two SMs share one 256 x 128 tile; each stages its own 128 activation rows and HALF of the
  // weight tile, so a quarter fewer bytes cross L2 -> SM and a quarter fewer operand bytes are read from shared memory
  // per FLOP.  Measured (tools/bench_tc_shapes.py): +1..3 % on the dense layers, -5 % on the ragged-T convolutions
  // (256-row tiles waste more of the last tile), so pairs are used for k = 1 only.
  if (splits == 1 && BN == 128 && p.Cout % 128 == 0 && p.k == 1) {
    const int64_t t256 = (int64_t)p.B * cdiv64(p.Tout, 256) * (p.Cout / 128);
    const double eff128 = (double)p.Tout / (128.0 * cdiv64(p.Tout, 128)), eff256 = (double)p.Tout / (256.0 * cdiv64(p.Tout, 256));
    pair = t256 >= (int64_t)(sms / 2) * 4 / 5 && eff256 >= 0.9 * eff128;
  }
  // halo form: one K-slab per tap (Cin <= SWB / 2), the activation tile + halo fits the 192-row buffer
  const bool halo_form = !pair && splits == 1 && p.out_shift == 0 && p.k > 1 && p.Cin <= SWB / 2 &&
                         halo + 128 <= CTC_HALO_ROWS &&   // (the halo kernel's epilogue has no K-split / transposed-conv paths)
                         ((SWB == 64 && BN == 32) || (SWB == 128 && BN == 64)) && p.Cout == BN;
  // ... as a CTA pair: an N = 32 / 64 MMA costs 41 / 48 cycles whatever its M (128 or 256: 52 cycles, measured with
  // tools/microbench/mma_floor2.cu), and these layers issue k * Cin / 16 * 3 of them per tile, so one instruction per 256
  // rows nearly halves their tensor-pipe time.  Measured: C = 64, k = 7: 0.415 -> 0.358 ms; C = 32: 0.424 -> 0.453 ms (its
  // tiles are paced by the epilogue, not by MMA issue; four accumulator buffers instead of two change nothing either:
  // profiles/r2r_tc_shapes.log, r2s_stages_halo_pair_modes.log, r2t_nacc4_ab.log) - so pairs serve the C = 64 stage only
  bool halo_pair = false;
  if (halo_form && SWB == 128) {
    const int64_t t256 = (int64_t)p.B * cdiv64(p.Tout, 256);
    const double eff128 = (double)p.Tout / (128.0 * cdiv64(p.Tout, 128)), eff256 = (double)p.Tout / (256.0 * cdiv64(p.Tout, 256));
    halo_pair = t256 >= (int64_t)(sms / 2) * 2 && eff256 >= 0.9 * eff128;
  }
  TcPlan pl;
  pl.SWB = SWB; pl.BN = BN; pl.splits = splits; pl.pair = pair; pl.halo_form = halo_form; pl.halo_pair = halo_pair;
  return pl;
}

int conv_tc(const mtts_conv_params& p, cudaStream_t st, LnFuse* ln) {
  if (ln) ln->done = 0;
  const int sms = cur_device_sms();
  const int fmt = p.tc_fmt;
  const int np = fmt == MTTS_TC_F16X2 ? 2 : 3;
  int32_t* ovf = tc_ovf_ptr();
  const int halo = p.dil * (p.k - 1);
  const int hl = p.pad, Tp = p.Tout + halo;
  const int64_t Tp_map = p.tc_rows_cap > 0 ? p.tc_rows_cap : (p.tc_in_tp > 0 ? p.tc_in_tp : Tp);     // descriptor rows (>= Tp)
  __nv_bfloat16* planes = reinterpret_cast<__nv_bfloat16*>((((uintptr_t)p.tc_scratch) + 1023) & ~(uintptr_t)1023);
  const int64_t plane_stride = (int64_t)p.B * Tp_map * p.Cin;
  if (!p.tc_presplit) {
    const int64_t total4 = (int64_t)p.B * Tp * p.Cin / 4;
    launch_k(split_pad_kernel, (unsigned)cdiv64(total4, 256), 256, 0, st, p.x, p.x_batch_stride, p.ldx, p.Tin, p.Cin, hl, Tp,
                                                                   p.pad_mode, p.pre_act, p.pre_slope, planes, plane_stride,
                                                                   total4, fmt, ovf);
    MTTS_CHECK_LAUNCH();
  }
  // the reduction of a split launch can carry the LayerNorm the caller asked for when a row is 3 / 4 / 6 / 8 x 128 wide
  const bool ln_rides = ln && ln->po.p && p.y && !p.tc_out_planes && (p.Cout == 1024 || p.Cout == 768 || p.Cout == 512 || p.Cout == 384);
  const TcPlan pl = tc_plan(sms, p, np, ln_rides);
  const int SWB = pl.SWB, BN = pl.BN, splits = pl.splits;
  const bool pair = pl.pair, halo_form = pl.halo_form, halo_pair = pl.halo_pair;
  const int b_rows = (pair || halo_pair) ? BN / 2 : BN;
  ConvTcMaps maps;
  for (int q = 0; q < np; ++q) {
    MTTS_TRY(cmap_get(planes + q * plane_stride, (uint64_t)p.Cin, (uint64_t)Tp_map, (uint64_t)p.B, SWB / 2,
                      halo_form ? 128 + halo : 128, SWB, fmt, &maps.a[q]));
    MTTS_TRY(cmap_get((const __nv_bfloat16*)p.w_tc + (int64_t)q * p.k * p.Cout * p.Cin, (uint64_t)p.Cin,
                      (uint64_t)p.k * p.Cout, 0, SWB / 2, b_rows, SWB, fmt, &maps.b[q]));
  }
  if (np == 2) { maps.a[2] = maps.a[1]; maps.b[2] = maps.b[1]; }
  ConvTcArgs a;
  a.B = p.B; a.T = p.Tout; a.Cin = p.Cin; a.Cout = p.Cout; a.k = p.k; a.dil = p.dil;
  a.bias = p.bias; a.res = p.res; a.res_sb = p.res_batch_stride; a.ldr = p.ldr;
  a.y = p.y; a.y_sb = p.y_batch_stride; a.ldy = p.ldy;
  a.post_act = p.post_act; a.post_slope = p.post_slope; a.out_scale = p.out_scale; a.accumulate = p.accumulate;
  a.out_shift = p.out_shift; a.ybe = p.y_batch_elems ? p.y_batch_elems : (int64_t)p.Tout * p.ldy;
  a.op = reinterpret_cast<__nv_bfloat16*>(p.tc_out_planes); a.op_stride = p.tc_out_plane_stride; a.op_ld = p.tc_out_ld;
  a.op_tp = p.tc_out_tp; a.op_hl = p.tc_out_hl; a.op_act = p.tc_out_act; a.op_slope = p.tc_out_slope;
  a.splits = splits; a.partial = reinterpret_cast<float*>(p.tc_partial);
  a.fmt = fmt; a.ovf = ovf; a.row0 = p.tc_in_row0;
  if (halo_pair) return np == 2 ? conv_tc_launch<64, 128, 1, 2, 1>(maps, a, st) : conv_tc_launch<64, 128, 1, 3, 1>(maps, a, st);
  if (halo_form) {
    if (SWB == 64) return np == 2 ? conv_tc_launch<32, 64, 0, 2, 1>(maps, a, st) : conv_tc_launch<32, 64, 0, 3, 1>(maps, a, st);
    return np == 2 ? conv_tc_launch<64, 128, 0, 2, 1>(maps, a, st) : conv_tc_launch<64, 128, 0, 3, 1>(maps, a, st);
  }
  if (splits > 1) {
    MTTS_TRY(np == 2 ? (conv_tc_launch<128, 128, 0, 2>(maps, a, st)) : (conv_tc_launch<128, 128, 0, 3>(maps, a, st)));
    // the rows' LayerNorm rides on the reduction when the caller asked for it and a row is 3 / 4 / 6 / 8 x 128 wide
    if (ln && ln->po.p && a.y && !a.op && a.out_shift == 0 && (p.Cout == 1024 || p.Cout == 768 || p.Cout == 512 || p.Cout == 384) &&
        p.ldy % 4 == 0 && ln->po.ld % 4 == 0 && ln->po.stride % 4 == 0) {
      const unsigned grid = (unsigned)cdiv64((int64_t)p.B * p.Tout, 4);      // 4 rows (warps) per CTA
      if (p.Cout == 1024) launch_k(tc_splitk_reduce_ln_kernel<8>, grid, 128, 0, st, a, ln->gamma, ln->beta, ln->eps, ln->po);
      else if (p.Cout == 768) launch_k(tc_splitk_reduce_ln_kernel<6>, grid, 128, 0, st, a, ln->gamma, ln->beta, ln->eps, ln->po);
      else if (p.Cout == 512) launch_k(tc_splitk_reduce_ln_kernel<4>, grid, 128, 0, st, a, ln->gamma, ln->beta, ln->eps, ln->po);
      else launch_k(tc_splitk_reduce_ln_kernel<3>, grid, 128, 0, st, a, ln->gamma, ln->beta, ln->eps, ln->po);
      MTTS_CHECK_LAUNCH();
      ln->done = 1;
      return 0;
    }
    const int64_t total4 = (int64_t)p.B * p.Tout * p.Cout / 4;
    launch_k(tc_splitk_reduce_kernel, (unsigned)cdiv64(total4, 256), 256, 0, st, a, total4);
    MTTS_CHECK_LAUNCH();
    return 0;
  }
  return np == 2 ? conv_tc_dispatch<2>(maps, a, BN, SWB, pair, st) : conv_tc_dispatch<3>(maps, a, BN, SWB, pair, st);
}

// diagnostics: the plan conv_tc() would pick for a stride-1 tap-GEMM of this shape on `sms` SMs; out = {BN, splits, pair,
// halo form (0 | 1 | 2 = as a CTA pair), K-slab bytes}
int tc_plan_query(int sms, int B, int T, int Cin, int Cout, int k, int dil, int fmt, int64_t partial_bytes, int ln_rides, int32_t* out5) {
  MTTS_REQUIRE(out5 && sms > 0 && B > 0 && T > 0 && Cin > 0 && Cout > 0 && k > 0 && dil > 0, "bad arguments");
  MTTS_REQUIRE(fmt == MTTS_TC_BF16X3 || fmt == MTTS_TC_F16X2, "unknown operand format");
  mtts_conv_params p;
  memset(&p, 0, sizeof(p));
  p.B = B; p.Tin = T + dil * (k - 1); p.Tout = T; p.Cin = Cin; p.Cout = Cout; p.k = k; p.stride = 1; p.dil = dil;
  static float dummy;
  p.y = &dummy;
  if (partial_bytes > 0) { p.tc_partial = &dummy; p.tc_partial_bytes = partial_bytes; }
  const TcPlan pl = tc_plan(sms, p, fmt == MTTS_TC_F16X2 ? 2 : 3, ln_rides != 0);
  out5[0] = pl.BN; out5[1] = pl.splits; out5[2] = pl.pair ? 1 : 0; out5[3] = pl.halo_form ? (pl.halo_pair ? 2 : 1) : 0; out5[4] = pl.SWB;
  return 0;
}

// fp32 (B, T, C) -> padded operand planes (B, hl + T + hr, C) at the 1024-byte-aligned start of `planes_base`
int split_pad(const float* x, int64_t x_sb, int ldx, int B, int T, int C, int hl, int hr, int pad_mode, int act, float slope,
              void* planes_base, int fmt, cudaStream_t st) {
  MTTS_REQUIRE(x && planes_base && C % 4 == 0 && ldx % 4 == 0 && x_sb % 4 == 0 && ((((uintptr_t)x) & 15) == 0), "bad arguments");
  if (B <= 0 || T <= 0) return 0;
  __nv_bfloat16* planes = reinterpret_cast<__nv_bfloat16*>((((uintptr_t)planes_base) + 1023) & ~(uintptr_t)1023);
  const int Tp = T + hl + hr;
  const int64_t total4 = (int64_t)B * Tp * C / 4;
  launch_k(split_pad_kernel, (unsigned)cdiv64(total4, 256), 256, 0, st, x, x_sb, ldx, T, C, hl, Tp, pad_mode, act, slope, planes,
           (int64_t)B * Tp * C, total4, fmt, tc_ovf_ptr());
  MTTS_CHECK_LAUNCH();
  return 0;
}

// fp32 (rows, C) -> operand planes (3 | 2, rows, C): the activation split, exposed for packing weights on the device
int split_planes(const float* x, int ldx, int64_t rows, int C, void* planes, int fmt, cudaStream_t st) {
  MTTS_REQUIRE(x && planes && C > 0 && C % 4 == 0 && ldx % 4 == 0 && ((((uintptr_t)x) | ((uintptr_t)planes)) & 15) == 0, "bad arguments");
  MTTS_REQUIRE(fmt == MTTS_TC_BF16X3 || fmt == MTTS_TC_F16X2, "unknown operand format");
  if (rows <= 0) return 0;
  MTTS_REQUIRE(rows < (int64_t)1 << 31, "too many rows");
  const int64_t total4 = rows * C / 4;
  launch_k(split_pad_kernel, (unsigned)cdiv64(total4, 256), 256, 0, st, x, 0, ldx, (int)rows, C, 0, (int)rows, MTTS_PAD_ZERO, MTTS_ACT_NONE, 0.f,
                                                                 reinterpret_cast<__nv_bfloat16*>(planes), rows * (int64_t)C, total4,
                                                                 fmt, tc_ovf_ptr());
  MTTS_CHECK_LAUNCH();
  return 0;
}

// nn.Linear on the tensor-core engine = the k = 1 case of the tap-GEMM
int64_t linear_tc_scratch_bytes(int64_t rows_cap, int K) { return 3 * rows_cap * (int64_t)K * 2 + 4096; }

int linear_tc(const float* x, int ldx, int64_t M, int K, const void* w_planes, int N, const float* bias,
              const float* res, int ldr, float* y, int ldy, int pre_act, float pre_slope, int post_act,
              float out_scale, void* scratch, int64_t scratch_bytes, int64_t rows_cap, int fmt, cudaStream_t st) {
  MTTS_REQUIRE(x && w_planes && y && scratch, "null pointer");
  mtts_conv_params p = linear_params(x, ldx, nullptr, bias, y, ldy, M, K, N);
  p.w = reinterpret_cast<const float*>(w_planes);     // unused on this path (non-null for validation only)
  p.res = res; p.ldr = ldr; p.pre_act = pre_act; p.pre_slope = pre_slope; p.post_act = post_act; p.out_scale = out_scale;
  p.w_tc = w_planes; p.tc_scratch = scratch; p.tc_scratch_bytes = scratch_bytes; p.tc_rows_cap = rows_cap; p.tc_fmt = fmt;
  if (!conv_tc_eligible(p))
    return fail(MTTS_ERR_UNSUPPORTED, "%s: shape not eligible for the tensor-core engine (M=%lld N=%lld)", "linear_tc", M, N);
  return conv_tc(p, st);
}

}  // namespace mtts
