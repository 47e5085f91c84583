// Tensor-core attention (tcgen05): softmax(Q K^T * scale + mask) V with fp32-grade accuracy from f16x2 split operands
// (kernels.h: x = x1 + x2' * 2^-11, three MMAs per product: x1*y1 | x1*y2' + x2'*y1, the correction accumulator scaled by
// 2^-11 when it is read back).  Replaces F.scaled_dot_product_attention at modules/transformer.py:52-53 for the head dims
// of the autoregressive stacks (PLM: 16 x 64, ADM: 8 x 96) whenever the sequence is long enough to feed a 128-row MMA.
//
// One CTA = one (batch item, head, 128-query tile), 128 threads, thread r owns query row r == TMEM lane r:
//   stage   Q (128 x dh) once, then per 64-key tile K (64 x dh) and V^T (dh x 64): fp32 global -> f16x2 planes in shared
//           memory, written directly in the UMMA K-major 64-byte-swizzle layout (what a TMA load with SWIZZLE_64B would
//           produce: 16-byte chunk c of row r lands at chunk c ^ ((r >> 1) & 3)); fence.proxy.async hands them to the MMA
//   S       one elected thread issues 3 * dh/16 MMAs (M 128, N 64) into two TMEM accumulators (main | correction)
//   softmax each thread reads ITS row of S from TMEM (tcgen05.ld 32x32b), scales, masks, keeps the running max / sum of
//           the online softmax in registers - no shuffles, no shared memory - and writes P (unnormalised, f16x2 planes)
//           as the A operand of the second product
//   O       3 * 4 MMAs (M 128, N dh, K 64 keys) into the SAME TMEM columns (S is dead by then); the tile's result is read
//           back and folded into the row's fp32 accumulator with the usual exp(m_old - m_new) rescale
//   out     acc / l  ->  fp32 rows and / or operand planes (bf16x3 | f16x2) for the out-projection GEMM
// Shared memory: 96 KB (dh 64) / 128 KB (dh 96) / 160 KB (dh 128); TMEM: 128 / 256 / 256 columns.
#include "kernels.h"
#include "tc_ptx.cuh"

namespace mtts {

namespace {

constexpr int ATC_NK = 64;     // keys per tile

__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// 8 consecutive fp32 values -> one 16-byte chunk per f16x2 plane
__device__ __forceinline__ void split8_f16x2(const float* v, uint4& p0, uint4& p1, bool& bad) {
  uint32_t a[4], b[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    uint16_t h0[2], h1[2];
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const float x = v[2 * i + e];
      const __half x1 = __float2half_rn(x);
      const __half x2 = __float2half_rn((x - __half2float(x1)) * F16X2_SCALE);
      h0[e] = __half_as_ushort(x1);
      h1[e] = __half_as_ushort(x2);
      bad |= !(fabsf(x) <= 65504.0f);
    }
    a[i] = (uint32_t)h0[0] | ((uint32_t)h0[1] << 16);
    b[i] = (uint32_t)h1[0] | ((uint32_t)h1[1] << 16);
  }
  p0 = make_uint4(a[0], a[1], a[2], a[3]);
  p1 = make_uint4(b[0], b[1], b[2], b[3]);
}

// byte offset of 16-byte chunk `c` (0..3) of row `r` inside a K-major slab of 64-byte rows with the 64-byte swizzle
__device__ __forceinline__ uint32_t sw64_off(int r, int c) { return (uint32_t)r * 64u + (uint32_t)((c ^ ((r >> 1) & 3)) << 4); }

template <int DH>
struct AtcCfg {
  static constexpr int NS = DH / 32;                      // 32-element (64-byte) K-slabs along dh
  static constexpr int Q_SLAB = 128 * 64;                 // bytes: 128 rows x 64 B
  static constexpr int K_SLAB = ATC_NK * 64;
  static constexpr int V_SLAB = DH * 64;                  // V^T: dh rows, one slab per 32 keys
  static constexpr int P_SLAB = 128 * 64;
  static constexpr int Q_PLANE = NS * Q_SLAB, K_PLANE = NS * K_SLAB, V_PLANE = 2 * V_SLAB, P_PLANE = 2 * P_SLAB;
  static constexpr int OFF_Q = 0, OFF_K = OFF_Q + 2 * Q_PLANE, OFF_V = OFF_K + 2 * K_PLANE, OFF_P = OFF_V + 2 * V_PLANE;
  static constexpr int SMEM = OFF_P + 2 * P_PLANE + 1024 + 64;      // + alignment slack + barrier / TMEM slot
  static constexpr int TMEM_COLS = (2 * DH > 128) ? 256 : 128;      // max(2 * 64 for S, 2 * dh for O), power of two
};

template <int DH>
__global__ void __launch_bounds__(128)
attn_tc_kernel(const mtts_attn_params p, int32_t* ovf) {
  using Cfg = AtcCfg<DH>;
  pdl_trigger();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar = base + Cfg::OFF_P + 2 * Cfg::P_PLANE;
  const uint32_t tmem_slot = bar + 16;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(sm + Cfg::OFF_P + 2 * Cfg::P_PLANE + 16);

  const int tid = threadIdx.x;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);        // warp-uniform for the compiler (uniform-register MMA operands)
  const int q0 = blockIdx.x * 128, h = blockIdx.y, b = blockIdx.z;
  const int qrow = q0 + tid;
  const bool qvalid = qrow < p.Tq;

  if (tid == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(Cfg::TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }

  pdl_wait();
  bool bad = false;
  // ---- stage Q: thread r splits its own row (rows past Tq are zero)
  {
    const float* src = p.q + (int64_t)b * p.q_sb + (int64_t)(qvalid ? qrow : 0) * p.q_st + (int64_t)h * DH;
#pragma unroll
    for (int c8 = 0; c8 < DH / 8; ++c8) {
      float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (qvalid) {
        const float4 a = *reinterpret_cast<const float4*>(src + c8 * 8);
        const float4 c = *reinterpret_cast<const float4*>(src + c8 * 8 + 4);
        v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
      }
      uint4 p0, p1;
      split8_f16x2(v, p0, p1, bad);
      const uint32_t off = (uint32_t)(c8 >> 2) * Cfg::Q_SLAB + sw64_off(tid, c8 & 3);
      *reinterpret_cast<uint4*>(sm + Cfg::OFF_Q + off) = p0;
      *reinterpret_cast<uint4*>(sm + Cfg::OFF_Q + Cfg::Q_PLANE + off) = p1;
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);
  const uint32_t leader = (warp == 0 && elect_one()) ? 1u : 0u;
  const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);      // this warp's TMEM lane quarter

  float m_run = -INFINITY, l_run = 0.f;
  float acc[DH];
#pragma unroll
  for (int d = 0; d < DH; ++d) acc[d] = 0.f;
  const float* mrow = p.mask ? p.mask + (int64_t)b * p.mask_sb + (int64_t)h * p.mask_sh + (int64_t)(qvalid ? qrow : 0) * p.mask_sq : nullptr;
  const float* kb = p.k + (int64_t)b * p.k_sb + (int64_t)h * DH;
  const float* vb = p.v + (int64_t)b * p.v_sb + (int64_t)h * DH;
  const uint64_t desc_hi = umma_desc_kmajor<64>(0u);
  constexpr uint32_t IDESC_S = (1u << 4) | ((uint32_t)(ATC_NK >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);   // f16 x f16 -> f32
  constexpr uint32_t IDESC_O = (1u << 4) | ((uint32_t)(DH >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  uint32_t phase = 0;

  for (int k0 = 0; k0 < p.Tk; k0 += ATC_NK) {
    // ---- stage the K tile (two threads per key row) and the V^T tile (lanes = consecutive keys, so that a warp fills
    //      one 64-byte row of V^T with 2-byte stores); keys past Tk are zero
    {
      const int key = tid >> 1, half = tid & 1;
      const bool kvalid = k0 + key < p.Tk;
      const float* src = kb + (int64_t)(kvalid ? k0 + key : 0) * p.k_st + half * (DH / 2);
#pragma unroll
      for (int i = 0; i < DH / 16; ++i) {
        float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (kvalid) {
          const float4 a = *reinterpret_cast<const float4*>(src + i * 8);
          const float4 c = *reinterpret_cast<const float4*>(src + i * 8 + 4);
          v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = c.x; v[5] = c.y; v[6] = c.z; v[7] = c.w;
        }
        uint4 p0, p1;
        split8_f16x2(v, p0, p1, bad);
        const int c8 = half * (DH / 16) + i;              // 16-byte chunk index along dh
        const uint32_t off = (uint32_t)(c8 >> 2) * Cfg::K_SLAB + sw64_off(key, c8 & 3);
        *reinterpret_cast<uint4*>(sm + Cfg::OFF_K + off) = p0;
        *reinterpret_cast<uint4*>(sm + Cfg::OFF_K + Cfg::K_PLANE + off) = p1;
      }
    }
    {
      const int key = tid & 63, dg = tid >> 6;            // dg: which half of dh this thread transposes
      const bool kvalid = k0 + key < p.Tk;
      const float* src = vb + (int64_t)(kvalid ? k0 + key : 0) * p.v_st + dg * (DH / 2);
      uint8_t* vt0 = sm + Cfg::OFF_V + (key >> 5) * Cfg::V_SLAB;
      const int kk = key & 31;
#pragma unroll
      for (int i = 0; i < DH / 8; ++i) {
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
        if (kvalid) a = *reinterpret_cast<const float4*>(src + i * 4);
        const float vv[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int d = dg * (DH / 2) + i * 4 + e;
          const __half x1 = __float2half_rn(vv[e]);
          const __half x2 = __float2half_rn((vv[e] - __half2float(x1)) * F16X2_SCALE);
          bad |= !(fabsf(vv[e]) <= 65504.0f);
          const uint32_t off = sw64_off(d, kk >> 3) + (uint32_t)(kk & 7) * 2u;
          *reinterpret_cast<uint16_t*>(vt0 + off) = __half_as_ushort(x1);
          *reinterpret_cast<uint16_t*>(vt0 + Cfg::V_PLANE + off) = __half_as_ushort(x2);
        }
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();       // every thread's TMEM reads of the previous tile (O) are complete before the MMAs overwrite it
    __syncthreads();
    // ---- S = Q K^T   (warp 0 walks the issue loop uniformly; its elected lane executes the MMAs)
    if (warp == 0) {
      tc_fence_after();
#pragma unroll
      for (int ks = 0; ks < DH / 16; ++ks) {
        const uint32_t qa = base + Cfg::OFF_Q + (ks >> 1) * Cfg::Q_SLAB + (ks & 1) * 32;
        const uint32_t ka = base + Cfg::OFF_K + (ks >> 1) * Cfg::K_SLAB + (ks & 1) * 32;
        const uint64_t a1 = desc_hi | (uint64_t)((qa >> 4) & 0x3FFF), a2 = desc_hi | (uint64_t)(((qa + Cfg::Q_PLANE) >> 4) & 0x3FFF);
        const uint64_t b1 = desc_hi | (uint64_t)((ka >> 4) & 0x3FFF), b2 = desc_hi | (uint64_t)(((ka + Cfg::K_PLANE) >> 4) & 0x3FFF);
        tc_mma_l(tmem + ATC_NK, a1, b2, IDESC_S, ks ? 1u : 0u, leader);      // correction: q1 k2' + q2' k1
        tc_mma_l(tmem + ATC_NK, a2, b1, IDESC_S, 1u, leader);
        tc_mma_l(tmem, a1, b1, IDESC_S, ks ? 1u : 0u, leader);               // main: q1 k1
      }
      tc_commit_l(bar, leader);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
    // ---- online softmax on this thread's row
    float s[ATC_NK];
#pragma unroll
    for (int u = 0; u < ATC_NK / 16; ++u) {
      uint32_t r[16], rc[16];
      tmem_ld16(lane_addr + u * 16, r);
      tmem_ld16(lane_addr + ATC_NK + u * 16, rc);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int key = k0 + u * 16 + j;
        float x = fmaf(__uint_as_float(rc[j]), F16X2_INV_SCALE, __uint_as_float(r[j])) * p.scale;
        if (mrow && key < p.Tk) x += mrow[key];
        s[u * 16 + j] = key < p.Tk ? x : -INFINITY;
      }
    }
    float tmax = s[0];
#pragma unroll
    for (int j = 1; j < ATC_NK; ++j) tmax = fmaxf(tmax, s[j]);
    const float m_new = fmaxf(m_run, tmax);
    const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
    const float alpha = expf(m_run - m_use);
    float psum = 0.f;
#pragma unroll
    for (int j = 0; j < ATC_NK; ++j) {
      s[j] = expf(s[j] - m_use);
      psum += s[j];
    }
    l_run = l_run * alpha + psum;
    m_run = m_new;
    bool pbad = false;     // p is in [0, 1]: never out of range
#pragma unroll
    for (int c8 = 0; c8 < ATC_NK / 8; ++c8) {
      uint4 p0, p1;
      split8_f16x2(s + c8 * 8, p0, p1, pbad);
      const uint32_t off = (uint32_t)(c8 >> 2) * Cfg::P_SLAB + sw64_off(tid, c8 & 3);
      *reinterpret_cast<uint4*>(sm + Cfg::OFF_P + off) = p0;
      *reinterpret_cast<uint4*>(sm + Cfg::OFF_P + Cfg::P_PLANE + off) = p1;
    }
    fence_proxy_async_smem();
    tc_fence_before();       // this thread's reads of S are complete before O overwrites the columns
    __syncthreads();
    // ---- O_tile = P V   (K = the tile's 64 keys: 4 k-steps)
    if (warp == 0) {
      tc_fence_after();
#pragma unroll
      for (int ks = 0; ks < ATC_NK / 16; ++ks) {
        const uint32_t pa = base + Cfg::OFF_P + (ks >> 1) * Cfg::P_SLAB + (ks & 1) * 32;
        const uint32_t va = base + Cfg::OFF_V + (ks >> 1) * Cfg::V_SLAB + (ks & 1) * 32;
        const uint64_t a1 = desc_hi | (uint64_t)((pa >> 4) & 0x3FFF), a2 = desc_hi | (uint64_t)(((pa + Cfg::P_PLANE) >> 4) & 0x3FFF);
        const uint64_t b1 = desc_hi | (uint64_t)((va >> 4) & 0x3FFF), b2 = desc_hi | (uint64_t)(((va + Cfg::V_PLANE) >> 4) & 0x3FFF);
        tc_mma_l(tmem + DH, a1, b2, IDESC_O, ks ? 1u : 0u, leader);
        tc_mma_l(tmem + DH, a2, b1, IDESC_O, 1u, leader);
        tc_mma_l(tmem, a1, b1, IDESC_O, ks ? 1u : 0u, leader);
      }
      tc_commit_l(bar, leader);
    }
    mbar_wait(bar, phase);
    phase ^= 1;
    tc_fence_after();
#pragma unroll
    for (int u = 0; u < DH / 16; ++u) {
      uint32_t r[16], rc[16];
      tmem_ld16(lane_addr + u * 16, r);
      tmem_ld16(lane_addr + DH + u * 16, rc);
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 16; ++j)
        acc[u * 16 + j] = fmaf(acc[u * 16 + j], alpha, fmaf(__uint_as_float(rc[j]), F16X2_INV_SCALE, __uint_as_float(r[j])));
    }
  }
  if (bad && ovf) *ovf = 1;

  // ---- output: this thread's row
  if (qvalid) {
    const float inv = 1.0f / l_run;
    if (p.o) {
      float* o = p.o + (int64_t)b * p.o_sb + (int64_t)qrow * p.o_st + (int64_t)h * DH;
#pragma unroll
      for (int d = 0; d < DH; d += 4)
        *reinterpret_cast<float4*>(o + d) = make_float4(acc[d] * inv, acc[d + 1] * inv, acc[d + 2] * inv, acc[d + 3] * inv);
    }
    if (p.o_planes) {
      __nv_bfloat16* pl = reinterpret_cast<__nv_bfloat16*>(p.o_planes);
      const int64_t off = ((int64_t)b * p.Tq + qrow) * p.o_planes_ld + (int64_t)h * DH;
#pragma unroll
      for (int d = 0; d < DH; d += 4) {
        const float v[4] = {acc[d] * inv, acc[d + 1] * inv, acc[d + 2] * inv, acc[d + 3] * inv};
        store_planes4(pl, p.o_plane_stride, off + d, v, p.o_planes_fmt, ovf);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(Cfg::TMEM_COLS) : "memory");
  }
}

template <int DH>
int attn_tc_launch(const mtts_attn_params& p, cudaStream_t st) {
  using Cfg = AtcCfg<DH>;
  static std::atomic<uint64_t> configured{0};
  const int dev = cur_device();
  if (!(configured.load(std::memory_order_relaxed) & (1ull << dev))) {
    cudaError_t e = cudaFuncSetAttribute(attn_tc_kernel<DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM);
    if (e != cudaSuccess) return fail(MTTS_ERR_CUDA, "%s: cudaFuncSetAttribute failed: %lld", "attention_tc", (long long)e);
    configured.fetch_or(1ull << dev, std::memory_order_relaxed);
  }
  dim3 grid((unsigned)cdiv64(p.Tq, 128), (unsigned)p.H, (unsigned)p.B);
  launch_k(attn_tc_kernel<DH>, grid, 128, Cfg::SMEM, st, p, tc_ovf_ptr());
  MTTS_CHECK_LAUNCH();
  return 0;
}

}  // namespace

// eligible: head dims of the AR stacks, 16-byte aligned fp32 views, output rows aligned for float4 / plane stores
bool attention_tc_eligible(const mtts_attn_params& p) {
  if (!(p.dh == 64 || p.dh == 96 || p.dh == 128)) return false;
  auto al = [](const void* q) { return (((uintptr_t)q) & 15) == 0; };
  if (!(al(p.q) && al(p.k) && al(p.v) && p.q_st % 4 == 0 && p.k_st % 4 == 0 && p.v_st % 4 == 0 && p.q_sb % 4 == 0 &&
        p.k_sb % 4 == 0 && p.v_sb % 4 == 0))
    return false;
  if (p.o && !(al(p.o) && p.o_st % 4 == 0 && p.o_sb % 4 == 0)) return false;
  if (p.o_planes && (p.o_planes_ld % 4 != 0 || p.o_plane_stride % 4 != 0)) return false;
  return p.B > 0 && p.H > 0 && p.Tq > 0 && p.Tk > 0 && p.H <= 65535 && p.B <= 65535;
}

int attention_tc(const mtts_attn_params& p, cudaStream_t st) {
  MTTS_REQUIRE(attention_tc_eligible(p), "shape / alignment not eligible for the tensor-core attention");
  if (p.dh == 64) return attn_tc_launch<64>(p, st);
  if (p.dh == 96) return attn_tc_launch<96>(p, st);
  return attn_tc_launch<128>(p, st);
}

}  // namespace mtts
