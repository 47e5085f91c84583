// HBM-bound and small kernels of the synthesis path: LayerNorm, attention (fp32),
// VQ search / gather, max-pool, embeddings + sine PE, length regulator, layout copies,
// and the per-step helpers of the PLM / ADM autoregressive loops.
#include <float.h>
#include <math.h>
#include <stdlib.h>

#include <atomic>

#include "kernels.h"

namespace mtts {

// ------------------------------------------------------------------------------------------
// LayerNorm: one warp per row, three passes over a row that stays in L1 (C <= 4096 floats).
// x / res may alias y (same element is read then written by the same lane only).
__global__ void __launch_bounds__(256)
layernorm_kernel(const float* x, int ldx, const float* __restrict__ gamma, const float* __restrict__ beta,
                 const float* res, int ldr, float* y, int ldy, int64_t rows, int C, float eps,
                 int post_act, int accumulate, int vec, const PlanesOut po) {
  pdl_entry();
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * ldx;
  float s = 0.f;
  if (vec) {
    for (int c = lane * 4; c < C; c += 128) {
      const float4 v = *reinterpret_cast<const float4*>(xr + c);
      s += (v.x + v.y) + (v.z + v.w);
    }
  } else {
    for (int c = lane; c < C; c += 32) s += xr[c];
  }
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
  if (vec) {
    for (int c = lane * 4; c < C; c += 128) {
      const float4 v = *reinterpret_cast<const float4*>(xr + c);
      const float a = v.x - mean, b = v.y - mean, d = v.z - mean, e = v.w - mean;
      q += (a * a + b * b) + (d * d + e * e);
    }
  } else {
    for (int c = lane; c < C; c += 32) {
      const float a = xr[c] - mean;
      q += a * a;
    }
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)C + eps);
  float* yr = y ? y + row * ldy : nullptr;
  const float* rr = res ? res + row * ldr : nullptr;
  if (vec) {
    for (int c = lane * 4; c < C; c += 128) {
      const float4 v = *reinterpret_cast<const float4*>(xr + c);
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
      const float4 bb = __ldg(reinterpret_cast<const float4*>(beta + c));
      float o[4] = {(v.x - mean) * rstd * g.x + bb.x, (v.y - mean) * rstd * g.y + bb.y,
                    (v.z - mean) * rstd * g.z + bb.z, (v.w - mean) * rstd * g.w + bb.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) o[e] = act_apply(o[e], post_act, 0.f);
      if (rr) {
        const float4 r = *reinterpret_cast<const float4*>(rr + c);
        o[0] += r.x; o[1] += r.y; o[2] += r.z; o[3] += r.w;
      }
      if (accumulate) {
        const float4 r = *reinterpret_cast<const float4*>(yr + c);
        o[0] += r.x; o[1] += r.y; o[2] += r.z; o[3] += r.w;
      }
      if (yr) *reinterpret_cast<float4*>(yr + c) = make_float4(o[0], o[1], o[2], o[3]);
      if (po.p) {
#pragma unroll
        for (int e = 0; e < 4; ++e) o[e] = act_apply(o[e], po.act, po.slope);
        store_planes4(po.p, po.stride, row * po.ld + c, o, po.fmt, po.ovf);
      }
    }
  } else {
    for (int c = lane; c < C; c += 32) {
      float o = act_apply((xr[c] - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c), post_act, 0.f);
      if (rr) o += rr[c];
      if (accumulate) o += yr[c];
      if (yr) yr[c] = o;
    }
  }
}

// Register-resident variant for the row widths of the path (C = 128*NV, NV float4 per lane): one global read
// of the row (NV independent 128-bit loads in flight), two shuffle reductions, one write.
template <int NV>
__global__ void __launch_bounds__(256)
layernorm_reg_kernel(const float* x, int ldx, const float* __restrict__ gamma, const float* __restrict__ beta,
                     const float* res, int ldr, float* y, int ldy, int64_t rows, float eps, int post_act,
                     int accumulate, const PlanesOut po) {
  pdl_entry();
  constexpr int C = 128 * NV;
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + row * ldx;
  float4 v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = *reinterpret_cast<const float4*>(xr + i * 128 + lane * 4);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  const float mean = warp_sum(s) / (float)C;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, d = v[i].z - mean, e = v[i].w - mean;
    q += (a * a + b * b) + (d * d + e * e);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) / (float)C + eps);
  float* yr = y ? y + row * ldy : nullptr;
  const float* rr = res ? res + row * ldr : nullptr;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = i * 128 + lane * 4;
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + c));
    const float4 bb = __ldg(reinterpret_cast<const float4*>(beta + c));
    float o[4] = {(v[i].x - mean) * rstd * g.x + bb.x, (v[i].y - mean) * rstd * g.y + bb.y,
                  (v[i].z - mean) * rstd * g.z + bb.z, (v[i].w - mean) * rstd * g.w + bb.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) o[e] = act_apply(o[e], post_act, 0.f);
    if (rr) {
      const float4 r = *reinterpret_cast<const float4*>(rr + c);
      o[0] += r.x; o[1] += r.y; o[2] += r.z; o[3] += r.w;
    }
    if (accumulate) {
      const float4 r = *reinterpret_cast<const float4*>(yr + c);
      o[0] += r.x; o[1] += r.y; o[2] += r.z; o[3] += r.w;
    }
    if (yr) *reinterpret_cast<float4*>(yr + c) = make_float4(o[0], o[1], o[2], o[3]);
    if (po.p) {
#pragma unroll
      for (int e = 0; e < 4; ++e) o[e] = act_apply(o[e], po.act, po.slope);
      store_planes4(po.p, po.stride, row * po.ld + c, o, po.fmt, po.ovf);
    }
  }
}

static inline bool al16(const void* p) { return (((uintptr_t)p) & 15) == 0; }

int layernorm_ex(const float* x, int ldx, const float* gamma, const float* beta, const float* res, int ldr,
                 float* y, int ldy, int64_t rows, int C, float eps, int post_act, int accumulate, PlanesOut po,
                 cudaStream_t st) {
  MTTS_REQUIRE(x && gamma && beta && (y || po.p), "null pointer");
  MTTS_REQUIRE(C > 0 && ldx >= C && (!y || ldy >= C), "bad dims");
  MTTS_REQUIRE(!(accumulate && !y), "accumulate needs a y buffer");
  MTTS_REQUIRE(post_act != MTTS_ACT_LEAKY, "leaky post-activation is not supported by LayerNorm (no slope argument)");
  if (rows <= 0) return 0;
  const int vec = (C % 4 == 0) && (ldx % 4 == 0) && (!y || ((ldy % 4 == 0) && al16(y))) && al16(x) && al16(gamma) &&
                  al16(beta) && (!res || ((ldr % 4 == 0) && al16(res)));
  MTTS_REQUIRE(!po.p || (vec && po.ld % 4 == 0 && po.stride % 4 == 0), "plane output needs the vector path");
  const int wpb = 8;
  const unsigned grid = (unsigned)cdiv64(rows, wpb);
#define MTTS_LN_REG(NV)                                                                                          \
  launch_k(layernorm_reg_kernel<NV>, grid, wpb * 32, 0, st, x, ldx, gamma, beta, res, ldr, y, ldy, rows, eps, post_act, \
                                                      accumulate, po)
  if (vec && C == 1024) MTTS_LN_REG(8);
  else if (vec && C == 768) MTTS_LN_REG(6);
  else if (vec && C == 512) MTTS_LN_REG(4);
  else if (vec && C == 384) MTTS_LN_REG(3);
  else
    launch_k(layernorm_kernel, grid, wpb * 32, 0, st, x, ldx, gamma, beta, res, ldr, y, ldy, rows, C, eps, post_act,
                                                accumulate, vec, po);
#undef MTTS_LN_REG
  MTTS_CHECK_LAUNCH();
  return 0;
}

int layernorm(const float* x, int ldx, const float* gamma, const float* beta, const float* res, int ldr,
              float* y, int ldy, int64_t rows, int C, float eps, int post_act, int accumulate,
              cudaStream_t st) {
  MTTS_REQUIRE(y, "null pointer");
  PlanesOut po{nullptr, 0, 0, 0, 0.f, 0, nullptr};
  return layernorm_ex(x, ldx, gamma, beta, res, ldr, y, ldy, rows, C, eps, post_act, accumulate, po, st);
}

// ------------------------------------------------------------------------------------------
// Attention, fp32, online softmax.  CTA = NW warps x RW query rows of one (b, h); K/V stream through
// shared memory 32*KPL keys at a time (float4 global loads when aligned); lane l scores keys l (+32 when KPL = 2:
// the broadcast Q loads of the score loop are then shared by two keys - that loop is shared-memory-bound), then owns
// output dims l + 32*i.  Head dims on the path: 64 (PLM), 96 (ADM), 256 (phone encoder), 512 (MRTE
// cross-attention, Tk ~ 32).  For dh <= 128 a CTA covers 64 query rows, i.e. a whole AR-step sequence:
// K and V are read once per (b, h).
// dh = 64 (NI = 2): capped at 80 registers so that three CTAs share an SM (49 vs 53 us at S = 64); the wider heads spill too
// much under that cap (dh 96: 44 vs 36 us) and keep two CTAs (gpurun call AT, profiles/r2at_attention_regs_ab.log)
template <int NI, int RW, int NW, int KPL>
__global__ void __launch_bounds__(NW * 32, (NI == 2 ? 3 : 2)) attn_kernel(const mtts_attn_params p, const int vec, int32_t* ovf) {
  pdl_entry();
  constexpr int DH = 32 * NI;
  constexpr int BQ = RW * NW, BKV = 32 * KPL, NT = NW * 32;
  extern __shared__ __align__(16) float sm[];
  float* Qs = sm;                        // [BQ][DH]
  constexpr int KS = DH + 4;             // K row stride: 16-byte aligned rows, conflict-free 128-bit reads (lane stride 4 banks)
  float* Ks = Qs + BQ * DH;              // [BKV][KS]
  float* Vs = Ks + BKV * KS;             // [BKV][DH]
  float* Ps = Vs + BKV * DH;             // [NW][RW][BKV]
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int q0 = blockIdx.x * BQ, h = blockIdx.y, b = blockIdx.z;
  const float* qb = p.q + (int64_t)b * p.q_sb + (int64_t)h * DH;
  const float* kb = p.k + (int64_t)b * p.k_sb + (int64_t)h * DH;
  const float* vb = p.v + (int64_t)b * p.v_sb + (int64_t)h * DH;

  if (vec) {
    for (int i = tid; i < BQ * (DH / 4); i += NT) {
      const int r = i / (DH / 4), d = (i - r * (DH / 4)) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q0 + r < p.Tq) v = *reinterpret_cast<const float4*>(qb + (int64_t)(q0 + r) * p.q_st + d);
      *reinterpret_cast<float4*>(Qs + r * DH + d) = v;
    }
  } else {
    for (int i = tid; i < BQ * DH; i += NT) {
      const int r = i / DH, d = i - r * DH;
      Qs[i] = (q0 + r < p.Tq) ? qb[(int64_t)(q0 + r) * p.q_st + d] : 0.f;
    }
  }
  float m_run[RW], l_run[RW], acc[RW][NI];
#pragma unroll
  for (int i = 0; i < RW; ++i) {
    m_run[i] = -INFINITY;
    l_run[i] = 0.f;
#pragma unroll
    for (int j = 0; j < NI; ++j) acc[i][j] = 0.f;
  }
  const float* mrow[RW];
#pragma unroll
  for (int i = 0; i < RW; ++i) {
    const int qr = min(q0 + w * RW + i, p.Tq - 1);
    mrow[i] = p.mask ? p.mask + (int64_t)b * p.mask_sb + (int64_t)h * p.mask_sh + (int64_t)qr * p.mask_sq : nullptr;
  }
  const bool warp_live = (q0 + w * RW) < p.Tq;   // warp-uniform: this warp owns at least one real query row

  for (int k0 = 0; k0 < p.Tk; k0 += BKV) {
    __syncthreads();   // previous tile fully consumed (also orders the Q fill)
    if (vec) {
      for (int i = tid; i < BKV * (DH / 4); i += NT) {
        const int r = i / (DH / 4), d = (i - r * (DH / 4)) * 4;
        float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
        if (k0 + r < p.Tk) {
          kv = *reinterpret_cast<const float4*>(kb + (int64_t)(k0 + r) * p.k_st + d);
          vv = *reinterpret_cast<const float4*>(vb + (int64_t)(k0 + r) * p.v_st + d);
        }
        *reinterpret_cast<float4*>(Ks + r * KS + d) = kv;
        *reinterpret_cast<float4*>(Vs + r * DH + d) = vv;
      }
    } else {
      for (int i = tid; i < BKV * DH; i += NT) {
        const int r = i / DH, d = i - r * DH;
        const bool ok = k0 + r < p.Tk;
        Ks[r * KS + d] = ok ? kb[(int64_t)(k0 + r) * p.k_st + d] : 0.f;
        Vs[r * DH + d] = ok ? vb[(int64_t)(k0 + r) * p.v_st + d] : 0.f;
      }
    }
    __syncthreads();
    if (!warp_live) continue;
    float s[RW][KPL];
#pragma unroll
    for (int i = 0; i < RW; ++i)
#pragma unroll
      for (int c = 0; c < KPL; ++c) s[i][c] = 0.f;
    // 128-bit shared loads: KPL key chunks per lane + RW broadcast Q chunks feed 4 * RW * KPL FMAs (the scalar form
    // issued 9 loads per 8 FMAs and was load-issue bound); the d order of every dot product is unchanged
    const float* kr = Ks + lane * KS;
    const float* qr = Qs + (w * RW) * DH;
#pragma unroll 4
    for (int d = 0; d < DH; d += 4) {
      float4 kv[KPL];
#pragma unroll
      for (int c = 0; c < KPL; ++c) kv[c] = *reinterpret_cast<const float4*>(kr + c * 32 * KS + d);
#pragma unroll
      for (int i = 0; i < RW; ++i) {
        const float4 qv = *reinterpret_cast<const float4*>(qr + i * DH + d);
#pragma unroll
        for (int c = 0; c < KPL; ++c) {
          s[i][c] = fmaf(qv.x, kv[c].x, s[i][c]);
          s[i][c] = fmaf(qv.y, kv[c].y, s[i][c]);
          s[i][c] = fmaf(qv.z, kv[c].z, s[i][c]);
          s[i][c] = fmaf(qv.w, kv[c].w, s[i][c]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < RW; ++i) {
      float v[KPL];
      float vmax = -INFINITY;
#pragma unroll
      for (int c = 0; c < KPL; ++c) {
        const int key = k0 + lane + 32 * c;
        const bool kvalid = key < p.Tk;
        float x = s[i][c] * p.scale;
        if (mrow[i]) x += kvalid ? mrow[i][key] : 0.f;
        v[c] = kvalid ? x : -INFINITY;
        vmax = fmaxf(vmax, v[c]);
      }
      const float m_new = fmaxf(m_run[i], warp_max(vmax));
      const float m_use = (m_new == -INFINITY) ? 0.f : m_new;
      float psum = 0.f;
#pragma unroll
      for (int c = 0; c < KPL; ++c) {
        const float pr = expf(v[c] - m_use);
        Ps[(w * RW + i) * BKV + lane + 32 * c] = pr;
        psum += pr;
      }
      const float alpha = expf(m_run[i] - m_use);
      l_run[i] = l_run[i] * alpha + warp_sum(psum);
      m_run[i] = m_new;
#pragma unroll
      for (int j = 0; j < NI; ++j) acc[i][j] *= alpha;
    }
    __syncwarp();
    const float* pw = Ps + (w * RW) * BKV;
#pragma unroll 2
    for (int j = 0; j < BKV; j += 4) {
      float4 pj[RW];
#pragma unroll
      for (int i = 0; i < RW; ++i) pj[i] = *reinterpret_cast<const float4*>(pw + i * BKV + j);
#pragma unroll
      for (int ii = 0; ii < NI; ++ii) {
        const float v0 = Vs[(j + 0) * DH + lane + 32 * ii], v1 = Vs[(j + 1) * DH + lane + 32 * ii];
        const float v2 = Vs[(j + 2) * DH + lane + 32 * ii], v3 = Vs[(j + 3) * DH + lane + 32 * ii];
#pragma unroll
        for (int i = 0; i < RW; ++i) {
          acc[i][ii] = fmaf(pj[i].x, v0, acc[i][ii]);
          acc[i][ii] = fmaf(pj[i].y, v1, acc[i][ii]);
          acc[i][ii] = fmaf(pj[i].z, v2, acc[i][ii]);
          acc[i][ii] = fmaf(pj[i].w, v3, acc[i][ii]);
        }
      }
    }
    __syncwarp();
  }
  if (p.o) {
#pragma unroll
    for (int i = 0; i < RW; ++i) {
      const int qr = q0 + w * RW + i;
      if (qr >= p.Tq) continue;
      float* o = p.o + (int64_t)b * p.o_sb + (int64_t)qr * p.o_st + (int64_t)h * DH;
      const float inv = 1.0f / l_run[i];
#pragma unroll
      for (int ii = 0; ii < NI; ++ii) o[lane + 32 * ii] = acc[i][ii] * inv;
    }
  }
  if (p.o_planes) {
    // bf16x3 planes for the following tensor-core GEMM: stage this warp's rows in its (now dead) Q rows so
    // that every lane can split 4 CONSECUTIVE dims and store 8 bytes per plane
    __syncwarp();
    float* stg = Qs + (w * RW) * DH;
#pragma unroll
    for (int i = 0; i < RW; ++i) {
      const float inv = 1.0f / l_run[i];
#pragma unroll
      for (int ii = 0; ii < NI; ++ii) stg[i * DH + lane + 32 * ii] = acc[i][ii] * inv;
    }
    __syncwarp();
    __nv_bfloat16* pl = reinterpret_cast<__nv_bfloat16*>(p.o_planes);
    for (int e = lane; e < RW * (DH / 4); e += 32) {
      const int i = e / (DH / 4), d = (e - i * (DH / 4)) * 4;
      const int qr = q0 + w * RW + i;
      if (qr >= p.Tq) continue;
      const float4 v = *reinterpret_cast<const float4*>(stg + i * DH + d);
      const float vv[4] = {v.x, v.y, v.z, v.w};
      store_planes4(pl, p.o_plane_stride, ((int64_t)b * p.Tq + qr) * p.o_planes_ld + (int64_t)h * DH + d, vv, p.o_planes_fmt, ovf);
    }
  }
}

template <int NI, int RW, int NW, int KPL = 1>
static int attn_launch(const mtts_attn_params& p, cudaStream_t st) {
  constexpr int DH = 32 * NI;
  constexpr int BQ = RW * NW, BKV = 32 * KPL;
  const size_t smem = sizeof(float) * (BQ * DH + BKV * (DH + 4) + BKV * DH + NW * RW * BKV);
  // the max-dynamic-shared-memory attribute is per device: one flag per (instantiation, device)
  static std::atomic<uint64_t> configured{0};
  const int dev = cur_device();
  if (!(configured.load(std::memory_order_relaxed) & (1ull << dev))) {
    cudaError_t e = cudaFuncSetAttribute(attn_kernel<NI, RW, NW, KPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail(MTTS_ERR_CUDA, "%s: cudaFuncSetAttribute failed: %lld", "attention", (long long)e);
    configured.fetch_or(1ull << dev, std::memory_order_relaxed);
  }
  auto al = [](const void* q) { return (((uintptr_t)q) & 15) == 0; };
  const int vec = al(p.q) && al(p.k) && al(p.v) && p.q_st % 4 == 0 && p.k_st % 4 == 0 && p.v_st % 4 == 0 &&
                  p.q_sb % 4 == 0 && p.k_sb % 4 == 0 && p.v_sb % 4 == 0;
  dim3 grid((unsigned)cdiv64(p.Tq, BQ), (unsigned)p.H, (unsigned)p.B);
  launch_k(attn_kernel<NI, RW, NW, KPL>, grid, NW * 32, smem, st, p, vec, p.o_planes ? tc_ovf_ptr() : nullptr);
  MTTS_CHECK_LAUNCH();
  return 0;
}

int attention(const mtts_attn_params& p, cudaStream_t st) {
  MTTS_REQUIRE(p.q && p.k && p.v && (p.o || p.o_planes), "null pointer");
  MTTS_REQUIRE(!p.o_planes || (p.o_planes_ld % 4 == 0 && p.o_plane_stride % 4 == 0), "plane output alignment");
  MTTS_REQUIRE(p.B >= 0 && p.H > 0 && p.Tq >= 0 && p.Tk > 0, "bad dims");
  MTTS_REQUIRE(p.H <= 65535 && p.B <= 65535, "grid too large");
  if (p.B == 0 || p.Tq == 0) return 0;
  // tensor-core path (attn_tc.cu): the head dims of the AR stacks once a sequence has more than 64 queries.  Measured at
  // the C4 step shapes (Tq = Tk <= 64, profiles/r2c_attention_tc_ab.md) the phase-serialised tensor-core kernel is 1.5x
  // SLOWER than this fp32 kernel (58 vs 38 us per launch: the problem is 64 x 64 x 64 per head, all latency), so the AR
  // steps of the benchmark stay here; longer sequences (teacher-forced forwards, config C3) go to the tensor cores.
  if (p.Tq >= 65 && attention_tc_eligible(p)) return attention_tc(p, st);
  // dh <= 128: one CTA of 8 warps covers a whole AR-step sequence (Tq <= 64), so K and V are read once per (b, h);
  // the rows are dealt evenly to the warps (RW = ceil(Tq / 8) rows each) - with a fixed 8 rows per warp a 35-row
  // step left three of the eight warps idle.  Row results do not depend on RW (each row's sums keep their order).
  if (p.dh == 64 || p.dh == 96 || p.dh == 128) {
    const int rw = p.Tq >= 64 ? 8 : (p.Tq + 7) / 8;
    const bool two = p.Tk > 32;          // two keys per lane: one 64-key tile instead of two 32-key tiles
#define MTTS_ATTN_RW(NI)                                                                    \
    switch (rw) {                                                                             \
      case 1: return two ? attn_launch<NI, 1, 8, 2>(p, st) : attn_launch<NI, 1, 8>(p, st);    \
      case 2: return two ? attn_launch<NI, 2, 8, 2>(p, st) : attn_launch<NI, 2, 8>(p, st);    \
      case 3: return two ? attn_launch<NI, 3, 8, 2>(p, st) : attn_launch<NI, 3, 8>(p, st);    \
      case 4: return two ? attn_launch<NI, 4, 8, 2>(p, st) : attn_launch<NI, 4, 8>(p, st);    \
      case 5: return two ? attn_launch<NI, 5, 8, 2>(p, st) : attn_launch<NI, 5, 8>(p, st);    \
      case 6: return two ? attn_launch<NI, 6, 8, 2>(p, st) : attn_launch<NI, 6, 8>(p, st);    \
      case 7: return two ? attn_launch<NI, 7, 8, 2>(p, st) : attn_launch<NI, 7, 8>(p, st);    \
      default: return two ? attn_launch<NI, 8, 8, 2>(p, st) : attn_launch<NI, 8, 8>(p, st);   \
    }
    if (p.dh == 64) { MTTS_ATTN_RW(2) }
    if (p.dh == 96) { MTTS_ATTN_RW(3) }
    MTTS_ATTN_RW(4)
#undef MTTS_ATTN_RW
  }
  switch (p.dh) {
    case 256: return attn_launch<8, 4, 4>(p, st);
    case 512: return attn_launch<16, 4, 4>(p, st);
    default: return fail(MTTS_ERR_UNSUPPORTED, "%s: head dim %lld not in {64,96,128,256,512}", "attention", p.dh);
  }
}

// ------------------------------------------------------------------------------------------
// VQ nearest-code search.  CTA = 8 rows x all K codes; warp w scans codes w, w+8, ...; lanes
// split D (float4 chunks) and butterfly-reduce; strict '<' keeps the first index on ties,
// matching torch.max(-dist) on CPU (core_vq.py:175-183).
template <int CH>   // D = 128 * CH
__global__ void __launch_bounds__(256)
vq_argmin_kernel(const float* __restrict__ x, int ldx, const float* __restrict__ embed, int64_t N, int K,
                 int64_t* __restrict__ idx) {
  pdl_entry();
  constexpr int R = 8, D = 128 * CH;
  __shared__ float sd[8][R];
  __shared__ int sk[8][R];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t r0 = (int64_t)blockIdx.x * R;
  float4 xv[R][CH];
  float xx[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      xv[r][c] = (r0 + r < N) ? *reinterpret_cast<const float4*>(x + (r0 + r) * ldx + c * 128 + lane * 4)
                               : make_float4(0.f, 0.f, 0.f, 0.f);
      s += (xv[r][c].x * xv[r][c].x + xv[r][c].y * xv[r][c].y) + (xv[r][c].z * xv[r][c].z + xv[r][c].w * xv[r][c].w);
    }
    xx[r] = warp_sum(s);
  }
  float best[R];
  int bestk[R];
#pragma unroll
  for (int r = 0; r < R; ++r) { best[r] = INFINITY; bestk[r] = 0x7fffffff; }
  for (int k = w; k < K; k += 8) {
    float4 ev[CH];
    float ee = 0.f;
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      ev[c] = __ldg(reinterpret_cast<const float4*>(embed + (int64_t)k * D + c * 128 + lane * 4));
      ee += (ev[c].x * ev[c].x + ev[c].y * ev[c].y) + (ev[c].z * ev[c].z + ev[c].w * ev[c].w);
    }
    ee = warp_sum(ee);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      float d = 0.f;
#pragma unroll
      for (int c = 0; c < CH; ++c)
        d += (xv[r][c].x * ev[c].x + xv[r][c].y * ev[c].y) + (xv[r][c].z * ev[c].z + xv[r][c].w * ev[c].w);
      d = warp_sum(d);
      const float dist = (xx[r] - 2.0f * d) + ee;
      if (dist < best[r]) { best[r] = dist; bestk[r] = k; }
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int r = 0; r < R; ++r) { sd[w][r] = best[r]; sk[w][r] = bestk[r]; }
  }
  __syncthreads();
  if (threadIdx.x < R && r0 + threadIdx.x < N) {
    float bd = sd[0][threadIdx.x];
    int bk = sk[0][threadIdx.x];
    for (int ww = 1; ww < 8; ++ww) {
      const float d = sd[ww][threadIdx.x];
      const int k = sk[ww][threadIdx.x];
      if (d < bd || (d == bd && k < bk)) { bd = d; bk = k; }
    }
    idx[r0 + threadIdx.x] = (int64_t)bk;
  }
}

int vq_argmin(const float* x, int ldx, const float* embed, int64_t N, int D, int K, int64_t* idx, cudaStream_t st) {
  MTTS_REQUIRE(x && embed && idx, "null pointer");
  MTTS_REQUIRE(K > 0 && D > 0 && ldx >= D, "bad dims");
  MTTS_REQUIRE(ldx % 4 == 0 && al16(x) && al16(embed), "x / embed must be 16-byte aligned with ldx % 4 == 0");
  if (N <= 0) return 0;
  const unsigned grid = (unsigned)cdiv64(N, 8);
  switch (D) {
    case 128: launch_k(vq_argmin_kernel<1>, grid, 256, 0, st, x, ldx, embed, N, K, idx); break;
    case 256: launch_k(vq_argmin_kernel<2>, grid, 256, 0, st, x, ldx, embed, N, K, idx); break;
    case 512: launch_k(vq_argmin_kernel<4>, grid, 256, 0, st, x, ldx, embed, N, K, idx); break;
    default: return fail(MTTS_ERR_UNSUPPORTED, "%s: codebook dim %lld not in {128,256,512}", "vq_argmin", D);
  }
  MTTS_CHECK_LAUNCH();
  return 0;
}

__global__ void vq_gather_kernel(const int64_t* __restrict__ idx, int idx_ld, const float* __restrict__ embed, int D,
                                 int K, int T_out, int repeat, float* __restrict__ y, int64_t y_sb, int ldy,
                                 int64_t total) {
  pdl_entry();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int d = (int)(i % D);
  const int64_t bt = i / D;
  const int t = (int)(bt % T_out);
  const int b = (int)(bt / T_out);
  int64_t code = idx[(int64_t)b * idx_ld + t / repeat];
  code = code < 0 ? 0 : (code >= K ? K - 1 : code);
  y[(int64_t)b * y_sb + (int64_t)t * ldy + d] = __ldg(embed + code * D + d);
}

int vq_gather(const int64_t* idx, int idx_ld, const float* embed, int D, int K, int B, int T_out, int repeat,
              float* y, int64_t y_sb, int ldy, cudaStream_t st) {
  MTTS_REQUIRE(idx && embed && y && repeat >= 1 && D > 0 && K > 0, "bad arguments");
  const int64_t total = (int64_t)B * T_out * D;
  if (total <= 0) return 0;
  launch_k(vq_gather_kernel, (unsigned)cdiv64(total, 256), 256, 0, st, idx, idx_ld, embed, D, K, T_out, repeat, y, y_sb, ldy, total);
  MTTS_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------
__global__ void maxpool_time_kernel(const float* __restrict__ x, int64_t x_sb, int ldx, float* __restrict__ y,
                                    int64_t y_sb, int ldy, int T, int To, int C, int k, int64_t total) {
  pdl_entry();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % C);
  const int64_t bt = i / C;
  const int to = (int)(bt % To);
  const int b = (int)(bt / To);
  const float* src = x + (int64_t)b * x_sb + c;
  float m = -INFINITY;
  for (int r = 0; r < k; ++r) {
    const int t = to * k + r;
    if (t < T) m = fmaxf(m, src[(int64_t)t * ldx]);
  }
  y[(int64_t)b * y_sb + (int64_t)to * ldy + c] = m;
}

int maxpool_time(const float* x, int64_t x_sb, int ldx, float* y, int64_t y_sb, int ldy, int B, int T, int C, int k,
                 cudaStream_t st) {
  MTTS_REQUIRE(x && y && k >= 1 && C > 0, "bad arguments");
  const int To = (T + k - 1) / k;
  const int64_t total = (int64_t)B * To * C;
  if (total <= 0) return 0;
  launch_k(maxpool_time_kernel, (unsigned)cdiv64(total, 256), 256, 0, st, x, x_sb, ldx, y, y_sb, ldy, T, To, C, k, total);
  MTTS_CHECK_LAUNCH();
  return 0;
}

__global__ void embed_pe_kernel(const int64_t* __restrict__ ids, int ids_ld, const float* __restrict__ table,
                                int vocab, int D, const float* __restrict__ pe, float alpha, int pe_offset, int T,
                                float* __restrict__ y, int64_t y_sb, int ldy, int64_t total) {
  pdl_entry();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int d = (int)(i % D);
  const int64_t bt = i / D;
  const int t = (int)(bt % T);
  const int b = (int)(bt / T);
  int64_t id = ids[(int64_t)b * ids_ld + t];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
  float v = __ldg(table + id * D + d);
  if (pe) v = v * 1.0f + alpha * __ldg(pe + (int64_t)(t + pe_offset) * D + d);
  y[(int64_t)b * y_sb + (int64_t)t * ldy + d] = v;
}

int embed_pe(const int64_t* ids, int ids_ld, const float* table, int vocab, int D, const float* pe, float alpha,
             int pe_offset, int B, int T, float* y, int64_t y_sb, int ldy, cudaStream_t st) {
  MTTS_REQUIRE(ids && table && y && D > 0 && vocab > 0, "bad arguments");
  const int64_t total = (int64_t)B * T * D;
  if (total <= 0) return 0;
  launch_k(embed_pe_kernel, (unsigned)cdiv64(total, 256), 256, 0, st, ids, ids_ld, table, vocab, D, pe, alpha, pe_offset, T, y, y_sb, ldy, total);
  MTTS_CHECK_LAUNCH();
  return 0;
}

__global__ void add_pe_kernel(const float* __restrict__ x, int64_t x_sb, int ldx, const float* __restrict__ pe,
                              float alpha, int T, int D, float* __restrict__ y, int64_t y_sb, int ldy, int64_t total) {
  pdl_entry();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int d = (int)(i % D);
  const int64_t bt = i / D;
  const int t = (int)(bt % T);
  const int b = (int)(bt / T);
  y[(int64_t)b * y_sb + (int64_t)t * ldy + d] =
      x[(int64_t)b * x_sb + (int64_t)t * ldx + d] * 1.0f + alpha * __ldg(pe + (int64_t)t * D + d);
}

int add_pe(const float* x, int64_t x_sb, int ldx, const float* pe, float alpha, int B, int T, int D, float* y,
           int64_t y_sb, int ldy, cudaStream_t st) {
  MTTS_REQUIRE(x && pe && y && D > 0, "bad arguments");
  const int64_t total = (int64_t)B * T * D;
  if (total <= 0) return 0;
  launch_k(add_pe_kernel, (unsigned)cdiv64(total, 256), 256, 0, st, x, x_sb, ldx, pe, alpha, T, D, y, y_sb, ldy, total);
  MTTS_CHECK_LAUNCH();
  return 0;
}

// LengthRegulator: CTA = 32 output rows of one utterance; thread 0 scans the durations of
// that utterance into shared memory, each warp binary-searches its rows.
__global__ void __launch_bounds__(256)
length_regulate_kernel(const float* __restrict__ x, int64_t x_sb, int ldx, const int32_t* __restrict__ dur, int dur_ld,
                       int Tp, int D, int L_out, float* __restrict__ y, int64_t y_sb, int ldy,
                       int32_t* __restrict__ totals) {
  pdl_entry();
  extern __shared__ int cum[];   // Tp + 1
  const int b = blockIdx.y;
  if (threadIdx.x == 0) {
    int s = 0;
    cum[0] = 0;
    for (int i = 0; i < Tp; ++i) {
      s += max(dur[(int64_t)b * dur_ld + i], 0);
      cum[i + 1] = s;
    }
    if (totals && blockIdx.x == 0) totals[b] = s;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int total = cum[Tp];
  for (int rr = w; rr < 32; rr += 8) {
    const int r = blockIdx.x * 32 + rr;
    if (r >= L_out) break;
    float* dst = y + (int64_t)b * y_sb + (int64_t)r * ldy;
    if (r >= total) {
      for (int d = lane; d < D; d += 32) dst[d] = 0.f;
      continue;
    }
    int lo = 0, hi = Tp;   // largest i with cum[i] <= r
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (cum[mid] <= r) lo = mid; else hi = mid;
    }
    const float* src = x + (int64_t)b * x_sb + (int64_t)lo * ldx;
    for (int d = lane; d < D; d += 32) dst[d] = src[d];
  }
}

int length_regulate(const float* x, int64_t x_sb, int ldx, const int32_t* dur, int dur_ld, int B, int Tp, int D,
                    int L_out, float* y, int64_t y_sb, int ldy, int32_t* totals, cudaStream_t st) {
  MTTS_REQUIRE(x && dur && D > 0 && Tp > 0 && B >= 0 && L_out >= 0, "bad arguments");
  MTTS_REQUIRE(Tp <= 8192, "Tp too large");
  if (B == 0) return 0;
  MTTS_REQUIRE(y || L_out == 0, "null output");
  dim3 grid((unsigned)(L_out > 0 ? cdiv64(L_out, 32) : 1), (unsigned)B);
  launch_k(length_regulate_kernel, grid, 256, (Tp + 1) * sizeof(int), st, x, x_sb, ldx, dur, dur_ld, Tp, D, L_out, y, y_sb, ldy, totals);
  MTTS_CHECK_LAUNCH();
  return 0;
}

// Generic strided (B,T,C) copy through a 32x32 shared tile so that both the read and the
// write are coalesced whichever of (t, c) is the unit-stride dim on each side.
__global__ void __launch_bounds__(256)
copy_strided_kernel(const float* __restrict__ x, int64_t x_sb, int64_t x_st, int64_t x_sc, float* __restrict__ y,
                    int64_t y_sb, int64_t y_st, int64_t y_sc, int T, int C, int pad_rep) {
  pdl_entry();
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int To = T + 2 * pad_rep;
  const int fx = threadIdx.x & 31, sy = threadIdx.x >> 5;   // 32 x 8
  const bool src_c_fast = (x_sc <= x_st);
  const bool dst_c_fast = (y_sc <= y_st);
  for (int s = sy; s < 32; s += 8) {
    const int tl = src_c_fast ? s : fx, cl = src_c_fast ? fx : s;
    const int t = t0 + tl, c = c0 + cl;
    if (t < To && c < C) {
      int ts = t - pad_rep;
      ts = ts < 0 ? 0 : (ts >= T ? T - 1 : ts);
      tile[tl][cl] = x[(int64_t)b * x_sb + (int64_t)ts * x_st + (int64_t)c * x_sc];
    }
  }
  __syncthreads();
  for (int s = sy; s < 32; s += 8) {
    const int tl = dst_c_fast ? s : fx, cl = dst_c_fast ? fx : s;
    const int t = t0 + tl, c = c0 + cl;
    if (t < To && c < C) y[(int64_t)b * y_sb + (int64_t)t * y_st + (int64_t)c * y_sc] = tile[tl][cl];
  }
}

int copy_strided(const float* x, int64_t x_sb, int64_t x_st, int64_t x_sc, float* y, int64_t y_sb, int64_t y_st,
                 int64_t y_sc, int B, int T, int C, int pad_rep, cudaStream_t st) {
  MTTS_REQUIRE(x && y && pad_rep >= 0, "bad arguments");
  if (B <= 0 || T <= 0 || C <= 0) return 0;
  MTTS_REQUIRE(B <= 65535 && cdiv64(C, 32) <= 65535, "grid too large");
  dim3 grid((unsigned)cdiv64(T + 2 * pad_rep, 32), (unsigned)cdiv64(C, 32), (unsigned)B);
  launch_k(copy_strided_kernel, grid, 256, 0, st, x, x_sb, x_st, x_sc, y, y_sb, y_st, y_sc, T, C, pad_rep);
  MTTS_CHECK_LAUNCH();
  return 0;
}

__global__ void mask_tail_kernel(float* __restrict__ x, int rows, int L, const int32_t* __restrict__ keep) {
  pdl_entry();
  const int b = blockIdx.z, r = blockIdx.y;
  const int k0 = max(keep[b], 0);
  float* xr = x + ((int64_t)b * rows + r) * L;
  for (int i = k0 + blockIdx.x * blockDim.x + threadIdx.x; i < L; i += gridDim.x * blockDim.x) xr[i] = 0.f;
}
int mask_tail(float* x, int B, int rows, int L, const int32_t* keep, cudaStream_t st) {
  MTTS_REQUIRE(x && keep && B >= 0 && rows >= 0 && L >= 0, "bad arguments");
  if (B == 0 || rows == 0 || L == 0) return 0;
  MTTS_REQUIRE(B <= 65535 && rows <= 65535, "grid too large");
  dim3 grid((unsigned)(cdiv64(L, 1024) < 64 ? cdiv64(L, 1024) : 64), (unsigned)rows, (unsigned)B);
  launch_k(mask_tail_kernel, grid, 256, 0, st, x, rows, L, keep);
  MTTS_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------
// Autoregressive-loop helpers (device-resident state: no host sync inside the loops).

// PLM step input (models/megatts2.py:173-175): X[b,s,:] = cat(tc[b,s,:], emb[codes[b,s]]) + alpha*pe[s]
__global__ void plm_build_input_kernel(const float* __restrict__ tc, int64_t tc_sb, int tc_ld, int tc_dim,
                                       const int64_t* __restrict__ codes, int codes_ld,
                                       const float* __restrict__ emb, int vq_dim, int vocab,
                                       const float* __restrict__ pe, float alpha, int S, float* __restrict__ X,
                                       int64_t total) {
  pdl_entry();
  const int D = tc_dim + vq_dim;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int d = (int)(i % D);
  const int64_t bs = i / D;
  const int s = (int)(bs % S);
  const int b = (int)(bs / S);
  float v;
  if (d < tc_dim) {
    v = tc[(int64_t)b * tc_sb + (int64_t)s * tc_ld + d];
  } else {
    int64_t id = codes[(int64_t)b * codes_ld + s];
    id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);
    v = __ldg(emb + id * vq_dim + (d - tc_dim));
  }
  X[i] = v * 1.0f + alpha * __ldg(pe + (int64_t)s * D + d);
}

int plm_build_input(const float* tc, int64_t tc_sb, int tc_ld, int tc_dim, const int64_t* codes, int codes_ld,
                    const float* emb, int vq_dim, int vocab, const float* pe, float alpha, int B, int S, float* X,
                    cudaStream_t st) {
  const int64_t total = (int64_t)B * S * (tc_dim + vq_dim);
  if (total <= 0) return 0;
  launch_k(plm_build_input_kernel, (unsigned)cdiv64(total, 256), 256, 0, st, tc, tc_sb, tc_ld, tc_dim, codes, codes_ld, emb, vq_dim, vocab, pe, alpha, S, X, total);
  MTTS_CHECK_LAUNCH();
  return 0;
}

// argmax over the last dim, first index on ties (torch.argmax on CPU); one warp per row.
// writes out_a[row*lda] and (optionally) out_b[row*ldb].
__global__ void argmax_rows_kernel(const float* __restrict__ x, int64_t ldx, int V, int rows, int64_t* out_a,
                                   int64_t lda, int64_t* out_b, int64_t ldb) {
  pdl_entry();
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const float* xr = x + (int64_t)row * ldx;
  float best = -INFINITY;
  int bi = 0x7fffffff;
  for (int i = lane; i < V; i += 32) {
    const float v = xr[i];
    if (v > best) { best = v; bi = i; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ob = __shfl_xor_sync(0xffffffffu, best, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ob > best || (ob == best && oi < bi)) { best = ob; bi = oi; }
  }
  if (lane == 0) {
    if (bi == 0x7fffffff) bi = 0;
    out_a[(int64_t)row * lda] = bi;
    if (out_b) out_b[(int64_t)row * ldb] = bi;
  }
}

int argmax_rows(const float* x, int64_t ldx, int V, int rows, int64_t* out_a, int64_t lda, int64_t* out_b, int64_t ldb,
                cudaStream_t st) {
  if (rows <= 0) return 0;
  launch_k(argmax_rows_kernel, (unsigned)cdiv64(rows, 4), 128, 0, st, x, ldx, V, rows, out_a, lda, out_b, ldb);
  MTTS_CHECK_LAUNCH();
  return 0;
}

__global__ void fill_i64_kernel(int64_t* p, int64_t stride, int n, int64_t v) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[(int64_t)i * stride] = v;
}
int fill_i64(int64_t* p, int64_t stride, int n, int64_t v, cudaStream_t st) {
  if (n <= 0) return 0;
  launch_k(fill_i64_kernel, (unsigned)cdiv64(n, 256), 256, 0, st, p, stride, n, v);
  MTTS_CHECK_LAUNCH();
  return 0;
}
__global__ void fill_f32_kernel(float* p, int64_t stride, int n, float v) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[(int64_t)i * stride] = v;
}
int fill_f32(float* p, int64_t stride, int n, float v, cudaStream_t st) {
  if (n <= 0) return 0;
  launch_k(fill_f32_kernel, (unsigned)cdiv64(n, 256), 256, 0, st, p, stride, n, v);
  MTTS_CHECK_LAUNCH();
  return 0;
}

// ADM step input (models/megatts2.py:265-269): X[b,s,:] = cat(tc_emb[b,s,:], p[b,s]*w_dt[:]) + alpha*pe[s]
__global__ void adm_build_input_kernel(const float* __restrict__ tc_emb, int64_t te_sb, int te_ld, int tc_emb_dim,
                                       const float* __restrict__ praw, int p_ld, const float* __restrict__ w_dt,
                                       int emb_dim, const float* __restrict__ pe, float alpha, int S,
                                       float* __restrict__ X, int64_t total) {
  pdl_entry();
  const int D = tc_emb_dim + emb_dim;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int d = (int)(i % D);
  const int64_t bs = i / D;
  const int s = (int)(bs % S);
  const int b = (int)(bs / S);
  float v;
  if (d < tc_emb_dim) v = tc_emb[(int64_t)b * te_sb + (int64_t)s * te_ld + d];
  else v = praw[(int64_t)b * p_ld + s] * __ldg(w_dt + (d - tc_emb_dim));
  X[i] = v * 1.0f + alpha * __ldg(pe + (int64_t)s * D + d);
}

int adm_build_input(const float* tc_emb, int64_t te_sb, int te_ld, int tc_emb_dim, const float* praw, int p_ld,
                    const float* w_dt, int emb_dim, const float* pe, float alpha, int B, int S, float* X,
                    cudaStream_t st) {
  const int64_t total = (int64_t)B * S * (tc_emb_dim + emb_dim);
  if (total <= 0) return 0;
  launch_k(adm_build_input_kernel, (unsigned)cdiv64(total, 256), 256, 0, st, tc_emb, te_sb, te_ld, tc_emb_dim, praw, p_ld, w_dt, emb_dim, pe, alpha, S, X, total);
  MTTS_CHECK_LAUNCH();
  return 0;
}

// ADM readout (models/megatts2.py:272-273): p[b, s_next] = x_last[b,:] . w_predict ; one warp per b
__global__ void adm_readout_kernel(const float* __restrict__ xl, int D, const float* __restrict__ w, int B,
                                   float* __restrict__ praw, int p_ld, int s_next) {
  pdl_entry();
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (b >= B) return;
  float s = 0.f;
  for (int d = lane; d < D; d += 32) s = fmaf(xl[(int64_t)b * D + d], __ldg(w + d), s);
  s = warp_sum(s);
  if (lane == 0) praw[(int64_t)b * p_ld + s_next] = s;
}
int adm_readout(const float* xl, int D, const float* w, int B, float* praw, int p_ld, int s_next, cudaStream_t st) {
  if (B <= 0) return 0;
  launch_k(adm_readout_kernel, (unsigned)cdiv64(B, 4), 128, 0, st, xl, D, w, B, praw, p_ld, s_next);
  MTTS_CHECK_LAUNCH();
  return 0;
}

// (p + 0.5).to(int32).clamp(1, 128)  (models/megatts2.py:275); praw row b holds [0, p_1..p_T]
__global__ void adm_finalize_kernel(const float* __restrict__ praw, int p_ld, int B, int T, int32_t* __restrict__ dur,
                                    float* __restrict__ raw_out) {
  pdl_entry();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * T) return;
  const int b = i / T, t = i - b * T;
  const float p = praw[(int64_t)b * p_ld + t + 1];
  int v = (int)(p + 0.5f);             // truncation toward zero, like Tensor.to(int32)
  v = v < 1 ? 1 : (v > 128 ? 128 : v);
  dur[i] = v;
  if (raw_out) raw_out[i] = p;
}
int adm_finalize(const float* praw, int p_ld, int B, int T, int32_t* dur, float* raw_out, cudaStream_t st) {
  if (B * T <= 0) return 0;
  launch_k(adm_finalize_kernel, (unsigned)cdiv64((int64_t)B * T, 256), 256, 0, st, praw, p_ld, B, T, dur, raw_out);
  MTTS_CHECK_LAUNCH();
  return 0;
}

}  // namespace mtts
