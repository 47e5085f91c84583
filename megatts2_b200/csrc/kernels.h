// Internal (C++) entry points shared by the drivers and the C ABI.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace mtts {
// Tensor-core operand formats ("planes": 2-byte elements in the activation's own (B, Tp, C) layout):
//   fmt 0  bf16x3: x = p0 + p1 + p2 (three bf16 terms, to ~2^-24); six MMAs per product
//   fmt 1  f16x2 : x = p0 + p1 * 2^-11 (two fp16 terms, the residual stored SCALED by 2^11 so it keeps the
//                  magnitude - and the normal range - of x; 22 significant bits); three MMAs per product
//                  (x0w0 | x0w1' + x1'w0, the second accumulator scaled by 2^-11 in the epilogue).  fp16 range:
//                  |x| > 65504 cannot be represented - the split then poisons the value (inf/NaN propagate to the
//                  output) and raises the caller-registered overflow flag (mtts_tc_overflow_bind).
enum { MTTS_TC_BF16X3 = 0, MTTS_TC_F16X2 = 1 };
constexpr float F16X2_SCALE = 2048.0f;           // 2^11
constexpr float F16X2_INV_SCALE = 1.0f / 2048.0f;

// optional plane output of a producer kernel (feeds the tensor-core engine without a split pass)
struct PlanesOut {
  __nv_bfloat16* p;      // plane 0; planes 1 (, 2) follow at +stride (, +2*stride) elements; 2-byte elements of `fmt`
  int64_t stride;
  int ld;                // row stride (elements)
  int act;               // activation applied to the planes copy (the consumer's pre-activation)
  float slope;
  int fmt;               // MTTS_TC_BF16X3 | MTTS_TC_F16X2
  int32_t* ovf;          // f16x2 range flag (device, may be null)
};

// 4 consecutive elements -> one 8-byte store per plane
__device__ __forceinline__ void store_planes4(__nv_bfloat16* planes, int64_t plane_stride, int64_t off, const float* v,
                                              int fmt = MTTS_TC_BF16X3, int32_t* ovf = nullptr) {
  if (fmt == MTTS_TC_F16X2) {
    // two elements per conversion instruction (cvt.rn.f16x2.f32); the range check is one NaN-propagating max per element
    const __half2 h01 = __floats2half2_rn(v[0], v[1]), h23 = __floats2half2_rn(v[2], v[3]);   // +-inf beyond the fp16 range
    const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
    const __half2 l01 = __floats2half2_rn((v[0] - f01.x) * F16X2_SCALE, (v[1] - f01.y) * F16X2_SCALE);   // exact difference,
    const __half2 l23 = __floats2half2_rn((v[2] - f23.x) * F16X2_SCALE, (v[3] - f23.y) * F16X2_SCALE);   // exact scaling
    uint2 o;
    o.x = *reinterpret_cast<const uint32_t*>(&h01);
    o.y = *reinterpret_cast<const uint32_t*>(&h23);
    *reinterpret_cast<uint2*>(planes + off) = o;
    o.x = *reinterpret_cast<const uint32_t*>(&l01);
    o.y = *reinterpret_cast<const uint32_t*>(&l23);
    *reinterpret_cast<uint2*>(planes + plane_stride + off) = o;
    if (ovf) {
      float m;
      asm("{\n\t.reg .f32 t0, t1, t2, t3;\n\tabs.f32 t0, %1;\n\tabs.f32 t1, %2;\n\tabs.f32 t2, %3;\n\tabs.f32 t3, %4;\n\t"
          "max.NaN.f32 t0, t0, t1;\n\tmax.NaN.f32 t2, t2, t3;\n\tmax.NaN.f32 %0, t0, t2;\n\t}"
          : "=f"(m) : "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]));
      if (!(m <= 65504.0f)) *ovf = 1;                                  // also NaN
    }
    return;
  }
  // bf16x3: round-to-nearest at every step
  __nv_bfloat16 p[3][4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    float a = v[e];
    p[0][e] = __float2bfloat16_rn(a);
    a -= __bfloat162float(p[0][e]);
    p[1][e] = __float2bfloat16_rn(a);
    a -= __bfloat162float(p[1][e]);
    p[2][e] = __float2bfloat16_rn(a);
  }
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    uint2 o;
    o.x = (uint32_t)__bfloat16_as_ushort(p[q][0]) | ((uint32_t)__bfloat16_as_ushort(p[q][1]) << 16);
    o.y = (uint32_t)__bfloat16_as_ushort(p[q][2]) | ((uint32_t)__bfloat16_as_ushort(p[q][3]) << 16);
    *reinterpret_cast<uint2*>(planes + q * plane_stride + off) = o;
  }
}
// the overflow flag registered for the current device (null if none) and the current device's id / SM count
int32_t* tc_ovf_ptr();
int cur_device();
int cur_device_sms();
int tc_plan_query(int sms, int B, int T, int Cin, int Cout, int k, int dil, int fmt, int64_t partial_bytes, int ln_rides, int32_t* out5);
static inline int tc_fmt_of_engine(int engine) { return engine == 2 ? MTTS_TC_F16X2 : MTTS_TC_BF16X3; }
int layernorm_ex(const float* x, int ldx, const float* gamma, const float* beta, const float* res, int ldr, float* y,
                 int ldy, int64_t rows, int C, float eps, int post_act, int accumulate, PlanesOut po, cudaStream_t st);
int conv1d_ffma(const mtts_conv_params& p, cudaStream_t st);
int conv1d(const mtts_conv_params& p, cudaStream_t st);   // engine dispatch (FFMA today)
bool conv_tc_eligible(const mtts_conv_params& p);
// Optional LayerNorm of the rows a split-K tap-GEMM has just reduced (the dense layers of the AR loops' early steps): the
// reduction kernel then also normalises each finished row and writes the next layer's operand planes, which saves the
// separate LayerNorm launch.  `done` is set when the fused kernel ran; the caller launches LayerNorm itself otherwise.
struct LnFuse {
  const float* gamma; const float* beta; float eps;
  PlanesOut po;
  int done;
};
int conv_tc(const mtts_conv_params& p, cudaStream_t st, LnFuse* ln = nullptr);
int halo_fill(void* planes_base, int B, int T, int C, int hl, int hr, int pad_mode, cudaStream_t st);
int64_t linear_tc_scratch_bytes(int64_t rows_cap, int K);
int linear_tc(const float* x, int ldx, int64_t M, int K, const void* w_planes, int N, const float* bias,
              const float* res, int ldr, float* y, int ldy, int pre_act, float pre_slope, int post_act,
              float out_scale, void* scratch, int64_t scratch_bytes, int64_t rows_cap, int fmt, cudaStream_t st);
int split_planes(const float* x, int ldx, int64_t rows, int C, void* planes, int fmt, cudaStream_t st);
int split_pad(const float* x, int64_t x_sb, int ldx, int B, int T, int C, int hl, int hr, int pad_mode, int act, float slope,
              void* planes_base, int fmt, cudaStream_t st);
int tc_overflow_bind(int32_t* flag);
int mask_tail(float* x, int B, int rows, int L, const int32_t* keep, cudaStream_t st);
int layernorm(const float* x, int ldx, const float* gamma, const float* beta, const float* res, int ldr, float* y,
              int ldy, int64_t rows, int C, float eps, int post_act, int accumulate, cudaStream_t st);
int attention(const mtts_attn_params& p, cudaStream_t st);
bool attention_tc_eligible(const mtts_attn_params& p);
int attention_tc(const mtts_attn_params& p, cudaStream_t st);
int vq_argmin(const float* x, int ldx, const float* embed, int64_t N, int D, int K, int64_t* idx, cudaStream_t st);
int vq_gather(const int64_t* idx, int idx_ld, const float* embed, int D, int K, int B, int T_out, int repeat, float* y,
              int64_t y_sb, int ldy, cudaStream_t st);
int maxpool_time(const float* x, int64_t x_sb, int ldx, float* y, int64_t y_sb, int ldy, int B, int T, int C, int k,
                 cudaStream_t st);
int embed_pe(const int64_t* ids, int ids_ld, const float* table, int vocab, int D, const float* pe, float alpha,
             int pe_offset, int B, int T, float* y, int64_t y_sb, int ldy, cudaStream_t st);
int add_pe(const float* x, int64_t x_sb, int ldx, const float* pe, float alpha, int B, int T, int D, float* y,
           int64_t y_sb, int ldy, cudaStream_t st);
int length_regulate(const float* x, int64_t x_sb, int ldx, const int32_t* dur, int dur_ld, int B, int Tp, int D,
                    int L_out, float* y, int64_t y_sb, int ldy, int32_t* totals, cudaStream_t st);
int copy_strided(const float* x, int64_t x_sb, int64_t x_st, int64_t x_sc, float* y, int64_t y_sb, int64_t y_st,
                 int64_t y_sc, int B, int T, int C, int pad_rep, cudaStream_t st);
int mel_spectrogram(const float* wav, int64_t wav_sb, int B, int L, const int32_t* lens, const float* window,
                    const float* fb_w, const int32_t* fb_off, const int32_t* fb_start, int n_mels, float clamp_min,
                    float* out, int64_t out_sb, int64_t out_sm, int64_t out_sf, cudaStream_t st);
// AR-loop helpers
int plm_build_input(const float* tc, int64_t tc_sb, int tc_ld, int tc_dim, const int64_t* codes, int codes_ld,
                    const float* emb, int vq_dim, int vocab, const float* pe, float alpha, int B, int S, float* X,
                    cudaStream_t st);
int argmax_rows(const float* x, int64_t ldx, int V, int rows, int64_t* out_a, int64_t lda, int64_t* out_b, int64_t ldb,
                cudaStream_t st);
int fill_i64(int64_t* p, int64_t stride, int n, int64_t v, cudaStream_t st);
int fill_f32(float* p, int64_t stride, int n, float v, cudaStream_t st);
int adm_build_input(const float* tc_emb, int64_t te_sb, int te_ld, int tc_emb_dim, const float* praw, int p_ld,
                    const float* w_dt, int emb_dim, const float* pe, float alpha, int B, int S, float* X,
                    cudaStream_t st);
int adm_readout(const float* xl, int D, const float* w, int B, float* praw, int p_ld, int s_next, cudaStream_t st);
int adm_finalize(const float* praw, int p_ld, int B, int T, int32_t* dur, float* raw_out, cudaStream_t st);

// convenience: dense linear layer  Y[M,N] = act(X[M,K] W + b) (+ res)
inline mtts_conv_params linear_params(const float* x, int ldx, const float* w, const float* bias, float* y, int ldy,
                                      int64_t M, int K, int N) {
  mtts_conv_params p;
  memset(&p, 0, sizeof(p));
  p.x = x; p.ldx = ldx; p.x_batch_stride = 0;
  p.w = w; p.bias = bias;
  p.y = y; p.ldy = ldy; p.y_batch_stride = 0;
  p.B = 1; p.Tin = (int32_t)M; p.Tout = (int32_t)M; p.Cin = K; p.Cout = N;
  p.k = 1; p.stride = 1; p.dil = 1; p.pad = 0; p.pad_mode = MTTS_PAD_ZERO;
  p.out_scale = 1.0f;
  return p;
}
// "same" stride-1 conv over (B, T, Cin) -> (B, T, Cout), contiguous buffers
inline mtts_conv_params conv_same_params(const float* x, const float* w, const float* bias, float* y, int B, int T,
                                         int Cin, int Cout, int k, int dil, int pad_mode) {
  mtts_conv_params p;
  memset(&p, 0, sizeof(p));
  p.x = x; p.ldx = Cin; p.x_batch_stride = (int64_t)T * Cin;
  p.w = w; p.bias = bias;
  p.y = y; p.ldy = Cout; p.y_batch_stride = (int64_t)T * Cout;
  p.B = B; p.Tin = T; p.Tout = T; p.Cin = Cin; p.Cout = Cout;
  p.k = k; p.stride = 1; p.dil = dil; p.pad = dil * (k - 1) / 2; p.pad_mode = pad_mode;
  p.out_scale = 1.0f;
  return p;
}
}  // namespace mtts
