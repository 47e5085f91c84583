// Composite drivers: whole sub-networks of the synthesis path enqueued from C++ (no Python
// per-kernel overhead, no host sync inside).  Buffers come from the caller's workspace.
#include <mutex>
#include <vector>

#include "kernels.h"

namespace mtts {

// Optional per-launch timing of the tap-GEMM kernels (bench.py's roofline leg): CUDA events on
// the launching stream around every conv1d launch; off by default, never on the timed path.
struct ProfRec { cudaEvent_t a, b; double flops; bool tc = false; };
static std::mutex g_prof_mu;
static bool g_prof_on = false;
static std::vector<ProfRec> g_prof;

int conv1d(const mtts_conv_params& p, cudaStream_t st) {
  const bool tc = conv_tc_eligible(p);
  if (!g_prof_on) return tc ? conv_tc(p, st) : conv1d_ffma(p, st);
  std::lock_guard<std::mutex> lk(g_prof_mu);
  ProfRec r;
  if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess)
    return fail(MTTS_ERR_CUDA, "%s: cudaEventCreate failed", "profile");
  r.flops = 2.0 * (double)p.B * p.Tout * p.Cout * p.Cin * p.k;
  r.tc = tc;
  cudaEventRecord(r.a, st);
  const int rc = tc ? conv_tc(p, st) : conv1d_ffma(p, st);
  cudaEventRecord(r.b, st);
  g_prof.push_back(r);
  return rc;
}

// tensor-core context of a composite driver call: engine switch + scratch for activation planes
struct ConvTc { int engine; void* scratch; int64_t bytes; };
static inline void attach_tc(mtts_conv_params& p, const void* w_tc, const ConvTc* tc) {
  if (tc && tc->engine >= 1 && w_tc && tc->scratch) {
    p.w_tc = w_tc; p.tc_scratch = tc->scratch; p.tc_scratch_bytes = tc->bytes; p.tc_fmt = tc_fmt_of_engine(tc->engine);
  }
}
static inline int64_t conv_tc_scratch_need(int64_t B, int64_t Tp, int64_t C) { return 6 * B * Tp * C + 4096; }

// scratch for the tensor-core engine's activation planes, carved once per driver call so that the
// (cached) TMA descriptors keep hitting across the steps of an autoregressive loop
struct TcScratch { void* p; int64_t bytes; int64_t rows_cap; int fmt; };

constexpr int64_t TC_PARTIAL_BYTES = 64ll << 20;
static inline int64_t tc_planes_bytes(const mtts_encoder* e, int64_t rows_cap) {
  return align_up(6 * rows_cap * ((int64_t)e->d_model + e->ff_dim) + 8192, 1024);
}
static int64_t tc_scratch_bytes(const mtts_encoder* e, int64_t rows_cap) {
  if (e->engine < 1) return 0;
  const int kmax = e->ff_dim > e->d_model ? e->ff_dim : e->d_model;
  // conv-FF (k = 5): padded planes need 4 halo rows per sequence; rows_cap + 4*rows_cap covers any batch split
  if (e->conv_ff) return linear_tc_scratch_bytes(5 * rows_cap + 64, kmax) + 4096;
  // linear FF, fused plane flow: P_a (rows_cap x D) and P_b (rows_cap x F), three bf16 planes each,
  // followed by the split-K partial-sum area (used when a layer has too few tiles to fill the GPU)
  return tc_planes_bytes(e, rows_cap) + TC_PARTIAL_BYTES;
}
static inline void tc_partial_area(const mtts_encoder* e, const TcScratch* tc, void** ptr, int64_t* bytes) {
  *ptr = nullptr; *bytes = 0;
  if (!tc || !tc->p || e->conv_ff) return;
  const int64_t off = tc_planes_bytes(e, tc->rows_cap);
  if (tc->bytes >= off + TC_PARTIAL_BYTES) { *ptr = (char*)tc->p + off; *bytes = TC_PARTIAL_BYTES; }
}

// tensor-core GEMM on planes that a producer kernel already wrote (no split pass); optional plane output
static int lin_planes(const TcScratch* tc, __nv_bfloat16* planes, int64_t M, int K, int N, const void* wtc,
                      const float* bias, const float* res, int ldr, float* y, int ldy, int post_act,
                      __nv_bfloat16* out_planes, int out_ld, cudaStream_t st, void* partial = nullptr,
                      int64_t partial_bytes = 0, LnFuse* ln = nullptr) {
  mtts_conv_params p = linear_params(nullptr, K, nullptr, bias, y, ldy, M, K, N);
  p.res = res; p.ldr = ldr; p.post_act = post_act;
  p.tc_partial = partial; p.tc_partial_bytes = partial_bytes;
  p.w_tc = wtc; p.tc_scratch = planes; p.tc_scratch_bytes = 6 * tc->rows_cap * (int64_t)K + 4096; p.tc_rows_cap = tc->rows_cap;
  p.tc_presplit = 1; p.tc_fmt = tc->fmt;
  if (out_planes) {
    p.tc_out_planes = out_planes; p.tc_out_plane_stride = tc->rows_cap * (int64_t)out_ld; p.tc_out_ld = out_ld;
    p.tc_out_tp = (int32_t)tc->rows_cap; p.tc_out_hl = 0; p.tc_out_act = MTTS_ACT_NONE;
  }
  if (!conv_tc_eligible(p))
    return fail(MTTS_ERR_UNSUPPORTED, "%s: fused tensor-core layer not eligible (M=%lld N=%lld)", "encoder", M, N);
  ProfRec r;
  const bool prof = g_prof_on;
  if (prof) {
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    r.flops = 2.0 * (double)M * N * K; r.tc = true;
    cudaEventRecord(r.a, st);
  }
  const int rc = conv_tc(p, st, ln);
  if (prof) {
    cudaEventRecord(r.b, st);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof.push_back(r);
  }
  return rc;
}

// dense layer dispatch: one tap-GEMM call; conv1d() picks the tcgen05 engine when planes + scratch are attached
// and the shape is eligible (M >= 128), else the exact FFMA engine
static int lin(const mtts_encoder* e, const TcScratch* tc, const float* x, int ldx, int64_t M, int K, int N,
               const float* w32, const void* wtc, const float* bias, const float* res, int ldr, float* y, int ldy,
               int post_act, cudaStream_t st) {
  mtts_conv_params p = linear_params(x, ldx, w32, bias, y, ldy, M, K, N);
  p.res = res; p.ldr = ldr; p.post_act = post_act;
  if (e->engine >= 1 && tc && tc->p && wtc) {
    p.w_tc = wtc; p.tc_scratch = tc->p; p.tc_scratch_bytes = tc->bytes; p.tc_rows_cap = tc->rows_cap; p.tc_fmt = tc->fmt;
  }
  return conv1d(p, st);
}

// ------------------------------------------------------------------------------------------
// TransformerEncoder.forward (modules/transformer.py:88-102, 119-133)
static int64_t encoder_ws_floats(const mtts_encoder* e, int B, int T) {
  const int64_t M = (int64_t)B * T, D = e->d_model, F = e->ff_dim;
  // xw, h, qkv(3D), a, f  (+ alignment slack)
  return M * (D + D + 3 * D + D + F) + 5 * 64;
}

static int encoder_forward(const mtts_encoder* e, const float* x, float* y, int B, int T, const float* mask,
                           int64_t mask_sb, int64_t mask_sh, int64_t mask_sq, int last_row_only, Arena& ar,
                           const TcScratch* tc, cudaStream_t st) {
  const int D = e->d_model, H = e->n_heads, F = e->ff_dim, dh = D / H;
  MTTS_REQUIRE(D % H == 0, "d_model not divisible by n_heads");
  MTTS_REQUIRE(!(last_row_only && e->conv_ff), "last_row_only needs a linear feed-forward");
  MTTS_REQUIRE(e->n_layers >= 1, "no layers");
  const int64_t M = (int64_t)B * T;
  if (M == 0) return 0;
  float* xw = last_row_only ? ar.take<float>(M * D) : y;   // running activations (B,T,D)
  float* h = ar.take<float>(M * D);
  float* qkv = ar.take<float>(M * 3 * D);
  float* a = ar.take<float>(M * D);
  float* f = ar.take<float>(M * F);
  if (!ar.ok()) return fail(MTTS_ERR_WORKSPACE, "%s: workspace too small (need %lld bytes)", "encoder", ar.off);
  const float scale = 1.0f / sqrtf((float)dh);
  const float* xin = x;
  // Fused plane flow (tensor-core engine, linear FF, M >= 128): LayerNorm / attention / the FF1 epilogue write
  // their result directly as bf16x3 planes, so no split pass and no fp32 round trip feeds the GEMMs.
  bool fused = e->engine >= 1 && !e->conv_ff && tc && tc->p && M >= 128 && D % 32 == 0 && F % 32 == 0 &&
               tc->bytes >= tc_planes_bytes(e, tc->rows_cap) && tc->rows_cap >= M;
  for (int l = 0; fused && l < e->n_layers; ++l)
    fused = e->layers[l].w_qkv_tc && e->layers[l].w_o_tc && e->layers[l].w_ff1_tc && e->layers[l].w_ff2_tc;
  __nv_bfloat16* Pa = nullptr;
  __nv_bfloat16* Pb = nullptr;
  if (fused) {
    Pa = reinterpret_cast<__nv_bfloat16*>((((uintptr_t)tc->p) + 1023) & ~(uintptr_t)1023);
    Pb = reinterpret_cast<__nv_bfloat16*>((((uintptr_t)(Pa + 3 * tc->rows_cap * (int64_t)D)) + 1023) & ~(uintptr_t)1023);
  }
  const PlanesOut pa_out{Pa, tc ? tc->rows_cap * (int64_t)D : 0, D, MTTS_ACT_NONE, 0.f, tc ? tc->fmt : 0, tc_ovf_ptr()};
  void* part = nullptr;
  int64_t part_bytes = 0;
  if (fused) tc_partial_area(e, tc, &part, &part_bytes);
  bool ln1_done = false;     // LN1 of the current layer was produced by the previous layer's split-K reduction
  for (int l = 0; l < e->n_layers; ++l) {
    const mtts_encoder_layer& L = e->layers[l];
    const bool last = last_row_only && (l == e->n_layers - 1);
    if (fused) {
      // (when the previous layer's FF2 was a split-K launch its reduction already normalised these rows into P_a)
      if (!ln1_done) MTTS_TRY(layernorm_ex(xin, D, L.ln1_g, L.ln1_b, nullptr, 0, nullptr, 0, M, D, 1e-5f, 0, 0, pa_out, st));
      ln1_done = false;
      MTTS_TRY(lin_planes(tc, Pa, M, D, 3 * D, L.w_qkv_tc, L.b_qkv, nullptr, 0, qkv, 3 * D, 0, nullptr, 0, st, part, part_bytes));
    } else {
      // h = LN1(x);  qkv = h Wqkv + b
      MTTS_TRY(layernorm(xin, D, L.ln1_g, L.ln1_b, nullptr, 0, h, D, M, D, 1e-5f, 0, 0, st));
      MTTS_TRY(lin(e, tc, h, D, M, D, 3 * D, L.w_qkv, L.w_qkv_tc, L.b_qkv, nullptr, 0, qkv, 3 * D, 0, st));
    }
    mtts_attn_params ap;
    memset(&ap, 0, sizeof(ap));
    ap.B = B; ap.H = H; ap.Tk = T; ap.dh = dh; ap.scale = scale;
    ap.k = qkv + D; ap.k_sb = (int64_t)T * 3 * D; ap.k_st = 3 * D;
    ap.v = qkv + 2 * D; ap.v_sb = (int64_t)T * 3 * D; ap.v_st = 3 * D;
    ap.mask = mask; ap.mask_sb = mask_sb; ap.mask_sh = mask_sh; ap.mask_sq = mask_sq;
    if (!last) {
      ap.q = qkv; ap.q_sb = (int64_t)T * 3 * D; ap.q_st = 3 * D; ap.Tq = T;
      if (fused) {
        ap.o = nullptr; ap.o_planes = Pa; ap.o_plane_stride = tc->rows_cap * (int64_t)D; ap.o_planes_ld = D; ap.o_planes_fmt = tc->fmt;
        MTTS_TRY(attention(ap, st));
        // out-projection (+ residual); a split-K launch's reduction kernel applies LN2 to the finished rows as well
        LnFuse ln2{L.ln2_g, L.ln2_b, 1e-5f, pa_out, 0};
        MTTS_TRY(lin_planes(tc, Pa, M, D, D, L.w_o_tc, L.b_o, xin, D, xw, D, 0, nullptr, 0, st, part, part_bytes, &ln2));
        if (!ln2.done) MTTS_TRY(layernorm_ex(xw, D, L.ln2_g, L.ln2_b, nullptr, 0, nullptr, 0, M, D, 1e-5f, 0, 0, pa_out, st));
        // FF1: relu(h W1 + b1) goes straight to planes P_b; FF2 reads them
        MTTS_TRY(lin_planes(tc, Pa, M, D, F, L.w_ff1_tc, L.b_ff1, nullptr, 0, nullptr, 0, MTTS_ACT_RELU, Pb, F, st, part, part_bytes));
        // FF2 (+ residual); likewise the NEXT layer's LN1 (all rows are consumed by it unless that layer is the pruned last one
        // - its LN1 still runs over all rows, only its later stages use the last row)
        const bool next_ln = l + 1 < e->n_layers;
        LnFuse ln1{next_ln ? e->layers[l + 1].ln1_g : nullptr, next_ln ? e->layers[l + 1].ln1_b : nullptr, 1e-5f, pa_out, 0};
        MTTS_TRY(lin_planes(tc, Pb, M, F, D, L.w_ff2_tc, L.b_ff2, xw, D, xw, D, 0, nullptr, 0, st, part, part_bytes,
                            next_ln ? &ln1 : nullptr));
        ln1_done = ln1.done != 0;
        xin = xw;
        continue;
      }
      ap.o = a; ap.o_sb = (int64_t)T * D; ap.o_st = D;
      MTTS_TRY(attention(ap, st));
      // x = x + a Wo + bo
      MTTS_TRY(lin(e, tc, a, D, M, D, D, L.w_o, L.w_o_tc, L.b_o, xin, D, xw, D, 0, st));
      if (e->conv_ff) {
        // x = LN2(x); x = x + conv5(relu(conv5(x)))       (transformer.py:96-98)
        MTTS_TRY(layernorm(xw, D, L.ln2_g, L.ln2_b, nullptr, 0, xw, D, M, D, 1e-5f, 0, 0, st));
        ConvTc ctc{e->engine, tc ? tc->p : nullptr, tc ? tc->bytes : 0};
        mtts_conv_params c1 = conv_same_params(xw, L.w_ff1, L.b_ff1, f, B, T, D, F, 5, 1, MTTS_PAD_ZERO);
        c1.post_act = MTTS_ACT_RELU;
        attach_tc(c1, L.w_ff1_tc, &ctc);
        MTTS_TRY(conv1d(c1, st));
        mtts_conv_params c2 = conv_same_params(f, L.w_ff2, L.b_ff2, xw, B, T, F, D, 5, 1, MTTS_PAD_ZERO);
        c2.res = xw; c2.res_batch_stride = (int64_t)T * D; c2.ldr = D;
        attach_tc(c2, L.w_ff2_tc, &ctc);
        MTTS_TRY(conv1d(c2, st));
      } else {
        // x = x + W2 relu(W1 LN2(x) + b1) + b2             (transformer.py:101)
        MTTS_TRY(layernorm(xw, D, L.ln2_g, L.ln2_b, nullptr, 0, h, D, M, D, 1e-5f, 0, 0, st));
        MTTS_TRY(lin(e, tc, h, D, M, D, F, L.w_ff1, L.w_ff1_tc, L.b_ff1, nullptr, 0, f, F, MTTS_ACT_RELU, st));
        MTTS_TRY(lin(e, tc, f, F, M, F, D, L.w_ff2, L.w_ff2_tc, L.b_ff2, xw, D, xw, D, 0, st));
      }
      xin = xw;
    } else {
      // final layer, last position only (exact: nothing else is consumed downstream)
      ap.q = qkv + (int64_t)(T - 1) * 3 * D; ap.q_sb = (int64_t)T * 3 * D; ap.q_st = 3 * D; ap.Tq = 1;
      if (mask) ap.mask = mask + (int64_t)(T - 1) * mask_sq;
      if (fused && B >= 32) {
        // the B last rows as one half-filled 128-row tile on the tensor cores (split-K fills the SMs): the attention rows,
        // LN2 and FF1 write operand planes like the full-sequence layers.  The exact-FFMA form below took 21 + 5 us per
        // dense layer at B = 64 (weight streaming through the FP32 pipe), 4 layers per AR step.
        ap.o = nullptr; ap.o_planes = Pa; ap.o_plane_stride = tc->rows_cap * (int64_t)D; ap.o_planes_ld = D; ap.o_planes_fmt = tc->fmt;
        MTTS_TRY(attention(ap, st));
        MTTS_TRY(lin_planes(tc, Pa, B, D, D, L.w_o_tc, L.b_o, xin + (int64_t)(T - 1) * D, T * D, y, D, 0, nullptr, 0, st, part, part_bytes));
        MTTS_TRY(layernorm_ex(y, D, L.ln2_g, L.ln2_b, nullptr, 0, nullptr, 0, B, D, 1e-5f, 0, 0, pa_out, st));
        MTTS_TRY(lin_planes(tc, Pa, B, D, F, L.w_ff1_tc, L.b_ff1, nullptr, 0, nullptr, 0, MTTS_ACT_RELU, Pb, F, st, part, part_bytes));
        MTTS_TRY(lin_planes(tc, Pb, B, F, D, L.w_ff2_tc, L.b_ff2, y, D, y, D, 0, nullptr, 0, st, part, part_bytes));
        continue;
      }
      ap.o = a; ap.o_sb = D; ap.o_st = D;
      MTTS_TRY(attention(ap, st));
      mtts_conv_params p;
      memset(&p, 0, sizeof(p));
      p.x = a; p.ldx = D; p.x_batch_stride = D;
      p.w = L.w_o; p.bias = L.b_o;
      p.res = xin + (int64_t)(T - 1) * D; p.res_batch_stride = (int64_t)T * D; p.ldr = D;
      p.y = y; p.ldy = D; p.y_batch_stride = D;
      p.B = B; p.Tin = 1; p.Tout = 1; p.Cin = D; p.Cout = D; p.k = 1; p.stride = 1; p.dil = 1;
      p.out_scale = 1.0f;
      // M = B rows only: the FFMA engine splits K across CTAs into the tensor-core scratch (when present)
      auto scratch = [&](mtts_conv_params& q) {
        if (tc && tc->p) { q.tc_scratch = tc->p; q.tc_scratch_bytes = tc->bytes; }
      };
      scratch(p);
      MTTS_TRY(conv1d(p, st));
      MTTS_TRY(layernorm(y, D, L.ln2_g, L.ln2_b, nullptr, 0, h, D, B, D, 1e-5f, 0, 0, st));
      mtts_conv_params p1 = linear_params(h, D, L.w_ff1, L.b_ff1, f, F, B, D, F);
      p1.post_act = MTTS_ACT_RELU;
      scratch(p1);
      MTTS_TRY(conv1d(p1, st));
      mtts_conv_params p2 = linear_params(f, F, L.w_ff2, L.b_ff2, y, D, B, F, D);
      p2.res = y; p2.ldr = D;
      scratch(p2);
      MTTS_TRY(conv1d(p2, st));
    }
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// MegaPLM.infer (models/megatts2.py:165-181)
static int64_t plm_ws_floats(const mtts_plm* m, int B, int T) {
  const int64_t D = m->enc.d_model;
  return encoder_ws_floats(&m->enc, B, T) + tc_scratch_bytes(&m->enc, (int64_t)B * T) / 4 + 512 + (int64_t)B * T * D + (int64_t)B * D + (int64_t)B * m->vq_bins +
         2 * ((int64_t)B * (T + 1) + 64) + 6 * 64;
}

static int plm_infer(const mtts_plm* m, const float* tc, int64_t tc_sb, int tc_ld, int B, int T, int64_t* codes_out,
                     float* logits_out, void* ws, int64_t ws_bytes, cudaStream_t st) {
  const int D = m->enc.d_model, V = m->vq_bins;
  MTTS_REQUIRE(D == m->tc_dim + m->vq_dim, "d_model != tc_dim + vq_dim");
  MTTS_REQUIRE(tc && codes_out && m->pc_embedding && m->w_predict && m->pe, "null pointer");
  if (B <= 0 || T <= 0) return 0;
  Arena top(ws, ws_bytes);
  float* X = top.take<float>((int64_t)B * T * D);
  float* xl = top.take<float>((int64_t)B * D);
  float* logits = top.take<float>((int64_t)B * V);
  int64_t* codes = top.take<int64_t>((int64_t)B * (T + 1));
  TcScratch tcs{nullptr, tc_scratch_bytes(&m->enc, (int64_t)B * T), (int64_t)B * T, tc_fmt_of_engine(m->enc.engine)};
  if (tcs.bytes) tcs.p = top.take<char>(tcs.bytes);
  const int64_t enc_off = align_up(top.off, 256);
  if (enc_off + encoder_ws_floats(&m->enc, B, T) * 4 > ws_bytes)
    return fail(MTTS_ERR_WORKSPACE, "%s: workspace too small (need %lld bytes)", "plm_infer",
                enc_off + encoder_ws_floats(&m->enc, B, T) * 4);
  MTTS_TRY(fill_i64(codes, T + 1, B, (int64_t)V, st));   // BOS = vq_bins (megatts2.py:170-171)
  for (int t = 0; t < T; ++t) {
    const int S = t + 1;
    MTTS_TRY(plm_build_input(tc, tc_sb, tc_ld, m->tc_dim, codes, T + 1, m->pc_embedding, m->vq_dim, V + 2, m->pe,
                             m->pe_alpha, B, S, X, st));
    Arena ar((char*)ws + enc_off, ws_bytes - enc_off);
    MTTS_TRY(encoder_forward(&m->enc, X, xl, B, S, nullptr, 0, 0, 0, 1, ar, &tcs, st));
    float* lg = logits_out ? logits_out + (int64_t)t * V : logits;
    const int64_t lg_sb = logits_out ? (int64_t)T * V : V;
    mtts_conv_params p;
    memset(&p, 0, sizeof(p));
    p.x = xl; p.ldx = D; p.x_batch_stride = D;
    p.w = m->w_predict;
    p.y = lg; p.ldy = V; p.y_batch_stride = lg_sb;
    p.B = B; p.Tin = 1; p.Tout = 1; p.Cin = D; p.Cout = V; p.k = 1; p.stride = 1; p.dil = 1; p.out_scale = 1.0f;
    if (tcs.p) { p.tc_scratch = tcs.p; p.tc_scratch_bytes = tcs.bytes; }
    MTTS_TRY(conv1d(p, st));
    MTTS_TRY(argmax_rows(lg, lg_sb, V, B, codes + (t + 1), T + 1, codes_out + t, T, st));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// MegaADM.infer (models/megatts2.py:257-275)
static int64_t adm_ws_floats(const mtts_adm* m, int B, int T) {
  const int64_t D = m->enc.d_model;
  return encoder_ws_floats(&m->enc, B, T) + tc_scratch_bytes(&m->enc, (int64_t)B * T) / 4 + 512 + (int64_t)B * T * D + (int64_t)B * D + (int64_t)B * T * m->tc_emb_dim +
         (int64_t)B * (T + 1) + 6 * 64;
}

static int adm_infer(const mtts_adm* m, const float* tc, int64_t tc_sb, int tc_ld, int B, int T, int32_t* dur_out,
                     float* raw_out, void* ws, int64_t ws_bytes, cudaStream_t st) {
  const int D = m->enc.d_model;
  MTTS_REQUIRE(D == m->emb_dim + m->tc_emb_dim, "d_model != emb_dim + tc_emb_dim");
  MTTS_REQUIRE(tc && dur_out && m->w_dt && m->w_tc && m->w_predict && m->pe, "null pointer");
  if (B <= 0 || T <= 0) return 0;
  Arena top(ws, ws_bytes);
  float* X = top.take<float>((int64_t)B * T * D);
  float* xl = top.take<float>((int64_t)B * D);
  float* tc_emb = top.take<float>((int64_t)B * T * m->tc_emb_dim);
  float* praw = top.take<float>((int64_t)B * (T + 1));
  TcScratch tcs{nullptr, tc_scratch_bytes(&m->enc, (int64_t)B * T), (int64_t)B * T, tc_fmt_of_engine(m->enc.engine)};
  if (tcs.bytes) tcs.p = top.take<char>(tcs.bytes);
  const int64_t enc_off = align_up(top.off, 256);
  if (enc_off + encoder_ws_floats(&m->enc, B, T) * 4 > ws_bytes)
    return fail(MTTS_ERR_WORKSPACE, "%s: workspace too small (need %lld bytes)", "adm_infer",
                enc_off + encoder_ws_floats(&m->enc, B, T) * 4);
  // tc_linear_emb(tc_latents[:, :t+1]) is step-invariant row by row: computed once (exact)
  {
    mtts_conv_params p;
    memset(&p, 0, sizeof(p));
    p.x = tc; p.ldx = tc_ld; p.x_batch_stride = tc_sb;
    p.w = m->w_tc;
    p.y = tc_emb; p.ldy = m->tc_emb_dim; p.y_batch_stride = (int64_t)T * m->tc_emb_dim;
    p.B = B; p.Tin = T; p.Tout = T; p.Cin = m->tc_dim; p.Cout = m->tc_emb_dim; p.k = 1; p.stride = 1; p.dil = 1;
    p.out_scale = 1.0f;
    MTTS_TRY(conv1d(p, st));
  }
  MTTS_TRY(fill_f32(praw, T + 1, B, 0.0f, st));   // p_code = [[0]] (megatts2.py:262-263)
  for (int t = 0; t < T; ++t) {
    const int S = t + 1;
    MTTS_TRY(adm_build_input(tc_emb, (int64_t)T * m->tc_emb_dim, m->tc_emb_dim, m->tc_emb_dim, praw, T + 1, m->w_dt,
                             m->emb_dim, m->pe, m->pe_alpha, B, S, X, st));
    Arena ar((char*)ws + enc_off, ws_bytes - enc_off);
    MTTS_TRY(encoder_forward(&m->enc, X, xl, B, S, nullptr, 0, 0, 0, 1, ar, &tcs, st));
    MTTS_TRY(adm_readout(xl, D, m->w_predict, B, praw, T + 1, t + 1, st));
  }
  MTTS_TRY(adm_finalize(praw, T + 1, B, T, dur_out, raw_out, st));
  return 0;
}

// ------------------------------------------------------------------------------------------
// Opt-in causal KV-cache decode (SURVEY.md 8f-1).  NOT the parity path of infer(): the reference's infer()
// re-runs the stack bidirectionally every step (megatts2.py:177, 271).  This decode follows the TRAINING
// semantics instead (causal=True, megatts2.py:158, 244): row t attends to rows <= t only, so rows < t never change
// and step t computes one row per utterance, appending its K/V to per-layer caches.  Its oracle is the
// teacher-forced causal forward (MegaPLM.forward / MegaADM.forward) evaluated on the decode's own prefix.
struct CausalBufs {
  float *x, *h, *qkv, *a, *f, *kv;     // (B,D) (B,D) (B,3D) (B,D) (B,F); kv: n_layers x (B, T, 2D) [k | v]
  char* scratch; int64_t scratch_bytes;
};

static int64_t causal_ws_floats(const mtts_encoder* e, int B, int T) {
  const int64_t D = e->d_model, F = e->ff_dim;
  const int64_t wide = 3 * D > F ? 3 * D : F;
  return (int64_t)B * (D + D + 3 * D + D + F) + (int64_t)e->n_layers * B * T * 2 * D + 16 * (int64_t)B * wide + 2048 + 8 * 64;
}

static int causal_take(const mtts_encoder* e, int B, int T, Arena& ar, CausalBufs& cb) {
  const int64_t D = e->d_model, F = e->ff_dim;
  const int64_t wide = 3 * D > F ? 3 * D : F;
  cb.x = ar.take<float>((int64_t)B * D);
  cb.h = ar.take<float>((int64_t)B * D);
  cb.qkv = ar.take<float>((int64_t)B * 3 * D);
  cb.a = ar.take<float>((int64_t)B * D);
  cb.f = ar.take<float>((int64_t)B * F);
  cb.kv = ar.take<float>((int64_t)e->n_layers * B * T * 2 * D);
  cb.scratch_bytes = 16 * (int64_t)B * wide * 4 + 4096;
  cb.scratch = ar.take<char>(cb.scratch_bytes);
  return ar.ok() ? 0 : fail(MTTS_ERR_WORKSPACE, "%s: workspace too small (need %lld bytes)", "causal decode", ar.off);
}

// one decode step: cb.x holds row t of the input (B,D) on entry and the stack's output row on return
static int causal_step(const mtts_encoder* e, int B, int T, int t, const CausalBufs& cb, cudaStream_t st) {
  const int D = e->d_model, H = e->n_heads, F = e->ff_dim, dh = D / H;
  const float scale = 1.0f / sqrtf((float)dh);
  auto skinny = [&](mtts_conv_params& q) { q.tc_scratch = cb.scratch; q.tc_scratch_bytes = cb.scratch_bytes; };   // split-K room
  for (int l = 0; l < e->n_layers; ++l) {
    const mtts_encoder_layer& L = e->layers[l];
    float* kv = cb.kv + (int64_t)l * B * T * 2 * D;
    MTTS_TRY(layernorm(cb.x, D, L.ln1_g, L.ln1_b, nullptr, 0, cb.h, D, B, D, 1e-5f, 0, 0, st));
    mtts_conv_params pq = linear_params(cb.h, D, L.w_qkv, L.b_qkv, cb.qkv, 3 * D, B, D, 3 * D);
    skinny(pq);
    MTTS_TRY(conv1d(pq, st));
    // append this row's [k | v] to the cache at position t
    MTTS_TRY(copy_strided(cb.qkv + D, 3 * D, 3 * D, 1, kv + (int64_t)t * 2 * D, (int64_t)T * 2 * D, 2 * D, 1, B, 1, 2 * D, 0, st));
    mtts_attn_params ap;
    memset(&ap, 0, sizeof(ap));
    ap.B = B; ap.H = H; ap.Tq = 1; ap.Tk = t + 1; ap.dh = dh; ap.scale = scale;
    ap.q = cb.qkv; ap.q_sb = 3 * D; ap.q_st = 3 * D;
    ap.k = kv; ap.k_sb = (int64_t)T * 2 * D; ap.k_st = 2 * D;
    ap.v = kv + D; ap.v_sb = (int64_t)T * 2 * D; ap.v_st = 2 * D;
    ap.o = cb.a; ap.o_sb = D; ap.o_st = D;
    MTTS_TRY(attention(ap, st));
    mtts_conv_params po = linear_params(cb.a, D, L.w_o, L.b_o, cb.x, D, B, D, D);
    po.res = cb.x; po.ldr = D;
    skinny(po);
    MTTS_TRY(conv1d(po, st));
    MTTS_TRY(layernorm(cb.x, D, L.ln2_g, L.ln2_b, nullptr, 0, cb.h, D, B, D, 1e-5f, 0, 0, st));
    mtts_conv_params p1 = linear_params(cb.h, D, L.w_ff1, L.b_ff1, cb.f, F, B, D, F);
    p1.post_act = MTTS_ACT_RELU;
    skinny(p1);
    MTTS_TRY(conv1d(p1, st));
    mtts_conv_params p2 = linear_params(cb.f, F, L.w_ff2, L.b_ff2, cb.x, D, B, F, D);
    p2.res = cb.x; p2.ldr = D;
    skinny(p2);
    MTTS_TRY(conv1d(p2, st));
  }
  return 0;
}

static int64_t plm_causal_ws_floats(const mtts_plm* m, int B, int T) {
  return causal_ws_floats(&m->enc, B, T) + (int64_t)B * m->vq_bins + 2 * ((int64_t)B * (T + 1) + 64) + 4 * 64;
}

static int plm_decode_causal(const mtts_plm* m, const float* tc, int64_t tc_sb, int tc_ld, int B, int T, int64_t* codes_out,
                             float* logits_out, void* ws, int64_t ws_bytes, cudaStream_t st) {
  const int D = m->enc.d_model, V = m->vq_bins;
  MTTS_REQUIRE(D == m->tc_dim + m->vq_dim, "d_model != tc_dim + vq_dim");
  MTTS_REQUIRE(tc && codes_out && m->pc_embedding && m->w_predict && m->pe, "null pointer");
  MTTS_REQUIRE(!m->enc.conv_ff && D % m->enc.n_heads == 0, "needs a linear feed-forward encoder");
  if (B <= 0 || T <= 0) return 0;
  Arena ar(ws, ws_bytes);
  float* logits = ar.take<float>((int64_t)B * V);
  int64_t* codes = ar.take<int64_t>((int64_t)B * (T + 1));
  CausalBufs cb;
  MTTS_TRY(causal_take(&m->enc, B, T, ar, cb));
  MTTS_TRY(fill_i64(codes, T + 1, B, (int64_t)V, st));   // BOS = vq_bins (megatts2.py:170-171)
  for (int t = 0; t < T; ++t) {
    // row t of the input: cat(tc[:, t], emb[codes[:, t]]) + alpha * pe[t]   (megatts2.py:154-157)
    MTTS_TRY(plm_build_input(tc + (int64_t)t * tc_ld, tc_sb, tc_ld, m->tc_dim, codes + t, T + 1, m->pc_embedding, m->vq_dim,
                             V + 2, m->pe + (int64_t)t * D, m->pe_alpha, B, 1, cb.x, st));
    MTTS_TRY(causal_step(&m->enc, B, T, t, cb, st));
    float* lg = logits_out ? logits_out + (int64_t)t * V : logits;
    const int64_t lg_sb = logits_out ? (int64_t)T * V : V;
    mtts_conv_params p = linear_params(cb.x, D, m->w_predict, nullptr, lg, V, B, D, V);
    p.y_batch_stride = lg_sb;
    p.B = B; p.Tin = 1; p.Tout = 1; p.x_batch_stride = D;
    p.tc_scratch = cb.scratch; p.tc_scratch_bytes = cb.scratch_bytes;
    MTTS_TRY(conv1d(p, st));
    MTTS_TRY(argmax_rows(lg, lg_sb, V, B, codes + (t + 1), T + 1, codes_out + t, T, st));
  }
  return 0;
}

static int64_t adm_causal_ws_floats(const mtts_adm* m, int B, int T) {
  return causal_ws_floats(&m->enc, B, T) + (int64_t)B * T * m->tc_emb_dim + (int64_t)B * (T + 1) + 4 * 64;
}

static int adm_decode_causal(const mtts_adm* m, const float* tc, int64_t tc_sb, int tc_ld, int B, int T, int32_t* dur_out,
                             float* raw_out, void* ws, int64_t ws_bytes, cudaStream_t st) {
  const int D = m->enc.d_model;
  MTTS_REQUIRE(D == m->emb_dim + m->tc_emb_dim, "d_model != emb_dim + tc_emb_dim");
  MTTS_REQUIRE(tc && dur_out && m->w_dt && m->w_tc && m->w_predict && m->pe, "null pointer");
  MTTS_REQUIRE(!m->enc.conv_ff && D % m->enc.n_heads == 0, "needs a linear feed-forward encoder");
  if (B <= 0 || T <= 0) return 0;
  Arena ar(ws, ws_bytes);
  float* tc_emb = ar.take<float>((int64_t)B * T * m->tc_emb_dim);
  float* praw = ar.take<float>((int64_t)B * (T + 1));
  CausalBufs cb;
  MTTS_TRY(causal_take(&m->enc, B, T, ar, cb));
  {
    mtts_conv_params p;
    memset(&p, 0, sizeof(p));
    p.x = tc; p.ldx = tc_ld; p.x_batch_stride = tc_sb;
    p.w = m->w_tc;
    p.y = tc_emb; p.ldy = m->tc_emb_dim; p.y_batch_stride = (int64_t)T * m->tc_emb_dim;
    p.B = B; p.Tin = T; p.Tout = T; p.Cin = m->tc_dim; p.Cout = m->tc_emb_dim; p.k = 1; p.stride = 1; p.dil = 1;
    p.out_scale = 1.0f;
    MTTS_TRY(conv1d(p, st));
  }
  MTTS_TRY(fill_f32(praw, T + 1, B, 0.0f, st));   // p_code = [[0]] (megatts2.py:262-263)
  for (int t = 0; t < T; ++t) {
    MTTS_TRY(adm_build_input(tc_emb + (int64_t)t * m->tc_emb_dim, (int64_t)T * m->tc_emb_dim, m->tc_emb_dim, m->tc_emb_dim,
                             praw + t, T + 1, m->w_dt, m->emb_dim, m->pe + (int64_t)t * D, m->pe_alpha, B, 1, cb.x, st));
    MTTS_TRY(causal_step(&m->enc, B, T, t, cb, st));
    MTTS_TRY(adm_readout(cb.x, D, m->w_predict, B, praw, T + 1, t + 1, st));
  }
  MTTS_TRY(adm_finalize(praw, T + 1, B, T, dur_out, raw_out, st));
  return 0;
}

// ------------------------------------------------------------------------------------------
// ConvNet family (modules/convnet.py), channels-last
struct StackBufs { float *tmp, *h1; };

// ResidualBlockStack.forward (convnet.py:69-72): x = x + ConvStack(x), n_stacks times.
// Reads `src` (never written), leaves the result in `dst` (may equal src); if final_dst is
// given, the LAST stack writes (x + y) there instead (optionally accumulating).
static int residual_stack(const mtts_conv_block* blocks, int n_stacks, int n_blocks, int C, int k, int B, int T,
                          const float* src, float* dst, float* final_dst, int final_accumulate, const StackBufs& sb,
                          const ConvTc* tc, cudaStream_t st) {
  const int64_t M = (int64_t)B * T;
  const float* cur = src;
  for (int s = 0; s < n_stacks; ++s) {
    const float* yin = cur;
    for (int b = 0; b < n_blocks; ++b) {
      const mtts_conv_block& bl = blocks[s * n_blocks + b];
      // ConvBlock (convnet.py:22-31): ReLU -> conv -> LN
      mtts_conv_params p = conv_same_params(yin, bl.w, bl.b, sb.tmp, B, T, C, C, k, 1, MTTS_PAD_ZERO);
      p.pre_act = MTTS_ACT_RELU;
      attach_tc(p, bl.w_tc, tc);
      MTTS_TRY(conv1d(p, st));
      if (b + 1 < n_blocks) {
        MTTS_TRY(layernorm(sb.tmp, C, bl.ln_g, bl.ln_b, nullptr, 0, sb.h1, C, M, C, 1e-5f, 0, 0, st));
        yin = sb.h1;
      } else {
        const bool fin = final_dst && (s == n_stacks - 1);
        float* out = fin ? final_dst : dst;
        MTTS_TRY(layernorm(sb.tmp, C, bl.ln_g, bl.ln_b, cur, C, out, C, M, C, 1e-5f, 0, fin ? final_accumulate : 0, st));
        cur = out;
      }
    }
  }
  return 0;
}

static int64_t convnet_ws_floats(const mtts_convnet* n, int B, int T) {
  return 3 * ((int64_t)B * T * n->hidden + 64) + (n->engine >= 1 ? conv_tc_scratch_need(B, T + n->k, n->hidden) / 4 + 64 : 0);
}

static int convnet_forward(const mtts_convnet* n, const float* x, int64_t x_sb, int ldx, float* y, int64_t y_sb,
                           int ldy, int B, int T, void* ws, int64_t ws_bytes, cudaStream_t st) {
  MTTS_REQUIRE(n->k % 2 == 1, "even kernel size");
  if (B <= 0 || T <= 0) return 0;
  Arena ar(ws, ws_bytes);
  const int64_t M = (int64_t)B * T;
  float* xc = ar.take<float>(M * n->hidden);
  StackBufs sb;
  sb.tmp = ar.take<float>(M * n->hidden);
  sb.h1 = ar.take<float>(M * n->hidden);
  ConvTc tc{n->engine, nullptr, n->engine >= 1 ? conv_tc_scratch_need(B, T + n->k, n->hidden) : 0};
  if (tc.bytes) tc.scratch = ar.take<char>(tc.bytes);
  if (!ar.ok()) return fail(MTTS_ERR_WORKSPACE, "%s: workspace too small (need %lld bytes)", "convnet", ar.off);
  mtts_conv_params p = conv_same_params(x, n->w_first, n->b_first, xc, B, T, n->in_channels, n->hidden, n->k, 1, MTTS_PAD_ZERO);
  p.ldx = ldx; p.x_batch_stride = x_sb;
  MTTS_TRY(conv1d(p, st));
  MTTS_TRY(residual_stack(n->blocks, n->n_stacks, n->n_blocks, n->hidden, n->k, B, T, xc, xc, nullptr, 0, sb, &tc, st));
  mtts_conv_params q = conv_same_params(xc, n->w_last, n->b_last, y, B, T, n->hidden, n->out_channels, n->k, 1, MTTS_PAD_ZERO);
  q.ldy = ldy; q.y_batch_stride = y_sb;
  MTTS_TRY(conv1d(q, st));
  return 0;
}

static int cnd_mid_len(const mtts_convnet_double* n, int T) {
  if (n->middle_kind == 0) return (T + n->middle_k - 1) / n->middle_k;
  return (T + 2 * n->middle_pad - n->middle_k) / n->middle_stride + 1;
}

static int64_t convnet_double_ws_floats(const mtts_convnet_double* n, int B, int T) {
  const int Tm = cnd_mid_len(n, T);
  return 4 * ((int64_t)B * T * n->hidden + 64) + 2 * ((int64_t)B * Tm * n->hidden + 64) +
         (n->engine >= 1 ? conv_tc_scratch_need(B, T + n->k, n->hidden) / 4 + 64 : 0);
}

static int convnet_double_forward(const mtts_convnet_double* n, const float* x, int64_t x_sb, int ldx, float* y,
                                  int64_t y_sb, int ldy, int B, int T, void* ws, int64_t ws_bytes, cudaStream_t st) {
  MTTS_REQUIRE(n->k % 2 == 1, "even kernel size");
  if (B <= 0 || T <= 0) return 0;
  const int H = n->hidden, Tm = cnd_mid_len(n, T);
  MTTS_REQUIRE(Tm >= 1, "input too short for the middle layer");
  Arena ar(ws, ws_bytes);
  const int64_t M = (int64_t)B * T, Mm = (int64_t)B * Tm;
  float* h0 = ar.take<float>(M * H);
  float* xc = ar.take<float>(M * H);
  StackBufs sb;
  sb.tmp = ar.take<float>(M * H);
  sb.h1 = ar.take<float>(M * H);
  float* xm = ar.take<float>(Mm * H);
  float* acc = ar.take<float>(Mm * H);
  ConvTc tc{n->engine, nullptr, n->engine >= 1 ? conv_tc_scratch_need(B, T + n->k, H) : 0};
  if (tc.bytes) tc.scratch = ar.take<char>(tc.bytes);
  if (!ar.ok()) return fail(MTTS_ERR_WORKSPACE, "%s: workspace too small (need %lld bytes)", "convnet_double", ar.off);
  mtts_conv_params p = conv_same_params(x, n->w_first, n->b_first, h0, B, T, n->in_channels, H, n->k, 1, MTTS_PAD_ZERO);
  p.ldx = ldx; p.x_batch_stride = x_sb;
  MTTS_TRY(conv1d(p, st));
  const int per = n->n_stacks * n->n_blocks;
  for (int l = 0; l < n->n_layers; ++l) {
    const mtts_conv_block* b1 = n->blocks + (int64_t)(l * 2 + 0) * per;
    const mtts_conv_block* b2 = n->blocks + (int64_t)(l * 2 + 1) * per;
    // every layer consumes the SAME first_layer output (convnet.py:205-207)
    MTTS_TRY(residual_stack(b1, n->n_stacks, n->n_blocks, H, n->k, B, T, h0, xc, nullptr, 0, sb, &tc, st));
    if (n->middle_kind == 0) {
      MTTS_TRY(maxpool_time(xc, (int64_t)T * H, H, xm, (int64_t)Tm * H, H, B, T, H, n->middle_k, st));
    } else {
      mtts_conv_params m;
      memset(&m, 0, sizeof(m));
      m.x = xc; m.ldx = H; m.x_batch_stride = (int64_t)T * H;
      m.w = n->w_middle; m.bias = n->b_middle;
      m.y = xm; m.ldy = H; m.y_batch_stride = (int64_t)Tm * H;
      m.B = B; m.Tin = T; m.Tout = Tm; m.Cin = H; m.Cout = H;
      m.k = n->middle_k; m.stride = n->middle_stride; m.dil = 1; m.pad = n->middle_pad; m.out_scale = 1.0f;
      MTTS_TRY(conv1d(m, st));
    }
    MTTS_TRY(residual_stack(b2, n->n_stacks, n->n_blocks, H, n->k, B, Tm, xm, xm, acc, l > 0 ? 1 : 0, sb, &tc, st));
  }
  mtts_conv_params q = conv_same_params(acc, n->w_last, n->b_last, y, B, Tm, H, n->out_channels, n->k, 1, MTTS_PAD_ZERO);
  q.ldy = ldy; q.y_batch_stride = y_sb;
  MTTS_TRY(conv1d(q, st));
  return 0;
}

// ------------------------------------------------------------------------------------------
// HiFi-GAN V1 generator (speechbrain HifiganGenerator.inference; SURVEY.md §2.4 K13)
static int64_t hifigan_ws_floats(const mtts_hifigan* h, int B, int T) {
  const int64_t Tp = T + 2 * h->inference_padding;
  int64_t L = Tp, C = h->ch0, big = Tp * C;
  for (int i = 0; i < h->n_ups; ++i) {
    L *= h->up_factor[i];
    C /= 2;
    if (L * C > big) big = L * C;
  }
  const int64_t tcb = h->engine >= 1 ? conv_tc_scratch_need(B, 1, big) + 6 * (int64_t)B * 64 * h->ch0 : 0;   // + halo rows
  return (int64_t)B * Tp * h->in_channels + 64 + 5 * ((int64_t)B * big + 64) + 3 * (tcb / 4 + 64);
}

static int hifigan_forward(const mtts_hifigan* h, const float* mel, int64_t mel_sb, int mel_ld, int B, int T, float* wav,
                           int64_t wav_sb, void* ws, int64_t ws_bytes, cudaStream_t st) {
  MTTS_REQUIRE(h->n_ups >= 1 && h->n_ups <= 4 && h->n_kernels >= 1, "bad generator config");
  if (B <= 0 || T <= 0) return 0;
  const int pad = h->inference_padding;
  const int Tp = T + 2 * pad;
  int64_t L = Tp, C = h->ch0, big = (int64_t)Tp * C;
  for (int i = 0; i < h->n_ups; ++i) {
    MTTS_REQUIRE(h->up_kernel[i] == 2 * h->up_factor[i], "transposed conv needs kernel == 2 * stride");
    L *= h->up_factor[i];
    C /= 2;
    if (L * C > big) big = L * C;
  }
  Arena ar(ws, ws_bytes);
  float* mp = ar.take<float>((int64_t)B * Tp * h->in_channels);
  float* bufs[5];
  for (int i = 0; i < 5; ++i) bufs[i] = ar.take<float>((int64_t)B * big);
  ConvTc tc{h->engine, nullptr, h->engine >= 1 ? conv_tc_scratch_need(B, 1, big) + 6 * (int64_t)B * 64 * h->ch0 : 0};
  char* planes2 = nullptr;                      // second plane buffer for the fused ResBlock flow
  char* planes0 = nullptr;                      // the stage input (up-sampled signal), split ONCE for its three ResBlocks
  if (tc.bytes) {
    tc.scratch = ar.take<char>(tc.bytes);
    planes2 = ar.take<char>(tc.bytes);
    planes0 = ar.take<char>(tc.bytes);
  }
  if (!ar.ok()) return fail(MTTS_ERR_WORKSPACE, "%s: workspace too small (need %lld bytes)", "hifigan", ar.off);
  bool fused = h->engine >= 1 && tc.scratch && planes2;
  const int hfmt = tc_fmt_of_engine(h->engine);
  for (int n = 0; fused && n < h->n_ups * h->n_kernels; ++n)
    for (int m = 0; m < 3; ++m) fused = fused && h->resblocks[n].w1_tc[m] && h->resblocks[n].w2_tc[m];
  // replicate-pad `pad` frames at both ends (HifiganGenerator.inference)
  MTTS_TRY(copy_strided(mel, mel_sb, mel_ld, 1, mp, (int64_t)Tp * h->in_channels, h->in_channels, 1, B, T,
                        h->in_channels, pad, st));
  float* o = bufs[0];     // stage input
  float* oup = bufs[1];   // after the transposed conv
  float* xr = bufs[2];    // resblock running value
  float* xt = bufs[3];    // resblock inner value
  float* z = bufs[4];     // mean of the resblocks -> next stage input
  {
    mtts_conv_params p = conv_same_params(mp, h->w_pre, h->b_pre, o, B, Tp, h->in_channels, h->ch0, 7, 1, MTTS_PAD_REFLECT);
    MTTS_TRY(conv1d(p, st));
  }
  int Lc = Tp, Cc = h->ch0;
  for (int i = 0; i < h->n_ups; ++i) {
    const int s = h->up_factor[i], Co = Cc / 2, Lo = Lc * s, pt = (h->up_kernel[i] - s) / 2;
    {
      // ConvTranspose1d(k = 2s, stride s, padding (k-s)/2) as a 2-tap conv with s*Co columns:
      // super-row u in [0, Lc]: out[u*s + r - pt, co] = x[u-1] W[:, co, r+s] + x[u] W[:, co, r]
      mtts_conv_params p;
      memset(&p, 0, sizeof(p));
      p.x = o; p.ldx = Cc; p.x_batch_stride = (int64_t)Lc * Cc;
      p.w = h->w_up[i]; p.bias = h->b_up[i];
      p.y = oup; p.ldy = s * Co; p.y_batch_stride = (int64_t)Lo * Co;
      p.B = B; p.Tin = Lc; p.Tout = Lc + 1; p.Cin = Cc; p.Cout = s * Co;
      p.k = 2; p.stride = 1; p.dil = 1; p.pad = 1; p.pad_mode = MTTS_PAD_ZERO;
      p.pre_act = MTTS_ACT_LEAKY; p.pre_slope = 0.1f;
      p.out_scale = 1.0f;
      p.out_shift = -(int64_t)pt * Co;
      p.y_batch_elems = (int64_t)Lo * Co;
      attach_tc(p, h->w_up_tc[i], &tc);
      MTTS_TRY(conv1d(p, st));
    }
    // one split of leaky(oup) with the LARGEST first-conv halo of the stage's ResBlocks; each ResBlock's first conv reads it
    // at its own row offset (three separate splits of the same signal were 6 % of the vocoder)
    const bool stage_fused = fused && (Co == 32 || Co == 64 || (Co >= 128 && Co % 32 == 0)) && (int64_t)B * Lo >= 128;
    int hmax = 0;
    for (int j = 0; j < h->n_kernels; ++j) {
      const mtts_hifigan_resblock& rbj = h->resblocks[i * h->n_kernels + j];
      hmax = rbj.dil[0] * (rbj.k - 1) / 2 > hmax ? rbj.dil[0] * (rbj.k - 1) / 2 : hmax;
    }
    const bool shared_split = stage_fused && planes0 && 6 * (int64_t)B * (Lo + 2 * hmax) * Co + 4096 <= tc.bytes;
    if (shared_split)
      MTTS_TRY(split_pad(oup, (int64_t)Lo * Co, Co, B, Lo, Co, hmax, hmax, MTTS_PAD_REFLECT, MTTS_ACT_LEAKY, 0.1f, planes0, hfmt, st));
    for (int j = 0; j < h->n_kernels; ++j) {
      const mtts_hifigan_resblock& rb = h->resblocks[i * h->n_kernels + j];
      const bool fuse_rb = stage_fused;
      if (fuse_rb) {
        // Fused plane flow: only the ResBlock input is split by a standalone pass; every conv epilogue writes
        // the NEXT conv's input planes (leaky applied, interior rows), halo_fill materialises the reflect padding.
        const int h2 = (rb.k - 1) / 2;
        const float* xcur = oup;
        for (int m = 0; m < 3; ++m) {
          const int h1 = rb.dil[m] * (rb.k - 1) / 2;
          mtts_conv_params c1 = conv_same_params(xcur, rb.w1[m], rb.b1[m], nullptr, B, Lo, Co, Co, rb.k, rb.dil[m], MTTS_PAD_REFLECT);
          c1.pre_act = MTTS_ACT_LEAKY; c1.pre_slope = 0.1f;
          c1.w_tc = rb.w1_tc[m]; c1.tc_scratch = tc.scratch; c1.tc_scratch_bytes = tc.bytes; c1.tc_fmt = hfmt;
          c1.tc_presplit = (m > 0);              // m == 0 without the shared split: split_pad(leaky(oup)) runs inside conv_tc
          if (m == 0 && shared_split) {
            c1.tc_presplit = 1; c1.tc_scratch = planes0; c1.tc_in_tp = Lo + 2 * hmax; c1.tc_in_row0 = hmax - h1;
          }
          c1.y = nullptr;
          c1.tc_out_planes = reinterpret_cast<void*>((((uintptr_t)planes2) + 1023) & ~(uintptr_t)1023);
          c1.tc_out_tp = Lo + 2 * h2; c1.tc_out_hl = h2; c1.tc_out_ld = Co;
          c1.tc_out_plane_stride = (int64_t)B * c1.tc_out_tp * Co;
          c1.tc_out_act = MTTS_ACT_LEAKY; c1.tc_out_slope = 0.1f;
          if (!conv_tc_eligible(c1)) return fail(MTTS_ERR_UNSUPPORTED, "%s: fused ResBlock conv not eligible (C=%lld L=%lld)", "hifigan", Co, Lo);
          MTTS_TRY(conv1d(c1, st));
          MTTS_TRY(halo_fill(planes2, B, Lo, Co, h2, h2, MTTS_PAD_REFLECT, st));
          const bool lastm = (m == 2);
          mtts_conv_params c2 = conv_same_params(nullptr, rb.w2[m], rb.b2[m], lastm ? z : xr, B, Lo, Co, Co, rb.k, 1, MTTS_PAD_REFLECT);
          c2.w_tc = rb.w2_tc[m]; c2.tc_scratch = planes2; c2.tc_scratch_bytes = tc.bytes; c2.tc_presplit = 1; c2.tc_fmt = hfmt;
          c2.res = xcur; c2.res_batch_stride = (int64_t)Lo * Co; c2.ldr = Co;
          if (lastm) {
            c2.out_scale = 1.0f / (float)h->n_kernels;
            c2.accumulate = (j > 0);
          } else {
            const int h1n = rb.dil[m + 1] * (rb.k - 1) / 2;
            c2.tc_out_planes = reinterpret_cast<void*>((((uintptr_t)tc.scratch) + 1023) & ~(uintptr_t)1023);
            c2.tc_out_tp = Lo + 2 * h1n; c2.tc_out_hl = h1n; c2.tc_out_ld = Co;
            c2.tc_out_plane_stride = (int64_t)B * c2.tc_out_tp * Co;
            c2.tc_out_act = MTTS_ACT_LEAKY; c2.tc_out_slope = 0.1f;
          }
          if (!conv_tc_eligible(c2)) return fail(MTTS_ERR_UNSUPPORTED, "%s: fused ResBlock conv not eligible (C=%lld L=%lld)", "hifigan", Co, Lo);
          MTTS_TRY(conv1d(c2, st));
          if (!lastm) MTTS_TRY(halo_fill(tc.scratch, B, Lo, Co, rb.dil[m + 1] * (rb.k - 1) / 2, rb.dil[m + 1] * (rb.k - 1) / 2, MTTS_PAD_REFLECT, st));
          (void)h1;
          xcur = xr;
        }
        continue;
      }
      const float* xcur = oup;
      for (int m = 0; m < 3; ++m) {
        mtts_conv_params c1 = conv_same_params(xcur, rb.w1[m], rb.b1[m], xt, B, Lo, Co, Co, rb.k, rb.dil[m], MTTS_PAD_REFLECT);
        c1.pre_act = MTTS_ACT_LEAKY; c1.pre_slope = 0.1f;
        attach_tc(c1, rb.w1_tc[m], &tc);
        MTTS_TRY(conv1d(c1, st));
        const bool lastm = (m == 2);
        mtts_conv_params c2 = conv_same_params(xt, rb.w2[m], rb.b2[m], lastm ? z : xr, B, Lo, Co, Co, rb.k, 1, MTTS_PAD_REFLECT);
        c2.pre_act = MTTS_ACT_LEAKY; c2.pre_slope = 0.1f;
        c2.res = xcur; c2.res_batch_stride = (int64_t)Lo * Co; c2.ldr = Co;
        if (lastm) {
          c2.out_scale = 1.0f / (float)h->n_kernels;
          c2.accumulate = (j > 0);
        }
        attach_tc(c2, rb.w2_tc[m], &tc);
        MTTS_TRY(conv1d(c2, st));
        xcur = xr;
      }
    }
    float* tswap = o; o = z; z = tswap;   // z (mean) becomes the next stage's input
    Lc = Lo; Cc = Co;
  }
  {
    mtts_conv_params p = conv_same_params(o, h->w_post, h->b_post, wav, B, Lc, Cc, 1, 7, 1, MTTS_PAD_REFLECT);
    p.pre_act = MTTS_ACT_LEAKY; p.pre_slope = 0.01f;
    p.post_act = MTTS_ACT_TANH;
    p.ldy = 1; p.y_batch_stride = wav_sb;
    MTTS_TRY(conv1d(p, st));
  }
  return 0;
}

}  // namespace mtts

// ==========================================================================================
// C ABI
using namespace mtts;

extern "C" {

static double g_last_split[6] = {0, 0, 0, 0, 0, 0};
/* {ffma_ms, ffma_flops, ffma_launches, tc_ms, tc_flops, tc_launches} of the last profile_end */
int mtts_profile_split(double* out6) {
  for (int i = 0; i < 6; ++i) out6[i] = g_last_split[i];
  return 0;
}
int mtts_profile_begin(void) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  for (auto& r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  g_prof.clear();
  g_prof_on = true;
  return 0;
}
int mtts_profile_end(double* gemm_ms, double* gemm_flops, int64_t* gemm_launches) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = false;
  double ms = 0.0, fl = 0.0;
  for (auto& r : g_prof) {
    float t = 0.f;
    if (cudaEventSynchronize(r.b) != cudaSuccess || cudaEventElapsedTime(&t, r.a, r.b) != cudaSuccess)
      return fail(MTTS_ERR_CUDA, "%s: event timing failed", "profile");
    ms += t;
    fl += r.flops;
  }
  if (gemm_ms) *gemm_ms = ms;
  if (gemm_flops) *gemm_flops = fl;
  if (gemm_launches) *gemm_launches = (int64_t)g_prof.size();
  g_last_split[0] = g_last_split[1] = g_last_split[2] = g_last_split[3] = g_last_split[4] = g_last_split[5] = 0.0;
  for (auto& r : g_prof) {
    float t = 0.f;
    cudaEventElapsedTime(&t, r.a, r.b);
    const int o = r.tc ? 3 : 0;
    g_last_split[o] += t; g_last_split[o + 1] += r.flops; g_last_split[o + 2] += 1.0;
  }
  for (auto& r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  g_prof.clear();
  return 0;
}

int64_t mtts_encoder_workspace_bytes(const mtts_encoder* enc, int32_t B, int32_t T) {
  return encoder_ws_floats(enc, B, T) * 4 + tc_scratch_bytes(enc, (int64_t)B * T) + 8192;
}
int mtts_encoder_forward_f32(const mtts_encoder* enc, const float* x, float* y, int32_t B, int32_t T, const float* mask,
                             int64_t mask_sb, int64_t mask_sh, int64_t mask_sq, int32_t last_row_only, void* workspace,
                             int64_t workspace_bytes, void* stream) {
  MTTS_REQUIRE(enc && enc->layers && x && y && workspace, "null pointer");
  Arena ar(workspace, workspace_bytes);
  TcScratch tcs{nullptr, tc_scratch_bytes(enc, (int64_t)B * T), (int64_t)B * T, tc_fmt_of_engine(enc->engine)};
  if (tcs.bytes) tcs.p = ar.take<char>(tcs.bytes);
  return encoder_forward(enc, x, y, B, T, mask, mask_sb, mask_sh, mask_sq, last_row_only, ar, &tcs,
                         (cudaStream_t)stream);
}

int64_t mtts_linear_tc_scratch_bytes(int64_t rows_cap, int32_t K) { return linear_tc_scratch_bytes(rows_cap, K); }
int mtts_linear_tc_f32(const float* x, int32_t ldx, int64_t M, int32_t K, const void* w_planes, int32_t N,
                       const float* bias, const float* res, int32_t ldr, float* y, int32_t ldy, int32_t pre_act,
                       float pre_slope, int32_t post_act, void* scratch, int64_t scratch_bytes, int64_t rows_cap,
                       int32_t fmt, void* stream) {
  return linear_tc(x, ldx, M, K, w_planes, N, bias, res, ldr, y, ldy, pre_act, pre_slope, post_act, 1.0f, scratch,
                   scratch_bytes, rows_cap, fmt, (cudaStream_t)stream);
}
int mtts_split_planes_f32(const float* x, int32_t ldx, int64_t rows, int32_t C, void* planes, int32_t fmt, void* stream) {
  return split_planes(x, ldx, rows, C, planes, fmt, (cudaStream_t)stream);
}
int mtts_tc_overflow_bind(int32_t* flag_dev) { return tc_overflow_bind(flag_dev); }
int mtts_tc_plan_query(int32_t n_sms, int32_t B, int32_t T, int32_t Cin, int32_t Cout, int32_t k, int32_t dil, int32_t fmt,
                       int64_t partial_bytes, int32_t ln_rides, int32_t* out5) {
  return tc_plan_query(n_sms, B, T, Cin, Cout, k, dil, fmt, partial_bytes, ln_rides, out5);
}

int64_t mtts_plm_infer_workspace_bytes(const mtts_plm* m, int32_t B, int32_t T) { return plm_ws_floats(m, B, T) * 4 + 8192; }
int mtts_plm_infer_f32(const mtts_plm* m, const float* tc_latent, int64_t tc_sb, int32_t tc_ld, int32_t B, int32_t T,
                       int64_t* codes_out, float* logits_out, void* workspace, int64_t workspace_bytes, void* stream) {
  MTTS_REQUIRE(m && m->enc.layers && workspace, "null pointer");
  return plm_infer(m, tc_latent, tc_sb, tc_ld, B, T, codes_out, logits_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

int64_t mtts_adm_infer_workspace_bytes(const mtts_adm* m, int32_t B, int32_t T) { return adm_ws_floats(m, B, T) * 4 + 8192; }
int mtts_adm_infer_f32(const mtts_adm* m, const float* tc_latent, int64_t tc_sb, int32_t tc_ld, int32_t B, int32_t T,
                       int32_t* dur_out, float* raw_out, void* workspace, int64_t workspace_bytes, void* stream) {
  MTTS_REQUIRE(m && m->enc.layers && workspace, "null pointer");
  return adm_infer(m, tc_latent, tc_sb, tc_ld, B, T, dur_out, raw_out, workspace, workspace_bytes, (cudaStream_t)stream);
}

int64_t mtts_plm_decode_causal_workspace_bytes(const mtts_plm* m, int32_t B, int32_t T) {
  return plm_causal_ws_floats(m, B, T) * 4 + 8192;
}
int mtts_plm_decode_causal_f32(const mtts_plm* m, const float* tc_latent, int64_t tc_sb, int32_t tc_ld, int32_t B, int32_t T,
                               int64_t* codes_out, float* logits_out, void* workspace, int64_t workspace_bytes, void* stream) {
  MTTS_REQUIRE(m && m->enc.layers && workspace, "null pointer");
  return plm_decode_causal(m, tc_latent, tc_sb, tc_ld, B, T, codes_out, logits_out, workspace, workspace_bytes,
                           (cudaStream_t)stream);
}
int64_t mtts_adm_decode_causal_workspace_bytes(const mtts_adm* m, int32_t B, int32_t T) {
  return adm_causal_ws_floats(m, B, T) * 4 + 8192;
}
int mtts_adm_decode_causal_f32(const mtts_adm* m, const float* tc_latent, int64_t tc_sb, int32_t tc_ld, int32_t B, int32_t T,
                               int32_t* dur_out, float* raw_out, void* workspace, int64_t workspace_bytes, void* stream) {
  MTTS_REQUIRE(m && m->enc.layers && workspace, "null pointer");
  return adm_decode_causal(m, tc_latent, tc_sb, tc_ld, B, T, dur_out, raw_out, workspace, workspace_bytes,
                           (cudaStream_t)stream);
}

int64_t mtts_convnet_workspace_bytes(const mtts_convnet* n, int32_t B, int32_t T) { return convnet_ws_floats(n, B, T) * 4 + 4096; }
int mtts_convnet_forward_f32(const mtts_convnet* n, const float* x, int64_t x_sb, int32_t ldx, float* y, int64_t y_sb,
                             int32_t ldy, int32_t B, int32_t T, void* workspace, int64_t workspace_bytes, void* stream) {
  MTTS_REQUIRE(n && n->blocks && x && y && workspace, "null pointer");
  return convnet_forward(n, x, x_sb, ldx, y, y_sb, ldy, B, T, workspace, workspace_bytes, (cudaStream_t)stream);
}

int32_t mtts_convnet_double_out_len(const mtts_convnet_double* n, int32_t T) { return cnd_mid_len(n, T); }
int64_t mtts_convnet_double_workspace_bytes(const mtts_convnet_double* n, int32_t B, int32_t T) {
  return convnet_double_ws_floats(n, B, T) * 4 + 4096;
}
int mtts_convnet_double_forward_f32(const mtts_convnet_double* n, const float* x, int64_t x_sb, int32_t ldx, float* y,
                                    int64_t y_sb, int32_t ldy, int32_t B, int32_t T, void* workspace,
                                    int64_t workspace_bytes, void* stream) {
  MTTS_REQUIRE(n && n->blocks && x && y && workspace, "null pointer");
  return convnet_double_forward(n, x, x_sb, ldx, y, y_sb, ldy, B, T, workspace, workspace_bytes, (cudaStream_t)stream);
}

int64_t mtts_hifigan_workspace_bytes(const mtts_hifigan* h, int32_t B, int32_t T) { return hifigan_ws_floats(h, B, T) * 4 + 4096; }
int mtts_hifigan_forward_f32(const mtts_hifigan* h, const float* mel, int64_t mel_sb, int32_t mel_ld, int32_t B, int32_t T,
                             float* wav, int64_t wav_sb, void* workspace, int64_t workspace_bytes, void* stream) {
  MTTS_REQUIRE(h && h->resblocks && mel && wav && workspace, "null pointer");
  return hifigan_forward(h, mel, mel_sb, mel_ld, B, T, wav, wav_sb, workspace, workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"
