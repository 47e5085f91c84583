/*
 * megatts2_b200.h - C ABI of libmegatts2_b200.so (sm_100a).
 *
 * The reference (LSimon95/megatts2 @ 2ab81a1) has no FFI layer: its replaceable surface
 * is the Python nn.Module API (SURVEY.md §8b).  This library is what those modules bind
 * through ctypes; every entry point names the reference function it replaces
 * (file:line relative to the reference repo).
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host; fp32 unless stated
 *  - activations are channels-last: (B, T, C) with an explicit row stride `ld` (elements)
 *    and batch stride; the Python layer converts from/to the reference's (B, C, T)
 *  - the caller owns every buffer (inputs, outputs, workspace); the library never
 *    allocates device memory and keeps no pointer after return
 *  - work is enqueued on `stream` (a cudaStream_t passed as void*); no hidden device sync
 *  - every function returns 0 on success or a negative mtts_status; mtts_last_error()
 *    returns a thread-local message.  There is NO CPU fallback anywhere.
 */
#ifndef MEGATTS2_B200_H
#define MEGATTS2_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MTTS_ABI_VERSION 4

typedef enum {
  MTTS_OK = 0,
  MTTS_ERR_BAD_ARG = -1,
  MTTS_ERR_UNSUPPORTED = -2,
  MTTS_ERR_CUDA = -3,
  MTTS_ERR_WORKSPACE = -4
} mtts_status;

int mtts_abi_version(void);
const char* mtts_last_error(void);
/* number of kernels this library has launched in this process (bench.py gpu_launches) */
int64_t mtts_launch_count(void);
/* measurement aid (bench.py roofline leg; off by default): between begin and end every
 * tap-GEMM launch is bracketed by CUDA events on its stream; end() synchronises and returns
 * the summed kernel time, the summed algorithmic FLOPs (2*M*N*Cin*k) and the launch count. */
int mtts_profile_begin(void);
int mtts_profile_end(double* gemm_ms, double* gemm_flops, int64_t* gemm_launches);
/* per-engine split of the last profile_end: {ffma_ms, ffma_flops, ffma_launches, tc_ms, tc_flops, tc_launches} */
int mtts_profile_split(double* out6);
/* diagnostics: per-launcher CUDA-event trace of everything enqueued between begin and end (single stream);
 * end synchronises and writes a text table "launcher launches total_ms share" into buf */
int mtts_trace_begin(void* stream);
int mtts_trace_end(char* buf, int32_t buf_len);

/* Tensor-core operand formats.  Both give fp32-grade results (the tests hold them to the same bars):
 *   BF16X3: x = x1 + x2 + x3 (bf16), products x1w1 + x1w2 + x2w1 + x2w2 + x1w3 + x3w1  -> 6 MMAs, fp32 range
 *   F16X2 : x = x1 + x2' * 2^-11 (fp16, residual stored scaled so it stays in the normal range), products
 *           x1w1 + (x1w2' + x2'w1) * 2^-11 -> 3 MMAs, 22 significant bits per operand; |x| must be <= 65504.
 * An activation outside the fp16 range poisons its result (inf/NaN) and sets the int32 flag registered here for
 * the current device (the caller owns the 4 bytes; NULL unbinds).  The Python layer checks it once per synthesis
 * and reruns the batch on BF16X3. */
enum { MTTS_TC_BF16X3 = 0, MTTS_TC_F16X2 = 1 };
int mtts_tc_overflow_bind(int32_t* flag_dev);
/* Diagnostics (host only, no CUDA call): the launch plan the tap-GEMM dispatcher picks for a stride-1 layer of this shape
 * (B x T output rows, k taps) on n_sms SMs, with partial_bytes of split-K partial-sum space and, if ln_rides, a LayerNorm
 * that the split's reduction can carry.  out5 = {N-tile width, K splits, CTA pair, halo form (0 | 1 | 2 = as a pair),
 * K-slab bytes}. */
int mtts_tc_plan_query(int32_t n_sms, int32_t B, int32_t T, int32_t Cin, int32_t Cout, int32_t k, int32_t dil, int32_t fmt,
                       int64_t partial_bytes, int32_t ln_rides, int32_t* out5);

/* activation / padding codes */
enum { MTTS_ACT_NONE = 0, MTTS_ACT_RELU = 1, MTTS_ACT_LEAKY = 2, MTTS_ACT_TANH = 3 };
enum { MTTS_PAD_ZERO = 0, MTTS_PAD_REFLECT = 1, MTTS_PAD_REPLICATE = 2 };

/* ------------------------------------------------------------------------------------------
 * Tap-GEMM: the one dense contraction of the path.  Covers nn.Linear (k = 1), nn.Conv1d
 * (modules/convnet.py:13-18,88-94; modules/transformer.py:76-78; modules/mrte.py:101-107
 * stride 16), dilated HiFi-GAN convs and ConvTranspose1d (as a 2-tap conv with s*Cout
 * columns):
 *   acc[b,t,n] = sum_{j<k} sum_{c<Cin} pre(X[b, t*stride + j*dil - pad, c]) * W[j][c][n]
 *   v = post(acc + bias[n]);  v += R[b,t,n];  v *= out_scale;  v += Y_old (accumulate)
 *   Y[b, t*ldy + n + out_shift] = v        (skipped when outside [0, y_batch_elems))
 * W is PRE-PACKED as (k, Cin, Cout) row-major (mtts_pack_* on the host side does that once).
 */
typedef struct {
  const float* x; int64_t x_batch_stride; int32_t ldx;
  const float* w;
  const float* bias;                       /* (Cout) or NULL */
  const float* res; int64_t res_batch_stride; int32_t ldr;   /* optional */
  float* y; int64_t y_batch_stride; int32_t ldy;
  int32_t B, Tin, Tout, Cin, Cout;
  int32_t k, stride, dil, pad;
  int32_t pad_mode;                        /* MTTS_PAD_* */
  int32_t pre_act; float pre_slope;        /* applied to X on load */
  int32_t post_act; float post_slope;
  float out_scale;
  int32_t accumulate;
  int64_t out_shift;                       /* 0 for ordinary convs */
  int64_t y_batch_elems;                   /* 0 -> Tout*ldy */
  const int32_t* in_lens;                  /* optional (B): rows >= len read as zero / reflect about len */
  /* tensor-core engine (optional): the same weights as three bf16 planes (3, k, Cout, Cin) and a scratch
   * buffer for the padded activation planes (>= 6*B*(Tout + dil*(k-1))*Cin + 2048 bytes).  Used when the
   * shape is eligible (stride 1, Cin % 8 == 0, Cin >= 32, Cout in {32, 64, >= 128 and % 32 == 0}). */
  const void* w_tc;
  void* tc_scratch; int64_t tc_scratch_bytes;
  int64_t tc_rows_cap;                     /* k == 1 only: row capacity of the scratch planes (>= B*Tin, 0 -> B*Tin);
                                              a stable capacity keeps the cached TMA descriptors valid across AR steps */
  /* plane fusion (tensor-core engine only).  tc_presplit = 1: the activation planes already sit in tc_scratch
   * (three planes of (B, Tout + dil*(k-1), Cin) bf16, padding materialised, pre-activation applied) - x is not
   * read.  tc_out_planes != NULL: the epilogue additionally writes act(result) as three bf16 planes for the next
   * tensor-core layer (row (b*tc_out_tp + tc_out_hl + t), stride tc_out_ld); y may then be NULL. */
  int32_t tc_presplit;
  void* tc_out_planes; int64_t tc_out_plane_stride;
  int32_t tc_out_ld, tc_out_tp, tc_out_hl, tc_out_act; float tc_out_slope;
  /* optional room for split-K partial sums (tensor-core engine, k == 1): when a dense layer has too few output tiles to
   * fill the GPU, K is split across CTAs into fp32 partials here and a second kernel reduces them in a fixed order and
   * applies the epilogue.  >= splits * B*Tout * Cout * 4 bytes; NULL -> never split. */
  void* tc_partial; int64_t tc_partial_bytes;
  /* operand format of w_tc / the activation planes: MTTS_TC_BF16X3 (three bf16 planes, 6 MMAs per product) or
   * MTTS_TC_F16X2 (two fp16 planes, residual scaled by 2^11, 3 MMAs per product; see mtts_tc_overflow_bind) */
  int32_t tc_fmt;
  /* tc_presplit only: the planes in tc_scratch may be a SHARED buffer with a larger halo than this conv needs -
   * tc_in_tp rows per batch item (0 -> Tout + dil*(k-1)) and this conv's first padded row at tc_in_row0 (HiFi-GAN: the
   * three ResBlocks of a stage read one split of the up-sampled signal, each at its own row offset) */
  int32_t tc_in_tp, tc_in_row0;
} mtts_conv_params;

int mtts_conv1d_f32(const mtts_conv_params* p, void* stream);

/* Tensor-core linear layer (tcgen05, sm_100a): Y[M,N] = post(pre(X)[M,K] . W[N,K]^T + bias) (+ R) with
 * fp32-grade accuracy from split operands (fp32 accumulation in TMEM).  w_planes: (3, N, K) bf16 [BF16X3] or
 * (2, N, K) fp16 [F16X2] row-major; scratch receives the activation planes
 * (mtts_linear_tc_scratch_bytes(rows_cap, K), rows_cap >= M).  K %% 8 == 0. */
int64_t mtts_linear_tc_scratch_bytes(int64_t rows_cap, int32_t K);
int mtts_linear_tc_f32(const float* x, int32_t ldx, int64_t M, int32_t K, const void* w_planes, int32_t N,
                       const float* bias, const float* res, int32_t ldr, float* y, int32_t ldy,
                       int32_t pre_act, float pre_slope, int32_t post_act,
                       void* scratch, int64_t scratch_bytes, int64_t rows_cap, int32_t fmt, void* stream);
/* fp32 (rows, C) with row stride ldx -> operand planes (3 | 2, rows, C) of `fmt` (the split the kernels apply to
 * activations; the host side uses it to pack weights once).  C %% 4 == 0, x 16-byte aligned. */
int mtts_split_planes_f32(const float* x, int32_t ldx, int64_t rows, int32_t C, void* planes, int32_t fmt, void* stream);

/* LayerNorm over the last dim (nn.LayerNorm, eps 1e-5; modules/convnet.py:28-30,
 * modules/transformer.py:67-68, modules/mrte.py:136):
 *   v = LN(x[row]) * gamma + beta;  v = post(v);  v += res[row];  v += y_old (accumulate) */
int mtts_layernorm_f32(const float* x, int32_t ldx, const float* gamma, const float* beta,
                       const float* res, int32_t ldr, float* y, int32_t ldy,
                       int64_t rows, int32_t C, float eps, int32_t post_act, int32_t accumulate,
                       void* stream);

/* softmax(Q K^T * scale + mask) V  (F.scaled_dot_product_attention at
 * modules/transformer.py:52-53).  q/k/v/o are (B, T, H, dh) views given by strides;
 * mask is additive fp32 with element strides (mask_sb, mask_sh, mask_sq, 1) or NULL.
 * dh in {64, 96, 128, 256, 512}.  q_row0/n_q select a row range of the queries. */
typedef struct {
  const float* q; int64_t q_sb; int32_t q_st;
  const float* k; int64_t k_sb; int32_t k_st;
  const float* v; int64_t v_sb; int32_t v_st;
  float* o; int64_t o_sb; int32_t o_st;
  const float* mask; int64_t mask_sb, mask_sh, mask_sq;
  int32_t B, H, Tq, Tk, dh;
  float scale;
  /* optional: write the output as three bf16 planes (row b*Tq + t, stride o_planes_ld) for a following
   * tensor-core GEMM; o may then be NULL */
  void* o_planes; int64_t o_plane_stride; int32_t o_planes_ld;
  int32_t o_planes_fmt;                    /* MTTS_TC_BF16X3 | MTTS_TC_F16X2 */
} mtts_attn_params;
int mtts_attention_f32(const mtts_attn_params* p, void* stream);

/* EuclideanCodebook.quantize (modules/quantization/core_vq.py:175-183): first index of
 * max_k -(|x|^2 - 2 x.e_k + |e_k|^2).  x (N, D) ld = ldx, embed (K, D) -> idx (N) int64 */
int mtts_vq_argmin_f32(const float* x, int32_t ldx, const float* embed, int64_t N, int32_t D, int32_t K,
                       int64_t* idx, void* stream);
/* EuclideanCodebook.dequantize / ResidualVectorQuantizer.decode (core_vq.py:188-190, 360-367)
 * with an optional time-repeat (vqpe.py:60-61, models/megatts2.py:362-364):
 *   y[b, t, :] = embed[idx[b, t / repeat], :]  for t < T_out;  y is (B, T_out, ldy) */
int mtts_vq_gather_f32(const int64_t* idx, int32_t idx_ld, const float* embed, int32_t D, int32_t K,
                       int32_t B, int32_t T_out, int32_t repeat, float* y, int64_t y_sb, int32_t ldy,
                       void* stream);

/* extract_mel_spec (modules/tokenizer.py:107-125; SURVEY.md Appendix B): reflect-padded
 * 1024-point STFT (hop 256, window table given), magnitude, banded mel filterbank,
 * log(max(., clamp)).  wav (B, L) -> out[b*out_sb + m*out_sm + f*out_sf], f < 1 + L/256.
 * The filterbank is passed in GROUPED banded form (the host packs it once, like a weight plane;
 * megatts2_b200/modules/tokenizer.py:pack_grouped_filterbank).  Mels are taken in groups of 4, G = ceil(n_mels / 4):
 *   fb_start[4 G]  first bin read for each mel, a multiple of 4 (slots past n_mels: 0)
 *   fb_off[G + 1]  float offset of each group's block in fb_w; a block holds 4 * len_g floats, len_g a multiple of 4
 *                  covering the longest (aligned) band of the group
 *   fb_w           16-byte aligned; block g, element i * len_g + t = weight of mel 4 g + i at bin fb_start[4 g + i] + t
 *                  (0 outside its band); fb_start[m] + len_g <= 516 for every mel (bins 513..515 read as zero).
 * n_fft must be 1024, hop 256, n_mels <= 128. */
int mtts_mel_spectrogram_f32(const float* wav, int64_t wav_sb, int32_t B, int32_t L,
                             const float* window, const float* fb_w, const int32_t* fb_off,
                             const int32_t* fb_start, int32_t n_mels, float clamp_min,
                             float* out, int64_t out_sb, int64_t out_sm, int64_t out_sf, void* stream);
/* Ragged batch for bulk extraction (MelSpecExtractor.extract over a corpus, modules/tokenizer.py:139-155,
 * prepare_ds.py:211-217; SURVEY.md 8f-2): clip b holds lens[b] <= L_max valid samples (device int32); its reflect
 * padding and frame count 1 + lens[b]/256 follow its own length; frames past that are not written. lens[b] > 512. */
int mtts_mel_spectrogram_ragged_f32(const float* wav, int64_t wav_sb, int32_t B, int32_t L_max, const int32_t* lens,
                                    const float* window, const float* fb_w, const int32_t* fb_off,
                                    const int32_t* fb_start, int32_t n_mels, float clamp_min,
                                    float* out, int64_t out_sb, int64_t out_sm, int64_t out_sf, void* stream);

/* nn.MaxPool1d(k, ceil_mode=True) over time, channels-last (modules/vqpe.py:38,
 * models/megatts2.py:357-358).  x (B, T, C) -> y (B, ceil(T/k), C) */
int mtts_maxpool_time_f32(const float* x, int64_t x_sb, int32_t ldx, float* y, int64_t y_sb, int32_t ldy,
                          int32_t B, int32_t T, int32_t C, int32_t k, void* stream);

/* TokenEmbedding + SinePositionalEmbedding (modules/embedding.py:41-47, 94-98):
 *   y[b,t,:] = table[ids[b,t],:] + alpha * pe[t + pe_offset,:]    (pe may be NULL) */
int mtts_embed_pe_f32(const int64_t* ids, int32_t ids_ld, const float* table, int32_t vocab, int32_t D,
                      const float* pe, float alpha, int32_t pe_offset, int32_t B, int32_t T,
                      float* y, int64_t y_sb, int32_t ldy, void* stream);
/* y = x + alpha * pe[t,:]  (SinePositionalEmbedding.forward on an existing tensor) */
int mtts_add_pe_f32(const float* x, int64_t x_sb, int32_t ldx, const float* pe, float alpha,
                    int32_t B, int32_t T, int32_t D, float* y, int64_t y_sb, int32_t ldy, void* stream);

/* LengthRegulator.forward (modules/mrte.py:23-31, 42-60) as a gather:
 *   y[b, sum_{j<i} d[b,j] + r, :] = x[b,i,:]; rows >= sum(d[b]) are zero.
 * totals (B) int32 receives sum(d[b]) (pass NULL to skip). y is (B, L_out, ldy). */
int mtts_length_regulate_f32(const float* x, int64_t x_sb, int32_t ldx, const int32_t* dur, int32_t dur_ld,
                             int32_t B, int32_t Tp, int32_t D, int32_t L_out,
                             float* y, int64_t y_sb, int32_t ldy, int32_t* totals, void* stream);

/* strided 2-D copy / transpose helpers used at the (B,C,T) <-> (B,T,C) module boundary:
 *   y[b, t, c] = x[b*x_sb + t*x_st + c*x_sc]   with optional replicate padding of `pad`
 *   rows at both ends of t (HiFi-GAN inference_padding) */
int mtts_copy_strided_f32(const float* x, int64_t x_sb, int64_t x_st, int64_t x_sc,
                          float* y, int64_t y_sb, int64_t y_st, int64_t y_sc,
                          int32_t B, int32_t T, int32_t C, int32_t pad_rep, void* stream);

/* ------------------------------------------------------------------------------------------
 * Audio front / back ends of Megatts.forward on the device (SURVEY.md 8f-3).
 *
 * mtts_resample_f32 - librosa.load(path, sr=16000) at models/megatts2.py:335 (and prepare_ds.py:113), the resampling
 * part: band-limited polyphase FIR, y[i*up + p] = sum_k xpad[i*down + k] * h[p][k] with xpad = x preceded by `width`
 * zeros; h is the (up, taps) filter table of torchaudio.functional.resample (built on the host in fp64:
 * megatts2_b200/audio.py).  x (B, L_in) with optional per-clip lengths; y (B, L_out), samples past lens_out[b] are zero.
 * mtts_peak_normalize_f32 - librosa.util.normalize(y) (:336): x[b] /= max|x[b]| in place (unchanged if the peak is below
 * FLT_MIN); scratch: B x 4 bytes.
 * mtts_pcm16_f32 - the integer encoding of the wav writer behind torchaudio.save (:375): round-to-nearest of x * 32768,
 * saturated. */
int mtts_resample_f32(const float* x, int64_t x_sb, int32_t B, int32_t L_in, const int32_t* lens_in, const float* h,
                      int32_t up, int32_t down, int32_t width, int32_t taps, float* y, int64_t y_sb, int32_t L_out,
                      const int32_t* lens_out, void* stream);
int mtts_peak_normalize_f32(float* x, int64_t x_sb, int32_t B, int32_t L, const int32_t* lens, void* scratch, void* stream);
int mtts_pcm16_f32(const float* x, int64_t n, int16_t* out, void* stream);

/* ------------------------------------------------------------------------------------------
 * Training-mode / backward kernels (SURVEY.md 8f-4): what autograd needs so that MegaPLMTrainer / MegaADMTrainer
 * .training_step (models/trainer.py:243-268, 334-355) run through the drop-in modules.  The dense contractions of the
 * backward pass (dX = dY W, dW = dY^T X) use mtts_linear_tc_f32 / mtts_conv1d_f32 like the forward; these are the rest.
 *
 * mtts_bmm_f32: C[z1,z2][m,n] = alpha * sum_k A[z1,z2][m,k] * B[z1,z2][k,n] (+ C), every operand given by element strides
 *   (transposes and (B,T,H,dh) head views are free) - the attention products Q K^T, P V and their gradients.
 * mtts_softmax_fwd_f32: rows of S (B,H,Tq,Tk) -> P = softmax(S + mask) and Pd = P * keep (keep = dropout keep-scale or
 *   NULL); mtts_softmax_bwd_f32: dS = P * (dPd * keep - <dPd * keep, P>)   (F.scaled_dot_product_attention with dropout,
 *   modules/transformer.py:52-53, unfused for training).
 * mtts_layernorm_bwd_f32: dx (rows, C) and per-CTA partials (ceil(rows / 8), 2, C) of d-gamma | d-beta
 *   (reduce with mtts_colsum_f32).  mtts_colsum_f32: out[c] (+)= sum_r in[r*ld + c], fixed row order.
 * mtts_relu_bwd_f32: dx = dy * (y > 0).  mtts_embedding_bwd_f32: dW[ids[r]] += dy[r] (nn.Embedding).
 * mtts_rowdot_f32: out[r] = <a[r, :], b[r % period, :]> (d-alpha of SinePositionalEmbedding). */
int mtts_bmm_f32(const float* a, int64_t a_s1, int64_t a_s2, int64_t a_sm, int64_t a_sk, const float* b, int64_t b_s1,
                 int64_t b_s2, int64_t b_sk, int64_t b_sn, float* c, int64_t c_s1, int64_t c_s2, int64_t c_sm, int64_t c_sn,
                 int32_t Z1, int32_t Z2, int32_t M, int32_t N, int32_t K, float alpha, int32_t accumulate, void* stream);
int mtts_softmax_fwd_f32(const float* S, const float* mask, int64_t m_sb, int64_t m_sh, int64_t m_sq, int32_t B, int32_t H,
                         int32_t Tq, int32_t Tk, const float* keep, float* P, float* Pd, void* stream);
int mtts_softmax_bwd_f32(const float* P, const float* dPd, const float* keep, float* dS, int32_t Tk, int64_t rows, void* stream);
int mtts_layernorm_bwd_f32(const float* x, const float* gamma, const float* dy, float* dx, float* partial, int64_t rows, int32_t C,
                           float eps, void* stream);
int mtts_colsum_f32(const float* in, int64_t ld, int64_t rows, int32_t C, float* out, int32_t accumulate, void* stream);
int mtts_relu_bwd_f32(const float* y, const float* dy, float* dx, int64_t n, void* stream);
int mtts_embedding_bwd_f32(const int64_t* ids, const float* dy, int64_t rows, int32_t D, int32_t vocab, float* dW, void* stream);
int mtts_rowdot_f32(const float* a, const float* b, int64_t rows, int32_t C, int32_t period, float* out, void* stream);

/* Training-only pieces of the VQ codebook (SURVEY.md 8f-4): EuclideanCodebook.forward in train mode and the
 * straight-through / commitment step of VectorQuantization.forward.
 * mtts_kmeans_assign_f32: idx[n] = first argmin_k sum_d (x[n,d] - means[k,d])^2 - the bucket step of kmeans()
 *   (modules/quantization/core_vq.py:81-86; direct differences, not the expanded form of quantize).  D <= 512.
 * mtts_vq_cluster_sum_f32: sum[k,:] = sum_{n: idx[n]=k} x[n,:] accumulated in sample order, cnt[k] = bucket size as
 *   float - bincount + scatter_add_ of kmeans (:87-92) and embed_onehot.sum(0) / x.t() @ embed_onehot of the EMA step
 *   (:220-222).
 * mtts_kmeans_update_f32: means[k] = cnt[k] > 0 ? sum[k] / cnt[k] : means[k]   (:88-95).
 * mtts_vq_ema_update_f32: cluster_size <- decay cs + (1-decay) cnt; embed_avg <- decay ea + (1-decay) sum;
 *   embed = embed_avg / ((cs + eps) / (sum(cs) + K eps) * sum(cs))   (ema_inplace, laplace_smoothing; :217-229).
 *   scratch: K floats.
 * mtts_vq_replace_rows_f32: embed[k] = samples[pick[k]] where cluster_size[k] < thr   (expire_codes_ / replace_, :151-169;
 *   the caller draws pick = sample_vectors' indices).
 * mtts_vq_ste_commit_f32: out = x + (q - x) (the straight-through value as the reference rounds it) and
 *   loss[0] = mean((out - x)^2) (F.mse_loss(quantize.detach(), x), :303-311); partials: 256 floats of scratch.
 * mtts_vq_ste_commit_bwd_f32: dx = g_out + g_loss[0] * scale * (x - out), scale = commitment_weight * 2 / numel;
 *   g_out or g_loss may be NULL. */
int mtts_kmeans_assign_f32(const float* x, const float* means, int32_t N, int32_t K, int32_t D, int64_t* idx, void* stream);
int mtts_vq_cluster_sum_f32(const float* x, const int64_t* idx, int32_t N, int32_t K, int32_t D, float* sum, float* cnt,
                            void* stream);
int mtts_kmeans_update_f32(float* means, const float* sum, const float* cnt, int32_t K, int32_t D, void* stream);
int mtts_vq_ema_update_f32(float* cluster_size, float* embed_avg, float* embed, const float* sum, const float* cnt,
                           int32_t K, int32_t D, float decay, float eps, float* scratch, void* stream);
int mtts_vq_replace_rows_f32(float* embed, const float* samples, const int64_t* pick, const float* cluster_size, float thr,
                             int32_t K, int32_t D, int32_t N, void* stream);
int mtts_vq_ste_commit_f32(const float* x, const float* q, int64_t n, float* out, float* partials, float* loss, void* stream);
int mtts_vq_ste_commit_bwd_f32(const float* x, const float* out, const float* g_out, const float* g_loss, float scale,
                               int64_t n, float* dx, void* stream);

/* x (B, rows, L) contiguous: x[b, r, keep[b]:] = 0 in place - speechbrain HIFIGAN.mask_noise behind
 * decode_batch(mel, mel_lens, hop_len) (reference call site models/megatts2.py:370). */
int mtts_mask_tail_f32(float* x, int32_t B, int32_t rows, int32_t L, const int32_t* keep, void* stream);

/* ------------------------------------------------------------------------------------------
 * Composite drivers: whole sub-networks enqueued by one call (C++ launch loop, no Python
 * per-kernel overhead).  Weight pointers refer to PRE-PACKED device buffers owned by the
 * caller.
 */
typedef struct {
  const float *ln1_g, *ln1_b, *ln2_g, *ln2_b;
  const float *w_qkv, *b_qkv;          /* (1, D, 3D) packed, (3D) */
  const float *w_o, *b_o;              /* (1, D, D), (D) */
  const float *w_ff1, *b_ff1;          /* linear: (1, D, F); conv-FF: (5, D, F) */
  const float *w_ff2, *b_ff2;          /* linear: (1, F, D); conv-FF: (5, F, D) */
  /* tensor-core engine (optional, linear layers only): the same weights as THREE bf16 planes
   * (3, N, K) row-major (w = w1 + w2 + w3, see mtts_linear_tc_f32); NULL -> exact FFMA engine */
  const void *w_qkv_tc, *w_o_tc, *w_ff1_tc, *w_ff2_tc;
} mtts_encoder_layer;

typedef struct {
  int32_t n_layers, d_model, n_heads, ff_dim, conv_ff;
  int32_t engine;                      /* 0: fp32 FFMA everywhere; tcgen05 for GEMMs with M >= 128: 1 = BF16X3, 2 = F16X2 operands */
  const mtts_encoder_layer* layers;    /* HOST array of n_layers entries */
} mtts_encoder;

/* TransformerEncoder.forward (modules/transformer.py:119-133).  x (B,T,D) -> y (B,T,D);
 * mask: optional additive (B,H,T,T) fp32 (utils/utils.py:21-39) given by strides.
 * last_row_only != 0: y is (B,1,D) = the last position's output (exact pruning of the final
 * layer; what MegaPLM.infer / MegaADM.infer consume, models/megatts2.py:178, 272). */
int64_t mtts_encoder_workspace_bytes(const mtts_encoder* enc, int32_t B, int32_t T);
int mtts_encoder_forward_f32(const mtts_encoder* enc, const float* x, float* y, int32_t B, int32_t T,
                             const float* mask, int64_t mask_sb, int64_t mask_sh, int64_t mask_sq,
                             int32_t last_row_only, void* workspace, int64_t workspace_bytes, void* stream);

/* MegaPLM.infer (models/megatts2.py:165-181): greedy AR decode, BOS = vq_bins, exactly T
 * steps, NON-causal full recompute per step (reference-faithful).  tc_latent (B,T,tc_dim);
 * codes_out (B,T) int64; logits_out optional (B,T,vq_bins) = last-position logits per step. */
typedef struct {
  mtts_encoder enc;
  const float* pc_embedding;   /* (vq_bins+2, vq_dim) */
  const float* w_predict;      /* packed (1, D, vq_bins) */
  const float* pe;             /* (>=T, D) sine table (modules/embedding.py:66-92) */
  float pe_alpha;
  int32_t vq_bins, vq_dim, tc_dim;
} mtts_plm;
int64_t mtts_plm_infer_workspace_bytes(const mtts_plm* m, int32_t B, int32_t T);
int mtts_plm_infer_f32(const mtts_plm* m, const float* tc_latent, int64_t tc_sb, int32_t tc_ld,
                       int32_t B, int32_t T, int64_t* codes_out, float* logits_out,
                       void* workspace, int64_t workspace_bytes, void* stream);

/* MegaADM.infer (models/megatts2.py:257-275): AR duration regression, raw float feedback,
 * final (p + 0.5) -> int32 -> clamp(1,128).  dur_out (B,T) int32; raw_out optional (B,T). */
typedef struct {
  mtts_encoder enc;
  const float* w_dt;           /* (emb_dim)   dt_linear_emb.weight[:,0] */
  const float* w_tc;           /* packed (1, tc_dim, tc_emb_dim) */
  const float* w_predict;      /* (D) predict_layer.weight[0,:] */
  const float* pe; float pe_alpha;
  int32_t emb_dim, tc_dim, tc_emb_dim;
} mtts_adm;
int64_t mtts_adm_infer_workspace_bytes(const mtts_adm* m, int32_t B, int32_t T);
int mtts_adm_infer_f32(const mtts_adm* m, const float* tc_latent, int64_t tc_sb, int32_t tc_ld,
                       int32_t B, int32_t T, int32_t* dur_out, float* raw_out,
                       void* workspace, int64_t workspace_bytes, void* stream);

/* Opt-in causal KV-cache decode (SURVEY.md 8f-1; NOT what the reference's infer() computes).  Follows the TRAINING
 * semantics of MegaPLM.forward / MegaADM.forward (causal=True, models/megatts2.py:158, 244): row t attends to rows <= t,
 * so a step computes one row per utterance and appends its K/V to per-layer caches - O(T) instead of the O(T^2) full
 * recompute.  Same arguments and outputs as the *_infer_f32 entry points; linear feed-forward encoders only. */
int64_t mtts_plm_decode_causal_workspace_bytes(const mtts_plm* m, int32_t B, int32_t T);
int mtts_plm_decode_causal_f32(const mtts_plm* m, const float* tc_latent, int64_t tc_sb, int32_t tc_ld,
                               int32_t B, int32_t T, int64_t* codes_out, float* logits_out,
                               void* workspace, int64_t workspace_bytes, void* stream);
int64_t mtts_adm_decode_causal_workspace_bytes(const mtts_adm* m, int32_t B, int32_t T);
int mtts_adm_decode_causal_f32(const mtts_adm* m, const float* tc_latent, int64_t tc_sb, int32_t tc_ld,
                               int32_t B, int32_t T, int32_t* dur_out, float* raw_out,
                               void* workspace, int64_t workspace_bytes, void* stream);

/* ConvNet family (modules/convnet.py).  One ConvBlock = ReLU -> Conv1d(C,C,k,same) -> LN(C). */
typedef struct { const float *w, *b, *ln_g, *ln_b; const void* w_tc; } mtts_conv_block;   /* w packed (k,C,C); w_tc (3,k,C,C) bf16 or NULL */

typedef struct {
  int32_t in_channels, out_channels, hidden, k, n_stacks, n_blocks;
  int32_t engine;                      /* 0: fp32 FFMA; tcgen05 for the eligible convs: 1 = BF16X3, 2 = F16X2 */
  const float *w_first, *b_first;      /* packed (k, Cin, hidden) */
  const float *w_last, *b_last;        /* packed (k, hidden, Cout) */
  const mtts_conv_block* blocks;       /* HOST array [n_stacks*n_blocks] */
} mtts_convnet;
/* ConvNet.forward (convnet.py:115-119): x (B,T,Cin) -> y (B,T,Cout), channels-last */
int64_t mtts_convnet_workspace_bytes(const mtts_convnet* n, int32_t B, int32_t T);
int mtts_convnet_forward_f32(const mtts_convnet* n, const float* x, int64_t x_sb, int32_t ldx,
                             float* y, int64_t y_sb, int32_t ldy, int32_t B, int32_t T,
                             void* workspace, int64_t workspace_bytes, void* stream);

typedef struct {
  int32_t in_channels, out_channels, hidden, k, n_layers, n_stacks, n_blocks;
  int32_t engine;
  int32_t middle_kind;                 /* 0: MaxPool1d(middle_k, ceil) ; 1: strided Conv1d(k=middle_k, stride, pad) */
  int32_t middle_k, middle_stride, middle_pad;
  const float *w_middle, *b_middle;    /* packed (middle_k, hidden, hidden) when middle_kind == 1 */
  const float *w_first, *b_first, *w_last, *b_last;
  const mtts_conv_block* blocks;       /* HOST array [n_layers][2][n_stacks*n_blocks] */
} mtts_convnet_double;
/* ConvNetDouble.forward (convnet.py:202-210): x (B,T,Cin) -> y (B,T_mid,Cout) */
int32_t mtts_convnet_double_out_len(const mtts_convnet_double* n, int32_t T);
int64_t mtts_convnet_double_workspace_bytes(const mtts_convnet_double* n, int32_t B, int32_t T);
int mtts_convnet_double_forward_f32(const mtts_convnet_double* n, const float* x, int64_t x_sb, int32_t ldx,
                                    float* y, int64_t y_sb, int32_t ldy, int32_t B, int32_t T,
                                    void* workspace, int64_t workspace_bytes, void* stream);

/* HiFi-GAN V1 generator (speechbrain HIFIGAN.decode_batch, called at
 * models/megatts2.py:370-372).  mel (B, T, 80) channels-last -> wav (B, 256*(T+2*pad)). */
typedef struct {
  const float *w1[3], *b1[3], *w2[3], *b2[3]; int32_t k; int32_t dil[3];
  const void *w1_tc[3], *w2_tc[3];     /* (3, k, C, C) bf16 planes or NULL */
} mtts_hifigan_resblock;
typedef struct {
  int32_t in_channels, ch0, n_ups, n_kernels, inference_padding;
  int32_t engine;
  int32_t up_factor[4], up_kernel[4];
  const float *w_pre, *b_pre;          /* packed (7, 80, ch0) */
  const float *w_up[4], *b_up[4];      /* packed (2, Cin, s*Cout), bias expanded to (s*Cout) */
  const void* w_up_tc[4];              /* (3, 2, s*Cout, Cin) bf16 planes or NULL */
  const mtts_hifigan_resblock* resblocks;  /* HOST array [n_ups*n_kernels] */
  const float *w_post, *b_post;        /* packed (7, C_last, 1) */
} mtts_hifigan;
int64_t mtts_hifigan_workspace_bytes(const mtts_hifigan* h, int32_t B, int32_t T);
int mtts_hifigan_forward_f32(const mtts_hifigan* h, const float* mel, int64_t mel_sb, int32_t mel_ld,
                             int32_t B, int32_t T, float* wav, int64_t wav_sb,
                             void* workspace, int64_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MEGATTS2_B200_H */
