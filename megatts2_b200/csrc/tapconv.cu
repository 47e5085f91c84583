// Tap-GEMM: implicit-GEMM 1-D convolution / linear layer, channels-last, fp32 FFMA path.
//
//   acc[b,t,n] = sum_{j<k} sum_{c<Cin} pre(X[b, t*stride + j*dil - pad, c]) * W[j][c][n]
//
// replaces nn.Linear / nn.Conv1d / nn.ConvTranspose1d calls of the reference
// (modules/convnet.py:13-18, modules/transformer.py:26-31,76-85, modules/mrte.py:101-107,
// HiFi-GAN generator).  This is the exact-fp32 engine: every product is an FFMA, so ids
// derived from it (VQ codes, PLM argmax) are as close to the CPU fp32 reference as fp32
// reassociation allows.  The tcgen05 3xTF32 engine (tapconv_tc.cu) shares this ABI.
//
// Tiling: BM x BN output tile per CTA, BK = 16 reduction slice, double-buffered shared
// memory with register prefetch; each thread owns a TM x TN micro-tile split into 4-wide
// groups so every shared-memory read is a conflict-free LDS.128.
#include "common.cuh"

namespace mtts {

struct ConvFlags {
  int vec_a, vec_b, vec_y;
  int kk_per_split;        // split-K: reduction slices per blockIdx.z (0 = no split)
  float* partial;          // split-K: raw partial sums [splits][M][Cout]
};

__device__ __forceinline__ int map_row(int ti, int len, int mode) {
  if (ti >= 0 && ti < len) return ti;
  if (mode == MTTS_PAD_ZERO || len <= 0) return -1;
  if (mode == MTTS_PAD_REPLICATE) return ti < 0 ? 0 : len - 1;
  if (ti < 0) ti = -ti;
  if (ti >= len) ti = 2 * (len - 1) - ti;
  return (ti >= 0 && ti < len) ? ti : -1;
}

template <int BM, int BN, int TM, int TN>
__global__ void __launch_bounds__((BM / TM) * (BN / TN), ((BM / TM) * (BN / TN) <= 256 ? 2 : 1))
tapconv_kernel(const mtts_conv_params p, const ConvFlags fl) {
  pdl_entry();
  constexpr int BK = 16;
  constexpr int NT = (BM / TM) * (BN / TN);
  constexpr int AP = BM + 4;
  constexpr int A_IT = (BM * BK / 4) / NT;
  constexpr int B_IT = (BK * BN / 4) / NT;
  static_assert(A_IT >= 1 && B_IT >= 1, "tile too small for the thread count");
  static_assert((BM * BK / 4) % NT == 0 && (BK * BN / 4) % NT == 0, "loader shape");
  __shared__ __align__(16) float As[2][BK][AP];
  __shared__ __align__(16) float Bs[2][BK][BN];

  const int tid = threadIdx.x;
  const int64_t M = (int64_t)p.B * p.Tout;
  const int64_t m0 = (int64_t)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;
  const int nchunk = (p.Cin + BK - 1) / BK;
  const int nk_all = p.k * nchunk;
  const int kk_lo = fl.kk_per_split ? blockIdx.z * fl.kk_per_split : 0;
  const int nk = fl.kk_per_split ? min(nk_all, kk_lo + fl.kk_per_split) : nk_all;

  // ---- per-thread A rows (fixed for the whole K loop)
  int64_t a_base[A_IT];
  int a_t0[A_IT], a_len[A_IT], a_row[A_IT], a_c4[A_IT];
#pragma unroll
  for (int i = 0; i < A_IT; ++i) {
    const int idx = tid + i * NT;
    a_row[i] = idx >> 2;
    a_c4[i] = (idx & 3) * 4;
    const int64_t m = m0 + a_row[i];
    if (m < M) {
      const int b = (int)(m / p.Tout);
      const int t = (int)(m - (int64_t)b * p.Tout);
      a_base[i] = (int64_t)b * p.x_batch_stride;
      a_t0[i] = t * p.stride - p.pad;
      a_len[i] = p.in_lens ? min(p.in_lens[b], p.Tin) : p.Tin;
    } else {
      a_base[i] = 0;
      a_t0[i] = 0;
      a_len[i] = 0;  // every row maps to "outside" -> zeros
    }
  }
  int b_krow[B_IT], b_n4[B_IT];
#pragma unroll
  for (int i = 0; i < B_IT; ++i) {
    const int idx = tid + i * NT;
    b_krow[i] = idx / (BN / 4);
    b_n4[i] = (idx % (BN / 4)) * 4;
  }

  float4 ra[A_IT], rb[B_IT];

  auto load_regs = [&](int kk) {
    const int j = kk / nchunk;
    const int c0 = (kk - j * nchunk) * BK;
#pragma unroll
    for (int i = 0; i < A_IT; ++i) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      const int ti = map_row(a_t0[i] + j * p.dil, a_len[i], p.pad_mode);
      const int c = c0 + a_c4[i];
      if (ti >= 0 && c < p.Cin) {
        const float* src = p.x + a_base[i] + (int64_t)ti * p.ldx + c;
        if (fl.vec_a) {
          v = __ldg(reinterpret_cast<const float4*>(src));
        } else {
          v.x = __ldg(src);
          if (c + 1 < p.Cin) v.y = __ldg(src + 1);
          if (c + 2 < p.Cin) v.z = __ldg(src + 2);
          if (c + 3 < p.Cin) v.w = __ldg(src + 3);
        }
        if (p.pre_act != MTTS_ACT_NONE) {
          v.x = act_apply(v.x, p.pre_act, p.pre_slope);
          v.y = act_apply(v.y, p.pre_act, p.pre_slope);
          v.z = act_apply(v.z, p.pre_act, p.pre_slope);
          v.w = act_apply(v.w, p.pre_act, p.pre_slope);
        }
      }
      ra[i] = v;
    }
#pragma unroll
    for (int i = 0; i < B_IT; ++i) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      const int c = c0 + b_krow[i];
      const int n = n0 + b_n4[i];
      if (c < p.Cin && n < p.Cout) {
        const float* src = p.w + ((int64_t)j * p.Cin + c) * p.Cout + n;
        if (fl.vec_b) {
          v = __ldg(reinterpret_cast<const float4*>(src));
        } else {
          v.x = __ldg(src);
          if (n + 1 < p.Cout) v.y = __ldg(src + 1);
          if (n + 2 < p.Cout) v.z = __ldg(src + 2);
          if (n + 3 < p.Cout) v.w = __ldg(src + 3);
        }
      }
      rb[i] = v;
    }
  };
  auto store_smem = [&](int buf) {
#pragma unroll
    for (int i = 0; i < A_IT; ++i) {
      As[buf][a_c4[i] + 0][a_row[i]] = ra[i].x;
      As[buf][a_c4[i] + 1][a_row[i]] = ra[i].y;
      As[buf][a_c4[i] + 2][a_row[i]] = ra[i].z;
      As[buf][a_c4[i] + 3][a_row[i]] = ra[i].w;
    }
#pragma unroll
    for (int i = 0; i < B_IT; ++i)
      *reinterpret_cast<float4*>(&Bs[buf][b_krow[i]][b_n4[i]]) = rb[i];
  };

  constexpr int TXN = BN / TN;
  const int ty = tid / TXN, tx = tid % TXN;
  constexpr int MG = TM / 4, NG = TN / 4;   // 4-wide groups per thread
  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  load_regs(kk_lo);
  store_smem(0);
  __syncthreads();
  int cur = 0;
  for (int kk = kk_lo; kk < nk; ++kk) {
    if (kk + 1 < nk) load_regs(kk + 1);
#pragma unroll
    for (int k = 0; k < BK; ++k) {
      float a[TM], b[TN];
#pragma unroll
      for (int g = 0; g < MG; ++g) {
        const float4 v = *reinterpret_cast<const float4*>(&As[cur][k][g * (BM / MG) + ty * 4]);
        a[g * 4 + 0] = v.x; a[g * 4 + 1] = v.y; a[g * 4 + 2] = v.z; a[g * 4 + 3] = v.w;
      }
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const float4 v = *reinterpret_cast<const float4*>(&Bs[cur][k][g * (BN / NG) + tx * 4]);
        b[g * 4 + 0] = v.x; b[g * 4 + 1] = v.y; b[g * 4 + 2] = v.z; b[g * 4 + 3] = v.w;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (kk + 1 < nk) store_smem(cur ^ 1);
    __syncthreads();
    cur ^= 1;
  }

  // ---- split-K: raw partial sums only (the epilogue runs in splitk_reduce_kernel)
  if (fl.partial) {
    float* part = fl.partial + (int64_t)blockIdx.z * M * p.Cout;
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int row = (i / 4) * (BM / MG) + ty * 4 + (i & 3);
      const int64_t m = m0 + row;
      if (m >= M) continue;
#pragma unroll
      for (int g = 0; g < NG; ++g) {
        const int n = n0 + g * (BN / NG) + tx * 4;
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (n + e < p.Cout) part[m * p.Cout + n + e] = acc[i][g * 4 + e];
      }
    }
    return;
  }
  // ---- epilogue
  const int64_t ybe = p.y_batch_elems ? p.y_batch_elems : (int64_t)p.Tout * p.ldy;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    const int row = (i / 4) * (BM / MG) + ty * 4 + (i & 3);
    const int64_t m = m0 + row;
    if (m >= M) continue;
    const int b = (int)(m / p.Tout);
    const int t = (int)(m - (int64_t)b * p.Tout);
#pragma unroll
    for (int g = 0; g < NG; ++g) {
      const int n = n0 + g * (BN / NG) + tx * 4;
      if (n >= p.Cout) continue;
      float v[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float x = acc[i][g * 4 + e];
        if (p.bias && n + e < p.Cout) x += __ldg(p.bias + n + e);
        v[e] = act_apply(x, p.post_act, p.post_slope);
      }
      const int64_t flat = (int64_t)t * p.ldy + n + p.out_shift;
      float* dst = p.y + (int64_t)b * p.y_batch_stride + flat;
      const float* rsrc = p.res ? p.res + (int64_t)b * p.res_batch_stride + (int64_t)t * p.ldr + n : nullptr;
      if (fl.vec_y) {
        if (flat < 0 || flat >= ybe) continue;
        if (rsrc) {
          const float4 r = *reinterpret_cast<const float4*>(rsrc);  // may alias y: plain load
          v[0] += r.x; v[1] += r.y; v[2] += r.z; v[3] += r.w;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e) v[e] *= p.out_scale;
        if (p.accumulate) {
          const float4 o = *reinterpret_cast<const float4*>(dst);
          v[0] += o.x; v[1] += o.y; v[2] += o.z; v[3] += o.w;
        }
        *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
      } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (n + e >= p.Cout) break;
          if (flat + e < 0 || flat + e >= ybe) continue;
          float x = v[e];
          if (rsrc) x += rsrc[e];
          x *= p.out_scale;
          if (p.accumulate) x += dst[e];
          dst[e] = x;
        }
      }
    }
  }
}



// Single-output-channel conv (HiFi-GAN conv_post: 32 -> 1, k = 7, tanh).  One thread per output sample walks
// its k x Cin window with float4 loads (neighbouring threads share rows through L1); weights sit in shared
// memory.  A 128x32 GEMM tile would waste 31/32 of its columns here.
__global__ void __launch_bounds__(256)
conv_cout1_kernel(const mtts_conv_params p) {
  pdl_entry();
  extern __shared__ __align__(16) float wsm[];       // [k][Cin]
  for (int i = threadIdx.x; i < p.k * p.Cin; i += 256) wsm[i] = __ldg(p.w + i);   // packed (k, Cin, 1)
  __syncthreads();
  const int64_t M = (int64_t)p.B * p.Tout;
  const int64_t m = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (m >= M) return;
  const int b = (int)(m / p.Tout), t = (int)(m - (int64_t)b * p.Tout);
  const int len = p.in_lens ? min(p.in_lens[b], p.Tin) : p.Tin;
  const float* xb = p.x + (int64_t)b * p.x_batch_stride;
  float acc = 0.f;
  for (int j = 0; j < p.k; ++j) {
    const int ti = map_row(t * p.stride + j * p.dil - p.pad, len, p.pad_mode);
    if (ti < 0) continue;
    const float4* xr = reinterpret_cast<const float4*>(xb + (int64_t)ti * p.ldx);
    const float4* wr = reinterpret_cast<const float4*>(wsm + j * p.Cin);
    for (int c = 0; c < p.Cin / 4; ++c) {
      float4 v = __ldg(xr + c);
      const float4 w = wr[c];
      if (p.pre_act != MTTS_ACT_NONE) {
        v.x = act_apply(v.x, p.pre_act, p.pre_slope); v.y = act_apply(v.y, p.pre_act, p.pre_slope);
        v.z = act_apply(v.z, p.pre_act, p.pre_slope); v.w = act_apply(v.w, p.pre_act, p.pre_slope);
      }
      acc = fmaf(v.x, w.x, acc); acc = fmaf(v.y, w.y, acc); acc = fmaf(v.z, w.z, acc); acc = fmaf(v.w, w.w, acc);
    }
  }
  if (p.bias) acc += __ldg(p.bias);
  acc = act_apply(acc, p.post_act, p.post_slope);
  if (p.res) acc += p.res[(int64_t)b * p.res_batch_stride + (int64_t)t * p.ldr];
  acc *= p.out_scale;
  float* dst = p.y + (int64_t)b * p.y_batch_stride + (int64_t)t * p.ldy;
  if (p.accumulate) acc += *dst;
  *dst = acc;
}

// The same layer with its input window staged in shared memory (stride 1): a CTA owns 256 consecutive outputs of one
// batch item and loads their 256 + (k - 1) dil input rows ONCE, coalesced, applying the pre-activation on the way; each
// thread then walks its window with conflict-free 128-bit shared loads (row stride Cin + 4 floats).  The per-thread form
// above fetched every row 7 times through L1 with one 16-byte piece of a different 128-byte line per lane (1.78 ms for
// the vocoder's 64 x 133 632 x 32 input, ten times its HBM time).  Same accumulation order, bit-identical results.
__global__ void __launch_bounds__(256)
conv_cout1_tiled_kernel(const mtts_conv_params p) {
  pdl_entry();
  extern __shared__ __align__(16) float wsm[];       // [k][Cin] weights, then the input window [rows][Cin + 4]
  const int XS = p.Cin + 4;
  const int rows = 256 + (p.k - 1) * p.dil;
  float* xs = wsm + ((p.k * p.Cin + 3) & ~3);
  for (int i = threadIdx.x; i < p.k * p.Cin; i += 256) wsm[i] = __ldg(p.w + i);   // packed (k, Cin, 1)
  const int b = blockIdx.y, t0 = blockIdx.x * 256;
  const int len = p.in_lens ? min(p.in_lens[b], p.Tin) : p.Tin;
  const float* xb = p.x + (int64_t)b * p.x_batch_stride;
  const int c4n = p.Cin >> 2;
  for (int i = threadIdx.x; i < rows * c4n; i += 256) {
    const int r = i / c4n, c4 = i - r * c4n;
    const int ti = map_row(t0 + r - p.pad, len, p.pad_mode);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ti >= 0) {
      v = __ldg(reinterpret_cast<const float4*>(xb + (int64_t)ti * p.ldx) + c4);
      if (p.pre_act != MTTS_ACT_NONE) {
        v.x = act_apply(v.x, p.pre_act, p.pre_slope); v.y = act_apply(v.y, p.pre_act, p.pre_slope);
        v.z = act_apply(v.z, p.pre_act, p.pre_slope); v.w = act_apply(v.w, p.pre_act, p.pre_slope);
      }
    }
    *reinterpret_cast<float4*>(xs + r * XS + 4 * c4) = v;
  }
  __syncthreads();
  const int t = t0 + threadIdx.x;
  if (t >= p.Tout) return;
  float acc = 0.f;
  for (int j = 0; j < p.k; ++j) {
    if (map_row(t + j * p.dil - p.pad, len, p.pad_mode) < 0) continue;      // rows outside a zero-padded input add nothing
    const float4* xr = reinterpret_cast<const float4*>(xs + (threadIdx.x + j * p.dil) * XS);
    const float4* wr = reinterpret_cast<const float4*>(wsm + j * p.Cin);
    for (int c = 0; c < c4n; ++c) {
      const float4 v = xr[c];
      const float4 w = wr[c];
      acc = fmaf(v.x, w.x, acc); acc = fmaf(v.y, w.y, acc); acc = fmaf(v.z, w.z, acc); acc = fmaf(v.w, w.w, acc);
    }
  }
  if (p.bias) acc += __ldg(p.bias);
  acc = act_apply(acc, p.post_act, p.post_slope);
  if (p.res) acc += p.res[(int64_t)b * p.res_batch_stride + (int64_t)t * p.ldr];
  acc *= p.out_scale;
  float* dst = p.y + (int64_t)b * p.y_batch_stride + (int64_t)t * p.ldy;
  if (p.accumulate) acc += *dst;
  *dst = acc;
}

// split-K second pass: fixed-order sum of the partials (deterministic), then the usual epilogue
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const mtts_conv_params p, const float* __restrict__ partial, int splits) {
  pdl_entry();
  const int64_t M = (int64_t)p.B * p.Tout;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * p.Cout) return;
  const int64_t m = i / p.Cout;
  const int n = (int)(i - m * p.Cout);
  float v = 0.f;
  for (int z = 0; z < splits; ++z) v += partial[((int64_t)z * M + m) * p.Cout + n];
  const int b = (int)(m / p.Tout), t = (int)(m - (int64_t)b * p.Tout);
  if (p.bias) v += __ldg(p.bias + n);
  v = act_apply(v, p.post_act, p.post_slope);
  if (p.res) v += p.res[(int64_t)b * p.res_batch_stride + (int64_t)t * p.ldr + n];
  v *= p.out_scale;
  float* dst = p.y + (int64_t)b * p.y_batch_stride + (int64_t)t * p.ldy + n;
  if (p.accumulate) v += *dst;
  *dst = v;
}

template <int BM, int BN, int TM, int TN>
static int launch_cfg(const mtts_conv_params& p, const ConvFlags& fl, cudaStream_t st) {
  const int64_t M = (int64_t)p.B * p.Tout;
  dim3 grid((unsigned)cdiv64(M, BM), (unsigned)cdiv64(p.Cout, BN));
  launch_k(tapconv_kernel<BM, BN, TM, TN>, grid, (BM / TM) * (BN / TN), 0, st, p, fl);
  MTTS_CHECK_LAUNCH();
  return 0;
}

static inline bool al16(const void* p) { return (((uintptr_t)p) & 15) == 0; }

int conv1d_ffma(const mtts_conv_params& p, cudaStream_t st) {
  MTTS_REQUIRE(p.x && p.w && p.y, "null pointer");
  MTTS_REQUIRE(p.B >= 0 && p.Tin >= 0 && p.Tout >= 0 && p.Cin > 0 && p.Cout > 0, "bad dims");
  MTTS_REQUIRE(p.k >= 1 && p.stride >= 1 && p.dil >= 1, "bad conv geometry");
  MTTS_REQUIRE(p.ldx >= p.Cin, "ldx < Cin");
  MTTS_REQUIRE(p.pad_mode >= 0 && p.pad_mode <= 2, "bad pad_mode");
  const int64_t M = (int64_t)p.B * p.Tout;
  if (M == 0) return 0;
  MTTS_REQUIRE(M < (int64_t)2147483647 * 32, "too many rows");
  ConvFlags fl;
  fl.kk_per_split = 0;
  fl.partial = nullptr;
  fl.vec_a = (p.Cin % 4 == 0) && (p.ldx % 4 == 0) && (p.x_batch_stride % 4 == 0) && al16(p.x);
  fl.vec_b = (p.Cout % 4 == 0) && al16(p.w);
  fl.vec_y = (p.Cout % 4 == 0) && (p.ldy % 4 == 0) && (p.y_batch_stride % 4 == 0) && al16(p.y) &&
             (p.out_shift % 4 == 0) && (p.y_batch_elems % 4 == 0) &&
             (!p.res || ((p.ldr % 4 == 0) && (p.res_batch_stride % 4 == 0) && al16(p.res)));
  if (p.Cout == 1 && p.out_shift == 0 && fl.vec_a && p.stride == 1 && (p.k * p.Cin) % 4 == 0 && p.Cin <= 128 && p.B <= 65535 &&
      M >= 4096) {
    const size_t smem = sizeof(float) * ((size_t)((p.k * p.Cin + 3) & ~3) + (size_t)(256 + (p.k - 1) * p.dil) * (p.Cin + 4));
    if (smem <= 48 * 1024) {
      dim3 grid((unsigned)cdiv64(p.Tout, 256), (unsigned)p.B);
      launch_k(conv_cout1_tiled_kernel, grid, 256, smem, st, p);
      MTTS_CHECK_LAUNCH();
      return 0;
    }
  }
  if (p.Cout == 1 && p.out_shift == 0 && fl.vec_a && p.k * p.Cin <= 8192 && M >= 4096) {
    launch_k(conv_cout1_kernel, (unsigned)cdiv64(M, 256), 256, (size_t)p.k * p.Cin * sizeof(float), st, p);
    MTTS_CHECK_LAUNCH();
    return 0;
  }
  // Small-M linear layers (the last-position GEMMs of the AR loops: M = batch rows): a 64x64 tile grid leaves
  // most SMs idle and every CTA walks all of K serially.  Split K over blockIdx.z into the caller's scratch and
  // reduce in a fixed order (bit-reproducible), so ~all SMs stream a slice of the weights.
  {
    const int64_t tiles64 = cdiv64(M, 64) * cdiv64(p.Cout, 64);
    const int nk = (p.Cin + 15) / 16;
    if (p.k == 1 && p.stride == 1 && p.pad == 0 && p.out_shift == 0 && !p.in_lens && M <= 256 && tiles64 <= 148 &&
        nk >= 16 && p.tc_scratch) {
      // two CTAs per SM: a lone 8-warp CTA cannot hide the L2 latency of its one-chunk-ahead prefetch
      constexpr int target = 296;
      int splits = (int)(target / tiles64);
      if (splits > 16) splits = 16;
      if (splits > nk / 4) splits = nk / 4;
      if (splits >= 2 && (int64_t)splits * M * p.Cout * 4 + 256 <= p.tc_scratch_bytes) {
        fl.kk_per_split = (nk + splits - 1) / splits;
        splits = (nk + fl.kk_per_split - 1) / fl.kk_per_split;
        fl.partial = reinterpret_cast<float*>((((uintptr_t)p.tc_scratch) + 255) & ~(uintptr_t)255);
        dim3 grid((unsigned)cdiv64(M, 64), (unsigned)cdiv64(p.Cout, 64), (unsigned)splits);
        launch_k(tapconv_kernel<64, 64, 4, 4>, grid, 256, 0, st, p, fl);
        MTTS_CHECK_LAUNCH();
        launch_k(splitk_reduce_kernel, (unsigned)cdiv64(M * p.Cout, 256), 256, 0, st, p, fl.partial, splits);
        MTTS_CHECK_LAUNCH();
        return 0;
      }
    }
  }
  const int64_t tiles128 = cdiv64(M, 128) * cdiv64(p.Cout, 128);
  if (p.Cout <= 32) return launch_cfg<128, 32, 8, 4>(p, fl, st);
  if (p.Cout <= 64) return launch_cfg<128, 64, 8, 4>(p, fl, st);
  if (tiles128 >= 120) return launch_cfg<128, 128, 8, 8>(p, fl, st);
  return launch_cfg<64, 64, 4, 4>(p, fl, st);
}

}  // namespace mtts
