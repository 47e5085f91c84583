// C ABI: op-level entry points + library state.  (Composite drivers export theirs from
// drivers.cu.)  No C++ exception crosses this boundary; errors are negative codes plus a
// thread-local message.
#include <algorithm>
#include <stdlib.h>

#include "kernels.h"

#include <map>
#include <mutex>
#include <string>
#include <vector>

namespace mtts {
thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("MEGATTS2_PDL");
    return !(e && e[0] == '0');
  }();
  return on;
}

bool g_trace_on = false;
static std::mutex g_trace_mu;
static std::vector<std::pair<std::string, cudaEvent_t>> g_trace;
void trace_record(const char* name, cudaStream_t st) {
  std::lock_guard<std::mutex> lk(g_trace_mu);
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, st);
  g_trace.emplace_back(name, e);
}
}  // namespace mtts

using namespace mtts;

extern "C" {

int mtts_abi_version(void) { return MTTS_ABI_VERSION; }
const char* mtts_last_error(void) { return g_err; }
int64_t mtts_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

/* diagnostics: begin records a start marker on `stream`; end synchronises and writes a table
 * "launcher  launches  total_ms" (sorted by time) into buf */
int mtts_trace_begin(void* stream) {
  std::lock_guard<std::mutex> lk(g_trace_mu);
  for (auto& t : g_trace) cudaEventDestroy(t.second);
  g_trace.clear();
  cudaEvent_t e;
  cudaEventCreate(&e);
  cudaEventRecord(e, (cudaStream_t)stream);
  g_trace.emplace_back("<begin>", e);
  g_trace_on = true;
  return 0;
}
int mtts_trace_end(char* buf, int32_t buf_len) {
  std::lock_guard<std::mutex> lk(g_trace_mu);
  g_trace_on = false;
  std::map<std::string, std::pair<int, double>> agg;
  double total = 0.0;
  for (size_t i = 1; i < g_trace.size(); ++i) {
    float ms = 0.f;
    cudaEventSynchronize(g_trace[i].second);
    cudaEventElapsedTime(&ms, g_trace[i - 1].second, g_trace[i].second);
    agg[g_trace[i].first].first += 1;
    agg[g_trace[i].first].second += ms;
    total += ms;
  }
  std::vector<std::pair<double, std::string>> order;
  for (auto& kv : agg) order.emplace_back(-kv.second.second, kv.first);
  std::sort(order.begin(), order.end());
  int off = 0;
  for (auto& o : order) {
    auto& v = agg[o.second];
    off += snprintf(buf + off, off < buf_len ? buf_len - off : 0, "%-28s %7d %10.3f ms %5.1f%%\n", o.second.c_str(), v.first,
                    v.second, 100.0 * v.second / (total > 0 ? total : 1));
    if (off >= buf_len) break;
  }
  if (off < buf_len) snprintf(buf + off, buf_len - off, "%-28s %7d %10.3f ms\n", "TOTAL", (int)g_trace.size() - 1, total);
  for (auto& t : g_trace) cudaEventDestroy(t.second);
  g_trace.clear();
  return 0;
}

int mtts_conv1d_f32(const mtts_conv_params* p, void* stream) {
  MTTS_REQUIRE(p, "null params");
  return conv1d(*p, (cudaStream_t)stream);
}

int mtts_layernorm_f32(const float* x, int32_t ldx, const float* gamma, const float* beta, const float* res, int32_t ldr,
                       float* y, int32_t ldy, int64_t rows, int32_t C, float eps, int32_t post_act, int32_t accumulate,
                       void* stream) {
  return layernorm(x, ldx, gamma, beta, res, ldr, y, ldy, rows, C, eps, post_act, accumulate, (cudaStream_t)stream);
}

int mtts_attention_f32(const mtts_attn_params* p, void* stream) {
  MTTS_REQUIRE(p, "null params");
  return attention(*p, (cudaStream_t)stream);
}

int mtts_vq_argmin_f32(const float* x, int32_t ldx, const float* embed, int64_t N, int32_t D, int32_t K, int64_t* idx,
                       void* stream) {
  return vq_argmin(x, ldx, embed, N, D, K, idx, (cudaStream_t)stream);
}

int mtts_vq_gather_f32(const int64_t* idx, int32_t idx_ld, const float* embed, int32_t D, int32_t K, int32_t B,
                       int32_t T_out, int32_t repeat, float* y, int64_t y_sb, int32_t ldy, void* stream) {
  return vq_gather(idx, idx_ld, embed, D, K, B, T_out, repeat, y, y_sb, ldy, (cudaStream_t)stream);
}

int mtts_mel_spectrogram_f32(const float* wav, int64_t wav_sb, int32_t B, int32_t L, const float* window,
                             const float* fb_w, const int32_t* fb_off, const int32_t* fb_start, int32_t n_mels,
                             float clamp_min, float* out, int64_t out_sb, int64_t out_sm, int64_t out_sf, void* stream) {
  return mel_spectrogram(wav, wav_sb, B, L, nullptr, window, fb_w, fb_off, fb_start, n_mels, clamp_min, out, out_sb, out_sm,
                         out_sf, (cudaStream_t)stream);
}

int mtts_mel_spectrogram_ragged_f32(const float* wav, int64_t wav_sb, int32_t B, int32_t L_max, const int32_t* lens,
                                    const float* window, const float* fb_w, const int32_t* fb_off, const int32_t* fb_start,
                                    int32_t n_mels, float clamp_min, float* out, int64_t out_sb, int64_t out_sm,
                                    int64_t out_sf, void* stream) {
  MTTS_REQUIRE(lens, "null lens");
  return mel_spectrogram(wav, wav_sb, B, L_max, lens, window, fb_w, fb_off, fb_start, n_mels, clamp_min, out, out_sb, out_sm,
                         out_sf, (cudaStream_t)stream);
}

int mtts_maxpool_time_f32(const float* x, int64_t x_sb, int32_t ldx, float* y, int64_t y_sb, int32_t ldy, int32_t B,
                          int32_t T, int32_t C, int32_t k, void* stream) {
  return maxpool_time(x, x_sb, ldx, y, y_sb, ldy, B, T, C, k, (cudaStream_t)stream);
}

int mtts_embed_pe_f32(const int64_t* ids, int32_t ids_ld, const float* table, int32_t vocab, int32_t D, const float* pe,
                      float alpha, int32_t pe_offset, int32_t B, int32_t T, float* y, int64_t y_sb, int32_t ldy,
                      void* stream) {
  return embed_pe(ids, ids_ld, table, vocab, D, pe, alpha, pe_offset, B, T, y, y_sb, ldy, (cudaStream_t)stream);
}

int mtts_add_pe_f32(const float* x, int64_t x_sb, int32_t ldx, const float* pe, float alpha, int32_t B, int32_t T,
                    int32_t D, float* y, int64_t y_sb, int32_t ldy, void* stream) {
  return add_pe(x, x_sb, ldx, pe, alpha, B, T, D, y, y_sb, ldy, (cudaStream_t)stream);
}

int mtts_length_regulate_f32(const float* x, int64_t x_sb, int32_t ldx, const int32_t* dur, int32_t dur_ld, int32_t B,
                             int32_t Tp, int32_t D, int32_t L_out, float* y, int64_t y_sb, int32_t ldy, int32_t* totals,
                             void* stream) {
  return length_regulate(x, x_sb, ldx, dur, dur_ld, B, Tp, D, L_out, y, y_sb, ldy, totals, (cudaStream_t)stream);
}

int mtts_mask_tail_f32(float* x, int32_t B, int32_t rows, int32_t L, const int32_t* keep, void* stream) {
  return mask_tail(x, B, rows, L, keep, (cudaStream_t)stream);
}

int mtts_copy_strided_f32(const float* x, int64_t x_sb, int64_t x_st, int64_t x_sc, float* y, int64_t y_sb, int64_t y_st,
                          int64_t y_sc, int32_t B, int32_t T, int32_t C, int32_t pad_rep, void* stream) {
  return copy_strided(x, x_sb, x_st, x_sc, y, y_sb, y_st, y_sc, B, T, C, pad_rep, (cudaStream_t)stream);
}

}  // extern "C"
