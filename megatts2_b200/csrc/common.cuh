// Shared helpers for libmegatts2_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>

#include "../../include/megatts2_b200.h"

namespace mtts {

extern thread_local char g_err[512];
extern std::atomic<int64_t> g_launches;

inline int fail(int code, const char* fmt, const char* a = "", long long b = 0, long long c = 0) {
  snprintf(g_err, sizeof(g_err), fmt, a, b, c);
  return code;
}

#define MTTS_REQUIRE(cond, msg)                                                      \
  do {                                                                               \
    if (!(cond)) return mtts::fail(MTTS_ERR_BAD_ARG, "%s: requirement failed: " msg, __func__); \
  } while (0)

// per-launch event trace (diagnostics; off by default): one event after every launch on its stream,
// duration(i) = event(i) - event(i-1) since everything runs on one stream
void trace_record(const char* name, cudaStream_t st);
extern bool g_trace_on;

#define MTTS_CHECK_LAUNCH()                                                          \
  do {                                                                               \
    mtts::g_launches.fetch_add(1, std::memory_order_relaxed);                        \
    if (mtts::g_trace_on) mtts::trace_record(__func__, st);                          \
    cudaError_t e__ = cudaGetLastError();                                            \
    if (e__ != cudaSuccess)                                                          \
      return mtts::fail(MTTS_ERR_CUDA, "%s: CUDA launch failed: %lld", __func__, (long long)e__); \
  } while (0)

#define MTTS_TRY(expr)                                                               \
  do {                                                                               \
    int r__ = (expr);                                                                \
    if (r__ != 0) return r__;                                                        \
  } while (0)

// ---- programmatic dependent launch (PDL).  Every kernel of the library starts with pdl_entry() (or, for the kernels with
// a real prologue - barrier init, TMEM allocation, descriptor prefetch - pdl_trigger() at entry and pdl_wait() before the
// first access to global memory): launch_dependents lets the NEXT kernel of the stream be scheduled while this one still
// runs, and the wait blocks it until this grid has completed and flushed, so only launch latency and prologues overlap -
// never data.  Launches go through launch_k(), which sets the stream-serialisation attribute (MEGATTS2_PDL=0 disables it;
// the device-side instructions are no-ops for a kernel launched without the attribute).
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_entry() {
  pdl_trigger();
  pdl_wait();
}
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);      // a failure is picked up by MTTS_CHECK_LAUNCH
}

static inline int64_t cdiv64(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline int64_t align_up(int64_t a, int64_t b) { return cdiv64(a, b) * b; }

// bump allocator over the caller-provided workspace
struct Arena {
  char* base;
  int64_t size, off;
  // the base is rounded up to 256 bytes, so a raw C caller's workspace need not be aligned (float4 / TMA carving is)
  Arena(void* p, int64_t n) : base((char*)((((uintptr_t)p) + 255) & ~(uintptr_t)255)), size(n - (int64_t)(base - (char*)p)), off(0) {}
  template <typename T>
  T* take(int64_t n) {
    off = align_up(off, 256);
    T* r = (T*)(base + off);
    off += n * (int64_t)sizeof(T);
    return r;
  }
  bool ok() const { return off <= size; }
};

__device__ __forceinline__ float act_apply(float v, int act, float slope) {
  if (act == MTTS_ACT_RELU) return fmaxf(v, 0.f);
  if (act == MTTS_ACT_LEAKY) return v > 0.f ? v : v * slope;   // (kept as a select: correct for any slope)
  if (act == MTTS_ACT_TANH) return tanhf(v);
  return v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace mtts
