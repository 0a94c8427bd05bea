// Shared helpers for libkccot (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <atomic>

#include "../../include/kccot.h"

namespace kccot {

void set_error(const char* fmt, ...);
extern std::atomic<unsigned long long> g_launches;
inline void count_launch(int n = 1) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }

#define KCCOT_CHECK_ARG(cond, ...)            \
  do {                                        \
    if (!(cond)) {                            \
      ::kccot::set_error(__VA_ARGS__);        \
      return KCCOT_EINVAL;                    \
    }                                         \
  } while (0)

#define KCCOT_CUDA(expr)                                                                  \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::kccot::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                         __LINE__);                                                       \
      return KCCOT_ECUDA;                                                                 \
    }                                                                                     \
  } while (0)

#define KCCOT_LAUNCH_CHECK()                                                             \
  do {                                                                                   \
    ::kccot::count_launch();                                                             \
    cudaError_t _e = cudaGetLastError();                                                 \
    if (_e != cudaSuccess) {                                                             \
      ::kccot::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e),      \
                         __FILE__, __LINE__);                                            \
      return KCCOT_ECUDA;                                                                \
    }                                                                                    \
  } while (0)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Function attributes (the opt-in to more than 48 KB of dynamic shared memory) are per DEVICE: a call site
// keeps one `static size_t cache[kMaxDevices]` and asks here whether the current device still needs
// cudaFuncSetAttribute for `want` bytes.  (A benign race between host threads costs a redundant call.)
constexpr int kMaxDevices = 64;
inline bool smem_attr_needed(size_t (&cache)[kMaxDevices], size_t want) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) return true;
  if (want <= cache[dev]) return false;
  cache[dev] = want;
  return true;
}

// Programmatic dependent launch (sm_90+).  A kernel launched with launch_pdl() may start while the previous
// kernel of the stream is still running, once every CTA of that kernel has executed pdl_launch_dependents()
// (or exited); it must execute pdl_wait() before touching anything the previous kernel writes.  Rule used
// throughout: a kernel calls pdl_launch_dependents() only AFTER its own pdl_wait(), so whatever a dependent
// reads before its wait was complete when its predecessor's wait returned (dependencies stay transitive).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
int num_sms();

// Shared-context hint of kccot_mixed_loss_fwd_ctx / _bwd_ctx (the reference builds fake = concat(real_in, fake_pred),
// kernel_train.py:225-226): columns c of the flattened [B, K] rows with (c % period) < len hold the same values in
// real and fake.  The entry points open a CtxScope; the tensor-core launchers read it (zero = no hint).
struct CtxHint { long long period, len; };
extern thread_local CtxHint t_ctx;
struct CtxScope {
  CtxHint prev;
  CtxScope(long long period, long long len) : prev(t_ctx) { t_ctx = CtxHint{period, len}; }
  ~CtxScope() { t_ctx = prev; }
};
// hint in units of 32-column boxes, or false when it cannot be used for this K
inline bool ctx_boxes(long long K, int* period_boxes, int* len_boxes) {
  const CtxHint h = t_ctx;
  if (h.len <= 0 || h.period <= h.len || h.period % 32 || h.len % 32 || K % h.period) return false;
  if (h.period / 32 > 0x7fffffffLL) return false;
  *period_boxes = (int)(h.period / 32);
  *len_boxes = (int)(h.len / 32);
  return true;
}

struct SideLane {
  cudaStream_t stream;
  cudaEvent_t fork, join;
};
SideLane* side_lane();   // per host thread and device; nullptr if the stream / events cannot be created

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

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
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_log2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// bf16 as raw bits (uint16_t): widening to fp32 is exact, narrowing rounds to nearest even
// four bf16 (element 0 in the low half of .x) -> fp32
__device__ __forceinline__ float4 widen_bf16x4(uint2 v) {
  return make_float4(__uint_as_float(v.x << 16), __uint_as_float(v.x & 0xffff0000u), __uint_as_float(v.y << 16),
                     __uint_as_float(v.y & 0xffff0000u));
}
// two fp32 -> two bf16 in one word (lo in the low half)
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}

}  // namespace kccot
