// Shared device/host helpers for libmra_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <string>
#include <map>
#include <mutex>
#include <utility>

#include "../../include/mra_gan_b200.h"

namespace mra {

typedef __nv_bfloat16 bf16;

// ---- error plumbing (thread-local message, negative return codes, nothing throws) ----
extern thread_local std::string g_last_error;
inline int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}
#define MRA_CHECK_CUDA(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess)                                                                \
      return ::mra::fail(-100 - (int)_e, "%s failed: %s (%s:%d)", #expr,                  \
                         cudaGetErrorString(_e), __FILE__, __LINE__);                     \
  } while (0)
#define MRA_REQUIRE(cond, ...)                                                            \
  do {                                                                                    \
    if (!(cond)) return ::mra::fail(-1, __VA_ARGS__);                                     \
  } while (0)
// every kernel launch site is followed by exactly one MRA_LAUNCH_CHECK(): it doubles as the launch counter
extern std::atomic<long long> g_launch_count;
#define MRA_LAUNCH_CHECK()                                                                \
  do {                                                                                    \
    ::mra::g_launch_count.fetch_add(1, std::memory_order_relaxed);                        \
    MRA_CHECK_CUDA(cudaGetLastError());                                                   \
  } while (0)

// ---- programmatic dependent launch (PDL) ----
// A step is ~1100 launches of persistent, one-CTA-per-SM kernels; between two dependent kernels the stream (or graph)
// pays the launch / dependency latency and the successor's prologue (barrier init, tensor-map prefetch, TMEM
// allocation) in series: ~5 us per boundary, ~5 % of the step (sum of kernel durations 116 ms vs a 122 ms step).
// The hot kernels therefore (a) let their successor launch at once (griddepcontrol.launch_dependents as their first
// instruction: its CTAs become resident SM by SM as ours retire and run their prologue), (b) wait for their
// predecessors (griddepcontrol.wait: full completion + memory visibility) after the prologue and BEFORE the first
// global-memory access -- reads of anything a predecessor wrote, and writes, which could hit a buffer a predecessor
// still reads.  Every PDL-launched kernel executes the wait, so ordering stays transitive.
// MEASURED (profiles/r02_pdl_ab.txt, driver command, A/B/A/B on one box): 123.15 / 123.39 ms with the attribute,
// 122.83 / 122.93 ms without -- no gain: a persistent one-CTA-per-SM kernel with ~200 KB of shared memory cannot
// become resident before its predecessor's CTA on that SM has retired, so there is no prologue to overlap.  The
// attribute is therefore OFF by default (MRA_PDL=1 switches it on; without it the device instructions are no-ops).
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
inline bool pdl_enabled() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("MRA_PDL"); on = (e && atoi(e) != 0) ? 1 : 0; }
  return on != 0;
}
// kernel<<<grid, block, smem, st>>>(args...) with the programmatic-stream-serialization attribute (+ an optional
// cluster dimension)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, int cluster_x,
                              Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (cluster_x > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = (unsigned)cluster_x; attr[na].val.clusterDim.y = 1; attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl_enabled()) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr; cfg.numAttrs = (unsigned)na;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

inline int num_sms() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

// largest dynamic shared memory a block may opt into (cudaFuncAttributeMaxDynamicSharedMemorySize) on this device
inline size_t max_optin_smem() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&n, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess || n <= 0)
      n = 48 * 1024;
  }
  return (size_t)n;
}

// ---- scalar / vector element access with fp32 math ----
template <typename T> __device__ __forceinline__ float to_f(T v);
template <> __device__ __forceinline__ float to_f<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f<bf16>(bf16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f(float v);
template <> __device__ __forceinline__ float from_f<float>(float v) { return v; }
template <> __device__ __forceinline__ bf16 from_f<bf16>(float v) { return __float2bfloat16_rn(v); }

// 8 consecutive elements <-> float[8] (pointer must be 8-element aligned: 16 B bf16 / 32 B fp32)
template <typename T> struct Vec8;
template <> struct Vec8<float> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[8]) {
    float4 a = __ldg(reinterpret_cast<const float4*>(p));
    float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[8]) {
    reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
  }
};
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
template <> struct Vec8<bf16> {
  static __device__ __forceinline__ void load(const bf16* p, float (&v)[8]) {
    uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      v[2 * i] = __uint_as_float(w[i] << 16);
      v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
  }
  static __device__ __forceinline__ void store(bf16* p, const float (&v)[8]) {
    uint4 r;
    r.x = pack_bf16x2(v[0], v[1]); r.y = pack_bf16x2(v[2], v[3]);
    r.z = pack_bf16x2(v[4], v[5]); r.w = pack_bf16x2(v[6], v[7]);
    *reinterpret_cast<uint4*>(p) = r;
  }
};

__device__ __forceinline__ float apply_act(float v, int act, float slope) {
  switch (act) {
    case MRA_ACT_RELU: return v > 0.f ? v : 0.f;
    case MRA_ACT_LRELU: return v > 0.f ? v : v * slope;
    case MRA_ACT_TANH: return tanhf(v);
    case MRA_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
    default: return v;
  }
}
// derivative expressed through the OUTPUT y of the activation
__device__ __forceinline__ float act_grad_from_output(float y, int act, float slope) {
  switch (act) {
    case MRA_ACT_RELU: return y > 0.f ? 1.f : 0.f;
    case MRA_ACT_LRELU: return y > 0.f ? 1.f : slope;
    case MRA_ACT_TANH: return 1.f - y * y;
    case MRA_ACT_SIGMOID: return y * (1.f - y);
    default: return 1.f;
  }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace mra
