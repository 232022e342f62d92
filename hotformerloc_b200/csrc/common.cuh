// Shared helpers for libhfl_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

#include "../../include/hfl.h"

namespace hfl {

extern thread_local char g_err[512];
extern std::atomic<long long> g_launches;

inline int fail(int code, const char* fmt, const char* a = "", long long b = 0) {
  snprintf(g_err, sizeof(g_err), fmt, a, b);
  return code;
}

#define HFL_CHECK_ARG(cond, msg)                                              \
  do {                                                                        \
    if (!(cond)) return ::hfl::fail(HFL_ERR_INVALID, "%s (%lld)", msg, (long long)__LINE__); \
  } while (0)

#define HFL_CUDA(expr)                                                        \
  do {                                                                        \
    cudaError_t e__ = (expr);                                                 \
    if (e__ != cudaSuccess)                                                   \
      return ::hfl::fail(HFL_ERR_CUDA, "CUDA error: %s (line %lld)",          \
                         cudaGetErrorString(e__), (long long)__LINE__);       \
  } while (0)

// kernel<<<...>>> launch + bookkeeping + launch-error check (no sync).  cudaGetLastError clears the
// error it reports, so a rejected launch (e.g. a bad configuration) fails this call only and not every later
// call of the thread; a sticky device fault stays visible to everyone whatever we do here.
#define HFL_LAUNCH(...)                                                       \
  do {                                                                        \
    __VA_ARGS__;                                                              \
    ::hfl::g_launches.fetch_add(1, std::memory_order_relaxed);                \
    HFL_CUDA(cudaGetLastError());                                             \
  } while (0)

// cudaFuncAttributeMaxDynamicSharedMemorySize is per device: remember the largest size requested per
// (call site, device) -- no process-wide flag that a second GPU or a racing first call could trip over
// (worst case two threads both set the attribute, which is idempotent).  __VA_ARGS__ = the kernel.
#define HFL_ENSURE_SMEM(bytes, ...)                                                               \
  do {                                                                                            \
    static std::atomic<int> set__[64];                                                            \
    int dev__ = 0;                                                                                \
    if (cudaGetDevice(&dev__) != cudaSuccess || dev__ < 0 || dev__ >= 64) dev__ = 0;              \
    if (set__[dev__].load(std::memory_order_relaxed) < (int)(bytes)) {                            \
      HFL_CUDA(cudaFuncSetAttribute(__VA_ARGS__, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
      set__[dev__].store((int)(bytes), std::memory_order_relaxed);                                \
    }                                                                                             \
  } while (0)

constexpr int kSMs = 148;      // B200; grid caps of the small row kernels (any multiple works)

// SM count of the current device (persistent tcgen05 kernels launch one CTA per SM); cached per device.
inline int sm_count() {
  static std::atomic<int> cached[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return kSMs;
  int v = cached[dev].load(std::memory_order_relaxed);
  if (v <= 0) {
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = kSMs;
    cached[dev].store(v, std::memory_order_relaxed);
  }
  return v;
}

__host__ __device__ inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

inline int grid_for(int64_t n, int threads, int max_blocks = kSMs * 32) {
  int64_t g = ceil_div(n, threads);
  if (g < 1) g = 1;
  if (g > max_blocks) g = max_blocks;
  return (int)g;
}

}  // namespace hfl
