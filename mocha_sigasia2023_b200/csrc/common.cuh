// Shared helpers for the mocha_b200 CUDA library (sm_100a only).
#pragma once
#include "../../include/mocha_b200.h"  // MOCHA_OK / MOCHA_ERR_* codes
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>

namespace mocha {

// ---------------------------------------------------------------------------------------------
// Error channel of the C ABI: every entry point returns 0 on success or a negative code and
// leaves a message readable through mocha_last_error(). No exceptions cross the boundary.
// ---------------------------------------------------------------------------------------------
int set_error(int code, const char* fmt, ...);
const char* last_error();

#define MOCHA_CHECK_ARG(cond, ...)                                     \
  do {                                                                 \
    if (!(cond)) return ::mocha::set_error(MOCHA_ERR_ARG, __VA_ARGS__); \
  } while (0)

#define MOCHA_CUDA(call)                                                               \
  do {                                                                                 \
    cudaError_t e__ = (call);                                                          \
    if (e__ != cudaSuccess)                                                            \
      return ::mocha::set_error(MOCHA_ERR_CUDA, "%s failed: %s (%s:%d)", #call, \
                                cudaGetErrorString(e__), __FILE__, __LINE__);          \
  } while (0)

#define MOCHA_LAUNCH_CHECK(name)                                                        \
  do {                                                                                 \
    cudaError_t e__ = cudaGetLastError();                                              \
    if (e__ != cudaSuccess)                                                            \
      return ::mocha::set_error(MOCHA_ERR_CUDA, "launch of %s failed: %s", name, \
                                cudaGetErrorString(e__));                              \
  } while (0)

#define MOCHA_TRY(expr)          \
  do {                           \
    int rc__ = (expr);           \
    if (rc__ != 0) return rc__;  \
  } while (0)

// launch counter (bench.py reports "gpu_launches" from it)
void count_launch(int n = 1);

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL): every kernel of the library is launched with the programmatic-stream-
// serialization attribute, so its CTAs may become resident as soon as the previous kernel's CTAs have called
// pdl_trigger() (or exited) and run their prologue (barrier init, TMEM allocation, descriptor prefetch, weight
// staging) under the previous kernel's tail. Contract, kept by every kernel:
//   * nothing produced by an earlier kernel is read, and no global memory is written, before pdl_wait() returns
//     (griddepcontrol.wait = the previous grid has completed and its memory is visible);
//   * every kernel executes pdl_wait() before it exits, so completion stays transitive along the stream.
// A ~110-launch frame captured in a CUDA graph keeps these edges as programmatic dependencies.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);   // errors surface through MOCHA_LAUNCH_CHECK
}

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Bump allocator over the caller-provided workspace (the library never cudaMallocs on the
// data path; see include/mocha_b200.h "Ownership").
struct Workspace {
  char* base;
  size_t cap;
  size_t off;
  bool overflow;
  Workspace(void* p, size_t n) : base((char*)p), cap(n), off(0), overflow(false) {}
  template <typename T>
  T* take(size_t count) {
    size_t bytes = align_up(count * sizeof(T), 256);
    if (off + bytes > cap) { overflow = true; off += bytes; return nullptr; }
    T* r = (T*)(base + off);
    off += bytes;
    return r;
  }
};

__device__ __forceinline__ float lrelu02(float x) { return x > 0.f ? x : 0.2f * x; }
__device__ __forceinline__ float gelu_erf(float x) {
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
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
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace mocha
