// Shared host/device helpers for libtm_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>

#include "tm_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libtm_b200 is written for sm_100a only"
#endif

namespace tmk {

extern thread_local char g_err[512];
extern std::atomic<long long> g_launches;

inline int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

inline int check_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail((int)e, "%s: %s", what, cudaGetErrorString(e));
  return 0;
}

#define TM_TRY(expr)            \
  do {                          \
    int _rc = (expr);           \
    if (_rc != 0) return _rc;   \
  } while (0)

#define TM_CUDA(expr)                                                                   \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) return tmk::fail((int)_e, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

#define TM_REQUIRE(cond, ...)                                   \
  do {                                                          \
    if (!(cond)) return tmk::fail(TM_EINVAL, __VA_ARGS__);       \
  } while (0)

inline int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// carve typed arrays out of a caller-provided workspace
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* p) : base((char*)p) {}
  template <typename T>
  T* take(size_t count) {
    off = align_up(off, 256);
    T* r = (T*)(base + off);
    off += count * sizeof(T);
    return r;
  }
};

#ifdef __CUDACC__
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ float4 f4add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float4 f4scale(float4 a, float s) { return make_float4(a.x * s, a.y * s, a.z * s, a.w * s); }
__device__ __forceinline__ float4 f4relu(float4 a) { return make_float4(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f), fmaxf(a.z, 0.f), fmaxf(a.w, 0.f)); }
// streaming 128-bit load that does not allocate in L1 (rows read once per kernel)
__device__ __forceinline__ float4 ld4_stream(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
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
#endif

}  // namespace tmk
