// Shared host/device helpers for the CFL B200 library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <math.h>
#include <type_traits>
#include "cfl_b200.h"

namespace cfl {

// ---- host-side error plumbing -----------------------------------------------------------
void set_error(const char* fmt, ...);          // api.cu
int  device_check();                           // api.cu: CFL_OK iff current device is sm_100
int  sm_count();                               // api.cu (cached per device)
void timer_record(int which, cudaStream_t st);  // api.cu: 0 = start, 1 = stop (no-op if unset)

#define CFL_REQUIRE(cond, status, ...)                                                    \
  do {                                                                                    \
    if (!(cond)) { ::cfl::set_error(__VA_ARGS__); return (status); }                      \
  } while (0)

#define CFL_CUDA(expr)                                                                    \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::cfl::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__,  \
                       __LINE__);                                                         \
      return CFL_ERR_CUDA;                                                                \
    }                                                                                     \
  } while (0)

#define CFL_LAUNCH_CHECK() CFL_CUDA(cudaGetLastError())

// Raises a kernel's dynamic shared-memory limit.  cudaFuncSetAttribute costs tens of microseconds of host time, and a
// ranking step would issue ten of them: remember the limit set per call site (= per kernel instantiation) and device,
// call the runtime only when the request grows.  (A race between host threads only repeats the call.)
#define CFL_SMEM_LIMIT(kern, bytes)                                                                     \
  do {                                                                                                  \
    static int _cfl_lim[16];                                                                            \
    int _cfl_dev = 0;                                                                                   \
    CFL_CUDA(cudaGetDevice(&_cfl_dev));                                                                 \
    const int _cfl_want = (int)(bytes);                                                                 \
    if (_cfl_want >= _cfl_lim[_cfl_dev & 15]) {                                                         \
      CFL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, _cfl_want));     \
      _cfl_lim[_cfl_dev & 15] = _cfl_want + 1;                                                          \
    }                                                                                                   \
  } while (0)

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// The one dispatch of a runtime K onto the kernels' compile-time K: f(std::integral_constant<int, K>{}) for K in
// [1, CFL_MAX_K], CFL_ERR_UNSUPPORTED otherwise.  f returns a CFL status.
template <class F>
int with_k(int K, F&& f) {
  static_assert(CFL_MAX_K == 8, "with_k lists K = 1..8");
  switch (K) {
    case 1: return f(std::integral_constant<int, 1>{});
    case 2: return f(std::integral_constant<int, 2>{});
    case 3: return f(std::integral_constant<int, 3>{});
    case 4: return f(std::integral_constant<int, 4>{});
    case 5: return f(std::integral_constant<int, 5>{});
    case 6: return f(std::integral_constant<int, 6>{});
    case 7: return f(std::integral_constant<int, 7>{});
    case 8: return f(std::integral_constant<int, 8>{});
  }
  set_error("K=%d outside [1,%d]", K, CFL_MAX_K);
  return CFL_ERR_UNSUPPORTED;
}

// Bump allocator over the caller's workspace.
struct Workspace {
  char* base; size_t size; size_t off;
  Workspace(void* p, size_t n) : base((char*)p), size(n), off(0) {}
  template <class T> T* take(size_t count) {
    off = align_up(off, 256);
    T* r = (T*)(base + off);
    off += count * sizeof(T);
    return r;
  }
  bool ok() const { return off <= size && (base != nullptr || off == 0); }
};

// ---- device helpers ---------------------------------------------------------------------
#ifdef __CUDACC__
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
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Monotone map float -> uint32 (total order matching <, with -0.0 canonicalised to +0.0).
__device__ __forceinline__ uint32_t f2ord(float f) {
  uint32_t u = __float_as_uint(f + 0.0f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t u) {
  u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  return __uint_as_float(u);
}
// (value, index) packed so that u64 '<' is the lexicographic (value, index) order.
__device__ __forceinline__ unsigned long long pack_key(float v, uint32_t idx) {
  return ((unsigned long long)f2ord(v) << 32) | idx;
}
#define CFL_KEY_INF 0xffffffffffffffffull

__device__ __forceinline__ float apply_act(float y, int act) {
  switch (act) {
    case CFL_ACT_TANH:    return tanhf(y);
    case CFL_ACT_SIGMOID: return 1.0f / (1.0f + expf(-y));
    case CFL_ACT_RELU:    return fmaxf(y, 0.0f);
    case CFL_ACT_LRELU:   return fmaxf(y, 0.0f) - 0.2f * fmaxf(-y, 0.0f);
    default:              return y;
  }
}
// d act / d pre, written with the post-activation value y.
__device__ __forceinline__ float act_grad_from_y(float y, int act) {
  switch (act) {
    case CFL_ACT_TANH:    return 1.0f - y * y;
    case CFL_ACT_SIGMOID: return y * (1.0f - y);
    case CFL_ACT_RELU:    return y > 0.0f ? 1.0f : 0.0f;
    case CFL_ACT_LRELU:   return y > 0.0f ? 1.0f : 0.2f;
    default:              return 1.0f;
  }
}
// TF's stable softplus: max(x,0) + log1p(exp(-|x|)).
__device__ __forceinline__ float softplusf(float x) {
  return fmaxf(x, 0.0f) + log1pf(expf(-fabsf(x)));
}
__device__ __forceinline__ float sigmoidf(float x) { return 1.0f / (1.0f + expf(-x)); }
#endif  // __CUDACC__

}  // namespace cfl
