// Shared helpers for the pwa kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/pwa.h"

namespace pwa {

void set_error(const char* fmt, ...);

#define PWA_CHECK_ARG(cond, ...)            \
  do {                                      \
    if (!(cond)) {                          \
      ::pwa::set_error(__VA_ARGS__);        \
      return PWA_ERR_ARG;                   \
    }                                       \
  } while (0)

#define PWA_CUDA_OK(expr)                                                        \
  do {                                                                           \
    cudaError_t _e = (expr);                                                     \
    if (_e != cudaSuccess) {                                                     \
      ::pwa::set_error("%s failed: %s", #expr, cudaGetErrorString(_e));          \
      return PWA_ERR_CUDA;                                                       \
    }                                                                            \
  } while (0)

// exact n / d for n < 2^16, d < 2^16 with m = 2^32 / d + 1
struct FastDiv {
  uint32_t d, m;
  __host__ __device__ FastDiv() : d(1), m(0) {}
  __host__ explicit FastDiv(uint32_t d_) : d(d_), m(d_ == 1 ? 0u : (uint32_t)((1ull << 32) / d_ + 1)) {}
  __device__ __forceinline__ uint32_t div(uint32_t n) const { return d == 1 ? n : __umulhi(n, m); }
  __device__ __forceinline__ void divmod(uint32_t n, uint32_t& q, uint32_t& r) const {
    q = div(n);
    r = n - q * d;
  }
};

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace pwa
