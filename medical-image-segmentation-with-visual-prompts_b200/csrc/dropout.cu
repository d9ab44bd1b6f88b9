// Seeded elementwise dropout: y = x * keep(i) / keep_rate with keep(i) a counter-based hash of two DEVICE seed words
// and the element index.  Replaces nn.Dropout(proj_drop) after the attention output projection
// (reference window_attention.py:33,60).  torch's dropout draws from the CUDA generator: an activation-checkpointed block
// (swin_block.py:257-260, the reference's example config) then has to save and restore the generator state to recompute
// the same mask, which a CUDA-graph capture cannot do.  Here the mask is a pure function of (seed words, index): the
// seed words are drawn OUTSIDE the checkpointed region by a device RNG op, the recomputation and the backward
// (dx = dy * same mask) see the same mask, nothing is stored, and a captured step gets fresh masks on every replay.
// The rate moves in steps of 1/256 like the attention dropout (csrc/attn.cuh); kept values are scaled by the exact
// inverse of the quantised keep rate.  One 32-bit hash per 4 consecutive elements, one byte each.
#include "common.cuh"

namespace pwa {

namespace {

__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x21f0aaadu; x ^= x >> 15; x *= 0x735a2d97u; x ^= x >> 15;
  return x;
}

// COLSUM: the tensor is [rows][C] and the column sums of y are wanted as well (backward use: y = dx of the Linear output in
// front of the dropout, its column sums = the gradient of that Linear's bias -- torch's generic reduction took 62 us for it
// at the first stage).  blockDim is a multiple of C / 4, so every thread meets the same four columns in every iteration:
// four register accumulators, one shared-memory atomic per thread and one global atomic per column and CTA at the end.
template <typename T, bool COLSUM>
__global__ void __launch_bounds__(256) dropout_kernel(const T* __restrict__ x, T* __restrict__ y, long n, uint32_t thresh,
                                                      float inv_keep, const uint32_t* __restrict__ seed, float* __restrict__ colsum,
                                                      int C) {
  __shared__ float cs_s[COLSUM ? 1024 : 1];
  const uint32_t s0 = seed[0], s1 = seed[1];
  const long quads = (n + 3) / 4;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  if (COLSUM) {
    for (int i = threadIdx.x; i < C; i += blockDim.x) cs_s[i] = 0.f;
    __syncthreads();
  }
  for (long q = (long)blockIdx.x * blockDim.x + threadIdx.x; q < quads; q += (long)gridDim.x * blockDim.x) {
    const uint32_t h = mix32(s0 + (uint32_t)q * 0x9E3779B1u + (uint32_t)(q >> 32) * 0x85EBCA77u) ^ s1;
    const uint32_t bits = mix32(h);
    const long i = q * 4;
    if (i + 3 < n) {
      T v[4];
      if constexpr (sizeof(T) == 2) *reinterpret_cast<uint2*>(v) = *reinterpret_cast<const uint2*>(x + i);
      else *reinterpret_cast<float4*>(v) = *reinterpret_cast<const float4*>(x + i);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float f = ((bits >> (8 * e)) & 0xffu) >= thresh ? to_f32(v[e]) * inv_keep : 0.f;
        v[e] = from_f32<T>(f);
        if (COLSUM) acc[e] += f;
      }
      if constexpr (sizeof(T) == 2) *reinterpret_cast<uint2*>(y + i) = *reinterpret_cast<const uint2*>(v);
      else *reinterpret_cast<float4*>(y + i) = *reinterpret_cast<const float4*>(v);
    } else {
      for (int e = 0; e < 4 && i + e < n; ++e)
        y[i + e] = from_f32<T>(((bits >> (8 * e)) & 0xffu) >= thresh ? to_f32(x[i + e]) * inv_keep : 0.f);
    }
  }
  if (COLSUM) {
    const int c0 = (int)(threadIdx.x % (unsigned)(C / 4)) * 4;     // (n is a multiple of C here: no ragged tail)
#pragma unroll
    for (int e = 0; e < 4; ++e) atomicAdd(&cs_s[c0 + e], acc[e]);
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(&colsum[i], cs_s[i]);
  }
}

}  // namespace

}  // namespace pwa

using namespace pwa;

static int dropout_launch(const void* x, void* y, int64_t n, float p_drop, const void* seed_dev, float* colsum, int C, int dtype,
                          void* stream);

extern "C" int pwa_dropout(const void* x, void* y, int64_t n, float p_drop, const void* seed_dev, int dtype, void* stream) {
  return dropout_launch(x, y, n, p_drop, seed_dev, nullptr, 0, dtype, stream);
}

extern "C" int pwa_dropout_colsum(const void* x, void* y, int64_t rows, int C, float p_drop, const void* seed_dev, float* colsum,
                                  int dtype, void* stream) {
  PWA_CHECK_ARG(colsum != nullptr && C > 0 && C % 4 == 0 && C <= 1024 && rows >= 0, "pwa_dropout_colsum: need C %% 4 == 0, C <= 1024 (C=%d)", C);
  PWA_CUDA_OK(cudaMemsetAsync(colsum, 0, (size_t)C * 4, (cudaStream_t)stream));
  return dropout_launch(x, y, rows * C, p_drop, seed_dev, colsum, C, dtype, stream);
}

static int dropout_launch(const void* x, void* y, int64_t n, float p_drop, const void* seed_dev, float* colsum, int C, int dtype,
                          void* stream) {
  PWA_CHECK_ARG(x && y && seed_dev, "pwa_dropout: null pointer");
  PWA_CHECK_ARG(n >= 0 && p_drop >= 0.f && p_drop < 1.f, "pwa_dropout: n=%lld p=%g", (long long)n, (double)p_drop);
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "pwa_dropout: bad dtype %d", dtype);
  PWA_CHECK_ARG(((uintptr_t)x & 15) == 0 && ((uintptr_t)y & 15) == 0, "pwa_dropout: buffers must be 16-byte aligned");
  if (n == 0) return PWA_OK;
  int t = (int)(p_drop * 256.f + 0.5f);
  if (t > 255) t = 255;
  if (p_drop > 0.f && t == 0) t = 1;
  const float inv_keep = 256.f / (float)(256 - t);
  const long quads = (n + 3) / 4;
  const int threads = colsum ? 256 / (C / 4) * (C / 4) : 256;      // a multiple of the quads per row (see COLSUM)
  long blocks = (quads + threads - 1) / threads;
  if (blocks > 148 * 8) blocks = 148 * 8;
  cudaStream_t st = (cudaStream_t)stream;
  const uint32_t* sd = (const uint32_t*)seed_dev;
  if (dtype == PWA_F32) {
    if (colsum) dropout_kernel<float, true><<<(unsigned)blocks, threads, 0, st>>>((const float*)x, (float*)y, (long)n, (uint32_t)t, inv_keep, sd, colsum, C);
    else dropout_kernel<float, false><<<(unsigned)blocks, threads, 0, st>>>((const float*)x, (float*)y, (long)n, (uint32_t)t, inv_keep, sd, nullptr, 0);
  } else if (dtype == PWA_BF16) {
    using B = __nv_bfloat16;
    if (colsum) dropout_kernel<B, true><<<(unsigned)blocks, threads, 0, st>>>((const B*)x, (B*)y, (long)n, (uint32_t)t, inv_keep, sd, colsum, C);
    else dropout_kernel<B, false><<<(unsigned)blocks, threads, 0, st>>>((const B*)x, (B*)y, (long)n, (uint32_t)t, inv_keep, sd, nullptr, 0);
  } else {
    using H = __half;
    if (colsum) dropout_kernel<H, true><<<(unsigned)blocks, threads, 0, st>>>((const H*)x, (H*)y, (long)n, (uint32_t)t, inv_keep, sd, colsum, C);
    else dropout_kernel<H, false><<<(unsigned)blocks, threads, 0, st>>>((const H*)x, (H*)y, (long)n, (uint32_t)t, inv_keep, sd, nullptr, 0);
  }
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}
