// Column sum of fp32 partials: dst[j] = sum_s src[s][j].
//
// The weight gradients of the block's Linear layers (reference swin_block.py:141-143, window_attention.py:28-32; torch
// autograd there) are computed here as a token-split batched GEMM: dW_s = dy_s^T x_s for ~72 slices s of the token axis
// (fp32 partials [S][Cout*Cin], 0.6-8 MB), which streams dy and x at 4-4.8 TB/s where one split-K GEMM reached 1.7-3.3.
// This kernel is the final sum over the slices.  torch's generic reduce kernel needs 7-10 us for it; all loads of a
// thread are independent here (S/8 rows each), so the kernel is one load round trip long.
#include "common.cuh"

namespace pwa {

namespace {

constexpr int kRowGroups = 8;

__global__ void __launch_bounds__(32 * kRowGroups) colsum_f32_kernel(const float* __restrict__ src, float* __restrict__ dst, int S, long n) {
  __shared__ float red[kRowGroups][33];
  const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
  const long c = (long)blockIdx.x * 32 + lane;
  float a = 0.f;
  if (c < n) {
#pragma unroll 4
    for (int s = g; s < S; s += kRowGroups) a += __ldg(src + (size_t)s * n + c);
  }
  red[g][lane] = a;
  __syncthreads();
  if (g == 0 && c < n) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < kRowGroups; ++k) t += red[k][lane];
    dst[c] = t;
  }
}

// Column sums of a token matrix: dst[c] = sum_r x[r][c], x [rows][C] bf16, fp16 or fp32, dst fp32.  This is the bias gradient of
// the q|k|v projection (reference window_attention.py:28-30: three nn.Linear with bias; torch autograd sums dy over the
// tokens there): dy = the packed dq|dk|dv rows the attention backward kernel wrote, 127 MB at the first stage.  torch's
// generic reduction needed 36-62 us per call for it (0.5-2.3 TB/s).  blockDim is a multiple of the 16-byte vectors per
// row, so a thread meets the same columns in every iteration: four independent vector loads in flight per thread,
// register accumulators, a shared-memory transposition and one global atomic per (CTA, column) at the end.
// X = Det<T>: the CTA's column sums go with plain stores to its own slot dst[blockIdx.x][C] instead, summed over the slots in
// a fixed order by pwa_colsum_rows_det (the in-CTA order is fixed either way).
template <typename X>
__global__ void __launch_bounds__(512) colsum_rows_kernel(const X* __restrict__ xin, float* __restrict__ dst, long nvec, int C) {
  using T = typename Elem<X>::type;
  const T* __restrict__ x = reinterpret_cast<const T*>(xin);
  constexpr int E = 16 / (int)sizeof(T);
  extern __shared__ float part_s[];                       // [blockDim][E] partial sums
  float acc[E];
#pragma unroll
  for (int e = 0; e < E; ++e) acc[e] = 0.f;
  const uint4* __restrict__ xv = reinterpret_cast<const uint4*>(x);
  const long stride = (long)gridDim.x * blockDim.x;
  long v = (long)blockIdx.x * blockDim.x + threadIdx.x;
  auto add = [&](const uint4& q) {
    T t[E];
    *reinterpret_cast<uint4*>(t) = q;
#pragma unroll
    for (int e = 0; e < E; ++e) acc[e] += to_f32(t[e]);
  };
  for (; v + 3 * stride < nvec; v += 4 * stride) {
    const uint4 q0 = __ldg(xv + v), q1 = __ldg(xv + v + stride), q2 = __ldg(xv + v + 2 * stride), q3 = __ldg(xv + v + 3 * stride);
    add(q0); add(q1); add(q2); add(q3);
  }
  for (; v < nvec; v += stride) add(__ldg(xv + v));
  // thread t holds columns (t % vpr) * E .. + E - 1: column c is summed over the blockDim / vpr threads that share it
  // (plain shared-memory reads: fp32 shared atomics are compare-and-swap loops and took longer than the main loop)
#pragma unroll
  for (int e = 0; e < E; ++e) part_s[threadIdx.x * E + e] = acc[e];
  __syncthreads();
  const int vpr = C / E, reps = blockDim.x / vpr;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int cg = c / E, e = c - cg * E;
    float t = 0.f;
    for (int r = 0; r < reps; ++r) t += part_s[(r * vpr + cg) * E + e];
    if constexpr (Elem<X>::det) dst[(size_t)blockIdx.x * C + c] = t;
    else atomicAdd(&dst[c], t);
  }
}

}  // namespace

}  // namespace pwa

using namespace pwa;

extern "C" int pwa_colsum_f32(const float* src, float* dst, int S, int64_t n, void* stream) {
  PWA_CHECK_ARG(src != nullptr && dst != nullptr, "pwa_colsum_f32: null pointer");
  PWA_CHECK_ARG(S >= 1 && n >= 1, "pwa_colsum_f32: S=%d n=%lld", S, (long long)n);
  const long blocks = (n + 31) / 32;
  colsum_f32_kernel<<<(unsigned)blocks, 32 * kRowGroups, 0, (cudaStream_t)stream>>>(src, dst, S, (long)n);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

struct ColsumRowsGrid {
  int threads;
  long nvec, blocks;
};

static ColsumRowsGrid colsum_rows_grid(int64_t rows, int C, int dtype) {
  const int E = dtype == PWA_F32 ? 4 : 8;
  const int vpr = C / E;
  ColsumRowsGrid g;
  g.threads = 512 / vpr * vpr;                          // a multiple of the vectors per row: fixed columns per thread
  g.nvec = (long)rows * vpr;
  g.blocks = (g.nvec + (long)g.threads * 4 - 1) / ((long)g.threads * 4);
  if (g.blocks > 148 * 2) g.blocks = 148 * 2;
  if (g.blocks < 1) g.blocks = 1;
  return g;
}

static int colsum_rows_check(const void* x, const float* dst, int64_t rows, int C, int dtype, const char* who) {
  PWA_CHECK_ARG(x != nullptr && dst != nullptr, "%s: null pointer", who);
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "%s: bad dtype %d", who, dtype);
  const int E = dtype == PWA_F32 ? 4 : 8;
  PWA_CHECK_ARG(rows >= 0 && C >= E && C % E == 0 && C / E <= 512, "%s: rows=%lld C=%d (need C %% %d == 0, C <= %d)", who,
                (long long)rows, C, E, 512 * E);
  PWA_CHECK_ARG(((uintptr_t)x & 15) == 0, "%s: x must be 16-byte aligned", who);
  return PWA_OK;
}

template <bool DET>
static int colsum_rows_launch(const void* x, float* dst, int64_t rows, int C, int dtype, cudaStream_t st) {
  const ColsumRowsGrid g = colsum_rows_grid(rows, C, dtype);
  const size_t smem = (size_t)g.threads * 16;
  const unsigned nb = (unsigned)g.blocks;
  using B = __nv_bfloat16;
  using H = __half;
  if (dtype == PWA_BF16) {
    if (DET) colsum_rows_kernel<Det<B>><<<nb, g.threads, smem * 2, st>>>((const Det<B>*)x, dst, g.nvec, C);
    else colsum_rows_kernel<B><<<nb, g.threads, smem * 2, st>>>((const B*)x, dst, g.nvec, C);
  } else if (dtype == PWA_F16) {
    if (DET) colsum_rows_kernel<Det<H>><<<nb, g.threads, smem * 2, st>>>((const Det<H>*)x, dst, g.nvec, C);
    else colsum_rows_kernel<H><<<nb, g.threads, smem * 2, st>>>((const H*)x, dst, g.nvec, C);
  } else {
    if (DET) colsum_rows_kernel<Det<float>><<<nb, g.threads, smem, st>>>((const Det<float>*)x, dst, g.nvec, C);
    else colsum_rows_kernel<float><<<nb, g.threads, smem, st>>>((const float*)x, dst, g.nvec, C);
  }
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

extern "C" int pwa_colsum_rows(const void* x, float* dst, int64_t rows, int C, int dtype, void* stream) {
  int rc = colsum_rows_check(x, dst, rows, C, dtype, "pwa_colsum_rows");
  if (rc != PWA_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  PWA_CUDA_OK(cudaMemsetAsync(dst, 0, (size_t)C * 4, st));
  if (rows == 0) return PWA_OK;
  return colsum_rows_launch<false>(x, dst, rows, C, dtype, st);
}

extern "C" int64_t pwa_colsum_rows_det_workspace_size(int64_t rows, int C, int dtype) {
  const int E = dtype == PWA_F32 ? 4 : 8;
  if (rows < 0 || C < E || C % E != 0 || C / E > 512) return PWA_ERR_ARG;
  return rows == 0 ? 0 : colsum_rows_grid(rows, C, dtype).blocks * C * 4;
}

extern "C" int pwa_colsum_rows_det(const void* x, float* dst, int64_t rows, int C, int dtype, void* workspace,
                                   int64_t workspace_bytes, void* stream) {
  int rc = colsum_rows_check(x, dst, rows, C, dtype, "pwa_colsum_rows_det");
  if (rc != PWA_OK) return rc;
  const int64_t need = pwa_colsum_rows_det_workspace_size(rows, C, dtype);
  PWA_CHECK_ARG(workspace_bytes >= need && (need == 0 || workspace != nullptr),
                "pwa_colsum_rows_det: workspace of %lld bytes, %lld needed", (long long)workspace_bytes, (long long)need);
  cudaStream_t st = (cudaStream_t)stream;
  if (rows == 0) {
    PWA_CUDA_OK(cudaMemsetAsync(dst, 0, (size_t)C * 4, st));
    return PWA_OK;
  }
  float* slots = (float*)workspace;
  rc = colsum_rows_launch<true>(x, slots, rows, C, dtype, st);
  if (rc != PWA_OK) return rc;
  return pwa_colsum_f32(slots, dst, (int)colsum_rows_grid(rows, C, dtype).blocks, C, stream);
}
