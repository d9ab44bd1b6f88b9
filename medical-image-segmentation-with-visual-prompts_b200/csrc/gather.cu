// Row gather between channels-last token arrangements (HBM-bound, 16-byte vectors, no transposition).
//
// Inside a ConsecutiveSwinBlocks pair the feature map never has to leave the channels-last token layout:
//   block0 output (window order g0)  ->  block1 input (shifted window order g1)
//       = window_reverse + roll back + crop + pad + roll + window_partition      (swin_block.py:228-253, 150-214)
//   block1 output (window order g1)  ->  PatchMerging rows [T'][8][C]
//       = window_reverse + roll back + crop + pad + 8 strided slices + cat        (swin_block.py:228-253, down.py:21-47)
//   channels-last feature map (the strides PatchMerging's final rearrange leaves, down.py:48-53) -> window tokens
// are all the same operation: dst row j of a sample = src row map[j] of that sample (or zeros for map[j] < 0),
// rows being C contiguous elements.  The maps are composed on the host from pwa_index_map() and cached per
// geometry; each is injective, so the adjoint is the same kernel with the inverse map.  An optional second
// source fuses the block's last residual add (swin_block.py:227): dst = a[map] + b[map], summed in fp32.
#include "common.cuh"

namespace pwa {

namespace {

template <int VB> struct VecT;
template <> struct VecT<16> { using type = uint4; };
template <> struct VecT<8> { using type = uint2; };
template <> struct VecT<4> { using type = uint32_t; };
template <> struct VecT<2> { using type = uint16_t; };

__device__ __forceinline__ uint32_t add_bf16x2(uint32_t a, uint32_t b) {
  const float2 fa = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&a));
  const float2 fb = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&b));
  const __nv_bfloat162 r = __floats2bfloat162_rn(fa.x + fb.x, fa.y + fb.y);
  return *reinterpret_cast<const uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t add_f16x2(uint32_t a, uint32_t b) {
  const float2 fa = __half22float2(*reinterpret_cast<const __half2*>(&a));
  const float2 fb = __half22float2(*reinterpret_cast<const __half2*>(&b));
  const __half2 r = __floats2half2_rn(fa.x + fb.x, fa.y + fb.y);
  return *reinterpret_cast<const uint32_t*>(&r);
}
__device__ __forceinline__ uint32_t add_f32(uint32_t a, uint32_t b) { return __float_as_uint(__uint_as_float(a) + __uint_as_float(b)); }

// EB = element bytes; H: the 16-bit elements are fp16 (else bf16)
template <int EB, bool H> __device__ __forceinline__ uint32_t add_w(uint32_t a, uint32_t b) {
  return EB == 4 ? add_f32(a, b) : (H ? add_f16x2(a, b) : add_bf16x2(a, b));
}

template <int EB, bool H> __device__ __forceinline__ uint4 vadd(uint4 a, uint4 b) {
  return make_uint4(add_w<EB, H>(a.x, b.x), add_w<EB, H>(a.y, b.y), add_w<EB, H>(a.z, b.z), add_w<EB, H>(a.w, b.w));
}
template <int EB, bool H> __device__ __forceinline__ uint2 vadd(uint2 a, uint2 b) { return make_uint2(add_w<EB, H>(a.x, b.x), add_w<EB, H>(a.y, b.y)); }
template <int EB, bool H> __device__ __forceinline__ uint32_t vadd(uint32_t a, uint32_t b) { return add_w<EB, H>(a, b); }
template <int EB, bool H> __device__ __forceinline__ uint16_t vadd(uint16_t a, uint16_t b) {   // one 16-bit element
  return (uint16_t)(add_w<EB, H>((uint32_t)a, (uint32_t)b) & 0xffffu);
}

__device__ __forceinline__ void vzero(uint4& v) { v = make_uint4(0, 0, 0, 0); }
__device__ __forceinline__ void vzero(uint2& v) { v = make_uint2(0, 0); }
__device__ __forceinline__ void vzero(uint32_t& v) { v = 0; }
__device__ __forceinline__ void vzero(uint16_t& v) { v = 0; }

constexpr int kUnroll = 4;

// exact n / d for every 32-bit n (round-up magic number, Granlund-Montgomery); d >= 1
struct Div32 {
  uint32_t d, m, s;
  Div32() : d(1), m(0), s(0) {}
  explicit Div32(uint32_t d_) : d(d_) {
    s = 0;
    while ((1ull << s) < d_) ++s;
    m = (uint32_t)((((1ull << s) - d_) << 32) / d_ + 1);
  }
  __device__ __forceinline__ void divmod(uint32_t n, uint32_t& q, uint32_t& r) const {
    const uint32_t t = __umulhi(n, m);
    q = d == 1 ? n : (t + ((n - t) >> 1)) >> (s - 1);
    r = n - q * d;
  }
};

// One thread = kUnroll vectors, strided by the grid so that a warp's accesses stay contiguous.
// vpr = vectors per row; chunk q -> (row, c) with row in [0, B * rows_dst).
template <int VB, int EB, bool ADD, bool H>
__global__ void __launch_bounds__(256) gather_rows_kernel(const typename VecT<VB>::type* __restrict__ a,
                                                          const typename VecT<VB>::type* __restrict__ b,
                                                          typename VecT<VB>::type* __restrict__ dst,
                                                          const int32_t* __restrict__ map, uint32_t total, Div32 vpr,
                                                          size_t src_sample, size_t dst_sample) {
  using V = typename VecT<VB>::type;
  // blockIdx.y = sample; `total` = vectors per sample on the dst side
  a += (size_t)blockIdx.y * src_sample;
  if (ADD) b += (size_t)blockIdx.y * src_sample;
  dst += (size_t)blockIdx.y * dst_sample;
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t q0 = blockIdx.x * blockDim.x + threadIdx.x; q0 < total; q0 += stride * kUnroll) {
    V va[kUnroll], vb[kUnroll];
    bool live[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      const uint32_t q = q0 + u * stride;
      live[u] = q < total && q >= q0;
      vzero(va[u]);
      vzero(vb[u]);
      if (live[u]) {
        uint32_t j, c;
        vpr.divmod(q, j, c);
        const int s = __ldg(map + j);
        if (s >= 0) {
          const size_t off = (size_t)(uint32_t)s * vpr.d + c;
          va[u] = __ldg(a + off);
          if (ADD) vb[u] = __ldg(b + off);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u)
      if (live[u]) dst[q0 + u * stride] = ADD ? vadd<EB, H>(va[u], vb[u]) : va[u];
  }
}

template <int VB, int EB, bool H = false>
int launch_gather(const void* a, const void* b, void* dst, const int32_t* map, int B, long long rows_src, long long rows_dst,
                  int row_bytes, cudaStream_t st) {
  using V = typename VecT<VB>::type;
  const uint32_t vpr = row_bytes / VB;
  const long long total = rows_dst * vpr;         // vectors per sample
  if (total == 0) return PWA_OK;
  long long blocks = (total + 256LL * kUnroll - 1) / (256LL * kUnroll);
  const long long cap = (148LL * 8 * 4 + B - 1) / B;   // a few waves of full-occupancy CTAs; the grid-stride loop covers the rest
  if (blocks > cap) blocks = cap;
  const Div32 dv(vpr);
  const dim3 grid((unsigned)blocks, (unsigned)B);
  const size_t ss = (size_t)rows_src * vpr, ds = (size_t)rows_dst * vpr;
  if (b)
    gather_rows_kernel<VB, EB, true, H><<<grid, 256, 0, st>>>((const V*)a, (const V*)b, (V*)dst, map, (uint32_t)total, dv, ss, ds);
  else
    gather_rows_kernel<VB, EB, false, false><<<grid, 256, 0, st>>>((const V*)a, nullptr, (V*)dst, map, (uint32_t)total, dv, ss, ds);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

}  // namespace

}  // namespace pwa

extern "C" int pwa_gather_rows(const void* src_a, const void* src_b, void* dst, const int32_t* map, int B, int64_t rows_src,
                               int64_t rows_dst, int C, int dtype, void* stream) {
  using namespace pwa;
  PWA_CHECK_ARG(src_a && dst && map, "pwa_gather_rows: null pointer");
  PWA_CHECK_ARG(B > 0 && C > 0 && rows_src > 0 && rows_dst > 0, "pwa_gather_rows: bad shape B=%d C=%d rows %lld -> %lld", B, C,
                (long long)rows_src, (long long)rows_dst);
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "pwa_gather_rows: bad dtype %d", dtype);
  const int eb = dtype == PWA_F32 ? 4 : 2;
  const int row_bytes = C * eb;
  const uintptr_t al = (uintptr_t)src_a | (uintptr_t)src_b | (uintptr_t)dst;
  int vb = eb;
  for (int cand = 16; cand > eb; cand >>= 1)
    if (row_bytes % cand == 0 && (al & (uintptr_t)(cand - 1)) == 0) { vb = cand; break; }
  const long long total = (long long)rows_dst * (row_bytes / vb);       // per sample; samples ride in blockIdx.y
  PWA_CHECK_ARG(total < (1LL << 31) && rows_src < (1LL << 31) && B < 65536,
                "pwa_gather_rows: sample too large for 32-bit vector indexing (%lld vectors)", total);
  cudaStream_t st = (cudaStream_t)stream;
  if (eb == 4) {
    switch (vb) {
      case 16: return launch_gather<16, 4>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
      case 8: return launch_gather<8, 4>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
      default: return launch_gather<4, 4>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
    }
  }
  if (dtype == PWA_F16 && src_b) {                                      // only the fused add depends on the 16-bit format
    switch (vb) {
      case 16: return launch_gather<16, 2, true>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
      case 8: return launch_gather<8, 2, true>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
      case 4: return launch_gather<4, 2, true>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
      default: return launch_gather<2, 2, true>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
    }
  }
  switch (vb) {
    case 16: return launch_gather<16, 2>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
    case 8: return launch_gather<8, 2>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
    case 4: return launch_gather<4, 2>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
    default: return launch_gather<2, 2>(src_a, src_b, dst, map, B, rows_src, rows_dst, row_bytes, st);
  }
}
