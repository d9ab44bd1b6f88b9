// LayerNorm over the channel axis of window tokens, forward and backward, fused with the residual adds
// that surround it in the block (reference swin_block.py:216 attn_norm, :222 `x + shortcut`, :227 mlp_norm).
// HBM-bound row kernels for small C (48..768): a row is handled by a sub-warp group of G lanes, each lane
// owning 4-element vectors, statistics by shuffle reduction in fp32 (two-pass over registers: exact mean,
// then centred variance -- matches torch's numerics closely).  gamma/beta stay fp32 (no per-call casts).
//   forward : s = x (+ res) ; y = (s - mean) * rstd * gamma + beta ; saves mean, rstd   (also writes s if res)
//   backward: dx = rstd * (g - mean(g) - xhat * mean(g * xhat)) (+ dres), g = dy * gamma ;
//             dgamma += sum_rows dy * xhat ; dbeta += sum_rows dy   (register partials -> smem -> fp32 atomics)
#include "common.cuh"

namespace pwa {

constexpr int kLnThreads = 256;

// 16-byte lane vectors where the row length allows (8 bf16 or fp16 / 4 fp32), else 8-byte (4 bf16 or fp16)
template <typename T, int EPV> struct Vec;      // 16-bit T (bf16, fp16) below; fp32 specialised
template <> struct Vec<float, 4> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[4]) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <typename T> __device__ __forceinline__ void unpack2(uint32_t w, float& a, float& b);
template <> __device__ __forceinline__ void unpack2<__nv_bfloat16>(uint32_t w, float& a, float& b) {
  a = __uint_as_float(w << 16);
  b = __uint_as_float(w & 0xffff0000u);
}
template <> __device__ __forceinline__ void unpack2<__half>(uint32_t w, float& a, float& b) {
  const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w));
  a = f.x;
  b = f.y;
}
template <typename T> __device__ __forceinline__ uint32_t pack2(float a, float b);
template <> __device__ __forceinline__ uint32_t pack2<__nv_bfloat16>(float a, float b) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&v);
}
template <> __device__ __forceinline__ uint32_t pack2<__half>(float a, float b) {
  const __half2 v = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&v);
}
template <typename T> struct Vec<T, 4> {
  static __device__ __forceinline__ void load(const T* p, float (&v)[4]) {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
    unpack2<T>(t.x, v[0], v[1]);
    unpack2<T>(t.y, v[2], v[3]);
  }
  static __device__ __forceinline__ void store(T* p, const float (&v)[4]) {
    *reinterpret_cast<uint2*>(p) = make_uint2(pack2<T>(v[0], v[1]), pack2<T>(v[2], v[3]));
  }
};
template <typename T> struct Vec<T, 8> {
  static __device__ __forceinline__ void load(const T* p, float (&v)[8]) {
    const uint4 t = __ldg(reinterpret_cast<const uint4*>(p));
    unpack2<T>(t.x, v[0], v[1]);
    unpack2<T>(t.y, v[2], v[3]);
    unpack2<T>(t.z, v[4], v[5]);
    unpack2<T>(t.w, v[6], v[7]);
  }
  static __device__ __forceinline__ void store(T* p, const float (&v)[8]) {
    *reinterpret_cast<uint4*>(p) = make_uint4(pack2<T>(v[0], v[1]), pack2<T>(v[2], v[3]), pack2<T>(v[4], v[5]), pack2<T>(v[6], v[7]));
  }
};
template <int EPV> __device__ __forceinline__ void loadf(const float* p, float (&v)[EPV]) {
#pragma unroll
  for (int e = 0; e < EPV; e += 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p + e));
    v[e] = t.x; v[e + 1] = t.y; v[e + 2] = t.z; v[e + 3] = t.w;
  }
}

template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// A row is handled by a group of G lanes, each lane owning NV vectors of EPV elements, with all of its loads issued
// before the first use (these kernels are pure HBM streams of 2-4 passes over [rows, C]).
template <typename T, int G, int NV, int EPV>
__global__ void __launch_bounds__(kLnThreads, (NV * EPV <= 16 ? 4 : (NV * EPV <= 32 ? 2 : 1))) ln_fwd_kernel(const T* __restrict__ x, const T* __restrict__ res,
                                                            const float* __restrict__ gamma, const float* __restrict__ beta,
                                                            T* __restrict__ sum_out, T* __restrict__ y,
                                                            float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                                            long rows, int C, float eps) {
  constexpr int GPB = kLnThreads / G;                  // groups per block
  const int gl = threadIdx.x % G, gr = threadIdx.x / G;
  const int nvec = C / EPV;
  float gm[NV][EPV], bt[NV][EPV];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int vi = gl + k * G;
    if (vi < nvec) {
      loadf<EPV>(gamma + vi * EPV, gm[k]);
      loadf<EPV>(beta + vi * EPV, bt[k]);
    }
  }
  const float invC = 1.f / (float)C;
  const bool has_res = res != nullptr;
  // the loop bound is uniform per CTA so that the sub-warp shuffles always run with all 32 lanes
  for (long base = (long)blockIdx.x * GPB; base < rows; base += (long)gridDim.x * GPB) {
    const long row = base + gr;
    float v[NV][EPV], rr[NV][EPV];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int vi = gl + k * G;
#pragma unroll
      for (int e = 0; e < EPV; ++e) v[k][e] = rr[k][e] = 0.f;
      if (vi < nvec && row < rows) {
        Vec<T, EPV>::load(x + row * C + vi * EPV, v[k]);
        if (has_res) Vec<T, EPV>::load(res + row * C + vi * EPV, rr[k]);
      }
    }
    const bool live = row < rows;
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int vi = gl + k * G;
      if (vi < nvec && live) {
        if (has_res) {
#pragma unroll
          for (int e = 0; e < EPV; ++e) v[k][e] += rr[k][e];
          // the residual sum is stored in the I/O dtype and the statistics use the STORED value
          Vec<T, EPV>::store(sum_out + row * C + vi * EPV, v[k]);
          if (sizeof(T) == 2) {
#pragma unroll
            for (int e = 0; e < EPV; ++e) v[k][e] = to_f32(from_f32<T>(v[k][e]));
          }
        }
#pragma unroll
        for (int e = 0; e < EPV; ++e) s += v[k][e];
      }
    }
    const float mean = group_sum<G>(s) * invC;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int vi = gl + k * G;
      if (vi < nvec) {
#pragma unroll
        for (int e = 0; e < EPV; ++e) {
          const float d = v[k][e] - mean;
          q = fmaf(d, d, q);
        }
      }
    }
    const float rstd = rsqrtf(group_sum<G>(q) * invC + eps);
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int vi = gl + k * G;
      if (vi < nvec && live) {
        float o[EPV];
#pragma unroll
        for (int e = 0; e < EPV; ++e) o[e] = fmaf((v[k][e] - mean) * rstd, gm[k][e], bt[k][e]);
        Vec<T, EPV>::store(y + row * C + vi * EPV, o);
      }
    }
    if (gl == 0 && live) {
      mean_out[row] = mean;
      rstd_out[row] = rstd;
    }
  }
}

// dres_colsum / dx_colsum (optional, fp32 [C]): column sums over all rows of the residual-path gradient and of the
// produced dx -- the gradients of the Linear biases on either side of this LayerNorm (swin_block.py:222,227: dx is
// the gradient of `proj(...) + bias`, dres that of `mlp(...) + bias`), which saves two full reduction passes.
// PLAIN: no residual-path gradient and no column sums (the PatchMerging norm, down.py:44: rows of 384-1536 channels, where
// the three extra per-column register arrays of the general kernel meant spills and one CTA per SM)
// X = Det<T>: dgamma, dbeta, dres_colsum and dx_colsum are slot arrays [gridDim][C]; the warps add their column sums to shared
// memory one warp after the other and the CTA stores its sums to its own slots (summed in a fixed order by pwa_ln_bwd2_det).
template <typename X, int G, int NV, int EPV, bool PLAIN = false>
__global__ void __launch_bounds__(kLnThreads, (NV * EPV <= 8 ? 4 : (NV * EPV <= 16 ? 2 : 1))) ln_bwd_kernel(const X* __restrict__ dyin, const X* __restrict__ xin,
                                                            const float* __restrict__ gamma, const float* __restrict__ mean_in,
                                                            const float* __restrict__ rstd_in, const X* __restrict__ dresin,
                                                            X* __restrict__ dxout, float* __restrict__ dgamma,
                                                            float* __restrict__ dbeta, float* __restrict__ dres_colsum,
                                                            float* __restrict__ dx_colsum, long rows, int C) {
  using T = typename Elem<X>::type;
  const T* __restrict__ dy = reinterpret_cast<const T*>(dyin);
  const T* __restrict__ x = reinterpret_cast<const T*>(xin);
  const T* __restrict__ dres = reinterpret_cast<const T*>(dresin);
  T* __restrict__ dx = reinterpret_cast<T*>(dxout);
  constexpr int GPB = kLnThreads / G;
  extern __shared__ float red[];                        // [4][C]
  const int gl = threadIdx.x % G, gr = threadIdx.x / G;
  const int nvec = C / EPV;
  const bool has_res = !PLAIN && dres != nullptr;
  const bool want_rs = !PLAIN && dres_colsum != nullptr && has_res, want_xs = !PLAIN && dx_colsum != nullptr;
  for (int i = threadIdx.x; i < 4 * C; i += kLnThreads) red[i] = 0.f;
  constexpr int NVX = PLAIN ? 1 : NV, EPX = PLAIN ? 1 : EPV;     // (PLAIN: the extra arrays are never touched)
  float gm[NV][EPV], ag[NV][EPV], ab[NV][EPV], ar[NVX][EPX], ax[NVX][EPX];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int vi = gl + k * G;
    if (vi < nvec) loadf<EPV>(gamma + vi * EPV, gm[k]);
#pragma unroll
    for (int e = 0; e < EPV; ++e) {
      ag[k][e] = ab[k][e] = 0.f;
      if constexpr (!PLAIN) ar[k][e] = ax[k][e] = 0.f;
    }
  }
  const float invC = 1.f / (float)C;
  for (long base = (long)blockIdx.x * GPB; base < rows; base += (long)gridDim.x * GPB) {
    const long row = base + gr;
    const bool live = row < rows;
    float d[NV][EPV], xv[NV][EPV], rs[NVX][EPX];
    const float mean = live ? __ldg(mean_in + row) : 0.f;
    const float rstd = live ? __ldg(rstd_in + row) : 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int vi = gl + k * G;
#pragma unroll
      for (int e = 0; e < EPV; ++e) {
        d[k][e] = xv[k][e] = 0.f;
        if constexpr (!PLAIN) rs[k][e] = 0.f;
      }
      if (vi < nvec && live) {
        Vec<T, EPV>::load(dy + row * C + vi * EPV, d[k]);
        Vec<T, EPV>::load(x + row * C + vi * EPV, xv[k]);
        if constexpr (!PLAIN) {
          if (has_res) Vec<T, EPV>::load(dres + row * C + vi * EPV, rs[k]);
        }
      }
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      if (gl + k * G >= nvec) continue;                 // (dead rows hold zeros and mean = rstd = 0: they add nothing)
#pragma unroll
      for (int e = 0; e < EPV; ++e) {
        const float xh = (xv[k][e] - mean) * rstd;
        const float g = d[k][e] * gm[k][e];
        xv[k][e] = xh;
        s1 += g;
        s2 = fmaf(g, xh, s2);
        ag[k][e] = fmaf(d[k][e], xh, ag[k][e]);
        ab[k][e] += d[k][e];
        d[k][e] = g;
      }
    }
    s1 = group_sum<G>(s1) * invC;
    s2 = group_sum<G>(s2) * invC;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const int vi = gl + k * G;
      if (vi < nvec && live) {
        float o[EPV];
#pragma unroll
        for (int e = 0; e < EPV; ++e) {
          o[e] = rstd * (d[k][e] - s1 - xv[k][e] * s2);
          if constexpr (!PLAIN) {
            o[e] += rs[k][e];
            ar[k][e] += rs[k][e];
            ax[k][e] += o[e];
          }
        }
        Vec<T, EPV>::store(dx + row * C + vi * EPV, o);
      }
    }
  }
  __syncthreads();
  if constexpr (Elem<X>::det) {
    // the same shuffles, then the warps add to shared memory in warp order, then plain stores to this CTA's slots
#pragma unroll
    for (int k = 0; k < NV; ++k) {
#pragma unroll
      for (int e = 0; e < EPV; ++e) {
#pragma unroll
        for (int o = G; o < 32; o <<= 1) {
          ag[k][e] += __shfl_xor_sync(0xffffffffu, ag[k][e], o);
          ab[k][e] += __shfl_xor_sync(0xffffffffu, ab[k][e], o);
          if constexpr (!PLAIN) {
            if (want_rs) ar[k][e] += __shfl_xor_sync(0xffffffffu, ar[k][e], o);
            if (want_xs) ax[k][e] += __shfl_xor_sync(0xffffffffu, ax[k][e], o);
          }
        }
      }
    }
    for (int w = 0; w < kLnThreads / 32; ++w) {
      if ((int)(threadIdx.x >> 5) == w && (threadIdx.x & 31) < G) {
#pragma unroll
        for (int k = 0; k < NV; ++k) {
          const int vi = gl + k * G;
          if (vi >= nvec) continue;
#pragma unroll
          for (int e = 0; e < EPV; ++e) {
            red[vi * EPV + e] += ag[k][e];
            red[C + vi * EPV + e] += ab[k][e];
            if constexpr (!PLAIN) {
              if (want_rs) red[2 * C + vi * EPV + e] += ar[k][e];
              if (want_xs) red[3 * C + vi * EPV + e] += ax[k][e];
            }
          }
        }
      }
      __syncthreads();
    }
    const size_t slot = (size_t)blockIdx.x * C;
    for (int i = threadIdx.x; i < C; i += kLnThreads) {
      dgamma[slot + i] = red[i];
      dbeta[slot + i] = red[C + i];
      if (want_rs) dres_colsum[slot + i] = red[2 * C + i];
      if (want_xs) dx_colsum[slot + i] = red[3 * C + i];
    }
  } else {
  // column sums: first across the 32/G row groups of a warp (lanes with equal gl) by shuffles, then one
  // shared-memory atomic per warp and column (8-way instead of 256/G-way contention), then one global atomic per CTA
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const int vi = gl + k * G;
#pragma unroll
    for (int e = 0; e < EPV; ++e) {
      float a = ag[k][e], b = ab[k][e], c = 0.f, d = 0.f;
      if constexpr (!PLAIN) { c = ar[k][e]; d = ax[k][e]; }
#pragma unroll
      for (int o = G; o < 32; o <<= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
        if (want_rs) c += __shfl_xor_sync(0xffffffffu, c, o);
        if (want_xs) d += __shfl_xor_sync(0xffffffffu, d, o);
      }
      if ((threadIdx.x & 31) < G && vi < nvec) {
        atomicAdd(&red[vi * EPV + e], a);
        atomicAdd(&red[C + vi * EPV + e], b);
        if (want_rs) atomicAdd(&red[2 * C + vi * EPV + e], c);
        if (want_xs) atomicAdd(&red[3 * C + vi * EPV + e], d);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += kLnThreads) {
    atomicAdd(&dgamma[i], red[i]);
    atomicAdd(&dbeta[i], red[C + i]);
    if (want_rs) atomicAdd(&dres_colsum[i], red[2 * C + i]);
    if (want_xs) atomicAdd(&dx_colsum[i], red[3 * C + i]);
  }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Bulk-copy variants (bf16 / fp16, one 16-byte vector per lane): the register kernels above keep one row per lane group in
// flight, i.e. 16-48 bytes per thread, and at 4 CTAs/SM (56-64 registers) that is 16-48 KB per SM -- Little's law
// wants ~45 KB for the measured 6.6 TB/s, and the plain forward sat at 2.9 TB/s.  Here the operand tiles of a CTA
// iteration (256/G consecutive rows = one contiguous 3-4 KB chunk per operand) are fetched by cp.async.bulk into a
// shared-memory ring (kMaxStages / operands deep) (one elected thread, mbarrier complete_tx), which decouples the bytes in flight
// from the register file; the lanes then read their vector from shared memory and run the same math.
constexpr int kMaxStages = 12;     // ring depth = kMaxStages / operands (12 / 6 / 4 tiles of 3-4 KB: ~36-48 KB per CTA in flight)

__device__ __forceinline__ uint32_t ln_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ln_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ln_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void ln_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ln_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ln_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(ln_smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   ln_smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(ln_smem_u32(bar)) : "memory");
}
template <typename T>
__device__ __forceinline__ void lds_vec8(const T* p, float (&v)[8]) {
  const uint4 t = *reinterpret_cast<const uint4*>(p);
  unpack2<T>(t.x, v[0], v[1]);
  unpack2<T>(t.y, v[2], v[3]);
  unpack2<T>(t.z, v[4], v[5]);
  unpack2<T>(t.w, v[6], v[7]);
}

// ring of `stages` buffers, each holding `nop` operand tiles of GPB rows; tile t of this CTA = blockIdx.x + t * gridDim.x
template <int GPB, typename T>
struct BulkRing {
  uint8_t* buf;
  uint64_t* full;
  uint32_t tile_bytes;      // GPB * C * 2
  int nop, C, stages;
  long rows, n_tiles;
  const T* src[3];
  __device__ __forceinline__ void issue(long tile, int s) const {      // one thread
    const long row0 = tile * GPB;
    const long left = rows - row0;
    const uint32_t bytes = (uint32_t)(left < GPB ? left : GPB) * (uint32_t)C * 2u;
    ln_mbar_expect_tx(&full[s], bytes * nop);
    for (int o = 0; o < nop; ++o) bulk_g2s(buf + ((size_t)s * nop + o) * tile_bytes, src[o] + row0 * C, bytes, &full[s]);
  }
  __device__ __forceinline__ const T* tile(int s, int o) const {
    return reinterpret_cast<const T*>(buf + ((size_t)s * nop + o) * tile_bytes);
  }
};

// R rows per lane group and iteration (tile = R * 256/G rows): the per-iteration overhead (mbarrier wait, block barrier,
// refill, addressing, loop) is paid once per R rows, and the shuffle reductions of the R rows interleave.
template <int G, int R, typename T>
__global__ void __launch_bounds__(kLnThreads, R == 1 ? 4 : 3) ln_fwd_bulk_kernel(const T* __restrict__ x, const T* __restrict__ res,
                                                                    const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                    T* __restrict__ sum_out, T* __restrict__ y,
                                                                    float* __restrict__ mean_out, float* __restrict__ rstd_out,
                                                                    long rows, int C, float eps) {
  constexpr int GPB = kLnThreads / G, TR = GPB * R, EPV = 8;
  extern __shared__ __align__(128) uint8_t ln_sm[];
  __shared__ __align__(8) uint64_t full[kMaxStages];
  const int gl = threadIdx.x % G, gr = threadIdx.x / G;
  const int nvec = C / EPV;
  const bool has_res = res != nullptr;
  BulkRing<TR, T> ring;
  ring.buf = ln_sm; ring.full = full; ring.tile_bytes = (uint32_t)TR * C * 2u; ring.nop = has_res ? 2 : 1; ring.C = C;
  ring.stages = kMaxStages / ring.nop / R;
  ring.rows = rows; ring.n_tiles = (rows + TR - 1) / TR;
  ring.src[0] = x; ring.src[1] = res; ring.src[2] = nullptr;
  if (threadIdx.x == 0) {
    for (int s = 0; s < ring.stages; ++s) ln_mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int s = 0; s < ring.stages; ++s) {
      const long t = blockIdx.x + (long)s * gridDim.x;
      if (t < ring.n_tiles) ring.issue(t, s);
    }
  }
  float gm[EPV], bt[EPV];
  const bool lane_live = gl < nvec;
  if (lane_live) {
    loadf<EPV>(gamma + gl * EPV, gm);
    loadf<EPV>(beta + gl * EPV, bt);
  }
  const float invC = 1.f / (float)C;
  int s = 0;
  uint32_t par = 0;
  for (long tile = blockIdx.x; tile < ring.n_tiles; tile += gridDim.x) {
    const long row0 = tile * TR + gr;
    ln_mbar_wait(&full[s], par);
    float v[R][EPV], rr[R][EPV];
#pragma unroll
    for (int r = 0; r < R; ++r) {
#pragma unroll
      for (int e = 0; e < EPV; ++e) v[r][e] = rr[r][e] = 0.f;
      if (lane_live && row0 + r * GPB < rows) {
        lds_vec8<T>(ring.tile(s, 0) + (r * GPB + gr) * C + gl * EPV, v[r]);
        if (has_res) lds_vec8<T>(ring.tile(s, 1) + (r * GPB + gr) * C + gl * EPV, rr[r]);
      }
    }
    __syncthreads();                                    // every lane holds its vectors: the buffer can be refilled
    if (threadIdx.x == 0) {
      const long nt = tile + (long)ring.stages * gridDim.x;
      if (nt < ring.n_tiles) ring.issue(nt, s);
    }
    if (++s == ring.stages) { s = 0; par ^= 1u; }
    float sum[R], q[R], mean[R], rstd[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const long row = row0 + r * GPB;
      const bool live = lane_live && row < rows;
      sum[r] = 0.f;
      if (live) {
        if (has_res) {
#pragma unroll
          for (int e = 0; e < EPV; ++e) v[r][e] += rr[r][e];
          // the residual sum is stored in the I/O dtype and the statistics use the STORED value
          Vec<T, EPV>::store(sum_out + row * C + gl * EPV, v[r]);
#pragma unroll
          for (int e = 0; e < EPV; ++e) v[r][e] = to_f32(from_f32<T>(v[r][e]));
        }
#pragma unroll
        for (int e = 0; e < EPV; ++e) sum[r] += v[r][e];
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) mean[r] = group_sum<G>(sum[r]) * invC;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      q[r] = 0.f;
      if (lane_live) {
#pragma unroll
        for (int e = 0; e < EPV; ++e) {
          const float d = v[r][e] - mean[r];
          q[r] = fmaf(d, d, q[r]);
        }
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) rstd[r] = rsqrtf(group_sum<G>(q[r]) * invC + eps);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const long row = row0 + r * GPB;
      if (lane_live && row < rows) {
        float o[EPV];
#pragma unroll
        for (int e = 0; e < EPV; ++e) o[e] = fmaf((v[r][e] - mean[r]) * rstd[r], gm[e], bt[e]);
        Vec<T, EPV>::store(y + row * C + gl * EPV, o);
        if (gl == 0) {
          mean_out[row] = mean[r];
          rstd_out[row] = rstd[r];
        }
      }
    }
  }
}

// X = Det<T>: dgamma, dbeta, dres_colsum and dx_colsum are slot arrays [gridDim][C] that the CTA stores its sums to (the in-CTA
// order is fixed either way); pwa_ln_bwd2_det sums the slots in a fixed order.
template <int G, int R, typename X>
__global__ void __launch_bounds__(kLnThreads, R == 1 ? 3 : 2) ln_bwd_bulk_kernel(const X* __restrict__ dyin, const X* __restrict__ xin,
                                                                    const float* __restrict__ gamma, const float* __restrict__ mean_in,
                                                                    const float* __restrict__ rstd_in, const X* __restrict__ dresin,
                                                                    X* __restrict__ dxout, float* __restrict__ dgamma,
                                                                    float* __restrict__ dbeta, float* __restrict__ dres_colsum,
                                                                    float* __restrict__ dx_colsum, long rows, int C) {
  using T = typename Elem<X>::type;
  const T* __restrict__ dy = reinterpret_cast<const T*>(dyin);
  const T* __restrict__ x = reinterpret_cast<const T*>(xin);
  const T* __restrict__ dres = reinterpret_cast<const T*>(dresin);
  T* __restrict__ dx = reinterpret_cast<T*>(dxout);
  constexpr int GPB = kLnThreads / G, TR = GPB * R, EPV = 8;
  extern __shared__ __align__(128) uint8_t ln_sm[];
  __shared__ __align__(8) uint64_t full[kMaxStages];
  const int gl = threadIdx.x % G, gr = threadIdx.x / G;
  const int nvec = C / EPV;
  const bool has_res = dres != nullptr;
  const bool want_rs = dres_colsum != nullptr && has_res, want_xs = dx_colsum != nullptr;
  BulkRing<TR, T> ring;
  ring.buf = ln_sm; ring.full = full; ring.tile_bytes = (uint32_t)TR * C * 2u; ring.nop = has_res ? 3 : 2; ring.C = C;
  ring.stages = kMaxStages / ring.nop / R;
  ring.rows = rows; ring.n_tiles = (rows + TR - 1) / TR;
  ring.src[0] = dy; ring.src[1] = x; ring.src[2] = dres;
  if (threadIdx.x == 0) {
    for (int s = 0; s < ring.stages; ++s) ln_mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int s = 0; s < ring.stages; ++s) {
      const long t = blockIdx.x + (long)s * gridDim.x;
      if (t < ring.n_tiles) ring.issue(t, s);
    }
  }
  const bool lane_live = gl < nvec;
  float gm[EPV], ag[EPV], ab[EPV], ar[EPV], ax[EPV];
#pragma unroll
  for (int e = 0; e < EPV; ++e) gm[e] = ag[e] = ab[e] = ar[e] = ax[e] = 0.f;
  if (lane_live) loadf<EPV>(gamma + gl * EPV, gm);
  const float invC = 1.f / (float)C;
  int s = 0;
  uint32_t par = 0;
  for (long tile = blockIdx.x; tile < ring.n_tiles; tile += gridDim.x) {
    const long row0 = tile * TR + gr;
    float mean[R], rstd[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const long row = row0 + r * GPB;
      mean[r] = row < rows ? __ldg(mean_in + row) : 0.f;
      rstd[r] = row < rows ? __ldg(rstd_in + row) : 0.f;
    }
    ln_mbar_wait(&full[s], par);
    float d[R][EPV], xv[R][EPV], rs[R][EPV];
#pragma unroll
    for (int r = 0; r < R; ++r) {
#pragma unroll
      for (int e = 0; e < EPV; ++e) d[r][e] = xv[r][e] = rs[r][e] = 0.f;
      if (lane_live && row0 + r * GPB < rows) {
        lds_vec8<T>(ring.tile(s, 0) + (r * GPB + gr) * C + gl * EPV, d[r]);
        lds_vec8<T>(ring.tile(s, 1) + (r * GPB + gr) * C + gl * EPV, xv[r]);
        if (has_res) lds_vec8<T>(ring.tile(s, 2) + (r * GPB + gr) * C + gl * EPV, rs[r]);
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      const long nt = tile + (long)ring.stages * gridDim.x;
      if (nt < ring.n_tiles) ring.issue(nt, s);
    }
    if (++s == ring.stages) { s = 0; par ^= 1u; }
    float s1[R], s2[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      s1[r] = s2[r] = 0.f;
      if (lane_live && row0 + r * GPB < rows) {             // (dead lanes / rows add nothing)
#pragma unroll
        for (int e = 0; e < EPV; ++e) {
          const float xh = (xv[r][e] - mean[r]) * rstd[r];
          const float g = d[r][e] * gm[e];
          xv[r][e] = xh;
          s1[r] += g;
          s2[r] = fmaf(g, xh, s2[r]);
          ag[e] = fmaf(d[r][e], xh, ag[e]);
          ab[e] += d[r][e];
          d[r][e] = g;
        }
      }
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      s1[r] = group_sum<G>(s1[r]) * invC;
      s2[r] = group_sum<G>(s2[r]) * invC;
    }
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const long row = row0 + r * GPB;
      if (lane_live && row < rows) {
        float o[EPV];
#pragma unroll
        for (int e = 0; e < EPV; ++e) {
          o[e] = rstd[r] * (d[r][e] - s1[r] - xv[r][e] * s2[r]) + rs[r][e];
          ar[e] += rs[r][e];
          ax[e] += o[e];
        }
        Vec<T, EPV>::store(dx + row * C + gl * EPV, o);
      }
    }
  }
  __syncthreads();
#pragma unroll
  for (int e = 0; e < EPV; ++e) {
    float a = ag[e], b = ab[e], c = ar[e], d = ax[e];
#pragma unroll
    for (int o = G; o < 32; o <<= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
      if (want_rs) c += __shfl_xor_sync(0xffffffffu, c, o);
      if (want_xs) d += __shfl_xor_sync(0xffffffffu, d, o);
    }
    // per-warp partial sums -> the (now idle) ring memory, [warp][array][C]: plain stores.  (fp32 shared-memory atomics
    // are compare-and-swap loops; 8 warps contending for every column made this epilogue a fixed ~5 us per CTA, a quarter
    // of the kernel at the late stages' row counts.)
    if ((threadIdx.x & 31) < G && lane_live) {
      float* part = reinterpret_cast<float*>(ln_sm) + (size_t)(threadIdx.x >> 5) * 4 * C;
      part[gl * EPV + e] = a;
      part[C + gl * EPV + e] = b;
      if (want_rs) part[2 * C + gl * EPV + e] = c;
      if (want_xs) part[3 * C + gl * EPV + e] = d;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C; i += kLnThreads) {
    const float* part = reinterpret_cast<const float*>(ln_sm);
    float a = 0.f, b = 0.f, c = 0.f, d = 0.f;
#pragma unroll
    for (int w = 0; w < kLnThreads / 32; ++w) {
      a += part[(w * 4 + 0) * C + i];
      b += part[(w * 4 + 1) * C + i];
      if (want_rs) c += part[(w * 4 + 2) * C + i];
      if (want_xs) d += part[(w * 4 + 3) * C + i];
    }
    if constexpr (Elem<X>::det) {
      const size_t slot = (size_t)blockIdx.x * C;
      dgamma[slot + i] = a;
      dbeta[slot + i] = b;
      if (want_rs) dres_colsum[slot + i] = c;
      if (want_xs) dx_colsum[slot + i] = d;
    } else {
      atomicAdd(&dgamma[i], a);
      atomicAdd(&dbeta[i], b);
      if (want_rs) atomicAdd(&dres_colsum[i], c);
      if (want_xs) atomicAdd(&dx_colsum[i], d);
    }
  }
}

struct LnArgs {
  const void *a, *b, *res;
  const float *gamma, *bm, *rstd;
  void *o1, *o2;
  float *f1, *f2, *f3, *f4;
  long rows;
  int C;
  float eps;
  float* det_ws;       // backward: non-NULL = the deterministic kernels, slot arrays [4][blocks][C] here (see ln_det_slots)
};

// grid of the register kernels
static long ln_reg_blocks(bool fwd, long rows, int G) {
  const int GPB = kLnThreads / G;
  long blocks = (rows + GPB - 1) / GPB;
  // backward: fewer CTAs -> fewer global atomics; with few rows (the late PatchMerging norms: 7 K rows of 768 channels) every
  // CTA should also run several iterations, or its epilogue (4C shared words zeroed, 2C..4C shared + global atomics)
  // outweighs its share of the rows: 48 -> see tools/bench_ln.py
  long cap = 148L * (fwd ? 8 : 4);
  if (!fwd) {
    const long few = blocks / 6 > 148 ? blocks / 6 : (blocks < 148 ? blocks : 148);
    if (few < cap) cap = few;
  }
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return blocks;
}

// Rows per lane group and iteration of the bulk kernels, measured (tools/bench_ln.py): R = 2 is 8-13 % faster in backward,
// within +-5 % in forward.  At most 4 CTAs per SM forward, 2 backward (the bytes in flight no longer depend on the occupancy).
constexpr int kBulkRF = 1, kBulkRB = 2;
static long ln_bulk_blocks(bool fwd, long rows, int G) {
  const int TR = kLnThreads / G * (fwd ? kBulkRF : kBulkRB);
  long blocks = (rows + TR - 1) / TR;
  const long cap = 148L * (fwd ? 4 : 2);
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return blocks;
}

// Deterministic backward: the kernel writes its column sums to the slot arrays [4][blocks][C] of a.det_ws (dgamma, dbeta,
// dres_colsum, dx_colsum), which ln_det_reduce then sums over the CTAs in a fixed order into the caller's outputs.
static LnArgs ln_det_slots(const LnArgs& a, long blocks) {
  LnArgs d = a;
  const size_t n = (size_t)blocks * a.C;
  d.f1 = a.det_ws;
  d.f2 = a.det_ws + n;
  d.f3 = a.f3 ? a.det_ws + 2 * n : nullptr;
  d.f4 = a.f4 ? a.det_ws + 3 * n : nullptr;
  return d;
}

static int ln_det_reduce(const LnArgs& a, long blocks, cudaStream_t st) {
  const size_t n = (size_t)blocks * a.C;
  float* out[4] = {a.f1, a.f2, a.f3, a.f4};
  for (int i = 0; i < 4; ++i) {
    if (out[i] == nullptr) continue;
    const int rc = pwa_colsum_f32(a.det_ws + i * n, out[i], (int)blocks, a.C, st);
    if (rc != PWA_OK) return rc;
  }
  return PWA_OK;
}

template <typename T, int G, int NV, int EPV>
static int ln_launch(bool fwd, const LnArgs& a0, cudaStream_t st) {
  const long blocks = ln_reg_blocks(fwd, a0.rows, G);
  const bool det = !fwd && a0.det_ws != nullptr;
  const LnArgs a = det ? ln_det_slots(a0, blocks) : a0;
  if (det) {
    using D = Det<T>;
    if constexpr (NV >= 2) {
      if (a.res == nullptr && a.f3 == nullptr && a.f4 == nullptr) {
        ln_bwd_kernel<D, G, NV, EPV, true><<<(unsigned)blocks, kLnThreads, 4 * a.C * sizeof(float), st>>>(
            (const D*)a.a, (const D*)a.b, a.gamma, a.bm, a.rstd, nullptr, (D*)a.o1, a.f1, a.f2, nullptr, nullptr, a.rows, a.C);
        PWA_CUDA_OK(cudaGetLastError());
        return ln_det_reduce(a0, blocks, st);
      }
    }
    ln_bwd_kernel<D, G, NV, EPV><<<(unsigned)blocks, kLnThreads, 4 * a.C * sizeof(float), st>>>(
        (const D*)a.a, (const D*)a.b, a.gamma, a.bm, a.rstd, (const D*)a.res, (D*)a.o1, a.f1, a.f2, a.f3, a.f4, a.rows, a.C);
    PWA_CUDA_OK(cudaGetLastError());
    return ln_det_reduce(a0, blocks, st);
  }
  if (fwd) {
    ln_fwd_kernel<T, G, NV, EPV><<<(unsigned)blocks, kLnThreads, 0, st>>>((const T*)a.a, (const T*)a.res, a.gamma, a.bm,
                                                                           (T*)a.o1, (T*)a.o2, a.f1, a.f2, a.rows, a.C, a.eps);
  } else {
    if constexpr (NV >= 2) {
      if (a.res == nullptr && a.f3 == nullptr && a.f4 == nullptr) {
        ln_bwd_kernel<T, G, NV, EPV, true><<<(unsigned)blocks, kLnThreads, 4 * a.C * sizeof(float), st>>>(
            (const T*)a.a, (const T*)a.b, a.gamma, a.bm, a.rstd, nullptr, (T*)a.o1, a.f1, a.f2, nullptr, nullptr, a.rows, a.C);
        PWA_CUDA_OK(cudaGetLastError());
        return PWA_OK;
      }
    }
    ln_bwd_kernel<T, G, NV, EPV><<<(unsigned)blocks, kLnThreads, 4 * a.C * sizeof(float), st>>>(
        (const T*)a.a, (const T*)a.b, a.gamma, a.bm, a.rstd, (const T*)a.res, (T*)a.o1, a.f1, a.f2, a.f3, a.f4, a.rows, a.C);
  }
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

template <int G, typename T>
static int ln_launch_bulk(bool fwd, const LnArgs& a0, cudaStream_t st) {
  constexpr int RF = kBulkRF, RB = kBulkRB;
  const int R = fwd ? RF : RB, TR = kLnThreads / G * R;
  const int nop = fwd ? (a0.res ? 2 : 1) : (a0.res ? 3 : 2);
  // (backward epilogue: the per-warp column sums, 8 x 4 x C floats, reuse the ring memory: >= 192 * C bytes for every G)
  const size_t smem = (size_t)(kMaxStages / nop / R) * nop * TR * a0.C * 2;
  const long blocks = ln_bulk_blocks(fwd, a0.rows, G);
  if (!fwd && a0.det_ws != nullptr) {
    using D = Det<T>;
    const LnArgs a = ln_det_slots(a0, blocks);
    PWA_CUDA_OK(cudaFuncSetAttribute(ln_bwd_bulk_kernel<G, RB, D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ln_bwd_bulk_kernel<G, RB, D><<<(unsigned)blocks, kLnThreads, smem, st>>>((const D*)a.a, (const D*)a.b, a.gamma, a.bm, a.rstd,
                                                                          (const D*)a.res, (D*)a.o1, a.f1, a.f2, a.f3, a.f4, a.rows, a.C);
    PWA_CUDA_OK(cudaGetLastError());
    return ln_det_reduce(a0, blocks, st);
  }
  const LnArgs& a = a0;
  if (fwd) {
    PWA_CUDA_OK(cudaFuncSetAttribute(ln_fwd_bulk_kernel<G, RF, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ln_fwd_bulk_kernel<G, RF, T><<<(unsigned)blocks, kLnThreads, smem, st>>>((const T*)a.a, (const T*)a.res, a.gamma, a.bm,
                                                                          (T*)a.o1, (T*)a.o2, a.f1, a.f2, a.rows, a.C, a.eps);
  } else {
    PWA_CUDA_OK(cudaFuncSetAttribute(ln_bwd_bulk_kernel<G, RB, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ln_bwd_bulk_kernel<G, RB, T><<<(unsigned)blocks, kLnThreads, smem, st>>>((const T*)a.a, (const T*)a.b, a.gamma, a.bm, a.rstd,
                                                                          (const T*)a.res, (T*)a.o1, a.f1, a.f2, a.f3, a.f4, a.rows, a.C);
  }
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

// lane group width of the row kernels for rows of nvec vectors (ln_dispatch_v)
static int ln_group(int nvec) { return nvec <= 4 ? 4 : (nvec <= 8 ? 8 : (nvec <= 16 ? 16 : 32)); }

template <typename T, int EPV>
static int ln_dispatch_v(bool fwd, const LnArgs& a, cudaStream_t st) {
  const int nvec = a.C / EPV;
#define LN_CASE(G, NV) return ln_launch<T, G, NV, EPV>(fwd, a, st)
  if constexpr (sizeof(T) == 2 && EPV == 8) {
    // one vector per lane, rows contiguous: the bulk-copy kernels
    if (nvec <= 4) return ln_launch_bulk<4, T>(fwd, a, st);
    if (nvec <= 8) return ln_launch_bulk<8, T>(fwd, a, st);
    if (nvec <= 16) return ln_launch_bulk<16, T>(fwd, a, st);
    if (nvec <= 32) return ln_launch_bulk<32, T>(fwd, a, st);
  } else {
    if (nvec <= 4) LN_CASE(4, 1);
    if (nvec <= 8) LN_CASE(8, 1);
    if (nvec <= 16) LN_CASE(16, 1);
    if (nvec <= 32) LN_CASE(32, 1);
  }
  if (nvec <= 64) LN_CASE(32, 2);
  if (nvec <= 128) LN_CASE(32, 4);
  // C in (1024, 2048]: PatchMerging norms of wide stages (8 * 192 = 1536, 4 * 384 = 1536, down.py:13-14); these rows
  // live in more registers than a thread has (spills) -- rare shapes, correctness over speed
  if (nvec <= 256) LN_CASE(32, 8);
  if (EPV == 4 && nvec <= 512) LN_CASE(32, 16);
#undef LN_CASE
  set_error("layer norm: C=%d too large (max 2048)", a.C);
  return PWA_ERR_UNSUPPORTED;
}

template <typename T>
static int ln_dispatch(bool fwd, const LnArgs& a, cudaStream_t st) {
  if constexpr (sizeof(T) == 2) {
    const uintptr_t al = (uintptr_t)a.a | (uintptr_t)a.b | (uintptr_t)a.res | (uintptr_t)a.o1 | (uintptr_t)a.o2;
    if (a.C % 8 == 0 && (al & 15) == 0) return ln_dispatch_v<T, 8>(fwd, a, st);
  }
  return ln_dispatch_v<T, 4>(fwd, a, st);
}

}  // namespace pwa

using namespace pwa;

extern "C" int pwa_ln_fwd(const void* x, const void* res, const float* gamma, const float* beta, void* sum_out, void* y,
                          float* mean, float* rstd, int64_t rows, int C, float eps, int dtype, void* stream) {
  PWA_CHECK_ARG(x && gamma && beta && y && mean && rstd, "pwa_ln_fwd: null pointer");
  PWA_CHECK_ARG(res == nullptr || sum_out != nullptr, "pwa_ln_fwd: residual given without sum_out");
  PWA_CHECK_ARG(rows >= 0 && C > 0 && C % 4 == 0 && C <= 2048, "pwa_ln_fwd: need C %% 4 == 0, C <= 2048 (C=%d)", C);
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "pwa_ln_fwd: bad dtype %d", dtype);
  if (rows == 0) return PWA_OK;
  cudaStream_t st = (cudaStream_t)stream;
  LnArgs a = {x, nullptr, res, gamma, beta, nullptr, sum_out, y, mean, rstd, nullptr, nullptr, (long)rows, C, eps, nullptr};
  if (dtype == PWA_F16) return ln_dispatch<__half>(true, a, st);
  return dtype == PWA_F32 ? ln_dispatch<float>(true, a, st) : ln_dispatch<__nv_bfloat16>(true, a, st);
}

extern "C" int pwa_ln_bwd2(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd,
                           const void* dres, void* dx, float* dgamma, float* dbeta, float* dres_colsum, float* dx_colsum,
                           int64_t rows, int C, int dtype, void* stream) {
  PWA_CHECK_ARG(dy && x && gamma && mean && rstd && dx && dgamma && dbeta, "pwa_ln_bwd: null pointer");
  PWA_CHECK_ARG(rows >= 0 && C > 0 && C % 4 == 0 && C <= 2048, "pwa_ln_bwd: need C %% 4 == 0, C <= 2048 (C=%d)", C);
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "pwa_ln_bwd: bad dtype %d", dtype);
  PWA_CHECK_ARG(dres_colsum == nullptr || dres != nullptr, "pwa_ln_bwd: dres_colsum without dres");
  cudaStream_t st = (cudaStream_t)stream;
  PWA_CUDA_OK(cudaMemsetAsync(dgamma, 0, (size_t)C * 4, st));
  PWA_CUDA_OK(cudaMemsetAsync(dbeta, 0, (size_t)C * 4, st));
  if (dres_colsum) PWA_CUDA_OK(cudaMemsetAsync(dres_colsum, 0, (size_t)C * 4, st));
  if (dx_colsum) PWA_CUDA_OK(cudaMemsetAsync(dx_colsum, 0, (size_t)C * 4, st));
  if (rows == 0) return PWA_OK;
  LnArgs a = {dy, x, dres, gamma, mean, rstd, dx, nullptr, dgamma, dbeta, dres_colsum, dx_colsum, (long)rows, C, 0.f, nullptr};
  if (dtype == PWA_F16) return ln_dispatch<__half>(false, a, st);
  return dtype == PWA_F32 ? ln_dispatch<float>(false, a, st) : ln_dispatch<__nv_bfloat16>(false, a, st);
}

// Slots of the deterministic backward: the grid of whichever kernel ln_dispatch picks.  16-bit rows with C % 8 == 0 take the
// EPV = 8 kernels when the pointers are 16-byte aligned and the EPV = 4 ones otherwise: the size covers both.
extern "C" int64_t pwa_ln_bwd2_det_workspace_size(int64_t rows, int C, int dtype) {
  if (rows < 0 || C <= 0 || C % 4 != 0 || C > 2048) return PWA_ERR_ARG;
  if (dtype != PWA_F32 && dtype != PWA_BF16 && dtype != PWA_F16) return PWA_ERR_ARG;
  if (rows == 0) return 0;
  long blocks = ln_reg_blocks(false, (long)rows, ln_group(C / 4));
  if (dtype != PWA_F32 && C % 8 == 0) {
    const int nvec = C / 8;
    const long b8 = nvec <= 32 ? ln_bulk_blocks(false, (long)rows, ln_group(nvec)) : ln_reg_blocks(false, (long)rows, 32);
    if (b8 > blocks) blocks = b8;
  }
  return (int64_t)blocks * 4 * C * 4;
}

extern "C" int pwa_ln_bwd2_det(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd,
                               const void* dres, void* dx, float* dgamma, float* dbeta, float* dres_colsum, float* dx_colsum,
                               int64_t rows, int C, int dtype, void* workspace, int64_t workspace_bytes, void* stream) {
  PWA_CHECK_ARG(dy && x && gamma && mean && rstd && dx && dgamma && dbeta, "pwa_ln_bwd2_det: null pointer");
  PWA_CHECK_ARG(rows >= 0 && C > 0 && C % 4 == 0 && C <= 2048, "pwa_ln_bwd2_det: need C %% 4 == 0, C <= 2048 (C=%d)", C);
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "pwa_ln_bwd2_det: bad dtype %d", dtype);
  PWA_CHECK_ARG(dres_colsum == nullptr || dres != nullptr, "pwa_ln_bwd2_det: dres_colsum without dres");
  const int64_t need = pwa_ln_bwd2_det_workspace_size(rows, C, dtype);
  PWA_CHECK_ARG(workspace_bytes >= need && (need == 0 || workspace != nullptr),
                "pwa_ln_bwd2_det: workspace of %lld bytes, %lld needed", (long long)workspace_bytes, (long long)need);
  cudaStream_t st = (cudaStream_t)stream;
  if (rows == 0) {
    PWA_CUDA_OK(cudaMemsetAsync(dgamma, 0, (size_t)C * 4, st));
    PWA_CUDA_OK(cudaMemsetAsync(dbeta, 0, (size_t)C * 4, st));
    if (dres_colsum) PWA_CUDA_OK(cudaMemsetAsync(dres_colsum, 0, (size_t)C * 4, st));
    if (dx_colsum) PWA_CUDA_OK(cudaMemsetAsync(dx_colsum, 0, (size_t)C * 4, st));
    return PWA_OK;
  }
  LnArgs a = {dy, x, dres, gamma, mean, rstd, dx, nullptr, dgamma, dbeta, dres_colsum, dx_colsum, (long)rows, C, 0.f, (float*)workspace};
  if (dtype == PWA_F16) return ln_dispatch<__half>(false, a, st);
  return dtype == PWA_F32 ? ln_dispatch<float>(false, a, st) : ln_dispatch<__nv_bfloat16>(false, a, st);
}

extern "C" int pwa_ln_bwd(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd,
                          const void* dres, void* dx, float* dgamma, float* dbeta, int64_t rows, int C, int dtype,
                          void* stream) {
  return pwa_ln_bwd2(dy, x, gamma, mean, rstd, dres, dx, dgamma, dbeta, nullptr, nullptr, rows, C, dtype, stream);
}
