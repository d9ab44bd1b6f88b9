// Token-domain GEMM with a fused LayerNorm / residual / dropout prologue on the 5th-gen tensor cores (SURVEY §8f-1):
//     s = dropout(x) + res          (both optional; s is written when a residual is given)
//     z = LayerNorm(s) * gamma + beta   (optional; z is written when asked for: the backward's weight-gradient operand)
//     y = z @ W^T + bias            tcgen05.mma kind::f16, A = z tile from shared memory, B = W resident in shared memory,
//                                   fp32 accumulator in TMEM
// Replaces, in one pass over the tokens, the reference's LayerNorm + Linear pairs of the block (swin_block.py:216 attn_norm +
// window_attention.py:42-44 to_q/to_k/to_v as ONE [C -> 3C] projection; swin_block.py:222-227 residual add + mlp_norm + the
// single-Linear "MLP", with window_attention.py:60's projection dropout in front) that ran as separate LayerNorm kernels
// and cuBLAS GEMMs with a round trip through HBM between them.
//
// One CTA = 128 threads = one 128-token tile at a time (thread = token row = TMEM lane), several CTAs per SM so that the
// phases of different tiles overlap:
//   bulk copy (cp.async.bulk, mbarrier complete_tx) of the contiguous x / res tiles -> shared memory
//   -> per-row statistics in registers (no shuffles: a thread owns its row; exact mean, then centred variance, computed on
//      the bf16 / fp16 values that are stored, like csrc/ln.cu) -> s / z tiles written back in place (bulk stores) and z into the
//      UMMA canonical K-major layout -> C/16 MMAs of N = NCH output channels -> tcgen05.ld, + bias, rounded, staged row-major
//      -> bulk stores of the output rows.
// Weights wider than fits beside the tiles are split into chunks of NCH output channels over CTAs (blockIdx % n_chunks);
// a CTA keeps its chunk resident for all of its tiles.
#include "common.cuh"
#include "tc_common.cuh"

namespace pwa {
using namespace tc;

namespace {

constexpr int kTM = 128;          // tokens per tile = threads per CTA

struct TokGemmParams {
  const __nv_bfloat16 *x, *res, *W, *bias;
  const float *gamma, *beta;
  __nv_bfloat16 *sum_out, *ln_out, *y;
  float *mean, *rstd;
  long T;
  int C, Cout, NCH, n_chunks;
  float eps;
  uint32_t drop_thresh;
  float inv_keep;
  const uint32_t* seed;
};

struct TokSmem {
  uint32_t bx, br, a, w, out, total;
};
__host__ __device__ inline TokSmem tok_layout(int C, int NCH) {
  TokSmem s;
  uint32_t o = 0;
  s.bx = o; o += kTM * C * 2;                // x tile, overwritten by s
  s.br = o; o += kTM * C * 2;                // res tile, overwritten by z (row-major copy for ln_out)
  s.a = o; o += kTM * C * 2;                 // z in the UMMA canonical layout [16-byte chunk][row]
  s.w = o; o += NCH * C * 2;                 // W chunk, canonical [16-byte chunk][output channel]
  s.out = o; o += kTM * NCH * 2;             // y tile, row-major
  s.total = o;
  return s;
}

__device__ __forceinline__ uint32_t mixd(uint32_t x) {
  x ^= x >> 16; x *= 0x21f0aaadu; x ^= x >> 15; x *= 0x735a2d97u; x ^= x >> 15;
  return x;
}
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
template <typename T> __device__ __forceinline__ void unpack8(const uint4& w, float (&v)[8]) {
  const uint32_t u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) unpack2t<T>(u[i], v[2 * i], v[2 * i + 1]);
}
template <typename T> __device__ __forceinline__ uint4 pack8(const float (&v)[8]) {
  return make_uint4(pack2t<T>(v[0], v[1]), pack2t<T>(v[2], v[3]), pack2t<T>(v[4], v[5]), pack2t<T>(v[6], v[7]));
}

// T: element type of every token tensor, W and bias (bf16 or fp16; the pointers of TokGemmParams only carry the 16-bit width)
template <typename T, bool HAS_LN, bool HAS_RES, bool HAS_DROP>
__global__ void __launch_bounds__(kTM) token_gemm_kernel(TokGemmParams p) {
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_ld, bar_mma;
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) float gam_s[192], bet_s[192], bias_s[256];      // per-CTA copies: read by every thread for every tile
  const int tid = threadIdx.x, warp = tid >> 5;
  const int C = p.C, NCH = p.NCH, NC8 = C / 8;
  const TokSmem L = tok_layout(C, NCH);
  uint8_t* bx = smem + L.bx;
  uint8_t* br = smem + L.br;
  uint8_t* As = smem + L.a;
  uint8_t* Ws = smem + L.w;
  uint8_t* Os = smem + L.out;
  const int chunk = blockIdx.x % p.n_chunks;
  const int n0 = chunk * NCH;                                     // first output channel of this CTA
  const int nvalid = min(NCH, p.Cout - n0);                       // (the last chunk may be narrower; its MMA still runs NCH wide)

  // ---- once per CTA: the weight chunk in the canonical K-major layout [k chunk][output channel][16 B] ----
  for (int i = tid; i < NCH * NC8; i += kTM) {
    const int n = i / NC8, kc = i - n * NC8;
    uint4 w = make_uint4(0, 0, 0, 0);
    if (n < nvalid) w = __ldg(reinterpret_cast<const uint4*>(p.W + (size_t)(n0 + n) * C) + kc);
    *reinterpret_cast<uint4*>(Ws + (kc * NCH + n) * 16) = w;
  }
  for (int i = tid; i < C; i += kTM) {
    gam_s[i] = HAS_LN ? p.gamma[i] : 1.f;
    bet_s[i] = HAS_LN ? p.beta[i] : 0.f;
  }
  for (int i = tid; i < NCH; i += kTM) bias_s[i] = (p.bias && i < nvalid) ? to_f32(reinterpret_cast<const T*>(p.bias)[n0 + i]) : 0.f;
  if (tid == 0) {
    mbar_init(&bar_ld, 1);
    mbar_init(&bar_mma, 1);
    fence_mbar_init();
  }
  uint32_t tcols = 32;
  while ((int)tcols < NCH) tcols <<= 1;
  if (warp == 0) tmem_alloc(&tmem_base_s, tcols);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  const uint32_t idesc = make_idesc<T>(128, NCH, 0, 0);
  const uint32_t s0 = HAS_DROP ? p.seed[0] : 0u, s1 = HAS_DROP ? p.seed[1] : 0u;
  const long n_tiles = (p.T + kTM - 1) / kTM;
  const int stride = gridDim.x / p.n_chunks;
  uint32_t phase = 0;

  for (long tile = blockIdx.x / p.n_chunks; tile < n_tiles; tile += stride) {
    const long row0 = tile * kTM;
    const int rows = (int)min((long)kTM, p.T - row0);
    const uint32_t tile_bytes = (uint32_t)rows * C * 2;
    // ---- load: the x (and res) tiles are contiguous in memory: one bulk copy each ----
    if (tid == 0) {
      bulk_wait_read_all();                                       // the previous tile's bulk stores have read their buffers
      mbar_expect_tx(&bar_ld, tile_bytes * (HAS_RES ? 2u : 1u));
      bulk_g2s(bx, p.x + row0 * C, tile_bytes, &bar_ld);
      if (HAS_RES) bulk_g2s(br, p.res + row0 * C, tile_bytes, &bar_ld);
      mbar_arrive(&bar_ld);
    }
    mbar_wait(&bar_ld, phase);
    const long row = row0 + tid;
    const bool live = tid < rows;
    uint4* xr = reinterpret_cast<uint4*>(bx + (size_t)tid * C * 2);
    uint4* rr = reinterpret_cast<uint4*>(br + (size_t)tid * C * 2);
    float mean = 0.f, rstd = 1.f;
    if (live) {
      // pass 1: s = dropout(x) + res, rounded to bf16 and stored in place; row sum of the STORED values
      float sum = 0.f;
      for (int c = 0; c < NC8; ++c) {
        float v[8];
        unpack8<T>(xr[c], v);
        if (HAS_DROP) {
          const long q0 = (row * C + c * 8) >> 2;                   // same mask as pwa_dropout: one hash per 4 elements
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const long q = q0 + h;
            const uint32_t bits = mixd(mixd(s0 + (uint32_t)q * 0x9E3779B1u + (uint32_t)(q >> 32) * 0x85EBCA77u) ^ s1);
#pragma unroll
            for (int e = 0; e < 4; ++e)
              v[h * 4 + e] = ((bits >> (8 * e)) & 0xffu) >= p.drop_thresh ? v[h * 4 + e] * p.inv_keep : 0.f;
          }
          if (!HAS_RES) {                                           // dropped values rounded as pwa_dropout stores them
            const uint4 w = pack8<T>(v);
            unpack8<T>(w, v);
          }
        }
        if (HAS_RES) {
          if (HAS_DROP) {                                           // pwa_dropout rounds its output to bf16 before the add
            const uint4 w = pack8<T>(v);
            unpack8<T>(w, v);
          }
          float r[8];
          unpack8<T>(rr[c], r);
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] += r[e];
        }
        if (HAS_RES || HAS_DROP) {
          const uint4 w = pack8<T>(v);
          xr[c] = w;
          unpack8<T>(w, v);
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) sum += v[e];
      }
      if (HAS_LN) {
        mean = sum / (float)C;
        float q = 0.f;
        for (int c = 0; c < NC8; ++c) {
          float v[8];
          unpack8<T>(xr[c], v);
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const float d = v[e] - mean;
            q = fmaf(d, d, q);
          }
        }
        rstd = rsqrtf(q / (float)C + p.eps);
        if (p.mean && chunk == 0) {
          p.mean[row] = mean;
          p.rstd[row] = rstd;
        }
      }
    }
    // pass 2: z = (s - mean) * rstd * gamma + beta -> row-major copy (ln_out) and the canonical A operand
    for (int c = 0; c < NC8; ++c) {
      float v[8];
      uint4 w = make_uint4(0, 0, 0, 0);
      if (live) {
        unpack8<T>(xr[c], v);
        if (HAS_LN) {
          const float4 g0 = *reinterpret_cast<const float4*>(gam_s + c * 8), g1 = *reinterpret_cast<const float4*>(gam_s + c * 8 + 4);
          const float4 b0 = *reinterpret_cast<const float4*>(bet_s + c * 8), b1 = *reinterpret_cast<const float4*>(bet_s + c * 8 + 4);
          const float gm[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w}, bt[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = fmaf((v[e] - mean) * rstd, gm[e], bt[e]);
        }
        w = pack8<T>(v);
        if (HAS_LN) rr[c] = w;
      }
      *reinterpret_cast<uint4*>(As + (c * kTM + tid) * 16) = w;   // rows beyond the tensor feed zeros
    }
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
      if ((HAS_RES || HAS_DROP) && p.sum_out && chunk == 0) bulk_s2g(p.sum_out + row0 * C, bx, tile_bytes);
      if (HAS_LN && p.ln_out && chunk == 0) bulk_s2g(p.ln_out + row0 * C, br, tile_bytes);
      tc_fence_after();
      for (int ks = 0; ks < C / 16; ++ks) {
        const uint64_t da = make_smem_desc(smem_u32(As) + ks * 2 * (kTM * 16), kTM * 16, 128);
        const uint64_t db = make_smem_desc(smem_u32(Ws) + ks * 2 * (NCH * 16), NCH * 16, 128);
        mma_ss(tmem, da, db, idesc, ks > 0);
      }
      mma_commit(&bar_mma);
    }
    mbar_wait(&bar_mma, phase);
    tc_fence_after();
    // ---- epilogue: + bias, bf16, staged row-major, bulk stores of the output rows ----
    for (int c = 0; c < NCH / 16; ++c) {
      uint32_t r[16];
      tmem_ld16(trow + c * 16, r);
      tmem_wait_ld();
      float v[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) v[e] = __uint_as_float(r[e]);
#pragma unroll
      for (int e = 0; e < 16; ++e) v[e] += bias_s[c * 16 + e];
      uint4* dst = reinterpret_cast<uint4*>(Os + ((size_t)tid * NCH + c * 16) * 2);
      const float lo[8] = {v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]}, hi[8] = {v[8], v[9], v[10], v[11], v[12], v[13], v[14], v[15]};
      dst[0] = pack8<T>(lo);
      dst[1] = pack8<T>(hi);
    }
    tc_fence_before();
    fence_proxy_async_smem();
    __syncthreads();
    if (nvalid == p.Cout) {                                       // one chunk = whole rows: the tile is contiguous in y
      if (tid == 0) bulk_s2g(p.y + row0 * p.Cout, Os, (uint32_t)rows * p.Cout * 2);
    } else if (live) {
      bulk_s2g(p.y + row * p.Cout + n0, Os + (size_t)tid * NCH * 2, (uint32_t)nvalid * 2);
    }
    bulk_commit();
    if (tid != 0) bulk_wait_read_all();                           // (per-row stores: every thread owns its group)
    phase ^= 1;
    __syncthreads();                                              // the output staging / tiles are free for the next iteration
  }
  if (tid == 0) bulk_wait_read_all();
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, tcols);
}

template <typename T>
void (*select_kernel(bool ln, bool rs, bool dr))(TokGemmParams) {
  if (ln && rs && dr) return token_gemm_kernel<T, true, true, true>;
  if (ln && rs) return token_gemm_kernel<T, true, true, false>;
  if (ln && dr) return token_gemm_kernel<T, true, false, true>;
  if (ln) return token_gemm_kernel<T, true, false, false>;
  if (rs && dr) return token_gemm_kernel<T, false, true, true>;
  if (rs) return token_gemm_kernel<T, false, true, false>;
  if (dr) return token_gemm_kernel<T, false, false, true>;
  return token_gemm_kernel<T, false, false, false>;
}

}  // namespace

}  // namespace pwa

using namespace pwa;

extern "C" int pwa_token_gemm_supported(int C, int Cout) {
  return (C % 16 == 0 && C >= 16 && C <= 192 && Cout % 16 == 0 && Cout >= 16) ? 1 : 0;
}

extern "C" int pwa_token_gemm_fwd(const void* x, const void* res, const float* gamma, const float* beta, const void* W,
                                  const void* bias, void* sum_out, void* ln_out, void* y, float* mean, float* rstd,
                                  int64_t T, int C, int Cout, float eps, float p_drop, const void* seed_dev, void* stream) {
  return pwa_token_gemm_fwd_dt(x, res, gamma, beta, W, bias, sum_out, ln_out, y, mean, rstd, T, C, Cout, eps, p_drop, seed_dev,
                               PWA_BF16, stream);
}

extern "C" int pwa_token_gemm_fwd_dt(const void* x, const void* res, const float* gamma, const float* beta, const void* W,
                                     const void* bias, void* sum_out, void* ln_out, void* y, float* mean, float* rstd,
                                     int64_t T, int C, int Cout, float eps, float p_drop, const void* seed_dev, int dtype,
                                     void* stream) {
  PWA_CHECK_ARG(x && W && y, "pwa_token_gemm_fwd: null pointer");
  PWA_CHECK_ARG(dtype == PWA_BF16 || dtype == PWA_F16, "pwa_token_gemm_fwd: bad dtype %d (bf16 or fp16)", dtype);
  PWA_CHECK_ARG(pwa_token_gemm_supported(C, Cout), "pwa_token_gemm_fwd: need C %% 16 == 0, 16 <= C <= 192, Cout %% 16 == 0 (C=%d Cout=%d)", C, Cout);
  PWA_CHECK_ARG((gamma == nullptr) == (beta == nullptr), "pwa_token_gemm_fwd: gamma and beta go together");
  PWA_CHECK_ARG(p_drop >= 0.f && p_drop < 1.f && (p_drop == 0.f || seed_dev), "pwa_token_gemm_fwd: dropout needs seed words");
  PWA_CHECK_ARG((mean == nullptr) == (rstd == nullptr), "pwa_token_gemm_fwd: mean and rstd go together");
  if (T == 0) return PWA_OK;
  TokGemmParams p = {};
  p.x = (const __nv_bfloat16*)x; p.res = (const __nv_bfloat16*)res; p.W = (const __nv_bfloat16*)W; p.bias = (const __nv_bfloat16*)bias;
  p.gamma = gamma; p.beta = beta;
  p.sum_out = (__nv_bfloat16*)sum_out; p.ln_out = (__nv_bfloat16*)ln_out; p.y = (__nv_bfloat16*)y;
  p.mean = mean; p.rstd = rstd;
  p.T = T; p.C = C; p.Cout = Cout; p.eps = eps;
  int t = (int)(p_drop * 256.f + 0.5f);
  if (t > 255) t = 255;
  if (p_drop > 0.f && t == 0) t = 1;
  p.drop_thresh = (uint32_t)t;
  p.inv_keep = 256.f / (float)(256 - t);
  p.seed = (const uint32_t*)seed_dev;
  // output-channel chunk: the widest multiple of 16 (<= 256, one MMA) whose tiles fit twice on an SM, else once
  int nch = Cout > 256 ? 256 : Cout;
  auto fits = [&](int n, size_t budget) { return tok_layout(C, n).total + 2048 <= budget; };
  while (nch > 16 && !fits(nch, 110 * 1024)) nch -= 16;
  if (nch < 96 && Cout > nch) {                                    // too narrow for two CTAs per SM: one CTA per SM, wider chunks
    nch = Cout > 256 ? 256 : Cout;
    while (nch > 16 && !fits(nch, 220 * 1024)) nch -= 16;
  }
  PWA_CHECK_ARG(fits(nch, 220 * 1024), "pwa_token_gemm_fwd: tile does not fit shared memory (C=%d)", C);
  p.NCH = nch;
  p.n_chunks = (Cout + nch - 1) / nch;
  const TokSmem L = tok_layout(C, nch);
  const int per_sm = (int)((227 * 1024) / (L.total + 2048));
  int tcols = 32;
  while (tcols < nch) tcols <<= 1;
  int ctas = per_sm < 1 ? 1 : (per_sm > 4 ? 4 : per_sm);
  if (ctas * tcols > 512) ctas = 512 / tcols;
  long grid = 148L * ctas;
  grid -= grid % p.n_chunks;
  const long n_tiles = (T + kTM - 1) / kTM;
  if (grid > n_tiles * p.n_chunks) grid = n_tiles * p.n_chunks;
  if (grid < p.n_chunks) grid = p.n_chunks;
  const bool ln = gamma != nullptr, rs = res != nullptr, dr = p.drop_thresh != 0;
  void (*kern)(TokGemmParams) = dtype == PWA_F16 ? select_kernel<__half>(ln, rs, dr) : select_kernel<__nv_bfloat16>(ln, rs, dr);
  PWA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
  kern<<<(unsigned)grid, kTM, L.total, (cudaStream_t)stream>>>(p);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}
