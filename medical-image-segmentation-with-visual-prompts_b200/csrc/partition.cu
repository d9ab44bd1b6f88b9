// (a) pad + cyclic roll + strided window partition / reverse for channels-first 3D feature maps.
//
// Replaces F.pad + torch.roll + einops window_partition + 'b p c h w d -> b p (h w d) c'
// (reference swin_transformer/swin_block.py:163,174-178,205-214) and its inverse
// (window_reverse + roll back + crop, :228-253).  Pure byte movement: bit-exact by construction.
//
// Layouts:  x      [B][C][H][W][D]            (D contiguous)
//           tokens [B][P][N][C]               (C contiguous), P = P1*P2*P3 windows, N = wh*ww*wd
// Window (p1,p2,p3) / token (t1,t2,t3) sits at rolled-frame coordinate (t_a*P_a + p_a) -- windows
// are STRIDED -- which is padded-frame coordinate (r + shift) mod Sp and unpadded r' = that - lo.
//
// Fast kernel: one CTA owns a (batch, rolled h coordinate, window column p2, channel chunk) slab,
// i.e. ww lines of the padded map x CT channels.  It is staged through shared memory as
// S[w'][rolled d][channel word] so that BOTH global sides are fully coalesced: the x side moves
// whole D-lines, the token side moves runs of ww*wd*CT contiguous elements per window.
// All traffic is 32-bit words (one fp32 or a pair of bf16 channels); bf16 needs a 2x2 in-register
// transpose (PRMT) because x is contiguous along D and tokens along C.
#include <stdlib.h>

#include "common.cuh"

namespace pwa {

int partition_tma_run(bool is_partition, const void* src, const void* src2, void* dst, int B, int C, const pwa_geom* g,
                      const int32_t* lo, int eb, bool f16, cudaStream_t st);   // partition_tma.cu

struct PartParams {
  int B, C;
  int H, W, D;
  int Hp, Wp, Dp;
  int P1, P2, P3;
  int wh, ww, wd;
  int sh, sw, sd;
  int loh, low, lod;
  int N, P;
  int CT;        // channels per CTA chunk
  int nchunk;    // C / CT
  int pitch;     // smem row pitch in 32-bit words (odd)
  int padded;
  FastDiv div_cw, div_wwwd, div_wd, div_dq, div_ww, div_ndg;   // div_ndg: d-vector groups per line (vector kernels)
};

// ---------------------------------------------------------------------------------------------
// generic element-wise kernels (any shape / alignment).  Also the on-GPU checker of the fast path.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void partition_generic_kernel(const T* __restrict__ x, T* __restrict__ tok, PartParams p, size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int c = (int)(i % p.C);
    size_t r = i / p.C;
    int n = (int)(r % p.N);
    r /= p.N;
    int win = (int)(r % p.P);
    int b = (int)(r / p.P);
    int t3 = n % p.wd, t2 = (n / p.wd) % p.ww, t1 = n / (p.wd * p.ww);
    int p3 = win % p.P3, p2 = (win / p.P3) % p.P2, p1 = win / (p.P3 * p.P2);
    int h = (t1 * p.P1 + p1 + p.sh) % p.Hp - p.loh;
    int w = (t2 * p.P2 + p2 + p.sw) % p.Wp - p.low;
    int d = (t3 * p.P3 + p3 + p.sd) % p.Dp - p.lod;
    T v = T(0);
    if (h >= 0 && h < p.H && w >= 0 && w < p.W && d >= 0 && d < p.D)
      v = x[(((size_t)b * p.C + c) * p.H + h) * p.W * p.D + (size_t)w * p.D + d];
    tok[i] = v;
  }
}

template <typename T>
__device__ __forceinline__ T add_elem(T a, T b);
template <> __device__ __forceinline__ uint32_t add_elem<uint32_t>(uint32_t a, uint32_t b) {
  return __float_as_uint(__uint_as_float(a) + __uint_as_float(b));
}
template <> __device__ __forceinline__ uint16_t add_elem<uint16_t>(uint16_t a, uint16_t b) {
  const float fa = __uint_as_float((uint32_t)a << 16), fb = __uint_as_float((uint32_t)b << 16);
  const __nv_bfloat16 r = __float2bfloat16_rn(fa + fb);
  return *reinterpret_cast<const uint16_t*>(&r);
}
template <> __device__ __forceinline__ __half add_elem<__half>(__half a, __half b) {
  return __float2half_rn(__half2float(a) + __half2float(b));
}

template <typename T>
__global__ void reverse_generic_kernel(const T* __restrict__ tok, const T* __restrict__ tok2, T* __restrict__ x, PartParams p,
                                       size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int d = (int)(i % p.D);
    size_t r = i / p.D;
    int w = (int)(r % p.W);
    r /= p.W;
    int h = (int)(r % p.H);
    r /= p.H;
    int c = (int)(r % p.C);
    int b = (int)(r / p.C);
    // unpadded -> padded -> rolled frame (inverse of roll(-s))
    int rh = (h + p.loh - p.sh + p.Hp) % p.Hp;
    int rw = (w + p.low - p.sw + p.Wp) % p.Wp;
    int rd = (d + p.lod - p.sd + p.Dp) % p.Dp;
    int t1 = rh / p.P1, p1 = rh % p.P1;
    int t2 = rw / p.P2, p2 = rw % p.P2;
    int t3 = rd / p.P3, p3 = rd % p.P3;
    int win = (p1 * p.P2 + p2) * p.P3 + p3;
    int n = (t1 * p.ww + t2) * p.wd + t3;
    const size_t t = (((size_t)b * p.P + win) * p.N + n) * p.C + c;
    x[i] = tok2 ? add_elem<T>(tok[t], tok2[t]) : tok[t];
  }
}

// ---------------------------------------------------------------------------------------------
// fast kernels
// ---------------------------------------------------------------------------------------------
// EB = element bytes (2: bf16, words hold two adjacent channels; 4: fp32).
// grid.x = B * Hp * P2 * nchunk ; block = 256 threads ; dynamic smem = ww * Dp * pitch * 4 bytes.
template <int EB>
struct Slab {
  int b, a, p2, chunk;      // a = rolled h coordinate
  int t1, p1;               // a = t1 * P1 + p1
  int h;                    // source row in the unpadded map (may be out of range)
  __device__ __forceinline__ Slab(const PartParams& p) {
    uint32_t r = blockIdx.x;
    chunk = r % p.nchunk;
    r /= p.nchunk;
    p2 = r % p.P2;
    r /= p.P2;
    a = r % p.Hp;
    b = r / p.Hp;
    t1 = a / p.P1;
    p1 = a - t1 * p.P1;
    h = (a + p.sh) % p.Hp - p.loh;
  }
};

// word-wise add of two token words: one fp32 or a pair of bf16 / fp16 (H) (computed in fp32, rounded once: same as torch)
template <int EB, bool H = false>
__device__ __forceinline__ uint32_t add_word(uint32_t a, uint32_t b) {
  if (EB == 4) return __float_as_uint(__uint_as_float(a) + __uint_as_float(b));
  if (H) {
    const float2 fx = __half22float2(*reinterpret_cast<const __half2*>(&a)), fy = __half22float2(*reinterpret_cast<const __half2*>(&b));
    const __half2 r = __floats2half2_rn(fx.x + fy.x, fx.y + fy.y);
    return *reinterpret_cast<const uint32_t*>(&r);
  }
  const __nv_bfloat162 x = *reinterpret_cast<const __nv_bfloat162*>(&a), y = *reinterpret_cast<const __nv_bfloat162*>(&b);
  const float2 fx = __bfloat1622float2(x), fy = __bfloat1622float2(y);
  const __nv_bfloat162 r = __floats2bfloat162_rn(fx.x + fy.x, fx.y + fy.y);
  return *reinterpret_cast<const uint32_t*>(&r);
}

__device__ __forceinline__ int roll_fwd(int d, int lo, int s, int S) {  // unpadded -> rolled frame
  int r = d + lo - s;
  r += (r < 0) ? S : 0;
  r -= (r >= S) ? S : 0;
  return r;
}

template <int EB>
__global__ void __launch_bounds__(256) partition_fast_kernel(const uint32_t* __restrict__ x, uint32_t* __restrict__ tok,
                                                             PartParams p) {
  extern __shared__ uint32_t smem[];
  const Slab<EB> s(p);
  const int tid = threadIdx.x;
  constexpr int EPW = 4 / EB;              // elements per word
  const int CW = p.CT / EPW;               // channel words per token in this chunk
  const int rows = p.ww * p.Dp;

  if (p.padded) {  // slots that no source voxel reaches must read as zero padding
    for (int i = tid; i < rows * p.pitch; i += 256) smem[i] = 0u;
    __syncthreads();
  }

  // ---- phase 1: x lines -> smem.  item = (channel word, w', d word), d fastest (coalesced) ----
  const bool h_ok = s.h >= 0 && s.h < p.H;
  if (h_ok) {
    const int DQ = p.D / EPW;  // words per D line
    const int items = CW * p.ww * DQ;
    const size_t plane = (size_t)p.H * p.W * p.D;  // elements per channel
    const size_t base_b = ((size_t)s.b * p.C + (size_t)s.chunk * p.CT) * plane + (size_t)s.h * p.W * p.D;
#pragma unroll 4
    for (int i = tid; i < items; i += 256) {
      uint32_t line, dq, cw, t2;
      p.div_dq.divmod(i, line, dq);
      p.div_ww.divmod(line, cw, t2);
      int w = (int)(t2 * p.P2) + s.p2 + p.sw;
      w = (w >= p.Wp ? w - p.Wp : w) - p.low;
      if (w < 0 || w >= p.W) continue;
      if (EB == 4) {
        size_t g = base_b + (size_t)cw * plane + (size_t)w * p.D + dq;
        uint32_t v = __ldg(x + g);
        int r = roll_fwd(dq, p.lod, p.sd, p.Dp);
        smem[(t2 * p.Dp + r) * p.pitch + cw] = v;
      } else {
        // two bf16 channels (2cw, 2cw+1) x two d positions (2dq, 2dq+1): 2x2 transpose in registers
        size_t g0 = base_b + (size_t)(2 * cw) * plane + (size_t)w * p.D + 2 * dq;  // element offset, even
        uint32_t v0 = __ldg(x + (g0 >> 1));
        uint32_t v1 = __ldg(x + ((g0 + plane) >> 1));
        uint32_t lo = __byte_perm(v0, v1, 0x5410);  // (c0,d0),(c1,d0)
        uint32_t hi = __byte_perm(v0, v1, 0x7632);  // (c0,d1),(c1,d1)
        int r0 = roll_fwd(2 * dq, p.lod, p.sd, p.Dp);
        int r1 = roll_fwd(2 * dq + 1, p.lod, p.sd, p.Dp);
        smem[(t2 * p.Dp + r0) * p.pitch + cw] = lo;
        smem[(t2 * p.Dp + r1) * p.pitch + cw] = hi;
      }
    }
  }
  __syncthreads();

  // ---- phase 2: smem -> tokens.  item = (p3, w', d', channel word), channel fastest ----
  {
    const int per_win = p.ww * p.wd * CW;
    const int items = p.P3 * per_win;
    const size_t tok_stride_w = (size_t)p.C / EPW;  // words per token
    const size_t win0 = ((size_t)s.b * p.P + ((size_t)s.p1 * p.P2 + s.p2) * p.P3);
    const size_t row0 = (size_t)s.t1 * p.ww * p.wd;  // first token of this h' row inside a window
    const size_t cw0 = (size_t)s.chunk * CW;
#pragma unroll 4
    for (int i = tid; i < items; i += 256) {
      uint32_t p3, rem, tk, cw, t2, t3;
      p.div_cw.divmod(i, tk, cw);          // tk = (p3, w', d') flattened
      p.div_wwwd.divmod(tk, p3, rem);
      p.div_wd.divmod(rem, t2, t3);
      uint32_t v = smem[(t2 * p.Dp + t3 * p.P3 + p3) * p.pitch + cw];
      size_t g = ((win0 + p3) * p.N + row0 + rem) * tok_stride_w + cw0 + cw;
      tok[g] = v;
    }
  }
}

template <int EB, bool H>
__global__ void __launch_bounds__(256) reverse_fast_kernel(const uint32_t* __restrict__ tok, const uint32_t* __restrict__ tok2,
                                                           uint32_t* __restrict__ x, PartParams p) {
  extern __shared__ uint32_t smem[];
  const Slab<EB> s(p);
  const int tid = threadIdx.x;
  constexpr int EPW = 4 / EB;
  const int CW = p.CT / EPW;
  const bool h_ok = s.h >= 0 && s.h < p.H;
  if (!h_ok) return;  // this rolled row is cropped away entirely (uniform per CTA)

  // ---- phase 1: tokens -> smem (channel fastest: coalesced) ----
  {
    const int per_win = p.ww * p.wd * CW;
    const int items = p.P3 * per_win;
    const size_t tok_stride_w = (size_t)p.C / EPW;
    const size_t win0 = ((size_t)s.b * p.P + ((size_t)s.p1 * p.P2 + s.p2) * p.P3);
    const size_t row0 = (size_t)s.t1 * p.ww * p.wd;
    const size_t cw0 = (size_t)s.chunk * CW;
#pragma unroll 4
    for (int i = tid; i < items; i += 256) {
      uint32_t p3, rem, tk, cw, t2, t3;
      p.div_cw.divmod(i, tk, cw);
      p.div_wwwd.divmod(tk, p3, rem);
      p.div_wd.divmod(rem, t2, t3);
      size_t g = ((win0 + p3) * p.N + row0 + rem) * tok_stride_w + cw0 + cw;
      uint32_t v = __ldg(tok + g);
      if (tok2) v = add_word<EB, H>(v, __ldg(tok2 + g));
      smem[(t2 * p.Dp + t3 * p.P3 + p3) * p.pitch + cw] = v;
    }
  }
  __syncthreads();

  // ---- phase 2: smem -> x lines (d fastest: coalesced) ----
  {
    const int DQ = p.D / EPW;
    const int items = CW * p.ww * DQ;
    const size_t plane = (size_t)p.H * p.W * p.D;
    const size_t base_b = ((size_t)s.b * p.C + (size_t)s.chunk * p.CT) * plane + (size_t)s.h * p.W * p.D;
#pragma unroll 4
    for (int i = tid; i < items; i += 256) {
      uint32_t line, dq, cw, t2;
      p.div_dq.divmod(i, line, dq);
      p.div_ww.divmod(line, cw, t2);
      int w = (int)(t2 * p.P2) + s.p2 + p.sw;
      w = (w >= p.Wp ? w - p.Wp : w) - p.low;
      if (w < 0 || w >= p.W) continue;
      if (EB == 4) {
        int r = roll_fwd(dq, p.lod, p.sd, p.Dp);
        uint32_t v = smem[(t2 * p.Dp + r) * p.pitch + cw];
        x[base_b + (size_t)cw * plane + (size_t)w * p.D + dq] = v;
      } else {
        int r0 = roll_fwd(2 * dq, p.lod, p.sd, p.Dp);
        int r1 = roll_fwd(2 * dq + 1, p.lod, p.sd, p.Dp);
        uint32_t lo = smem[(t2 * p.Dp + r0) * p.pitch + cw];  // (c0,d0),(c1,d0)
        uint32_t hi = smem[(t2 * p.Dp + r1) * p.pitch + cw];  // (c0,d1),(c1,d1)
        uint32_t v0 = __byte_perm(lo, hi, 0x5410);            // (c0,d0),(c0,d1)
        uint32_t v1 = __byte_perm(lo, hi, 0x7632);            // (c1,d0),(c1,d1)
        size_t g0 = base_b + (size_t)(2 * cw) * plane + (size_t)w * p.D + 2 * dq;
        x[g0 >> 1] = v0;
        x[(g0 + plane) >> 1] = v1;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// vector kernels: same slab decomposition and smem tile as the word kernels above, but the x side moves
// 16-byte vectors (8 bf16 / 4 fp32 along D) and all index arithmetic is hoisted to once per warp-iteration.
// Lane mapping on the x side: bf16: lane = (channel pair & 7) + 8 * (d vector & 3)   -> 8 pairs x 64 B runs
//                             fp32: lane = (channel & 3)      + 4 * (d vector & 7)   -> 4 channels x 128 B runs
// which makes the transposing smem accesses bank-conflict free for an odd word pitch.
// Token side: a warp owns a (window p3, w') pair = wd consecutive tokens; lanes run over their channel words.
// ---------------------------------------------------------------------------------------------
constexpr int kTokK = 8;  // max 32-word chunks per (p3, w') token run

template <int EB>
struct VecCfg {
  static constexpr int EPV = 16 / EB;            // elements (d positions) per 16-byte vector
  static constexpr int CL = EB == 2 ? 8 : 4;     // channel-word lanes
  static constexpr int DL = 32 / CL;             // d-vector lanes
  static constexpr int CPW = 4 / EB;             // channels per word
};

struct TokMap {
  int soff[kTokK];
  int goff[kTokK];
  int nk;
};

__device__ __forceinline__ TokMap make_tok_map(const PartParams& p, int CW, int lane, int tok_w) {
  TokMap m;
  const int total = p.wd * CW;
  m.nk = (total + 31) / 32;
#pragma unroll
  for (int k = 0; k < kTokK; ++k) {
    const int idx = lane + 32 * k;
    const int t3 = (int)p.div_cw.div((uint32_t)idx), cw = idx - t3 * CW;
    const bool ok = idx < total;
    m.soff[k] = ok ? t3 * p.P3 * p.pitch + cw : -1;
    m.goff[k] = t3 * tok_w + cw;
  }
  return m;
}

template <int EB>
__global__ void __launch_bounds__(256) partition_vec_kernel(const uint32_t* __restrict__ x, uint32_t* __restrict__ tok,
                                                            PartParams p) {
  using V = VecCfg<EB>;
  extern __shared__ uint32_t smem[];
  const Slab<EB> s(p);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int CW = p.CT / V::CPW;
  const int rows = p.ww * p.Dp;
  if (p.padded) {
    for (int i = tid; i < rows * p.pitch; i += 256) smem[i] = 0u;
    __syncthreads();
  }
  // ---- phase 1: x lines -> smem ----
  if (s.h >= 0 && s.h < p.H) {
    const int DV = p.D / V::EPV;
    const int n_cg = (CW + V::CL - 1) / V::CL, n_dg = (DV + V::DL - 1) / V::DL;
    const int items = n_cg * p.ww * n_dg;
    const size_t plane = (size_t)p.H * p.W * p.D;
    const uint32_t* xb = x + (((size_t)s.b * p.C + (size_t)s.chunk * p.CT) * plane + (size_t)s.h * p.W * p.D) / V::CPW;
    const size_t plane_w = plane / V::CPW;                  // words per channel plane
    const int cl = lane % V::CL, dl = lane / V::CL;
    for (int it = warp; it < items; it += 8) {
      uint32_t r, dg, cg, t2;
      p.div_ndg.divmod((uint32_t)it, r, dg);
      p.div_ww.divmod(r, cg, t2);
      int w = (int)t2 * p.P2 + s.p2 + p.sw;          // < 2 * Wp
      w = (w >= p.Wp ? w - p.Wp : w) - p.low;
      const int cw = cg * V::CL + cl, dvec = dg * V::DL + dl;
      if (w < 0 || w >= p.W || cw >= CW || dvec >= DV) continue;
      int rr = roll_fwd(dvec * V::EPV, p.lod, p.sd, p.Dp);
      uint32_t* srow = smem + (t2 * p.Dp) * p.pitch + cw;
      if (EB == 4) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(xb + (size_t)cw * plane_w + (size_t)w * p.D + dvec * 4));
        const uint32_t vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          srow[rr * p.pitch] = vv[j];
          rr = (rr + 1 == p.Dp) ? 0 : rr + 1;
        }
      } else {
        const uint32_t* g0 = xb + (size_t)(2 * cw) * plane_w + ((size_t)w * p.D + dvec * 8) / 2;
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(g0));
        const uint4 b = __ldg(reinterpret_cast<const uint4*>(g0 + plane_w));
        const uint32_t av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          srow[rr * p.pitch] = __byte_perm(av[j], bv[j], 0x5410);
          rr = (rr + 1 == p.Dp) ? 0 : rr + 1;
          srow[rr * p.pitch] = __byte_perm(av[j], bv[j], 0x7632);
          rr = (rr + 1 == p.Dp) ? 0 : rr + 1;
        }
      }
    }
  }
  __syncthreads();
  // ---- phase 2: smem -> tokens ----
  {
    const int tok_w = p.C / V::CPW;
    const TokMap m = make_tok_map(p, CW, lane, tok_w);
    const size_t win0 = ((size_t)s.b * p.P + ((size_t)s.p1 * p.P2 + s.p2) * p.P3);
    const size_t row0 = (size_t)s.t1 * p.ww * p.wd;
    const size_t cw0 = (size_t)s.chunk * CW;
    const int items = p.P3 * p.ww;
    for (int it = warp; it < items; it += 8) {
      uint32_t p3, t2;
      p.div_ww.divmod((uint32_t)it, p3, t2);
      const uint32_t* sb = smem + (t2 * p.Dp + p3) * p.pitch;
      uint32_t* gb = tok + ((win0 + p3) * p.N + row0 + (size_t)t2 * p.wd) * tok_w + cw0;
#pragma unroll
      for (int k = 0; k < kTokK; ++k)
        if (k < m.nk && m.soff[k] >= 0) gb[m.goff[k]] = sb[m.soff[k]];
    }
  }
}

template <int EB, bool H>
__global__ void __launch_bounds__(256) reverse_vec_kernel(const uint32_t* __restrict__ tok, const uint32_t* __restrict__ tok2,
                                                          uint32_t* __restrict__ x, PartParams p) {
  using V = VecCfg<EB>;
  extern __shared__ uint32_t smem[];
  const Slab<EB> s(p);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int CW = p.CT / V::CPW;
  if (!(s.h >= 0 && s.h < p.H)) return;
  // ---- phase 1: tokens -> smem ----
  {
    const int tok_w = p.C / V::CPW;
    const TokMap m = make_tok_map(p, CW, lane, tok_w);
    const size_t win0 = ((size_t)s.b * p.P + ((size_t)s.p1 * p.P2 + s.p2) * p.P3);
    const size_t row0 = (size_t)s.t1 * p.ww * p.wd;
    const size_t cw0 = (size_t)s.chunk * CW;
    const int items = p.P3 * p.ww;
    for (int it = warp; it < items; it += 8) {
      uint32_t p3, t2;
      p.div_ww.divmod((uint32_t)it, p3, t2);
      uint32_t* sb = smem + (t2 * p.Dp + p3) * p.pitch;
      const size_t goff0 = ((win0 + p3) * p.N + row0 + (size_t)t2 * p.wd) * tok_w + cw0;
      const uint32_t* gb = tok + goff0;
#pragma unroll
      for (int k = 0; k < kTokK; ++k)
        if (k < m.nk && m.soff[k] >= 0) {
          uint32_t v = __ldg(gb + m.goff[k]);
          if (tok2) v = add_word<EB, H>(v, __ldg(tok2 + goff0 + m.goff[k]));
          sb[m.soff[k]] = v;
        }
    }
  }
  __syncthreads();
  // ---- phase 2: smem -> x lines ----
  {
    const int DV = p.D / V::EPV;
    const int n_cg = (CW + V::CL - 1) / V::CL, n_dg = (DV + V::DL - 1) / V::DL;
    const int items = n_cg * p.ww * n_dg;
    const size_t plane = (size_t)p.H * p.W * p.D;
    uint32_t* xb = x + (((size_t)s.b * p.C + (size_t)s.chunk * p.CT) * plane + (size_t)s.h * p.W * p.D) / V::CPW;
    const size_t plane_w = plane / V::CPW;
    const int cl = lane % V::CL, dl = lane / V::CL;
    for (int it = warp; it < items; it += 8) {
      uint32_t r, dg, cg, t2;
      p.div_ndg.divmod((uint32_t)it, r, dg);
      p.div_ww.divmod(r, cg, t2);
      int w = (int)t2 * p.P2 + s.p2 + p.sw;          // < 2 * Wp
      w = (w >= p.Wp ? w - p.Wp : w) - p.low;
      const int cw = cg * V::CL + cl, dvec = dg * V::DL + dl;
      if (w < 0 || w >= p.W || cw >= CW || dvec >= DV) continue;
      int rr = roll_fwd(dvec * V::EPV, p.lod, p.sd, p.Dp);
      const uint32_t* srow = smem + (t2 * p.Dp) * p.pitch + cw;
      if (EB == 4) {
        uint32_t vv[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          vv[j] = srow[rr * p.pitch];
          rr = (rr + 1 == p.Dp) ? 0 : rr + 1;
        }
        *reinterpret_cast<uint4*>(xb + (size_t)cw * plane_w + (size_t)w * p.D + dvec * 4) = make_uint4(vv[0], vv[1], vv[2], vv[3]);
      } else {
        uint32_t av[4], bv[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint32_t lo = srow[rr * p.pitch];
          rr = (rr + 1 == p.Dp) ? 0 : rr + 1;
          const uint32_t hi = srow[rr * p.pitch];
          rr = (rr + 1 == p.Dp) ? 0 : rr + 1;
          av[j] = __byte_perm(lo, hi, 0x5410);
          bv[j] = __byte_perm(lo, hi, 0x7632);
        }
        uint32_t* g0 = xb + (size_t)(2 * cw) * plane_w + ((size_t)w * p.D + dvec * 8) / 2;
        *reinterpret_cast<uint4*>(g0) = make_uint4(av[0], av[1], av[2], av[3]);
        *reinterpret_cast<uint4*>(g0 + plane_w) = make_uint4(bv[0], bv[1], bv[2], bv[3]);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int fill_params(PartParams& p, int B, int C, const pwa_geom* g, int use_crop_lo, int eb, bool* fast, bool* vec) {
  p.B = B; p.C = C;
  p.H = g->dims[0]; p.W = g->dims[1]; p.D = g->dims[2];
  p.Hp = g->sp[0]; p.Wp = g->sp[1]; p.Dp = g->sp[2];
  p.P1 = g->nwin[0]; p.P2 = g->nwin[1]; p.P3 = g->nwin[2];
  p.wh = g->ws[0]; p.ww = g->ws[1]; p.wd = g->ws[2];
  p.sh = g->shift[0]; p.sw = g->shift[1]; p.sd = g->shift[2];
  const int32_t* lo = (use_crop_lo & 1) ? g->crop_lo : g->data_lo;
  p.loh = lo[0]; p.low = lo[1]; p.lod = lo[2];
  p.N = g->N; p.P = g->P;
  p.padded = g->padded;
  const int epw = 4 / eb;
  // fast path needs whole 32-bit words on both sides
  bool ok = (C % epw == 0) && (p.D % epw == 0);
  // channel chunk: largest divisor of C that is <= 64 and a whole number of words
  int ct = 0;
  for (int c = (C < 64 ? C : 64); c >= epw; --c)
    if (C % c == 0 && c % epw == 0) { ct = c; break; }
  if (ct == 0) ok = false;
  if (ok) {
    p.CT = ct;
    p.nchunk = C / ct;
    int cw = ct / epw;
    p.pitch = cw | 1;  // odd word pitch: conflict-free for both access directions
    size_t smem = (size_t)p.ww * p.Dp * p.pitch * 4;
    size_t items = (size_t)p.P3 * p.ww * p.wd * cw;
    if (smem > 200 * 1024 || items >= 65536 || (size_t)cw * p.ww * (p.D / epw) >= 65536) ok = false;
    p.div_cw = FastDiv(cw);
    p.div_wwwd = FastDiv(p.ww * p.wd);
    p.div_wd = FastDiv(p.wd);
    p.div_dq = FastDiv(p.D / epw);
    p.div_ww = FastDiv(p.ww);
    const int dl = eb == 2 ? 4 : 8, dv = p.D / (16 / eb);
    p.div_ndg = FastDiv((dv + dl - 1) / dl > 0 ? (dv + dl - 1) / dl : 1);
  }
  *fast = ok;
  // vector path: whole 16-byte vectors along D, token runs that fit the per-lane offset table
  *vec = ok && ((p.D * eb) % 16 == 0) && (p.wd * (p.CT / epw) <= 32 * kTokK) &&
         ((size_t)p.H * p.W * p.D * eb) % 16 == 0;
  return 0;
}

template <int EB, bool H = false>
static int launch_vec(bool is_partition, const void* src, const void* src2, void* dst, const PartParams& p, cudaStream_t st) {
  size_t smem = (size_t)p.ww * p.Dp * p.pitch * 4;
  dim3 grid((unsigned)((size_t)p.B * p.Hp * p.P2 * p.nchunk));
  if (is_partition) {
    // (the attribute is per DEVICE: set it on every launch -- cheap, capture-safe, correct for one process driving several GPUs)
    PWA_CUDA_OK(cudaFuncSetAttribute(partition_vec_kernel<EB>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    partition_vec_kernel<EB><<<grid, 256, smem, st>>>((const uint32_t*)src, (uint32_t*)dst, p);
  } else {
    // (the attribute is per DEVICE: set it on every launch -- cheap, capture-safe, correct for one process driving several GPUs)
    PWA_CUDA_OK(cudaFuncSetAttribute(reverse_vec_kernel<EB, H>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    reverse_vec_kernel<EB, H><<<grid, 256, smem, st>>>((const uint32_t*)src, (const uint32_t*)src2, (uint32_t*)dst, p);
  }
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

template <int EB, bool H = false>
static int launch_fast(bool is_partition, const void* src, const void* src2, void* dst, const PartParams& p, cudaStream_t st) {
  size_t smem = (size_t)p.ww * p.Dp * p.pitch * 4;
  dim3 grid((unsigned)((size_t)p.B * p.Hp * p.P2 * p.nchunk));
  if (is_partition) {
    // (the attribute is per DEVICE: set it on every launch -- cheap, capture-safe, correct for one process driving several GPUs)
    PWA_CUDA_OK(cudaFuncSetAttribute(partition_fast_kernel<EB>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    partition_fast_kernel<EB><<<grid, 256, smem, st>>>((const uint32_t*)src, (uint32_t*)dst, p);
  } else {
    // (the attribute is per DEVICE: set it on every launch -- cheap, capture-safe, correct for one process driving several GPUs)
    PWA_CUDA_OK(cudaFuncSetAttribute(reverse_fast_kernel<EB, H>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    reverse_fast_kernel<EB, H><<<grid, 256, smem, st>>>((const uint32_t*)src, (const uint32_t*)src2, (uint32_t*)dst, p);
  }
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

template <typename T, typename TA = T>
static int launch_generic(bool is_partition, const void* src, const void* src2, void* dst, const PartParams& p, cudaStream_t st) {
  size_t total = is_partition ? (size_t)p.B * p.P * p.N * p.C : (size_t)p.B * p.C * p.H * p.W * p.D;
  if (total == 0) return PWA_OK;
  unsigned blocks = (unsigned)((total + 255) / 256);
  if (blocks > 148u * 32u) blocks = 148u * 32u;
  if (is_partition)
    partition_generic_kernel<T><<<blocks, 256, 0, st>>>((const T*)src, (T*)dst, p, total);
  else
    reverse_generic_kernel<TA><<<blocks, 256, 0, st>>>((const TA*)src, (const TA*)src2, (TA*)dst, p, total);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

static int run(bool is_partition, const void* src, const void* src2, void* dst, int B, int C, const pwa_geom* g,
               int use_crop_lo, int dtype, void* stream) {
  PWA_CHECK_ARG(src && dst && g, "pwa_partition/reverse: null pointer");
  PWA_CHECK_ARG(B > 0 && C > 0, "pwa_partition/reverse: bad B=%d C=%d", B, C);
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "pwa_partition/reverse: bad dtype %d", dtype);
  const int eb = dtype == PWA_F32 ? 4 : 2;
  PartParams p;
  bool fast = false, vec = false;
  fill_params(p, B, C, g, use_crop_lo, eb, &fast, &vec);
  // `use_crop_lo & 2` forces the generic kernel, `& 4` the word kernel, `& 8` the vector kernel (tests cross-check
  // the paths); otherwise the TMA-staged kernel (partition_tma.cu) takes every shape inside its envelope
  cudaStream_t st0 = (cudaStream_t)stream;
  static const bool no_tma = getenv("PWA_NO_TMA") != nullptr;
  if (!(use_crop_lo & (2 | 4 | 8)) && !no_tma) {
    const int32_t* lo = (use_crop_lo & 1) ? g->crop_lo : g->data_lo;
    const int rc = partition_tma_run(is_partition, src, src2, dst, B, C, g, lo, eb, dtype == PWA_F16, st0);
    if (rc != PWA_ERR_UNSUPPORTED) return rc;
  }
  if (use_crop_lo & 2) fast = vec = false;
  if (use_crop_lo & 4) vec = false;
  if (((uintptr_t)src | (uintptr_t)src2 | (uintptr_t)dst) & 3) fast = false;   // staged paths move aligned 32-bit words
  if (((uintptr_t)src | (uintptr_t)src2 | (uintptr_t)dst) & 15) vec = false;   // ... or aligned 16-byte vectors
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == PWA_F16 && src2) {                        // only the fused add of reverse_add depends on the 16-bit format
    if (fast && vec) return launch_vec<2, true>(false, src, src2, dst, p, st);
    if (fast) return launch_fast<2, true>(false, src, src2, dst, p, st);
    return launch_generic<uint16_t, __half>(false, src, src2, dst, p, st);
  }
  if (fast && vec) return eb == 4 ? launch_vec<4>(is_partition, src, src2, dst, p, st) : launch_vec<2>(is_partition, src, src2, dst, p, st);
  if (fast) return eb == 4 ? launch_fast<4>(is_partition, src, src2, dst, p, st) : launch_fast<2>(is_partition, src, src2, dst, p, st);
  return eb == 4 ? launch_generic<uint32_t>(is_partition, src, src2, dst, p, st)
                 : launch_generic<uint16_t>(is_partition, src, src2, dst, p, st);
}

}  // namespace pwa

extern "C" int pwa_partition(const void* x, void* tokens, int B, int C, const pwa_geom* g, int use_crop_lo, int dtype,
                             void* stream) {
  return pwa::run(true, x, nullptr, tokens, B, C, g, use_crop_lo, dtype, stream);
}

extern "C" int pwa_reverse(const void* tokens, void* x, int B, int C, const pwa_geom* g, int use_crop_lo, int dtype,
                           void* stream) {
  return pwa::run(false, tokens, nullptr, x, B, C, g, use_crop_lo, dtype, stream);
}

extern "C" int pwa_reverse_add(const void* tokens_a, const void* tokens_b, void* x, int B, int C, const pwa_geom* g,
                               int use_crop_lo, int dtype, void* stream) {
  return pwa::run(false, tokens_a, tokens_b, x, B, C, g, use_crop_lo, dtype, stream);
}
