// (b)/(c) prompted window attention with fp32 arithmetic on the CUDA cores.
//
// This is the accuracy path (fp32 within rtol 1e-4 of the reference, which itself runs true fp32
// matmuls) and the fall-back for shapes the tcgen05 kernel does not cover.  bf16 I/O is supported
// (math stays fp32).  One CTA = one (sample, window, head); K/V (content + prompt rows) of that head
// live in shared memory; each thread owns one query row (forward, dQ) or one key column (dK/dV), so
// no cross-thread reductions are needed except for the tiny bias-table gradients.
//
// Semantics (reference multi_head_attention/window_attention.py:49-58, swin_block.py:187-196):
//   logits[n][m] = (q_n . k_m * scale + bias[n][m]) * mask[n][m]       (mask multiplicative, pre-softmax)
//   bias[n][m]   = th[ih][jh] + tw[iw][jw] + td[id][jd]  for content columns, tok[m-N] for prompt columns
//   mask[n][m]   = ids[n] == ids[m] for content columns, 1 for prompt columns
//   out_n        = softmax_m(logits) @ v
#include "attn.cuh"

namespace pwa {

constexpr int kThreads = 128;
constexpr int kMaxWd = 8;

struct SmemLayout {
  // offsets in floats
  int a, b;            // two [rows][DH] tiles
  int th, tw, td, tok; // bias tables of this head
  int gth, gtw, gtd, gtok;  // gradient accumulators (dq kernel)
  int lse, delta;      // [N] each (dkv kernel)
  int ids;             // N bytes, stored at float offset
  int total;
};

__host__ __device__ inline SmemLayout make_layout(int rows_a, int rows_b, int DH, int wh, int ww, int wd, int I, int N) {
  SmemLayout L;
  int o = 0;
  L.a = o; o += rows_a * DH;
  L.b = o; o += rows_b * DH;
  L.th = o; o += wh * wh;
  L.tw = o; o += ww * ww;
  L.td = o; o += wd * wd;
  L.tok = o; o += I;
  L.gth = o; o += wh * wh;
  L.gtw = o; o += ww * ww;
  L.gtd = o; o += wd * wd;
  L.gtok = o; o += I;
  L.lse = o; o += N;
  L.delta = o; o += N;
  L.ids = o; o += (N + 3) / 4;
  L.total = o;
  return L;
}

template <typename T>
__device__ __forceinline__ const T* kv_row(const AttnParams& p, const void* content, const void* prompt, int b, int win,
                                           int j, int head, int DH) {
  if (j < p.N) return (const T*)content + (((size_t)b * p.P + win) * p.N + j) * p.ldq + head * DH;
  return (const T*)prompt + ((size_t)b * p.I + (j - p.N)) * p.ldp + head * DH;
}

__device__ __forceinline__ void load_tables(const AttnParams& p, const SmemLayout& L, float* sm, int head, int win,
                                            bool zero_grads) {
  const int tid = threadIdx.x;
  for (int i = tid; i < p.wh * p.wh; i += kThreads) sm[L.th + i] = p.th[head * p.wh * p.wh + i];
  for (int i = tid; i < p.ww * p.ww; i += kThreads) sm[L.tw + i] = p.tw[head * p.ww * p.ww + i];
  for (int i = tid; i < p.wd * p.wd; i += kThreads) sm[L.td + i] = p.td[head * p.wd * p.wd + i];
  for (int i = tid; i < p.I; i += kThreads) sm[L.tok + i] = p.tok[head * p.I + i];
  if (zero_grads) {
    for (int i = tid; i < p.wh * p.wh; i += kThreads) sm[L.gth + i] = 0.f;
    for (int i = tid; i < p.ww * p.ww; i += kThreads) sm[L.gtw + i] = 0.f;
    for (int i = tid; i < p.wd * p.wd; i += kThreads) sm[L.gtd + i] = 0.f;
    for (int i = tid; i < p.I; i += kThreads) sm[L.gtok + i] = 0.f;
  }
  uint8_t* ids_s = (uint8_t*)(sm + L.ids);
  if (p.ids)
    for (int i = tid; i < p.N; i += kThreads) ids_s[i] = p.ids[(size_t)win * p.N + i];
}

// ------------------------------------------------------------------------------------------------
// forward: thread = query row, online softmax over the N+I keys
// ------------------------------------------------------------------------------------------------
template <typename T, int DH>
__global__ void __launch_bounds__(kThreads) attn_fwd_f32_kernel(AttnParams p) {
  extern __shared__ float sm[];
  const int bw = blockIdx.x, head = blockIdx.y;
  const int b = bw / p.P, win = bw - b * p.P;
  const int tid = threadIdx.x;
  const SmemLayout L = make_layout(p.NK, p.NK, DH, p.wh, p.ww, p.wd, p.I, p.N);
  float* Ks = sm + L.a;
  float* Vs = sm + L.b;
  const uint8_t* ids_s = (const uint8_t*)(sm + L.ids);
  const bool masked = p.ids != nullptr;
  const bool drop = p.drop_thresh != 0;
  const DropThresh dth = drop_thresh_planes(p.drop_thresh);
  const uint32_t seed0 = p.drop_seed ? p.drop_seed[0] : p.seed_host[0], seed1 = p.drop_seed ? p.drop_seed[1] : p.seed_host[1];

  for (int i = tid; i < p.NK * DH; i += kThreads) {
    int j = i / DH, d = i - j * DH;
    Ks[i] = to_f32(kv_row<T>(p, p.k, p.kp, b, win, j, head, DH)[d]);
    Vs[i] = to_f32(kv_row<T>(p, p.v, p.vp, b, win, j, head, DH)[d]);
  }
  load_tables(p, L, sm, head, win, false);
  __syncthreads();

  for (int n = tid; n < p.N; n += kThreads) {
    const size_t row = (((size_t)b * p.P + win) * p.N + n);
    const T* qg = (const T*)p.q + row * p.ldq + head * DH;
    float qr[DH], o[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) {
      qr[d] = to_f32(qg[d]) * p.scale;
      o[d] = 0.f;
    }
    const int id_ = n % p.wd, iw = (n / p.wd) % p.ww, ih = n / (p.wd * p.ww);
    const int rid = masked ? ids_s[n] : 0;
    const uint32_t rhash = drop ? drop_row_hash(seed0, seed1, bw, p.heads, head, p.N, n) : 0u;
    uint32_t kword = 0;
    int kchunk = -1;
    float m = -1e30f, l = 0.f;
    auto step = [&](int j, float bias, bool keep) {
      float s = bias;
      const float* kr = Ks + j * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) s = fmaf(qr[d], kr[d], s);
      if (!keep) s = 0.f;
      if (s > m) {
        float c = __expf(m - s);
        l *= c;
#pragma unroll
        for (int d = 0; d < DH; ++d) o[d] *= c;
        m = s;
      }
      float pr = __expf(s - m);
      l += pr;                                            // the softmax denominator is not affected by dropout
      if (drop) {
        if ((j >> 5) != kchunk) {                         // one keep word per 32 keys (csrc/attn.cuh)
          kchunk = j >> 5;
          kword = drop_keep_word(rhash, (uint32_t)kchunk, dth);
        }
        if (!drop_keep_elem(kword, (uint32_t)j)) pr = 0.f;   // (kept ones are scaled once, below)
      }
      const float* vr = Vs + j * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) o[d] = fmaf(pr, vr[d], o[d]);
    };
    int j = 0;
    for (int jh = 0; jh < p.wh; ++jh) {
      const float bh = sm[L.th + ih * p.wh + jh];
      for (int jw = 0; jw < p.ww; ++jw) {
        const float bhw = bh + sm[L.tw + iw * p.ww + jw];
        for (int jd = 0; jd < p.wd; ++jd, ++j) {
          const float bias = bhw + sm[L.td + id_ * p.wd + jd];
          step(j, bias, !masked || ids_s[j] == rid);
        }
      }
    }
    for (int i = 0; i < p.I; ++i) step(p.N + i, sm[L.tok + i], true);

    const float inv = (drop ? p.inv_keep : 1.f) / l;
    T* og = (T*)p.out + row * p.C + head * DH;
#pragma unroll
    for (int d = 0; d < DH; ++d) og[d] = from_f32<T>(o[d] * inv);
    p.lse[(((size_t)b * p.P + win) * p.heads + head) * p.N + n] = m + __logf(l);
  }
}

// ------------------------------------------------------------------------------------------------
// backward, pass 1: thread = query row -> dQ, delta, bias-table gradients
// ------------------------------------------------------------------------------------------------
template <typename T, int DH>
__global__ void __launch_bounds__(kThreads) attn_bwd_dq_f32_kernel(AttnParams p) {
  extern __shared__ float sm[];
  const int bw = blockIdx.x, head = blockIdx.y;
  const int b = bw / p.P, win = bw - b * p.P;
  const int tid = threadIdx.x;
  const SmemLayout L = make_layout(p.NK, p.NK, DH, p.wh, p.ww, p.wd, p.I, p.N);
  float* Ks = sm + L.a;
  float* Vs = sm + L.b;
  const uint8_t* ids_s = (const uint8_t*)(sm + L.ids);
  const bool masked = p.ids != nullptr;
  const bool drop = p.drop_thresh != 0;
  const DropThresh dth = drop_thresh_planes(p.drop_thresh);
  const uint32_t seed0 = p.drop_seed ? p.drop_seed[0] : p.seed_host[0], seed1 = p.drop_seed ? p.drop_seed[1] : p.seed_host[1];

  for (int i = tid; i < p.NK * DH; i += kThreads) {
    int j = i / DH, d = i - j * DH;
    Ks[i] = to_f32(kv_row<T>(p, p.k, p.kp, b, win, j, head, DH)[d]);
    Vs[i] = to_f32(kv_row<T>(p, p.v, p.vp, b, win, j, head, DH)[d]);
  }
  load_tables(p, L, sm, head, win, true);
  __syncthreads();

  // every thread runs the same number of outer iterations so that the warp reductions stay convergent
  const int n_iter = (p.N + kThreads - 1) / kThreads;
  for (int it = 0; it < n_iter; ++it) {
    const int n = it * kThreads + tid;
    const bool live = n < p.N;
    const int nn = live ? n : 0;
    const size_t row = (((size_t)b * p.P + win) * p.N + nn);
    const T* qg = (const T*)p.q + row * p.ldq + head * DH;
    const T* og = (const T*)p.out + row * p.C + head * DH;
    const T* dog = (const T*)p.dout + row * p.C + head * DH;
    float qr[DH], dor[DH], dqr[DH];
    float delta = 0.f;
#pragma unroll
    for (int d = 0; d < DH; ++d) {
      qr[d] = to_f32(qg[d]) * p.scale;
      dor[d] = live ? to_f32(dog[d]) : 0.f;
      delta = fmaf(dor[d], to_f32(og[d]), delta);
      dqr[d] = 0.f;
    }
    const size_t stat = (((size_t)b * p.P + win) * p.heads + head) * p.N + nn;
    const float lse = p.lse[stat];
    if (live) p.delta[stat] = delta;
    const int id_ = nn % p.wd, iw = (nn / p.wd) % p.ww, ih = nn / (p.wd * p.ww);
    const int rid = masked ? ids_s[nn] : 0;
    const uint32_t rhash = drop ? drop_row_hash(seed0, seed1, bw, p.heads, head, p.N, nn) : 0u;
    uint32_t kword = 0;
    int kchunk = -1;

    auto grad = [&](int j, float bias, bool keep) -> float {
      float s = bias;
      const float* kr = Ks + j * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) s = fmaf(qr[d], kr[d], s);
      if (!keep) s = 0.f;
      const float pr = __expf(s - lse);
      const float* vr = Vs + j * DH;
      float dp = 0.f;
#pragma unroll
      for (int d = 0; d < DH; ++d) dp = fmaf(dor[d], vr[d], dp);
      if (drop) {   // d P = d P_dropped * mask / keep_rate ; delta = rowsum(dO * O) is unchanged
        if ((j >> 5) != kchunk) {
          kchunk = j >> 5;
          kword = drop_keep_word(rhash, (uint32_t)kchunk, dth);
        }
        dp = drop_keep_elem(kword, (uint32_t)j) ? dp * p.inv_keep : 0.f;
      }
      const float g = keep ? pr * (dp - delta) : 0.f;  // d logits / d (q.k*scale + bias) = mask
#pragma unroll
      for (int d = 0; d < DH; ++d) dqr[d] = fmaf(g, kr[d], dqr[d]);
      return g;
    };

    float acc_d[kMaxWd];
#pragma unroll
    for (int x = 0; x < kMaxWd; ++x) acc_d[x] = 0.f;
    int j = 0;
    for (int jh = 0; jh < p.wh; ++jh) {
      const float bh = sm[L.th + ih * p.wh + jh];
      float acc_h = 0.f;
      for (int jw = 0; jw < p.ww; ++jw) {
        const float bhw = bh + sm[L.tw + iw * p.ww + jw];
        float acc_w = 0.f;
#pragma unroll
        for (int jd = 0; jd < kMaxWd; ++jd) {
          if (jd < p.wd) {
            const float bias = bhw + sm[L.td + id_ * p.wd + jd];
            const float g = grad(j, bias, !masked || ids_s[j] == rid);
            acc_w += g;
            acc_d[jd] += g;
            ++j;
          }
        }
        if (live) atomicAdd(&sm[L.gtw + iw * p.ww + jw], acc_w);
        acc_h += acc_w;
      }
      if (live) atomicAdd(&sm[L.gth + ih * p.wh + jh], acc_h);
    }
#pragma unroll
    for (int jd = 0; jd < kMaxWd; ++jd)
      if (jd < p.wd && live) atomicAdd(&sm[L.gtd + id_ * p.wd + jd], acc_d[jd]);
    for (int i = 0; i < p.I; ++i) {
      float g = grad(p.N + i, sm[L.tok + i], true);
      g = warp_sum(live ? g : 0.f);
      if ((tid & 31) == 0) atomicAdd(&sm[L.gtok + i], g);
    }
    if (live) {
      T* dqg = (T*)p.dq + row * p.ldq + head * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) dqg[d] = from_f32<T>(dqr[d] * p.scale);
    }
  }
  __syncthreads();
  for (int i = tid; i < p.wh * p.wh; i += kThreads) atomicAdd(&p.dth[head * p.wh * p.wh + i], sm[L.gth + i]);
  for (int i = tid; i < p.ww * p.ww; i += kThreads) atomicAdd(&p.dtw[head * p.ww * p.ww + i], sm[L.gtw + i]);
  for (int i = tid; i < p.wd * p.wd; i += kThreads) atomicAdd(&p.dtd[head * p.wd * p.wd + i], sm[L.gtd + i]);
  for (int i = tid; i < p.I; i += kThreads) atomicAdd(&p.dtok[head * p.I + i], sm[L.gtok + i]);
}

// ------------------------------------------------------------------------------------------------
// backward, pass 2: thread = key column -> dK, dV (prompt columns accumulate over windows)
// ------------------------------------------------------------------------------------------------
template <typename T, int DH>
__global__ void __launch_bounds__(kThreads) attn_bwd_dkv_f32_kernel(AttnParams p) {
  extern __shared__ float sm[];
  const int bw = blockIdx.x, head = blockIdx.y;
  const int b = bw / p.P, win = bw - b * p.P;
  const int tid = threadIdx.x;
  const SmemLayout L = make_layout(p.N, p.N, DH, p.wh, p.ww, p.wd, p.I, p.N);
  float* Qs = sm + L.a;
  float* dOs = sm + L.b;
  const uint8_t* ids_s = (const uint8_t*)(sm + L.ids);
  const bool masked = p.ids != nullptr;
  const bool drop = p.drop_thresh != 0;
  const DropThresh dth = drop_thresh_planes(p.drop_thresh);
  const uint32_t seed0 = p.drop_seed ? p.drop_seed[0] : p.seed_host[0], seed1 = p.drop_seed ? p.drop_seed[1] : p.seed_host[1];

  for (int i = tid; i < p.N * DH; i += kThreads) {
    int n = i / DH, d = i - n * DH;
    const size_t row = (((size_t)b * p.P + win) * p.N + n);
    Qs[i] = to_f32(((const T*)p.q)[row * p.ldq + head * DH + d]) * p.scale;
    dOs[i] = to_f32(((const T*)p.dout)[row * p.C + head * DH + d]);
  }
  const size_t stat0 = (((size_t)b * p.P + win) * p.heads + head) * p.N;
  for (int i = tid; i < p.N; i += kThreads) {
    sm[L.lse + i] = p.lse[stat0 + i];
    sm[L.delta + i] = p.delta[stat0 + i];
  }
  load_tables(p, L, sm, head, win, false);
  __syncthreads();

  for (int j = tid; j < p.NK; j += kThreads) {
    const bool content = j < p.N;
    const T* kg = kv_row<T>(p, p.k, p.kp, b, win, j, head, DH);
    const T* vg = kv_row<T>(p, p.v, p.vp, b, win, j, head, DH);
    float kr[DH], vr[DH], dkr[DH], dvr[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) {
      kr[d] = to_f32(kg[d]);
      vr[d] = to_f32(vg[d]);
      dkr[d] = 0.f;
      dvr[d] = 0.f;
    }
    const int jd = j % p.wd, jw = (j / p.wd) % p.ww, jh = content ? j / (p.wd * p.ww) : 0;
    const int cid = (masked && content) ? ids_s[j] : -1;
    const float tokb = content ? 0.f : sm[L.tok + (j - p.N)];
    uint32_t dbits = 0;
    int n = 0;
    for (int ih = 0; ih < p.wh; ++ih) {
      const float bh = content ? sm[L.th + ih * p.wh + jh] : tokb;
      for (int iw = 0; iw < p.ww; ++iw) {
        const float bhw = content ? bh + sm[L.tw + iw * p.ww + jw] : tokb;
        for (int id_ = 0; id_ < p.wd; ++id_, ++n) {
          const float bias = content ? bhw + sm[L.td + id_ * p.wd + jd] : tokb;
          const float* qr = Qs + n * DH;
          const float* dor = dOs + n * DH;
          float s = bias;
#pragma unroll
          for (int d = 0; d < DH; ++d) s = fmaf(qr[d], kr[d], s);
          const bool keep = cid < 0 || ids_s[n] == cid;
          if (!keep) s = 0.f;
          const float pr = __expf(s - sm[L.lse + n]);
          float dp = 0.f;
#pragma unroll
          for (int d = 0; d < DH; ++d) dp = fmaf(dor[d], vr[d], dp);
          float prd = pr;
          if (drop) {
            // (this kernel walks along queries with one thread per key: a keep word per element -- the fp32-math path
            //  trades speed for simplicity here; the tcgen05 backward transposes 32x32 bit tiles instead)
            const uint32_t kword = drop_keep_word(drop_row_hash(seed0, seed1, bw, p.heads, head, p.N, n), (uint32_t)j >> 5, dth);
            const float kf = drop_keep_elem(kword, (uint32_t)j) ? p.inv_keep : 0.f;
            prd *= kf;
            dp *= kf;
          }
#pragma unroll
          for (int d = 0; d < DH; ++d) dvr[d] = fmaf(prd, dor[d], dvr[d]);
          const float g = keep ? pr * (dp - sm[L.delta + n]) : 0.f;
#pragma unroll
          for (int d = 0; d < DH; ++d) dkr[d] = fmaf(g, qr[d], dkr[d]);
        }
      }
    }
    if (content) {
      const size_t row = (((size_t)b * p.P + win) * p.N + j);
      T* dkg = (T*)p.dk + row * p.ldq + head * DH;
      T* dvg = (T*)p.dv + row * p.ldq + head * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) {
        dkg[d] = from_f32<T>(dkr[d]);
        dvg[d] = from_f32<T>(dvr[d]);
      }
    } else {
      float* dkg = p.dkp + ((size_t)b * p.I + (j - p.N)) * p.C + head * DH;
      float* dvg = p.dvp + ((size_t)b * p.I + (j - p.N)) * p.C + head * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) {
        atomicAdd(dkg + d, dkr[d]);
        atomicAdd(dvg + d, dvr[d]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// host dispatch
// ------------------------------------------------------------------------------------------------
template <typename T, int DH>
static int launch_fwd(const AttnParams& p, cudaStream_t st) {
  SmemLayout L = make_layout(p.NK, p.NK, DH, p.wh, p.ww, p.wd, p.I, p.N);
  size_t smem = (size_t)L.total * 4;
  PWA_CHECK_ARG(smem <= 227 * 1024, "attention window too large for shared memory (%zu bytes)", smem);
  PWA_CUDA_OK(cudaFuncSetAttribute(attn_fwd_f32_kernel<T, DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  attn_fwd_f32_kernel<T, DH><<<dim3(p.B * p.P, p.heads), kThreads, smem, st>>>(p);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

template <typename T, int DH>
static int launch_bwd(const AttnParams& p, cudaStream_t st) {
  SmemLayout L1 = make_layout(p.NK, p.NK, DH, p.wh, p.ww, p.wd, p.I, p.N);
  SmemLayout L2 = make_layout(p.N, p.N, DH, p.wh, p.ww, p.wd, p.I, p.N);
  size_t s1 = (size_t)L1.total * 4, s2 = (size_t)L2.total * 4;
  PWA_CHECK_ARG(s1 <= 227 * 1024, "attention window too large for shared memory (%zu bytes)", s1);
  PWA_CUDA_OK(cudaFuncSetAttribute(attn_bwd_dq_f32_kernel<T, DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s1));
  PWA_CUDA_OK(cudaFuncSetAttribute(attn_bwd_dkv_f32_kernel<T, DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s2));
  attn_bwd_dq_f32_kernel<T, DH><<<dim3(p.B * p.P, p.heads), kThreads, s1, st>>>(p);
  PWA_CUDA_OK(cudaGetLastError());
  attn_bwd_dkv_f32_kernel<T, DH><<<dim3(p.B * p.P, p.heads), kThreads, s2, st>>>(p);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

#define PWA_DISPATCH_DH(DHV, FN, ...)                                   \
  switch (DHV) {                                                        \
    case 3: return FN<T, 3>(__VA_ARGS__);                               \
    case 6: return FN<T, 6>(__VA_ARGS__);                               \
    case 8: return FN<T, 8>(__VA_ARGS__);                               \
    case 12: return FN<T, 12>(__VA_ARGS__);                             \
    case 16: return FN<T, 16>(__VA_ARGS__);                             \
    case 24: return FN<T, 24>(__VA_ARGS__);                             \
    case 32: return FN<T, 32>(__VA_ARGS__);                             \
    case 48: return FN<T, 48>(__VA_ARGS__);                             \
    default:                                                            \
      set_error("head_dim %d not instantiated (have 3,6,8,12,16,24,32,48)", DHV); \
      return PWA_ERR_UNSUPPORTED;                                       \
  }

template <typename T> static int fwd_t(const AttnParams& p, int dh, cudaStream_t st) { PWA_DISPATCH_DH(dh, launch_fwd, p, st) }
template <typename T> static int bwd_t(const AttnParams& p, int dh, cudaStream_t st) { PWA_DISPATCH_DH(dh, launch_bwd, p, st) }

int attn_f32_forward(const AttnParams& p, int dtype, cudaStream_t st) {
  const int dh = p.C / p.heads;
  return dtype == PWA_F32 ? fwd_t<float>(p, dh, st) : dtype == PWA_BF16 ? fwd_t<__nv_bfloat16>(p, dh, st) : fwd_t<__half>(p, dh, st);
}

int attn_f32_backward(const AttnParams& p, int dtype, cudaStream_t st) {
  const int dh = p.C / p.heads;
  return dtype == PWA_F32 ? bwd_t<float>(p, dh, st) : dtype == PWA_BF16 ? bwd_t<__nv_bfloat16>(p, dh, st) : bwd_t<__half>(p, dh, st);
}

}  // namespace pwa
