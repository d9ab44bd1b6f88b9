// Window attention with DENSE position-bias / mask tensors: the literal argument form of the reference's
// WindowAttention.forward(q, k, v, pos_bias, mask) (multi_head_attention/window_attention.py:35-58).
//
// The block never builds those tensors here (separable bias tables and region ids feed the fused kernels), but a caller
// that holds a dense bias [.., h, n_q, n_k] or a dense 0/1 mask [.., n_q, n_k] -- any shape that broadcasts against
// [b, p, h, n_q, n_k], as torch would accept it -- gets the same semantics on the device:
//     logits[i][j] = (scale * q_i . k_j + bias[b, p, h, i, j]) * mask[b, p, h, i, j]      (mask multiplicative, BEFORE softmax)
//     out_i        = dropout(softmax_j(logits)) @ v
// Every row of q is a query (prompt rows included, as in the reference; n_q and n_k are free).  fp32 arithmetic on the
// CUDA cores, fp32, bf16 or fp16 I/O; one CTA = one (sample, window, head) with the head's K / V (or Q / dO) slices in shared
// memory, one thread per query row (forward, dQ + dbias) or per key (dK / dV): the layout of attn_f32.cu, with global
// reads of the dense tensors in place of table lookups.  Broadcast dimensions are strides of 0; the bias gradient is
// accumulated with fp32 atomics into a buffer of the bias's own (broadcast) shape.
// Dropout uses the generator of the fused kernels (csrc/attn.cuh) with n_q rows per (window, head).
#include "attn.cuh"

namespace pwa {

namespace {

constexpr int kThreadsD = 128;

struct DenseParams {
  const void *q, *k, *v, *out, *dout;
  void *o, *dq, *dk, *dv;
  const float *bias, *mask;
  float *lse, *delta, *dbias;
  int B, P, heads, nq, nk;
  int ldq, ldk, ldv;
  long bs[4], ms[4];                 // strides of bias / mask over (b, p, head, i)
  float scale;
  uint32_t drop_thresh;
  float inv_keep;
  const uint32_t* seed;
};

__device__ __forceinline__ const float* dense_row(const float* base, const long* st, int b, int w, int head, int i) {
  return base ? base + st[0] * b + st[1] * w + st[2] * head + st[3] * i : nullptr;
}

// forward: thread = query row, online softmax over the keys
template <typename T, int DH>
__global__ void __launch_bounds__(kThreadsD) attn_dense_fwd_kernel(DenseParams p) {
  extern __shared__ float sm[];
  float* Ks = sm;
  float* Vs = sm + (size_t)p.nk * DH;
  const int bw = blockIdx.x, head = blockIdx.y, b = bw / p.P, w = bw - b * p.P;
  const bool drop = p.drop_thresh != 0;
  const DropThresh dth = drop_thresh_planes(p.drop_thresh);
  const uint32_t s0 = drop ? p.seed[0] : 0u, s1 = drop ? p.seed[1] : 0u;
  for (int i = threadIdx.x; i < p.nk * DH; i += kThreadsD) {
    const int j = i / DH, d = i - j * DH;
    Ks[i] = to_f32(((const T*)p.k)[((size_t)bw * p.nk + j) * p.ldk + head * DH + d]);
    Vs[i] = to_f32(((const T*)p.v)[((size_t)bw * p.nk + j) * p.ldv + head * DH + d]);
  }
  __syncthreads();
  for (int n = threadIdx.x; n < p.nq; n += kThreadsD) {
    const size_t row = (size_t)bw * p.nq + n;
    const T* qg = (const T*)p.q + row * p.ldq + head * DH;
    float qr[DH], o[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) {
      qr[d] = to_f32(qg[d]) * p.scale;
      o[d] = 0.f;
    }
    const float* brow = dense_row(p.bias, p.bs, b, w, head, n);
    const float* mrow = dense_row(p.mask, p.ms, b, w, head, n);
    const uint32_t rhash = drop ? drop_row_hash(s0, s1, bw, p.heads, head, p.nq, n) : 0u;
    uint32_t kword = 0;
    float m = -1e30f, l = 0.f;
    for (int j = 0; j < p.nk; ++j) {
      float s = brow ? __ldg(brow + j) : 0.f;
      const float* kr = Ks + j * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) s = fmaf(qr[d], kr[d], s);
      if (mrow) s *= __ldg(mrow + j);
      if (s > m) {
        const float c = __expf(m - s);
        l *= c;
#pragma unroll
        for (int d = 0; d < DH; ++d) o[d] *= c;
        m = s;
      }
      float pr = __expf(s - m);
      l += pr;
      if (drop) {
        if ((j & 31) == 0) kword = drop_keep_word(rhash, (uint32_t)(j >> 5), dth);
        if (!drop_keep_elem(kword, (uint32_t)j)) pr = 0.f;
      }
      const float* vr = Vs + j * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) o[d] = fmaf(pr, vr[d], o[d]);
    }
    const float inv = (drop ? p.inv_keep : 1.f) / l;
    T* og = (T*)p.o + row * (size_t)(p.heads * DH) + head * DH;
#pragma unroll
    for (int d = 0; d < DH; ++d) og[d] = from_f32<T>(o[d] * inv);
    p.lse[((size_t)bw * p.heads + head) * p.nq + n] = m + __logf(l);
  }
}

// backward, pass 1: thread = query row -> dQ, delta, dbias
template <typename T, int DH>
__global__ void __launch_bounds__(kThreadsD) attn_dense_bwd_dq_kernel(DenseParams p) {
  extern __shared__ float sm[];
  float* Ks = sm;
  float* Vs = sm + (size_t)p.nk * DH;
  const int bw = blockIdx.x, head = blockIdx.y, b = bw / p.P, w = bw - b * p.P;
  const bool drop = p.drop_thresh != 0;
  const DropThresh dth = drop_thresh_planes(p.drop_thresh);
  const uint32_t s0 = drop ? p.seed[0] : 0u, s1 = drop ? p.seed[1] : 0u;
  for (int i = threadIdx.x; i < p.nk * DH; i += kThreadsD) {
    const int j = i / DH, d = i - j * DH;
    Ks[i] = to_f32(((const T*)p.k)[((size_t)bw * p.nk + j) * p.ldk + head * DH + d]);
    Vs[i] = to_f32(((const T*)p.v)[((size_t)bw * p.nk + j) * p.ldv + head * DH + d]);
  }
  __syncthreads();
  const int C = p.heads * DH;
  for (int n = threadIdx.x; n < p.nq; n += kThreadsD) {
    const size_t row = (size_t)bw * p.nq + n;
    const T* qg = (const T*)p.q + row * p.ldq + head * DH;
    const T* og = (const T*)p.out + row * (size_t)C + head * DH;
    const T* gg = (const T*)p.dout + row * (size_t)C + head * DH;
    float qr[DH], go[DH], dq[DH];
    float delta = 0.f;
#pragma unroll
    for (int d = 0; d < DH; ++d) {
      qr[d] = to_f32(qg[d]) * p.scale;
      go[d] = to_f32(gg[d]);
      delta = fmaf(go[d], to_f32(og[d]), delta);
      dq[d] = 0.f;
    }
    const size_t li = ((size_t)bw * p.heads + head) * p.nq + n;
    const float lse = p.lse[li];
    p.delta[li] = delta;
    const float* brow = dense_row(p.bias, p.bs, b, w, head, n);
    const float* mrow = dense_row(p.mask, p.ms, b, w, head, n);
    float* dbrow = p.dbias ? p.dbias + p.bs[0] * b + p.bs[1] * w + p.bs[2] * head + p.bs[3] * n : nullptr;
    const uint32_t rhash = drop ? drop_row_hash(s0, s1, bw, p.heads, head, p.nq, n) : 0u;
    uint32_t kword = 0;
    for (int j = 0; j < p.nk; ++j) {
      float s = brow ? __ldg(brow + j) : 0.f;
      const float* kr = Ks + j * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) s = fmaf(qr[d], kr[d], s);
      const float mk = mrow ? __ldg(mrow + j) : 1.f;
      s *= mk;
      const float pr = __expf(s - lse);
      float dp = 0.f;
      const float* vr = Vs + j * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) dp = fmaf(go[d], vr[d], dp);
      if (drop) {
        if ((j & 31) == 0) kword = drop_keep_word(rhash, (uint32_t)(j >> 5), dth);
        dp = drop_keep_elem(kword, (uint32_t)j) ? dp * p.inv_keep : 0.f;
      }
      const float ds = pr * (dp - delta) * mk;           // gradient of (scale q.k + bias)
      if (dbrow) atomicAdd(dbrow + j, ds);
#pragma unroll
      for (int d = 0; d < DH; ++d) dq[d] = fmaf(ds, kr[d], dq[d]);
    }
    T* dqg = (T*)p.dq + row * p.ldq + head * DH;
#pragma unroll
    for (int d = 0; d < DH; ++d) dqg[d] = from_f32<T>(dq[d] * p.scale);
  }
}

// backward, pass 2: thread = key -> dK, dV (Q and dO of the head in shared memory)
template <typename T, int DH>
__global__ void __launch_bounds__(kThreadsD) attn_dense_bwd_dkv_kernel(DenseParams p) {
  extern __shared__ float sm[];
  float* Qs = sm;
  float* Gs = sm + (size_t)p.nq * DH;
  float* lse_s = Gs + (size_t)p.nq * DH;
  float* del_s = lse_s + p.nq;
  const int bw = blockIdx.x, head = blockIdx.y, b = bw / p.P, w = bw - b * p.P;
  const bool drop = p.drop_thresh != 0;
  const DropThresh dth = drop_thresh_planes(p.drop_thresh);
  const uint32_t s0 = drop ? p.seed[0] : 0u, s1 = drop ? p.seed[1] : 0u;
  const int C = p.heads * DH;
  for (int i = threadIdx.x; i < p.nq * DH; i += kThreadsD) {
    const int n = i / DH, d = i - n * DH;
    const size_t row = (size_t)bw * p.nq + n;
    Qs[i] = to_f32(((const T*)p.q)[row * p.ldq + head * DH + d]) * p.scale;
    Gs[i] = to_f32(((const T*)p.dout)[row * (size_t)C + head * DH + d]);
  }
  for (int n = threadIdx.x; n < p.nq; n += kThreadsD) {
    const size_t li = ((size_t)bw * p.heads + head) * p.nq + n;
    lse_s[n] = p.lse[li];
    del_s[n] = p.delta[li];
  }
  __syncthreads();
  for (int j = threadIdx.x; j < p.nk; j += kThreadsD) {
    const T* kg = (const T*)p.k + ((size_t)bw * p.nk + j) * p.ldk + head * DH;
    const T* vg = (const T*)p.v + ((size_t)bw * p.nk + j) * p.ldv + head * DH;
    float kr[DH], vr[DH], dk[DH], dv[DH];
#pragma unroll
    for (int d = 0; d < DH; ++d) {
      kr[d] = to_f32(kg[d]);
      vr[d] = to_f32(vg[d]);
      dk[d] = dv[d] = 0.f;
    }
    for (int n = 0; n < p.nq; ++n) {
      const float* brow = dense_row(p.bias, p.bs, b, w, head, n);
      const float* mrow = dense_row(p.mask, p.ms, b, w, head, n);
      float s = brow ? __ldg(brow + j) : 0.f;
      const float* qr = Qs + n * DH;
      const float* go = Gs + n * DH;
#pragma unroll
      for (int d = 0; d < DH; ++d) s = fmaf(qr[d], kr[d], s);
      const float mk = mrow ? __ldg(mrow + j) : 1.f;
      s *= mk;
      const float pr = __expf(s - lse_s[n]);
      float dp = 0.f;
#pragma unroll
      for (int d = 0; d < DH; ++d) dp = fmaf(go[d], vr[d], dp);
      float pd = pr;
      if (drop) {
        const uint32_t kword = drop_keep_word(drop_row_hash(s0, s1, bw, p.heads, head, p.nq, n), (uint32_t)(j >> 5), dth);
        const bool keep = drop_keep_elem(kword, (uint32_t)j);
        pd = keep ? pr * p.inv_keep : 0.f;
        dp = keep ? dp * p.inv_keep : 0.f;
      }
      const float ds = pr * (dp - del_s[n]) * mk;
#pragma unroll
      for (int d = 0; d < DH; ++d) {
        dv[d] = fmaf(pd, go[d], dv[d]);
        dk[d] = fmaf(ds, qr[d], dk[d]);                   // (qr carries the scale)
      }
    }
    T* dkg = (T*)p.dk + ((size_t)bw * p.nk + j) * p.ldk + head * DH;
    T* dvg = (T*)p.dv + ((size_t)bw * p.nk + j) * p.ldv + head * DH;
#pragma unroll
    for (int d = 0; d < DH; ++d) {
      dkg[d] = from_f32<T>(dk[d]);
      dvg[d] = from_f32<T>(dv[d]);
    }
  }
}

template <typename T, int DH>
int launch_dense_fwd(const DenseParams& p, cudaStream_t st) {
  const size_t smem = (size_t)p.nk * DH * 2 * 4;
  PWA_CHECK_ARG(smem <= 227 * 1024, "pwa_attn_dense: n_k * head_dim too large for shared memory (%zu bytes)", smem);
  PWA_CUDA_OK(cudaFuncSetAttribute(attn_dense_fwd_kernel<T, DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  attn_dense_fwd_kernel<T, DH><<<dim3(p.B * p.P, p.heads), kThreadsD, smem, st>>>(p);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

template <typename T, int DH>
int launch_dense_bwd(const DenseParams& p, cudaStream_t st) {
  const size_t s1 = (size_t)p.nk * DH * 2 * 4, s2 = ((size_t)p.nq * DH * 2 + 2 * (size_t)p.nq) * 4;
  PWA_CHECK_ARG(s1 <= 227 * 1024 && s2 <= 227 * 1024, "pwa_attn_dense: window too large for shared memory (%zu / %zu bytes)", s1, s2);
  PWA_CUDA_OK(cudaFuncSetAttribute(attn_dense_bwd_dq_kernel<T, DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s1));
  PWA_CUDA_OK(cudaFuncSetAttribute(attn_dense_bwd_dkv_kernel<T, DH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s2));
  attn_dense_bwd_dq_kernel<T, DH><<<dim3(p.B * p.P, p.heads), kThreadsD, s1, st>>>(p);
  PWA_CUDA_OK(cudaGetLastError());
  attn_dense_bwd_dkv_kernel<T, DH><<<dim3(p.B * p.P, p.heads), kThreadsD, s2, st>>>(p);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

#define PWA_DENSE_DH(DHV, FN, ...)                                                     \
  switch (DHV) {                                                                       \
    case 3: return FN<T, 3>(__VA_ARGS__);                                              \
    case 6: return FN<T, 6>(__VA_ARGS__);                                              \
    case 8: return FN<T, 8>(__VA_ARGS__);                                              \
    case 12: return FN<T, 12>(__VA_ARGS__);                                            \
    case 16: return FN<T, 16>(__VA_ARGS__);                                            \
    case 24: return FN<T, 24>(__VA_ARGS__);                                            \
    case 32: return FN<T, 32>(__VA_ARGS__);                                            \
    case 48: return FN<T, 48>(__VA_ARGS__);                                            \
    default:                                                                           \
      set_error("pwa_attn_dense: head_dim %d not instantiated (have 3,6,8,12,16,24,32,48)", DHV); \
      return PWA_ERR_UNSUPPORTED;                                                      \
  }

template <typename T> int dense_fwd_t(const DenseParams& p, int dh, cudaStream_t st) { PWA_DENSE_DH(dh, launch_dense_fwd, p, st) }
template <typename T> int dense_bwd_t(const DenseParams& p, int dh, cudaStream_t st) { PWA_DENSE_DH(dh, launch_dense_bwd, p, st) }

int fill_params(DenseParams& p, const pwa_dense_attn* s, const float* bias, const float* mask, const char* who) {
  PWA_CHECK_ARG(s != nullptr, "%s: null shape", who);
  PWA_CHECK_ARG(s->B >= 1 && s->P >= 1 && s->heads >= 1 && s->dh >= 1 && s->nq >= 1 && s->nk >= 1, "%s: bad sizes", who);
  PWA_CHECK_ARG(s->ld_q >= s->heads * s->dh && s->ld_k >= s->heads * s->dh && s->ld_v >= s->heads * s->dh, "%s: row strides below heads * dh", who);
  PWA_CHECK_ARG(s->p_drop >= 0.f && s->p_drop < 1.f, "%s: p_drop=%g", who, (double)s->p_drop);
  p.B = s->B; p.P = s->P; p.heads = s->heads; p.nq = s->nq; p.nk = s->nk;
  p.ldq = s->ld_q; p.ldk = s->ld_k; p.ldv = s->ld_v;
  for (int i = 0; i < 4; ++i) {
    PWA_CHECK_ARG(s->bias_stride[i] >= 0 && s->mask_stride[i] >= 0, "%s: negative stride", who);
    p.bs[i] = (long)s->bias_stride[i];
    p.ms[i] = (long)s->mask_stride[i];
  }
  p.bias = bias; p.mask = mask;
  p.scale = s->scale;
  int t = (int)(s->p_drop * 256.f + 0.5f);
  if (t > 255) t = 255;
  if (s->p_drop > 0.f && t == 0) t = 1;
  p.drop_thresh = (uint32_t)t;
  p.inv_keep = 256.f / (float)(256 - t);
  p.seed = (const uint32_t*)s->seed_dev;
  PWA_CHECK_ARG(t == 0 || p.seed != nullptr, "%s: dropout needs seed_dev (two uint32 words on the device)", who);
  return PWA_OK;
}

}  // namespace

}  // namespace pwa

using namespace pwa;

extern "C" int pwa_attn_dense_fwd(const void* q, const void* k, const void* v, const float* bias, const float* mask, void* out,
                                  float* lse, const pwa_dense_attn* s, int dtype, void* stream) {
  PWA_CHECK_ARG(q && k && v && out && lse, "pwa_attn_dense_fwd: null pointer");
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "pwa_attn_dense_fwd: bad dtype %d", dtype);
  DenseParams p{};
  if (int rc = fill_params(p, s, bias, mask, "pwa_attn_dense_fwd")) return rc;
  p.q = q; p.k = k; p.v = v; p.o = out; p.lse = lse;
  cudaStream_t st = (cudaStream_t)stream;
  return dtype == PWA_F32 ? dense_fwd_t<float>(p, s->dh, st) : dtype == PWA_BF16 ? dense_fwd_t<__nv_bfloat16>(p, s->dh, st) : dense_fwd_t<__half>(p, s->dh, st);
}

extern "C" int pwa_attn_dense_bwd(const void* q, const void* k, const void* v, const float* bias, const float* mask, const void* out,
                                  const float* lse, const void* dout, void* dq, void* dk, void* dv, float* dbias, float* delta,
                                  const pwa_dense_attn* s, int dtype, void* stream) {
  PWA_CHECK_ARG(q && k && v && out && lse && dout && dq && dk && dv && delta, "pwa_attn_dense_bwd: null pointer");
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "pwa_attn_dense_bwd: bad dtype %d", dtype);
  PWA_CHECK_ARG(dbias == nullptr || bias != nullptr, "pwa_attn_dense_bwd: dbias without bias");
  DenseParams p{};
  if (int rc = fill_params(p, s, bias, mask, "pwa_attn_dense_bwd")) return rc;
  p.q = q; p.k = k; p.v = v; p.out = out; p.lse = const_cast<float*>(lse); p.dout = dout;
  p.dq = dq; p.dk = dk; p.dv = dv; p.dbias = dbias; p.delta = delta;
  cudaStream_t st = (cudaStream_t)stream;
  return dtype == PWA_F32 ? dense_bwd_t<float>(p, s->dh, st) : dtype == PWA_BF16 ? dense_bwd_t<__nv_bfloat16>(p, s->dh, st) : dense_bwd_t<__half>(p, s->dh, st);
}
