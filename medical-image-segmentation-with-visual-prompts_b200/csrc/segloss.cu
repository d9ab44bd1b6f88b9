// Segmentation losses: fused Dice / focal sums forward and their gradient backward (include/pwa.h, "segmentation losses").
//
// The downstream trainer and the phase-2 trainer train the segmentation heads with MONAI's DiceLoss / FocalLoss /
// DiceFocalLoss (softmax or sigmoid, one-hot of an integer label map).  Every option of those losses reduces to four
// per-(sample, class) sums over the voxels: I = sum p*y, P = sum p (or p^2), G = sum y and F = sum focal; the losses are then
// a few torch operations on [B][K] (pwa_b200.trainer.seg_losses).  The forward reads the logits and labels once and writes
// the sums; the backward reads them once more, recomputes the activation per voxel and writes dlogits once.
//
// A thread covers runs of V consecutive voxels of one sample (V = 16 bytes of logits for K <= 8, where the K x V logits of a
// run stay in registers; one voxel for K > 8) and accumulates its sums in voxel order.  CTA (x, b) reduces its threads in a
// fixed order (warp shuffles, then warps in index order) and stores to its own slot of the workspace [S][4][B][K];
// pwa_colsum_f32 then sums the slots in index order.  No float atomics: the sums are bitwise reproducible.  S depends on
// (B, nvox) only, so the workspace query needs no GPU and no pointer.
#include <math.h>

#include "common.cuh"

namespace pwa {

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kGridUnit = 8;              // voxels per thread-run in the grid rule (the 16-bit run length)
constexpr int kCtaTarget = 148 * 2;       // CTAs over all samples: 2 per SM of a B200, one wave for K <= 8

struct SegArgs {
  int B, K;
  long nvox;
  int act, squared, focal, skip_bg, has_alpha;
  float gamma, alpha;
  int label_dt;
  int vec;        // logits (and dlogits) rows are read / written as 16-byte vectors
  int lvec;       // labels are read as vectors
};

// voxels per run: 16 bytes of logits while K <= 8 (K x 16 bytes in registers), one voxel above
template <typename T, int KB> __host__ __device__ constexpr int run_len() { return KB <= 8 ? 16 / (int)sizeof(T) : 1; }

// K <= 8: two CTAs per SM (at most 128 registers); K > 8 keeps up to 255 registers for its 2K register accumulators and K logits
template <int KB> __host__ __device__ constexpr int kMinCtas() { return KB <= 8 ? 2 : 1; }

long slots_per_sample(int B, long nvox) {
  const long runs = (nvox + kGridUnit - 1) / kGridUnit;
  long s = (runs + kThreads - 1) / kThreads;
  long cap = kCtaTarget / B;
  if (cap < 1) cap = 1;
  if (s > cap) s = cap;
  return s < 1 ? 1 : s;
}

__device__ __forceinline__ float sigmoid_f(float x) {
  if (x >= 0.f) return 1.f / (1.f + expf(-x));
  const float e = expf(x);
  return e / (1.f + e);
}

// labels of a run -> class index in [0, K), or -1 (outside [0, K): an all-zero one-hot row)
template <typename L, int V>
__device__ __forceinline__ void load_labels_t(const L* __restrict__ p, bool vec, int nval, int K, int (&t)[V]) {
  alignas(16) L buf[V];
  constexpr int BYTES = V * (int)sizeof(L);
  if (vec && BYTES >= 4) {
    if constexpr (BYTES >= 16) {
#pragma unroll
      for (int q = 0; q < BYTES / 16; ++q) reinterpret_cast<uint4*>(buf)[q] = __ldg(reinterpret_cast<const uint4*>(p) + q);
    } else if constexpr (BYTES == 8) {
      *reinterpret_cast<uint2*>(buf) = __ldg(reinterpret_cast<const uint2*>(p));
    } else if constexpr (BYTES == 4) {
      *reinterpret_cast<unsigned*>(buf) = __ldg(reinterpret_cast<const unsigned*>(p));
    }
  } else {
#pragma unroll
    for (int e = 0; e < V; ++e) buf[e] = e < nval ? p[e] : (L)0;
  }
#pragma unroll
  for (int e = 0; e < V; ++e) {
    const long v = (long)buf[e];
    t[e] = (v >= 0 && v < K) ? (int)v : -1;
  }
}

template <int V>
__device__ __forceinline__ void load_labels(const void* lab, const SegArgs& a, long off, int nval, int (&t)[V]) {
  if (a.label_dt == PWA_LABEL_U8) load_labels_t<uint8_t, V>(static_cast<const uint8_t*>(lab) + off, a.lvec, nval, a.K, t);
  else if (a.label_dt == PWA_LABEL_I32) load_labels_t<int32_t, V>(static_cast<const int32_t*>(lab) + off, a.lvec, nval, a.K, t);
  else load_labels_t<int64_t, V>(static_cast<const int64_t*>(lab) + off, a.lvec, nval, a.K, t);
}

// the K x V logits of a run (classes >= K and voxels >= nval are not read)
template <typename T, int KB, int V>
__device__ __forceinline__ void load_logits(const T* __restrict__ x, const SegArgs& a, int b, long v0, int nval, T (&xr)[KB][V]) {
#pragma unroll
  for (int k = 0; k < KB; ++k) {
    if (k >= a.K) continue;
    const T* row = x + ((long)b * a.K + k) * a.nvox + v0;
    if (V * sizeof(T) == 16 && a.vec) {
      *reinterpret_cast<uint4*>(xr[k]) = __ldg(reinterpret_cast<const uint4*>(row));
    } else {
#pragma unroll
      for (int e = 0; e < V; ++e) xr[k][e] = e < nval ? row[e] : from_f32<T>(0.f);
    }
  }
}

// per-voxel softmax statistics: (m, log s) over all K channels and over the focal channels c0 .. K-1
struct VoxelStats {
  float m, inv_s;     // activation softmax: p_k = exp(x_k - m) * inv_s
  float mf, lsf;      // focal softmax: log q_k = x_k - mf - lsf
};

template <typename T, int KB, int V>
__device__ __forceinline__ VoxelStats voxel_stats(const SegArgs& a, const T (&xr)[KB][V], int e) {
  VoxelStats st{0.f, 1.f, 0.f, 0.f};
  const bool all = a.act == PWA_ACT_SOFTMAX || (a.focal == PWA_FOCAL_SOFTMAX && !a.skip_bg);
  if (all) {
    float m = -INFINITY, s = 0.f;
#pragma unroll
    for (int k = 0; k < KB; ++k)
      if (k < a.K) m = fmaxf(m, to_f32(xr[k][e]));
#pragma unroll
    for (int k = 0; k < KB; ++k)
      if (k < a.K) s += expf(to_f32(xr[k][e]) - m);
    st.m = m;
    st.inv_s = 1.f / s;
    st.mf = m;
    st.lsf = logf(s);
  }
  if (a.focal == PWA_FOCAL_SOFTMAX && a.skip_bg) {
    float m = -INFINITY, s = 0.f;
#pragma unroll
    for (int k = 1; k < KB; ++k)
      if (k < a.K) m = fmaxf(m, to_f32(xr[k][e]));
#pragma unroll
    for (int k = 1; k < KB; ++k)
      if (k < a.K) s += expf(to_f32(xr[k][e]) - m);
    st.mf = m;
    st.lsf = logf(s);
  }
  return st;
}

__device__ __forceinline__ float activate(const SegArgs& a, const VoxelStats& st, float x) {
  return a.act == PWA_ACT_NONE ? x : a.act == PWA_ACT_SIGMOID ? sigmoid_f(x) : expf(x - st.m) * st.inv_s;
}

// softplus(z) and softplus(-z) of z = x (y = 1) or -x (y = 0): the sigmoid focal term is exp(-gamma sp(z)) * sp(-z)
__device__ __forceinline__ void softplus_pair(float z, float& sp_z, float& sp_nz) {
  const float l = log1pf(expf(-fabsf(z)));
  sp_z = fmaxf(z, 0.f) + l;
  sp_nz = fmaxf(-z, 0.f) + l;
}

__device__ __forceinline__ float alpha_factor(const SegArgs& a, bool y_or_fg) {
  return a.has_alpha ? (y_or_fg ? a.alpha : 1.f - a.alpha) : 1.f;
}

template <typename T, int KB>
__global__ void __launch_bounds__(kThreads, kMinCtas<KB>()) segloss_fwd_kernel(const T* __restrict__ x, const void* __restrict__ labels, SegArgs a,
                                                               float* __restrict__ slots) {
  constexpr int V = run_len<T, KB>();
  // I and G grow at the voxel's label class only: they live in shared memory, one column per thread (conflict-free, and each
  // column is updated by its own thread in voxel order); P and F grow at every class and stay in registers.
  extern __shared__ float col_s[];           // [2][KB][kThreads]: I, G
  float(*colI)[kThreads] = reinterpret_cast<float(*)[kThreads]>(col_s);
  float(*colG)[kThreads] = reinterpret_cast<float(*)[kThreads]>(col_s + KB * kThreads);
  __shared__ float red[kWarps][4 * KB];
  const int b = blockIdx.y, tid = threadIdx.x;
  float accP[KB], accF[KB];
#pragma unroll
  for (int k = 0; k < KB; ++k) {
    accP[k] = accF[k] = 0.f;
    colI[k][tid] = colG[k][tid] = 0.f;
  }
  const int c0 = a.skip_bg ? 1 : 0;
  const long runs = (a.nvox + V - 1) / V;
  for (long r = (long)blockIdx.x * blockDim.x + tid; r < runs; r += (long)gridDim.x * blockDim.x) {
    const long v0 = r * V;
    const int nval = a.nvox - v0 < V ? (int)(a.nvox - v0) : V;
    int t[V];
    load_labels<V>(labels, a, (long)b * a.nvox + v0, nval, t);
    alignas(16) T xr[KB][V];
    load_logits<T, KB, V>(x, a, b, v0, nval, xr);
#pragma unroll
    for (int e = 0; e < V; ++e) {
      if (e < nval) {
        const VoxelStats st = voxel_stats<T, KB, V>(a, xr, e);
        float pt = 0.f;
#pragma unroll
        for (int k = 0; k < KB; ++k) {
          if (k < a.K) {
            const float xk = to_f32(xr[k][e]);
            const bool yk = k == t[e];
            const float p = activate(a, st, xk);
            pt = yk ? p : pt;
            accP[k] += a.squared ? p * p : p;
            if (a.focal == PWA_FOCAL_SIGMOID) {
              float sp_z, sp_nz;
              softplus_pair(yk ? xk : -xk, sp_z, sp_nz);
              accF[k] += expf(-a.gamma * sp_z) * sp_nz * alpha_factor(a, yk);
            } else if (a.focal == PWA_FOCAL_SOFTMAX && yk && k >= c0) {
              const float lq = xk - st.mf - st.lsf;
              accF[k] += -alpha_factor(a, k > 0) * powf(-expm1f(lq), a.gamma) * lq;
            }
          }
        }
        if (t[e] >= 0) {
          colI[t[e]][tid] += pt;
          colG[t[e]][tid] += 1.f;
        }
      }
    }
  }
  // fixed-order CTA reduction: xor-shuffle tree in each warp, then the warps in index order
  const int lane = tid & 31, w = tid >> 5;
#pragma unroll
  for (int k = 0; k < KB; ++k) {
    if (k < a.K) {
      const float sI = warp_sum(colI[k][tid]), sP = warp_sum(accP[k]), sG = warp_sum(colG[k][tid]), sF = warp_sum(accF[k]);
      if (lane == 0) {
        red[w][k] = sI;
        red[w][KB + k] = sP;
        red[w][2 * KB + k] = sG;
        red[w][3 * KB + k] = sF;
      }
    }
  }
  __syncthreads();
  for (int j = tid; j < 4 * a.K; j += blockDim.x) {
    const int q = j / a.K, k = j - q * a.K;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < kWarps; ++i) s += red[i][q * KB + k];
    slots[(((long)blockIdx.x * 4 + q) * a.B + b) * a.K + k] = s;
  }
}

template <typename T, int KB>
__global__ void __launch_bounds__(kThreads, kMinCtas<KB>()) segloss_bwd_kernel(const T* __restrict__ x, const void* __restrict__ labels, SegArgs a,
                                                               const float* __restrict__ dsums, T* __restrict__ dx) {
  constexpr int V = run_len<T, KB>();
  __shared__ float dI[KB], dP[KB], dF[KB];
  const int b = blockIdx.y;
  for (int k = threadIdx.x; k < KB; k += blockDim.x) {
    const bool in = k < a.K;
    dI[k] = in ? dsums[((long)0 * a.B + b) * a.K + k] : 0.f;
    dP[k] = in ? dsums[((long)1 * a.B + b) * a.K + k] : 0.f;
    dF[k] = in ? dsums[((long)3 * a.B + b) * a.K + k] : 0.f;
  }
  __syncthreads();
  const int c0 = a.skip_bg ? 1 : 0;
  const long runs = (a.nvox + V - 1) / V;
  for (long r = (long)blockIdx.x * blockDim.x + threadIdx.x; r < runs; r += (long)gridDim.x * blockDim.x) {
    const long v0 = r * V;
    const int nval = a.nvox - v0 < V ? (int)(a.nvox - v0) : V;
    int t[V];
    load_labels<V>(labels, a, (long)b * a.nvox + v0, nval, t);
    alignas(16) T xr[KB][V];
    load_logits<T, KB, V>(x, a, b, v0, nval, xr);
#pragma unroll
    for (int e = 0; e < V; ++e) {
      if (e >= nval) continue;
      const VoxelStats st = voxel_stats<T, KB, V>(a, xr, e);
      // dL/dp_k = dI_k y_k + dP_k (1 or 2 p_k); the softmax Jacobian needs sum_k p_k dL/dp_k.  The softmax focal term of the
      // voxel is one class t: D = dF_t * d focal_t / d log q_t, and d log q_t / d x_j = [j == t] - q_j.
      float pg = 0.f, D = 0.f;
#pragma unroll
      for (int k = 0; k < KB; ++k) {
        if (k >= a.K) continue;
        const float xk = to_f32(xr[k][e]);
        const bool yk = k == t[e];
        if (a.act == PWA_ACT_SOFTMAX) {
          const float p = activate(a, st, xk);
          pg += p * ((yk ? dI[k] : 0.f) + dP[k] * (a.squared ? 2.f * p : 1.f));
        }
        if (a.focal == PWA_FOCAL_SOFTMAX && yk && k >= c0) {
          const float lq = xk - st.mf - st.lsf;
          const float q = expf(lq), omq = -expm1f(lq);
          // q d/dq [-(1 - q)^gamma log q] = -[(1 - q)^gamma - gamma q (1 - q)^(gamma - 1) log q]; the second part -> 0 as q -> 1
          const float second = (a.gamma == 0.f || lq == 0.f) ? 0.f : a.gamma * q * lq * powf(omq, a.gamma - 1.f);
          D = dF[k] * -alpha_factor(a, k > 0) * (powf(omq, a.gamma) - second);
        }
      }
#pragma unroll
      for (int k = 0; k < KB; ++k) {
        if (k >= a.K) continue;
        const float xk = to_f32(xr[k][e]);
        const bool yk = k == t[e];
        const float p = activate(a, st, xk);
        const float g = (yk ? dI[k] : 0.f) + dP[k] * (a.squared ? 2.f * p : 1.f);
        float d = a.act == PWA_ACT_NONE ? g : a.act == PWA_ACT_SIGMOID ? g * p * (1.f - p) : p * (g - pg);
        if (a.focal == PWA_FOCAL_SIGMOID) {
          // f(z) = sigma(-z)^gamma softplus(-z), z = +-x:  df/dz = -sigma(-z)^gamma (gamma sigma(z) softplus(-z) + sigma(-z))
          float sp_z, sp_nz;
          softplus_pair(yk ? xk : -xk, sp_z, sp_nz);
          const float dfdz = -expf(-a.gamma * sp_z) * (a.gamma * expf(-sp_nz) * sp_nz + expf(-sp_z));
          d += dF[k] * alpha_factor(a, yk) * (yk ? dfdz : -dfdz);
        } else if (a.focal == PWA_FOCAL_SOFTMAX && k >= c0) {
          const float q = expf(xk - st.mf - st.lsf);
          d += D * ((yk ? 1.f : 0.f) - q);
        }
        xr[k][e] = from_f32<T>(d);    // the gradient replaces the logit (read above, not read again), written below
      }
    }
#pragma unroll
    for (int k = 0; k < KB; ++k) {
      if (k >= a.K) continue;
      T* row = dx + ((long)b * a.K + k) * a.nvox + v0;
      if (V * sizeof(T) == 16 && a.vec) {
        *reinterpret_cast<uint4*>(row) = *reinterpret_cast<const uint4*>(xr[k]);
      } else {
#pragma unroll
        for (int e = 0; e < V; ++e)
          if (e < nval) row[e] = xr[k][e];
      }
    }
  }
}

bool float_dt(int dt) { return dt == PWA_F32 || dt == PWA_BF16 || dt == PWA_F16; }
bool label_dt_ok(int dt) { return dt == PWA_LABEL_U8 || dt == PWA_LABEL_I32 || dt == PWA_LABEL_I64; }
int label_size(int dt) { return dt == PWA_LABEL_U8 ? 1 : dt == PWA_LABEL_I32 ? 4 : 8; }

int check_shape(const char* who, const pwa_segloss* s) {
  PWA_CHECK_ARG(s != nullptr, "%s: null shape", who);
  PWA_CHECK_ARG(s->K >= 2 && s->K <= PWA_SEGLOSS_MAX_K, "%s: K=%d (2 .. %d)", who, s->K, PWA_SEGLOSS_MAX_K);
  PWA_CHECK_ARG(s->B >= 1 && s->B <= 65535, "%s: B=%d (1 .. 65535)", who, s->B);
  PWA_CHECK_ARG(s->nvox >= 1 && s->nvox <= (1LL << 40), "%s: nvox=%lld", who, (long long)s->nvox);
  PWA_CHECK_ARG(s->act == PWA_ACT_NONE || s->act == PWA_ACT_SIGMOID || s->act == PWA_ACT_SOFTMAX, "%s: act=%d", who, s->act);
  PWA_CHECK_ARG(s->squared_pred == 0 || s->squared_pred == 1, "%s: squared_pred=%d", who, s->squared_pred);
  PWA_CHECK_ARG(s->focal == PWA_FOCAL_OFF || s->focal == PWA_FOCAL_SIGMOID || s->focal == PWA_FOCAL_SOFTMAX, "%s: focal=%d", who,
                s->focal);
  PWA_CHECK_ARG(s->focal_skip_bg == 0 || (s->focal_skip_bg == 1 && s->focal == PWA_FOCAL_SOFTMAX),
                "%s: focal_skip_bg=%d is defined for the softmax focal form only", who, s->focal_skip_bg);
  const bool has_alpha = !isnan(s->alpha);
  PWA_CHECK_ARG(!has_alpha || (s->focal != PWA_FOCAL_OFF && isfinite(s->alpha)), "%s: alpha needs a focal term and a finite value", who);
  PWA_CHECK_ARG(!has_alpha || !s->focal_skip_bg, "%s: alpha is not defined for the softmax focal form without background", who);
  PWA_CHECK_ARG(s->focal == PWA_FOCAL_OFF || (isfinite(s->gamma) && s->gamma >= 0.f), "%s: gamma=%g (finite, >= 0)", who,
                (double)s->gamma);
  return PWA_OK;
}

int check_tensors(const char* who, const void* logits, int dtype, const void* labels, int label_dtype) {
  PWA_CHECK_ARG(logits != nullptr && labels != nullptr, "%s: null logits / labels", who);
  PWA_CHECK_ARG(float_dt(dtype), "%s: bad logits dtype %d", who, dtype);
  PWA_CHECK_ARG(label_dt_ok(label_dtype), "%s: bad label dtype %d", who, label_dtype);
  return PWA_OK;
}

SegArgs seg_args(const pwa_segloss* s, int dtype, int label_dtype, const void* logits, const void* labels, const void* dlogits) {
  SegArgs a;
  a.B = s->B;
  a.K = s->K;
  a.nvox = (long)s->nvox;
  a.act = s->act;
  a.squared = s->squared_pred;
  a.focal = s->focal;
  a.skip_bg = s->focal_skip_bg;
  a.has_alpha = !isnan(s->alpha);
  a.gamma = s->focal == PWA_FOCAL_OFF ? 0.f : s->gamma;
  a.alpha = a.has_alpha ? s->alpha : 0.f;
  a.label_dt = label_dtype;
  const int esz = dtype == PWA_F32 ? 4 : 2;
  const int V = s->K <= 8 ? 16 / esz : 1;
  const int lb = V * label_size(label_dtype), lalign = lb < 16 ? lb : 16;
  a.vec = V > 1 && a.nvox % V == 0 && ((uintptr_t)logits & 15) == 0 && (dlogits == nullptr || ((uintptr_t)dlogits & 15) == 0);
  a.lvec = V > 1 && a.nvox % V == 0 && ((uintptr_t)labels % lalign) == 0;
  return a;
}

template <typename T, bool FWD>
void launch_t(const void* logits, const void* labels, const SegArgs& a, float* f32, void* dx, dim3 grid, cudaStream_t st) {
  const T* x = (const T*)logits;
#define PWA_SEGLOSS_LAUNCH(KB)                                                                            \
  do {                                                                                                    \
    if (FWD) {                                                                                            \
      const int smem = 2 * KB * kThreads * (int)sizeof(float);                                            \
      if (smem > 48 * 1024)                                                                               \
        cudaFuncSetAttribute(segloss_fwd_kernel<T, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); \
      segloss_fwd_kernel<T, KB><<<grid, kThreads, smem, st>>>(x, labels, a, f32);                         \
    } else {                                                                                              \
      segloss_bwd_kernel<T, KB><<<grid, kThreads, 0, st>>>(x, labels, a, (const float*)f32, (T*)dx);      \
    }                                                                                                     \
  } while (0)
  if (a.K <= 2) PWA_SEGLOSS_LAUNCH(2);
  else if (a.K <= 4) PWA_SEGLOSS_LAUNCH(4);
  else if (a.K <= 8) PWA_SEGLOSS_LAUNCH(8);
  else if (a.K <= 16) PWA_SEGLOSS_LAUNCH(16);
  else PWA_SEGLOSS_LAUNCH(32);
#undef PWA_SEGLOSS_LAUNCH
}

template <bool FWD>
void launch(int dtype, const void* logits, const void* labels, const SegArgs& a, float* f32, void* dx, dim3 grid, cudaStream_t st) {
  if (dtype == PWA_F32) launch_t<float, FWD>(logits, labels, a, f32, dx, grid, st);
  else if (dtype == PWA_BF16) launch_t<__nv_bfloat16, FWD>(logits, labels, a, f32, dx, grid, st);
  else launch_t<__half, FWD>(logits, labels, a, f32, dx, grid, st);
}

}  // namespace

}  // namespace pwa

using namespace pwa;

extern "C" int64_t pwa_segloss_workspace_size(const pwa_segloss* s) {
  if (s == nullptr || s->B < 1 || s->B > 65535 || s->K < 2 || s->K > PWA_SEGLOSS_MAX_K || s->nvox < 1) return PWA_ERR_ARG;
  return (int64_t)slots_per_sample(s->B, (long)s->nvox) * 4 * s->B * s->K * (int64_t)sizeof(float);
}

extern "C" int pwa_segloss_fwd(const void* logits, int dtype, const void* labels, int label_dtype, const pwa_segloss* s, float* sums,
                               void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = check_shape("pwa_segloss_fwd", s);
  if (rc != PWA_OK) return rc;
  rc = check_tensors("pwa_segloss_fwd", logits, dtype, labels, label_dtype);
  if (rc != PWA_OK) return rc;
  PWA_CHECK_ARG(sums != nullptr, "pwa_segloss_fwd: null sums");
  const int64_t need = pwa_segloss_workspace_size(s);
  PWA_CHECK_ARG(workspace != nullptr && workspace_bytes >= need, "pwa_segloss_fwd: workspace of %lld bytes, %lld needed",
                (long long)workspace_bytes, (long long)need);
  const SegArgs a = seg_args(s, dtype, label_dtype, logits, labels, nullptr);
  const long S = slots_per_sample(s->B, (long)s->nvox);
  cudaStream_t st = (cudaStream_t)stream;
  launch<true>(dtype, logits, labels, a, (float*)workspace, nullptr, dim3((unsigned)S, (unsigned)s->B), st);
  PWA_CUDA_OK(cudaGetLastError());
  return pwa_colsum_f32((const float*)workspace, sums, (int)S, (int64_t)4 * s->B * s->K, stream);
}

extern "C" int pwa_segloss_bwd(const void* logits, int dtype, const void* labels, int label_dtype, const pwa_segloss* s,
                               const float* dsums, void* dlogits, void* stream) {
  int rc = check_shape("pwa_segloss_bwd", s);
  if (rc != PWA_OK) return rc;
  rc = check_tensors("pwa_segloss_bwd", logits, dtype, labels, label_dtype);
  if (rc != PWA_OK) return rc;
  PWA_CHECK_ARG(dsums != nullptr && dlogits != nullptr, "pwa_segloss_bwd: null dsums / dlogits");
  const SegArgs a = seg_args(s, dtype, label_dtype, logits, labels, dlogits);
  const long S = slots_per_sample(s->B, (long)s->nvox);
  launch<false>(dtype, logits, labels, a, (float*)dsums, dlogits, dim3((unsigned)S, (unsigned)s->B), (cudaStream_t)stream);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}
