// Relative-position bias tables (reference multi_head_attention/relative_positional_encoding.py:99-142) in the
// compact form the attention kernels consume, forward and backward, one tiny launch each:
//   T_a[h][i][j] = (E^-0.5 / 3) * sum_c weights_content_a[h][c] * enc_content_a[clamp(j - i + cap_a - 1)][c]   a in {h,w,d}
//   tok[h][i]    =  E^-0.5      * sum_c weights_token[h][c]     * enc_token[i][c]
// The reference gathers [w,w,E] embeddings, runs three einsums and an 8-D broadcast add into [1,h,N,N] on every
// forward (:101-123); here the separable tables (a few KB) are the final product.  fp32 throughout.
#include "common.cuh"

namespace pwa {

struct BiasArgs {
  const float* enc[3];
  const float* wc[3];
  const float* enc_tok;
  const float* w_tok;
  float* tab[3];        // fwd: out tables ; bwd: incoming table gradients
  float* tok;           // fwd: out ; bwd: incoming gradient
  float* denc[3];
  float* dwc[3];
  float* denc_tok;
  float* dw_tok;
  int heads, E, I;
  int ws[3], cap[3];
};

__device__ __forceinline__ int rel_index(int i, int j, int cap) {
  int r = j - i + cap - 1;
  r = r < 0 ? 0 : r;
  const int mx = 2 * (cap - 1);
  return r > mx ? mx : r;
}

// grid = (4 [three content axes + token], heads), block = 256
__global__ void __launch_bounds__(256) bias_tables_fwd_kernel(BiasArgs a) {
  extern __shared__ float sm[];                                  // per_dist [R] of this head
  const int ax = blockIdx.x, hd = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float scale = rsqrtf((float)a.E);
  if (ax < 3) {
    const int w = a.ws[ax], cap = a.cap[ax], R = 2 * cap - 1;
    for (int r = warp; r < R; r += 8) {
      float s = 0.f;
      for (int c = lane; c < a.E; c += 32) s = fmaf(a.wc[ax][hd * a.E + c], a.enc[ax][r * a.E + c], s);
      s = warp_sum(s);
      if (lane == 0) sm[r] = s * (scale / 3.f);
    }
    __syncthreads();
    for (int ij = tid; ij < w * w; ij += 256) {
      const int i = ij / w, j = ij - i * w;
      a.tab[ax][hd * w * w + ij] = sm[rel_index(i, j, cap)];
    }
  } else if (a.I > 0) {
    for (int i = warp; i < a.I; i += 8) {
      float s = 0.f;
      for (int c = lane; c < a.E; c += 32) s = fmaf(a.w_tok[hd * a.E + c], a.enc_tok[i * a.E + c], s);
      s = warp_sum(s);
      if (lane == 0) a.tok[hd * a.I + i] = s * scale;
    }
  }
}

// grid = (4, kBwdSplit): every block rebuilds the tiny dper table, then owns a slice of the output elements.
// DET: dper[h][r] is summed by one thread over the (i, j) of its distance in index order, without shared atomics (the
// only cross-thread reduction of this kernel; nothing crosses CTAs).
constexpr int kBwdSplit = 16;
// (tid: the wrapper's threadIdx.x, which carries the range its launch bounds give it)
template <bool DET>
__device__ __forceinline__ void bias_tables_bwd_body(const BiasArgs& a, const int tid) {
  extern __shared__ float sm[];                                  // dper [heads][R] (content) / unused (token)
  const int ax = blockIdx.x;
  const int gt = blockIdx.y * 256 + tid, gn = kBwdSplit * 256;   // thread id / count across the blockIdx.y slices
  const float scale = rsqrtf((float)a.E);
  if (ax < 3) {
    const int w = a.ws[ax], cap = a.cap[ax], R = 2 * cap - 1;
    const float f = scale / 3.f;
    if constexpr (DET) {
      for (int o = tid; o < a.heads * R; o += 256) {
        const int hd = o / R, r = o - hd * R;
        float s = 0.f;
        for (int ij = 0; ij < w * w; ++ij) {
          const int i = ij / w, j = ij - i * w;
          if (rel_index(i, j, cap) == r) s += a.tab[ax][hd * w * w + ij];
        }
        sm[o] = s;
      }
    } else {
      for (int o = tid; o < a.heads * R; o += 256) sm[o] = 0.f;
      __syncthreads();
      for (int o = tid; o < a.heads * w * w; o += 256) {
        const int hd = o / (w * w), ij = o - hd * w * w, i = ij / w, j = ij - i * w;
        atomicAdd(&sm[hd * R + rel_index(i, j, cap)], a.tab[ax][o]);
      }
    }
    __syncthreads();
    for (int o = gt; o < R * a.E; o += gn) {                     // d enc[r][c] = f * sum_h dper[h][r] * W[h][c]
      const int r = o / a.E, c = o - r * a.E;
      float s = 0.f;
      for (int hd = 0; hd < a.heads; ++hd) s = fmaf(sm[hd * R + r], a.wc[ax][hd * a.E + c], s);
      a.denc[ax][o] = s * f;
    }
    for (int o = gt; o < a.heads * a.E; o += gn) {               // d W[h][c] = f * sum_r dper[h][r] * enc[r][c]
      const int hd = o / a.E, c = o - hd * a.E;
      float s = 0.f;
      for (int r = 0; r < R; ++r) s = fmaf(sm[hd * R + r], a.enc[ax][r * a.E + c], s);
      a.dwc[ax][o] = s * f;
    }
  } else if (a.I > 0) {
    for (int o = gt; o < a.I * a.E; o += gn) {
      const int i = o / a.E, c = o - i * a.E;
      float s = 0.f;
      for (int hd = 0; hd < a.heads; ++hd) s = fmaf(a.tok[hd * a.I + i], a.w_tok[hd * a.E + c], s);
      a.denc_tok[o] = s * scale;
    }
    for (int o = gt; o < a.heads * a.E; o += gn) {
      const int hd = o / a.E, c = o - hd * a.E;
      float s = 0.f;
#pragma unroll 8
      for (int i = 0; i < a.I; ++i) s = fmaf(a.tok[hd * a.I + i], a.enc_tok[i * a.E + c], s);
      a.dw_tok[o] = s * scale;
    }
  }
}

__global__ void __launch_bounds__(256) bias_tables_bwd_kernel(BiasArgs a) { bias_tables_bwd_body<false>(a, threadIdx.x); }
__global__ void __launch_bounds__(256) bias_tables_bwd_det_kernel(BiasArgs a) { bias_tables_bwd_body<true>(a, threadIdx.x); }

static int check_common(const BiasArgs& a, const char* who) {
  PWA_CHECK_ARG(a.heads > 0 && a.E > 0 && a.I >= 0, "%s: bad heads/E/I", who);
  for (int x = 0; x < 3; ++x) {
    PWA_CHECK_ARG(a.enc[x] && a.wc[x] && a.tab[x], "%s: null content pointer", who);
    PWA_CHECK_ARG(a.ws[x] > 0 && a.cap[x] > 0 && a.ws[x] <= 64 && a.cap[x] <= 64, "%s: bad window/cap", who);
  }
  PWA_CHECK_ARG(a.I == 0 || (a.enc_tok && a.w_tok && a.tok), "%s: null token pointer", who);
  return PWA_OK;
}

}  // namespace pwa

using namespace pwa;

extern "C" int pwa_bias_tables_fwd(const float* enc_h, const float* enc_w, const float* enc_d, const float* wc_h,
                                   const float* wc_w, const float* wc_d, const float* enc_tok, const float* w_tok,
                                   float* th, float* tw, float* td, float* tok, int heads, int E, const int32_t ws[3],
                                   const int32_t cap[3], int I, void* stream) {
  BiasArgs a = {};
  a.enc[0] = enc_h; a.enc[1] = enc_w; a.enc[2] = enc_d;
  a.wc[0] = wc_h; a.wc[1] = wc_w; a.wc[2] = wc_d;
  a.enc_tok = enc_tok; a.w_tok = w_tok;
  a.tab[0] = th; a.tab[1] = tw; a.tab[2] = td; a.tok = tok;
  a.heads = heads; a.E = E; a.I = I;
  PWA_CHECK_ARG(ws && cap, "pwa_bias_tables_fwd: null ws/cap");
  int maxR = 1;
  for (int x = 0; x < 3; ++x) { a.ws[x] = ws[x]; a.cap[x] = cap[x]; maxR = max(maxR, 2 * cap[x] - 1); }
  int rc = check_common(a, "pwa_bias_tables_fwd");
  if (rc != PWA_OK) return rc;
  bias_tables_fwd_kernel<<<dim3(4, heads), 256, (size_t)maxR * 4, (cudaStream_t)stream>>>(a);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

static int bias_tables_bwd(const float* enc_h, const float* enc_w, const float* enc_d, const float* wc_h, const float* wc_w,
                           const float* wc_d, const float* enc_tok, const float* w_tok, const float* dth, const float* dtw,
                           const float* dtd, const float* dtok, float* denc_h, float* denc_w, float* denc_d, float* dwc_h,
                           float* dwc_w, float* dwc_d, float* denc_tok, float* dw_tok, int heads, int E, const int32_t ws[3],
                           const int32_t cap[3], int I, void* stream, bool det) {
  BiasArgs a = {};
  a.enc[0] = enc_h; a.enc[1] = enc_w; a.enc[2] = enc_d;
  a.wc[0] = wc_h; a.wc[1] = wc_w; a.wc[2] = wc_d;
  a.enc_tok = enc_tok; a.w_tok = w_tok;
  a.tab[0] = const_cast<float*>(dth); a.tab[1] = const_cast<float*>(dtw); a.tab[2] = const_cast<float*>(dtd);
  a.tok = const_cast<float*>(dtok);
  a.denc[0] = denc_h; a.denc[1] = denc_w; a.denc[2] = denc_d;
  a.dwc[0] = dwc_h; a.dwc[1] = dwc_w; a.dwc[2] = dwc_d;
  a.denc_tok = denc_tok; a.dw_tok = dw_tok;
  a.heads = heads; a.E = E; a.I = I;
  PWA_CHECK_ARG(ws && cap, "pwa_bias_tables_bwd: null ws/cap");
  int maxR = 1;
  for (int x = 0; x < 3; ++x) { a.ws[x] = ws[x]; a.cap[x] = cap[x]; maxR = max(maxR, 2 * cap[x] - 1); }
  int rc = check_common(a, "pwa_bias_tables_bwd");
  if (rc != PWA_OK) return rc;
  for (int x = 0; x < 3; ++x) PWA_CHECK_ARG(a.denc[x] && a.dwc[x], "pwa_bias_tables_bwd: null gradient pointer");
  PWA_CHECK_ARG(I == 0 || (denc_tok && dw_tok), "pwa_bias_tables_bwd: null token gradient pointer");
  (det ? bias_tables_bwd_det_kernel : bias_tables_bwd_kernel)<<<dim3(4, kBwdSplit), 256, (size_t)heads * maxR * 4, (cudaStream_t)stream>>>(a);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

extern "C" int pwa_bias_tables_bwd(const float* enc_h, const float* enc_w, const float* enc_d, const float* wc_h,
                                   const float* wc_w, const float* wc_d, const float* enc_tok, const float* w_tok,
                                   const float* dth, const float* dtw, const float* dtd, const float* dtok,
                                   float* denc_h, float* denc_w, float* denc_d, float* dwc_h, float* dwc_w, float* dwc_d,
                                   float* denc_tok, float* dw_tok, int heads, int E, const int32_t ws[3],
                                   const int32_t cap[3], int I, void* stream) {
  return bias_tables_bwd(enc_h, enc_w, enc_d, wc_h, wc_w, wc_d, enc_tok, w_tok, dth, dtw, dtd, dtok, denc_h, denc_w, denc_d,
                         dwc_h, dwc_w, dwc_d, denc_tok, dw_tok, heads, E, ws, cap, I, stream, false);
}

// Every CTA of this backward computes its outputs alone (no cross-CTA sums): the deterministic form needs no workspace.
extern "C" int64_t pwa_bias_tables_bwd_det_workspace_size(int heads, int E, const int32_t ws[3], const int32_t cap[3], int I) {
  if (heads <= 0 || E <= 0 || I < 0 || ws == nullptr || cap == nullptr) return PWA_ERR_ARG;
  return 0;
}

extern "C" int pwa_bias_tables_bwd_det(const float* enc_h, const float* enc_w, const float* enc_d, const float* wc_h,
                                       const float* wc_w, const float* wc_d, const float* enc_tok, const float* w_tok,
                                       const float* dth, const float* dtw, const float* dtd, const float* dtok,
                                       float* denc_h, float* denc_w, float* denc_d, float* dwc_h, float* dwc_w, float* dwc_d,
                                       float* denc_tok, float* dw_tok, int heads, int E, const int32_t ws[3],
                                       const int32_t cap[3], int I, void* workspace, int64_t workspace_bytes, void* stream) {
  (void)workspace;
  PWA_CHECK_ARG(workspace_bytes >= 0, "pwa_bias_tables_bwd_det: workspace_bytes=%lld", (long long)workspace_bytes);
  return bias_tables_bwd(enc_h, enc_w, enc_d, wc_h, wc_w, wc_d, enc_tok, w_tok, dth, dtw, dtd, dtok, denc_h, denc_w, denc_d,
                         dwc_h, dwc_w, dwc_d, denc_tok, dw_tok, heads, E, ws, cap, I, stream, true);
}
