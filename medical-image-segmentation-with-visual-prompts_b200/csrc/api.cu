// C-ABI entry points of the attention path: argument validation + dispatch.
#include <stdlib.h>

#include "attn.cuh"

namespace pwa {

static int fill(AttnParams& p, const pwa_attn_shape* s, const char* who) {
  PWA_CHECK_ARG(s != nullptr, "%s: null shape", who);
  PWA_CHECK_ARG(s->B > 0 && s->P > 0 && s->C > 0 && s->heads > 0 && s->I >= 0, "%s: bad shape B=%d P=%d C=%d h=%d I=%d",
                who, s->B, s->P, s->C, s->heads, s->I);
  // same check (and message) as the reference's WindowAttention.__init__ (window_attention.py:19-22)
  PWA_CHECK_ARG(s->C % s->heads == 0, "WindowAttention: The dimension is not compatible with the number of heads!");
  PWA_CHECK_ARG(s->ws[0] > 0 && s->ws[1] > 0 && s->ws[2] > 0 && s->ws[2] <= 8, "%s: window (%d,%d,%d) unsupported (need wd <= 8)",
                who, s->ws[0], s->ws[1], s->ws[2]);
  PWA_CHECK_ARG(s->p_drop >= 0.f && s->p_drop < 1.f, "%s: p_drop=%g outside [0, 1)", who, (double)s->p_drop);
  {
    // dropout probability in steps of 1/256 (0.1 -> 26/256 = 0.1016); the kept entries are scaled by the exact inverse
    // of the QUANTISED keep rate, so the estimator stays unbiased
    int t = (int)(s->p_drop * 256.f + 0.5f);
    if (t > 255) t = 255;
    if (s->p_drop > 0.f && t == 0) t = 1;
    p.drop_thresh = (uint32_t)t;
    p.drop_planes = drop_thresh_planes(p.drop_thresh);
    p.inv_keep = 256.f / (float)(256 - t);
    p.drop_seed = (const uint32_t*)s->seed_dev;
    p.work = (unsigned int*)s->work;
    p.sel = (const uint32_t*)s->sel_table;
    p.seed_host[0] = (uint32_t)(s->seed ^ (s->offset << 32)) ^ (uint32_t)(s->offset >> 7);
    p.seed_host[1] = (uint32_t)(s->seed >> 32) ^ (uint32_t)s->offset * 0x9E3779B1u;
  }
  p.B = s->B; p.P = s->P; p.C = s->C; p.heads = s->heads; p.I = s->I;
  p.wh = s->ws[0]; p.ww = s->ws[1]; p.wd = s->ws[2];
  p.N = p.wh * p.ww * p.wd;
  p.NK = p.N + p.I;
  p.scale = s->scale;
  p.ldq = s->ld_qkv > 0 ? s->ld_qkv : s->C;
  p.ldp = s->ld_p > 0 ? s->ld_p : s->C;
  PWA_CHECK_ARG(p.ldq >= s->C && p.ldp >= s->C, "%s: row strides must be >= C", who);
#ifdef PWA_TIMELINE_BUILD
  static const int dbg = getenv("PWA_TIMELINE") != nullptr;
  p.debug = dbg;
#endif
  return PWA_OK;
}

}  // namespace pwa

using namespace pwa;

#ifdef PWA_TIMELINE_BUILD
// Debug builds only (`make TIMELINE=1`, include/pwa_debug.h): the product library neither exports this symbol nor contains
// the allocation / synchronous copy below -- its entry points never allocate or synchronise (include/pwa.h).
static void* g_fwd_timeline = nullptr;

extern "C" int pwa_debug_fwd_timeline(void* host_dst, int bytes) {
  if (!g_fwd_timeline || bytes > (1 << 20)) return 0;
  if (cudaMemcpy(host_dst, g_fwd_timeline, bytes, cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return bytes;
}
#endif

extern "C" int pwa_attn_tc_supported(const pwa_attn_shape* s, int dtype) {
  AttnParams p = {};
  if (fill(p, s, "pwa_attn_tc_supported") != PWA_OK) return 0;
  return attn_tc_supported(p, dtype) ? 1 : 0;
}

extern "C" int pwa_attn_fwd(const void* q, const void* k, const void* v, const void* kp, const void* vp, const float* th,
                            const float* tw, const float* td, const float* tok, const uint8_t* ids, void* out, float* lse,
                            const pwa_attn_shape* s, int dtype, int impl, void* stream) {
  AttnParams p = {};
  int rc = fill(p, s, "pwa_attn_fwd");
  if (rc != PWA_OK) return rc;
  PWA_CHECK_ARG(q && k && v && th && tw && td && out && lse, "pwa_attn_fwd: null pointer");
  PWA_CHECK_ARG(p.I == 0 || (kp && vp && tok), "pwa_attn_fwd: prompt tensors missing for I=%d", p.I);
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "pwa_attn_fwd: bad dtype %d", dtype);
  p.q = q; p.k = k; p.v = v; p.kp = kp; p.vp = vp;
  p.th = th; p.tw = tw; p.td = td; p.tok = tok; p.ids = ids;
  p.out = out; p.lse = lse;
  cudaStream_t st = (cudaStream_t)stream;
#ifdef PWA_TIMELINE_BUILD
  if (p.debug) {   // PWA_TIMELINE=1 (debug build): CTA 0 of the forward kernel writes clock64 stamps / cycle counters here
    static void* tl = nullptr;
    if (!tl) PWA_CUDA_OK(cudaMalloc(&tl, 1 << 20));
    PWA_CUDA_OK(cudaMemsetAsync(tl, 0, 1 << 20, st));
    p.delta = (float*)tl;
    g_fwd_timeline = tl;
  }
#endif
  const bool tc_ok = attn_tc_supported(p, dtype);
  if (impl == 2 && !tc_ok) {
    set_error("pwa_attn_fwd: tcgen05 kernel does not support this shape/dtype");
    return PWA_ERR_UNSUPPORTED;
  }
  if (impl == 2 || (impl == 0 && tc_ok)) {
    // PWA_FWD_WS=0 (test infrastructure): the round-1 kernel (four 128-thread CTAs per SM) for A/B measurements -- bf16
    // only: fp16 always runs the warp-specialised kernel (tc_ok implies that it takes the shape)
    static const int use_ws = getenv("PWA_FWD_WS") ? atoi(getenv("PWA_FWD_WS")) : 1;
    if ((use_ws || dtype == PWA_F16) && attn_ws_supported(p, dtype)) return attn_ws_forward(p, dtype, st);
    return attn_tc_forward(p, st);
  }
  return attn_f32_forward(p, dtype, st);
}

extern "C" int pwa_attn_bwd(const void* q, const void* k, const void* v, const void* kp, const void* vp, const float* th,
                            const float* tw, const float* td, const float* tok, const uint8_t* ids, const void* out,
                            const float* lse, const void* dout, void* dq, void* dk, void* dv, float* dkp, float* dvp,
                            float* dth, float* dtw, float* dtd, float* dtok, float* delta, const pwa_attn_shape* s,
                            int dtype, int impl, void* stream) {
  AttnParams p = {};
  int rc = fill(p, s, "pwa_attn_bwd");
  if (rc != PWA_OK) return rc;
  PWA_CHECK_ARG(q && k && v && th && tw && td && out && lse && dout && dq && dk && dv && dth && dtw && dtd && delta,
                "pwa_attn_bwd: null pointer");
  PWA_CHECK_ARG(p.I == 0 || (kp && vp && tok && dkp && dvp && dtok), "pwa_attn_bwd: prompt tensors missing for I=%d", p.I);
  PWA_CHECK_ARG(dtype == PWA_F32 || dtype == PWA_BF16 || dtype == PWA_F16, "pwa_attn_bwd: bad dtype %d", dtype);
  p.q = q; p.k = k; p.v = v; p.kp = kp; p.vp = vp;
  p.th = th; p.tw = tw; p.td = td; p.tok = tok; p.ids = ids;
  p.out = const_cast<void*>(out); p.lse = const_cast<float*>(lse); p.dout = dout;
  p.dq = dq; p.dk = dk; p.dv = dv; p.dkp = dkp; p.dvp = dvp;
  p.dth = dth; p.dtw = dtw; p.dtd = dtd; p.dtok = dtok; p.delta = delta;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t hh = (size_t)p.heads;
  PWA_CUDA_OK(cudaMemsetAsync(dth, 0, hh * p.wh * p.wh * 4, st));
  PWA_CUDA_OK(cudaMemsetAsync(dtw, 0, hh * p.ww * p.ww * 4, st));
  PWA_CUDA_OK(cudaMemsetAsync(dtd, 0, hh * p.wd * p.wd * 4, st));
  if (p.I > 0) {
    PWA_CUDA_OK(cudaMemsetAsync(dtok, 0, hh * p.I * 4, st));
    PWA_CUDA_OK(cudaMemsetAsync(dkp, 0, (size_t)p.B * p.I * p.C * 4, st));
    PWA_CUDA_OK(cudaMemsetAsync(dvp, 0, (size_t)p.B * p.I * p.C * 4, st));
  }
  const bool tc_ok = attn_tc_bwd_supported(p, dtype);
  if (impl == 2 && !tc_ok) {
    set_error("pwa_attn_bwd: tcgen05 kernel does not support this shape/dtype");
    return PWA_ERR_UNSUPPORTED;
  }
  if (impl == 2 || (impl == 0 && tc_ok)) return attn_tc_backward(p, dtype, st);
  return attn_f32_backward(p, dtype, st);
}
