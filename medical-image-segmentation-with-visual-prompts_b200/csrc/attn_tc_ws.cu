// (b) fused prompted window attention forward, warp-specialised (tcgen05 + TMEM, bf16 or fp16 I/O).
//
// One persistent CTA per SM (768 threads = 24 warps, 6 per scheduler) = one fixed head, walking (sample, window) pairs.
// The softmax of this path is bound by the MUFU pipe (one ex2 per logit, 16 / clk / SM), so everything else is taken off
// the threads that compute exponentials and hidden behind them with mbarrier hand-offs:
//     warps 0-15        softmax: group = warp / 8 owns query tile 0 / 1 (128 rows = 128 TMEM lanes) of the current window,
//                       set = (warp / 4) % 2 takes alternate UNITS of 64 keys of the group's stream, lane quadrant = warp % 4.
//                       Per unit: wait for S, tcgen05.ld -> exp2 (FFMA2 + MUFU + pack) -> shift mask (one PRMT per packed
//                       pair) -> dropout (one AND per pair) -> tcgen05.st of the bf16 probabilities over the consumed S
//                       columns; per window: drain O, normalise, write the output rows and the log-sum-exp.
//     warps 16 / 17     MMA issuer of group 0 / 1 (warp-uniform loop, elect.sync picks the issuing lane so that descriptors
//                       stay in uniform registers): S = Q'.K'^T of unit n + 2 is issued while the group still works on
//                       unit n (three S buffers per group in TMEM), O += P.[V | 1] as soon as a unit's P is stored.  A
//                       thread's tcgen05.mma instructions execute in issue order, so S(n + 3) may overwrite the buffer
//                       whose P fed PV(n) without a further barrier.  The next window is opened with a NON-blocking
//                       try_wait on its operand barrier, so PV MMAs of the current window are never held back by it.
//     warps 18-19       idle (they round the CTA up to 6 warps per scheduler)
//     warps 20-23       staging (the highest ids: the scheduler prefers them): the NEXT windows' Q / K / [V | 1] head slices
//                       go global -> shared memory as 8-byte cp.async pieces straight into the UMMA canonical layouts (up
//                       to three operand sets in flight), |q|^2 per row and max |k|^2 (stabiliser), region ids and the
//                       PRMT selector table of the window (one cp.async.bulk of a host-built table, pwa_attn_sel_table);
//                       they also fetch the next window index from the per-head work counter.
// The arithmetic: no row-max pass (norm-bound stabiliser with an exact-max sweep as the rare fallback), no online
// rescaling, relative-position bias folded into the QK^T MMA through one-hot / table columns, multiplicative pre-softmax
// shift mask (window_attention.py:49-58), ones column of V for the softmax denominator, bit-sliced dropout keep words
// (csrc/attn.cuh).  TMEM: per group 3 x 64 columns of S / P plus 1-2 O accumulators.
#include <type_traits>

#include "attn.cuh"
#include "tc_common.cuh"

namespace pwa {
using namespace tc;

namespace {

constexpr int kN = 256;           // content tokens per window
constexpr int kIds = 28;          // region ids 0..26 and 100 (-> 27)
// Warp roles (the scheduler favours high warp ids among eligible warps).
constexpr int kThreadsW = 768;    // 24 warps = 6 per scheduler
constexpr int kStage0 = 20;       // staging warps 20-23: the HIGHEST ids -- they are few, on the critical path of every window,
                                  // and must not wait for issue slots behind sixteen always-eligible softmax warps
constexpr int kIssue0 = 16;       // issuer warps 16 (group 0) and 17 (group 1); warps 18, 19 idle
constexpr int kSoft0 = 0;         // softmax warps 0-15: group = warp / 8, set = (warp / 4) % 2, TMEM lane quadrant
                                  // = warp % 4.  The two SETS of a group take alternate units of the group's unit stream, so
                                  // that four softmax warps per scheduler feed the MUFU pipe (one warp alone issues an ex2
                                  // only every ~8 clk and leaves the pipe idle between its unpack / pack instructions)
constexpr int kStageThreads = 128;
constexpr int kUK = 64;           // keys per unit
constexpr int kNSB = 3;           // S / P buffers per group
constexpr float kMaxBoundW = 40.f;

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// volatile: keeps the 32 exponentials of a chunk back to back in program order.  Left to itself ptxas pairs every pack
// with the two MUFUs just in front of it, and the pack then waits out the MUFU latency 16 times per chunk (ncu: the F2FP
// lines carried as many stall samples as the MUFU lines).
__device__ __forceinline__ float ex2f_v(float x) {
  float y;
  asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t prmt3(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}
__device__ __forceinline__ int id_slot_w(uint32_t id) { return id < (uint32_t)(kIds - 1) ? (int)id : kIds - 1; }
__device__ __forceinline__ void ffma2w(float& d0, float& d1, float a0, float a1, float b, float c) {
  unsigned long long a, bb, cc, d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %1};" : "=l"(bb) : "f"(b));
  asm("mov.b64 %0, {%1, %1};" : "=l"(cc) : "f"(c));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(bb), "l"(cc));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(d));
}
__device__ __forceinline__ void fadd2w(float& s0, float& s1, float a0, float a1) {
  unsigned long long a, s, d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(s) : "f"(s0), "f"(s1));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(s), "l"(a));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(s0), "=f"(s1) : "l"(d));
}

__device__ __forceinline__ uint32_t hadd2_bf16(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("add.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t hadd2_f16(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("add.rn.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
template <typename T> __device__ __forceinline__ uint32_t hadd2t(uint32_t a, uint32_t b) {
  return std::is_same<T, __half>::value ? hadd2_f16(a, b) : hadd2_bf16(a, b);
}

// Stabiliser of the element type.  P = exp2(S c - mb) with mb an upper bound of the row's logits (norm bound, or the exact
// row maximum after the sweep) is rounded to T before the PV MMA.  bf16 has fp32's exponent range: a row whose largest P
// is 2^-80 still normalises.  fp16 flushes below 2^-24 (normal from 2^-14), so the fp16 kernel forms P = exp2(S c - mb + 10)
// (largest P <= 2^10: a 32-key partial sum of the dropout denominator stays <= 2^15 < 65504) and sweeps for the exact row
// maximum as soon as the bound may sit more than 24 binades above it: the row's largest P is then >= 2^(10 - 24) = 2^-14,
// a normal fp16 number, and whatever still flushes lies below the rounding error of that largest term.
template <typename T> struct WsStab {
  static constexpr float shift = 0.f, max_gap = 2.f * kMaxBoundW;
};
template <> struct WsStab<__half> {
  static constexpr float shift = 10.f, max_gap = 24.f;
};
// Dropout on the 16 packed pairs of a 32-key chunk + the chunk's share of the softmax denominator (the undropped values,
// after the shift mask).  The ALU pipe (shifts, logic, PRMT) is what saturates in the dropout variants (ncu: 64 % busy next
// to 25 % on the FMA pipe), so the sum is formed where it is cheapest there: four pairs are first added as packed bf16 on
// the FMA pipe (HADD2.BF16; partial sums of <= 4 probabilities, 2^-9 relative each, averaging out over the row's 40
// groups) and only every fourth pair is unpacked into the fp32 accumulators.
template <typename T, int G = 0>
__device__ __forceinline__ void drop_apply16w(uint32_t (&pk)[16], uint32_t kw, float& s0, float& s1) {
  if constexpr (G < 16) {
    const uint32_t part = hadd2t<T>(hadd2t<T>(pk[G], pk[G + 1]), hadd2t<T>(pk[G + 2], pk[G + 3]));
    float f0, f1;
    unpack2t<T>(part, f0, f1);
    fadd2w(s0, s1, f0, f1);
    pk[G] &= drop_pair_mask<G>(kw);
    pk[G + 1] &= drop_pair_mask<G + 1>(kw);
    pk[G + 2] &= drop_pair_mask<G + 2>(kw);
    pk[G + 3] &= drop_pair_mask<G + 3>(kw);
    drop_apply16w<T, G + 4>(pk, kw, s0, s1);
  }
}

template <int DH> struct WCfg {
  static constexpr int DHP = (DH + 1 + 15) / 16 * 16;      // V / O width (PV MMA N) incl. the ones column at DH
  static constexpr int NDC = DHP / 8;
  static constexpr int KS = (DH + 4 + 15) / 16;            // k-steps of the staged [q | onehot_d] operand
  static constexpr int NOB = DHP <= 32 ? 2 : 1;            // O accumulators per group
  static constexpr int GC = kNSB * kUK + NOB * DHP;        // TMEM columns per group
  static_assert(2 * GC <= 512, "TMEM column budget");
};

struct WsHeader {
  int bw;          // (sample * P + window) of this operand set, -1 = no more work
  int exact;       // 1: some row's stabiliser bound is loose -> exact row-max sweep first
  float kmax;      // max |k| over the window's keys (content + prompt) of this head
  int next_bw;
};

struct WsSmem {
  uint32_t qaug, kaug, rowb;                                // shared by all windows
  uint32_t q, k, v, sel, ids, qn2, hdr, part, opnd_bytes;   // per operand buffer
  uint32_t opnd0;
  int opb;
  uint32_t total;
};

__host__ __device__ inline WsSmem ws_layout(int KS, int DHP, int NKT, bool masked) {
  WsSmem s;
  uint32_t o = 0;
  s.q = o; o += KS * 2 * kN * 16;
  s.k = o; o += KS * 2 * NKT * 16;
  s.v = o; o += NKT * DHP * 2;
  s.sel = o; o += masked ? kIds * (kN / 4) * 4 : 0;
  s.ids = o; o += kN;
  s.qn2 = o; o += kN * 4;
  s.hdr = o; o += 32;
  s.part = o; o += 2 * kN * 4;                              // per (set, query row): partial softmax denominator / row maximum
  s.opnd_bytes = (o + 127) & ~127u;
  uint32_t sh = 0;
  s.qaug = sh; sh += 2 * kN * 16;
  s.kaug = sh; sh += 2 * NKT * 16;
  s.rowb = sh; sh += kN * 4;
  sh = (sh + 127) & ~127u;
  s.opnd0 = sh;
  s.opb = (sh + 3 * s.opnd_bytes <= 200u * 1024u) ? 3 : ((sh + 2 * s.opnd_bytes <= 200u * 1024u) ? 2 : 1);
  s.total = sh + s.opb * s.opnd_bytes;
  return s;
}

template <int DH, typename T>
__device__ __forceinline__ void load_row_w(const T* src, T (&dst)[DH]) {
  if constexpr (DH % 4 == 0) {
    const uint2* s2 = reinterpret_cast<const uint2*>(src);
    uint2* d2 = reinterpret_cast<uint2*>(dst);
#pragma unroll
    for (int i = 0; i < DH / 4; ++i) d2[i] = __ldg(s2 + i);
  } else {
#pragma unroll
    for (int i = 0; i < DH; ++i) dst[i] = src[i];
  }
}
template <int DH, typename T>
__device__ __forceinline__ float sumsq_w(const T (&r)[DH]) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < DH; ++i) {
    const float v = to_f32(r[i]);
    s = fmaf(v, v, s);
  }
  return s;
}
// staged K-dim layout of one head: [real DH | up to 4 extra columns | zero pad] -> KS k-steps of 16
template <int DH, int KS, typename T>
__device__ __forceinline__ void store_chunks_w(uint8_t* base, uint32_t chunk_stride, int row, const T (&real)[DH],
                                               const T (&extra)[4], int n_extra) {
#pragma unroll
  for (int c = 0; c < KS * 2; ++c) {
    __align__(16) T tmp[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int col = c * 8 + e;
      const int x = col - DH;
      T v = from_f32<T>(0.f);
      if (col < DH) v = real[col < DH ? col : 0];
      else if (x < 4 && x < n_extra) v = extra[x & 3];
      tmp[e] = v;
    }
    *reinterpret_cast<uint4*>(base + c * chunk_stride + row * 16) = *reinterpret_cast<const uint4*>(tmp);
  }
}

__device__ __forceinline__ void stage_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kStageThreads) : "memory"); }

// cycle accounting of CTA 0 (make TIMELINE=1, PWA_TIMELINE=1 in the environment; tools/ws_profile.py): every role adds
// the clocks it spends per phase to private counters and writes them out at the end of the kernel
#ifdef PWA_TIMELINE_BUILD
#define WS_PROF_DECL(n) long long prof_[n] = {}; long long prof_t_ = clock64()
#define WS_PROF(i) do { const long long t_ = clock64(); prof_[i] += t_ - prof_t_; prof_t_ = t_; } while (0)
#define WS_PROF_OUT(base, n) do { if (p.debug && p.delta && blockIdx.x == 0) { long long* o_ = reinterpret_cast<long long*>(p.delta) + (base); for (int i_ = 0; i_ < (n); ++i_) o_[i_] = prof_[i_]; } } while (0)
#else
#define WS_PROF_DECL(n) do { } while (0)
#define WS_PROF(i) do { } while (0)
#define WS_PROF_OUT(base, n) do { } while (0)
#endif

// bSFull: 6 per group, indexed by unit % 6 -- a set waits only for its own (every second) unit, and with one barrier per
// S buffer it would skip a phase between two waits, which a parity wait cannot tell apart; unit % 6 is always the same set
enum { bOpFull = 0, bOpFree = 3, bSFull = 6, bPReady = 18, bOFull = 24, bOFree = 28, bLsum = 32, kNumBarsW = 38 };

template <int DH, bool MASKED, bool DROP, typename T>
__global__ void __launch_bounds__(kThreadsW, 1) attn_fwd_ws_kernel(AttnParams p) {
  constexpr int DHP = WCfg<DH>::DHP, NDC = WCfg<DH>::NDC, KS = WCfg<DH>::KS, NOB = WCfg<DH>::NOB, GC = WCfg<DH>::GC;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar[kNumBarsW];
  __shared__ uint32_t tmem_base_s;
  __shared__ uint32_t kmax_w[3][4];
  __shared__ float tab_s[16 * 16 + 4 * 4 + 128 + 4];            // th | tw (wh + ww <= 16) | td (wd <= 4) | tok (I <= 128) | max tok

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NKT = kN + p.I;
  const WsSmem L = ws_layout(KS, DHP, NKT, MASKED);
  const int OPB = L.opb;
  uint8_t* Qa = smem + L.qaug;
  uint8_t* Ka = smem + L.kaug;
  float* rowb_s = reinterpret_cast<float*>(smem + L.rowb);
  const int head = blockIdx.x % p.heads;
  const float inv_scale = 1.f / p.scale;
  const float c2 = p.scale * 1.4426950408889634f;          // logits -> log2 domain
  const T one = from_f32<T>(1.f), zero = from_f32<T>(0.f);
  const int n_units = (NKT + kUK - 1) / kUK;
  const int last_nk = NKT - kUK * (n_units - 1);            // 64 or 32
  const int n_pairs = p.B * p.P;
  const int stride = gridDim.x / p.heads;

  // ---- once per CTA: bias tables of this head -> smem, window-independent halves of Q' and K', per-row bias bound ----
  float* th_s = tab_s;
  float* tw_s = th_s + p.wh * p.wh;
  float* td_s = tw_s + p.ww * p.ww;
  float* tok_s = td_s + p.wd * p.wd;
  for (int i = tid; i < p.wh * p.wh; i += kThreadsW) th_s[i] = p.th[head * p.wh * p.wh + i];
  for (int i = tid; i < p.ww * p.ww; i += kThreadsW) tw_s[i] = p.tw[head * p.ww * p.ww + i];
  for (int i = tid; i < p.wd * p.wd; i += kThreadsW) td_s[i] = p.td[head * p.wd * p.wd + i];
  for (int i = tid; i < p.I; i += kThreadsW) tok_s[i] = p.tok[head * p.I + i];
  __syncthreads();
  if (warp == 0) {
    float bt = -1e30f;
    for (int j = lane; j < p.I; j += 32) bt = fmaxf(bt, tok_s[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bt = fmaxf(bt, __shfl_xor_sync(0xffffffffu, bt, o));
    if (lane == 0) tok_s[p.I] = bt;
  }
  __syncthreads();
  for (int n = tid; n < kN; n += kThreadsW) {
    const int id_ = n % p.wd, iw = (n / p.wd) % p.ww, ih = n / (p.wd * p.ww);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      __align__(16) T tmp[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int col = c * 8 + e;
        tmp[e] = (col < p.wh) ? (col == ih ? one : zero) : ((col - p.wh < p.ww && col - p.wh == iw) ? one : zero);
      }
      *reinterpret_cast<uint4*>(Qa + c * (kN * 16) + n * 16) = *reinterpret_cast<const uint4*>(tmp);
    }
    float bh = -1e30f, bw_ = -1e30f, bd = -1e30f;
    const float bt = tok_s[p.I];
    for (int j = 0; j < p.wh; ++j) bh = fmaxf(bh, th_s[ih * p.wh + j]);
    for (int j = 0; j < p.ww; ++j) bw_ = fmaxf(bw_, tw_s[iw * p.ww + j]);
    for (int j = 0; j < p.wd; ++j) bd = fmaxf(bd, td_s[id_ * p.wd + j]);
    rowb_s[n] = (p.I > 0 ? fmaxf(bh + bw_ + bd, bt) : bh + bw_ + bd) * inv_scale;   // max_j bias[n][j] / scale
  }
  for (int j = tid; j < NKT; j += kThreadsW) {
    const bool content = j < kN;
    const int jw = (j / p.wd) % p.ww, jh = j / (p.wd * p.ww);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      __align__(16) T tmp[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int col = c * 8 + e;
        float v = 0.f;
        if (content) {
          if (col < p.wh) v = th_s[col * p.wh + jh];
          else if (col - p.wh < p.ww) v = tw_s[(col - p.wh) * p.ww + jw];
        } else if (col < p.wh) {
          v = tok_s[j - kN];
        }
        tmp[e] = from_f32<T>(v * inv_scale);
      }
      *reinterpret_cast<uint4*>(Ka + c * (NKT * 16) + j * 16) = *reinterpret_cast<const uint4*>(tmp);
    }
  }
  if (tid == 0) {
    for (int i = 0; i < 3; ++i) {
      mbar_init(&bar[bOpFull + i], kStageThreads);
      mbar_init(&bar[bOpFree + i], 512);
      mbar_init(&bar[bLsum + 2 * i], 256);
      mbar_init(&bar[bLsum + 2 * i + 1], 256);
    }
    for (int i = 0; i < 12; ++i) mbar_init(&bar[bSFull + i], 1);
    for (int i = 0; i < 6; ++i) mbar_init(&bar[bPReady + i], 128);
    for (int i = 0; i < 4; ++i) {
      mbar_init(&bar[bOFull + i], 1);
      mbar_init(&bar[bOFree + i], 128);
    }
    fence_mbar_init();
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;

  if (warp < kSoft0 + 16) {
    // =============================================================================================
    // softmax warps: group g (query tile g of the window), set (alternate units of the group's stream)
    // =============================================================================================
    const int g = (warp - kSoft0) >> 3;
    const uint32_t set = (uint32_t)((warp - kSoft0) >> 2) & 1u;
    const int tg = (warp & 3) * 32 + lane;                          // row within the tile = TMEM lane
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(g * GC);
    const uint32_t seed0 = DROP ? (p.drop_seed ? p.drop_seed[0] : p.seed_host[0]) : 0u;
    const uint32_t seed1 = DROP ? (p.drop_seed ? p.drop_seed[1] : p.seed_host[1]) : 0u;
    const DropThresh& dth = p.drop_planes;          // constant bank (filled by the dispatcher)
    uint32_t ucount = 0, tcount = 0;                                // units / tiles of this GROUP so far (both sets count all)
    WS_PROF_DECL(8);          // 0 wait operands, 1 window setup, 3 unit loop, 5 wait O, 6 epilogue
    for (int it = 0;; ++it) {
      const int ob = it % OPB;
      uint8_t* opnd = smem + L.opnd0 + ob * L.opnd_bytes;
      WS_PROF(6);
      mbar_wait(&bar[bOpFull + ob], (it / OPB) & 1);
      WS_PROF(0);
      const WsHeader* hdr = reinterpret_cast<const WsHeader*>(opnd + L.hdr);
      const int bw = hdr->bw;
      if (bw < 0) break;
      const bool exact = hdr->exact != 0;
      const uint32_t* sel_s = reinterpret_cast<const uint32_t*>(opnd + L.sel);
      const uint8_t* ids_s = opnd + L.ids;
      float* part_s = reinterpret_cast<float*>(opnd + L.part);     // [set][query row of the window]
      const int rown = g * 128 + tg;
      const uint32_t rid = MASKED ? ids_s[rown] : 0;
      float mb;
      {
        const float qk = sqrtf(reinterpret_cast<const float*>(opnd + L.qn2)[rown]) * hdr->kmax, rb = rowb_s[rown];
        mb = c2 * 1.01f * (qk + fmaxf(rb, 0.f));
      }
      if (exact) {
        // rare path: exact row maximum of the masked logits (masked entries count as 0, as in the reference); the issuer
        // runs the S MMAs of every unit once more for the real pass.  Each set sees its own units: the two partial maxima
        // meet in shared memory (named barrier over the group's 256 threads).
        float mx = -1e30f;
        for (int u = 0; u < n_units; ++u, ++ucount) {
          if ((ucount & 1u) != set) continue;
          const uint32_t buf = ucount % kNSB, sb = ucount % 6u;
          mbar_wait(&bar[bSFull + g * 6 + sb], (ucount / 6u) & 1);
          tc_fence_after();
          const int nk = u == n_units - 1 ? last_nk : kUK;
          const bool do_mask = MASKED && u * kUK < kN;
          for (int c = 0; c < nk / 32; ++c) {
            uint32_t r[32];
            tmem_ld32(trow + buf * kUK + c * 32, r);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              float s = __uint_as_float(r[e]);
              if (do_mask && ids_s[u * kUK + c * 32 + e] != rid) s = 0.f;
              mx = fmaxf(mx, s);
            }
          }
          tc_fence_before();
          mbar_arrive(&bar[bPReady + g * kNSB + buf]);
        }
        part_s[set * kN + rown] = mx;
        asm volatile("bar.sync %0, 256;" ::"r"(2 + g) : "memory");
        mx = fmaxf(mx, part_s[(set ^ 1u) * kN + rown]);
        asm volatile("bar.sync %0, 256;" ::"r"(2 + g) : "memory");  // both partials read before the denominators reuse the slots
        mb = mx * c2;
      }
      if constexpr (WsStab<T>::shift != 0.f) mb -= WsStab<T>::shift;
      const uint32_t rhash = DROP ? drop_row_hash(seed0, seed1, (uint32_t)bw, (uint32_t)p.heads, (uint32_t)head, kN, (uint32_t)rown) : 0u;
      float lsum0 = 0.f, lsum1 = 0.f;
      const float e0 = ex2f(-mb);                                  // weight of every masked (zeroed) logit
      const uint32_t e0pair = pack2t<T>(e0, e0);
      const uint32_t* selrow = sel_s + id_slot_w(rid) * (kN / 4);
      WS_PROF(1);

      bool last_mine = false;                                       // this set handled the window's last unit -> epilogue
      for (int u = 0; u < n_units; ++u, ++ucount) {
        if ((ucount & 1u) != set) continue;
        last_mine = u == n_units - 1;
        const uint32_t buf = ucount % kNSB, sb = ucount % 6u;
        mbar_wait(&bar[bSFull + g * 6 + sb], (ucount / 6u) & 1);
        tc_fence_after();
        const int nk = u == n_units - 1 ? last_nk : kUK;
        const bool do_mask = MASKED && u * kUK < kN;
        for (int c = 0; c < nk / 32; ++c) {
          uint32_t r[32];
          tmem_ld32(trow + buf * kUK + c * 32, r);
          tmem_wait_ld();
          uint32_t pk[16];
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            float x0, x1;
            ffma2w(x0, x1, __uint_as_float(r[2 * q]), __uint_as_float(r[2 * q + 1]), c2, -mb);
            const float p0 = ex2f(x0), p1 = ex2f(x1);
            pk[q] = pack2t<T>(p0, p1);
          }
          if (do_mask) {
            const uint4* sp = reinterpret_cast<const uint4*>(selrow + u * (kUK / 4) + c * 8);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const uint4 s4 = sp[h];
              const uint32_t sw[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
              for (int w = 0; w < 4; ++w) {
                pk[h * 8 + w * 2] = prmt3(pk[h * 8 + w * 2], e0pair, sw[w]);
                pk[h * 8 + w * 2 + 1] = prmt3(pk[h * 8 + w * 2 + 1], e0pair, sw[w] >> 16);
              }
            }
          }
          if (DROP) {
            const uint32_t kw = drop_keep_word(rhash, (uint32_t)(u * (kUK / 32) + c), dth);
            drop_apply16w<T>(pk, kw, lsum0, lsum1);
          }
          tmem_st16(trow + buf * kUK + c * 16, pk);
        }
        tmem_wait_st();
        tc_fence_before();
        mbar_arrive(&bar[bPReady + g * kNSB + buf]);
      }
      WS_PROF(3);
      if (DROP) {                                                   // the two sets' shares of the softmax denominator
        part_s[set * kN + rown] = lsum0 + lsum1;
        mbar_arrive(&bar[bLsum + ob * 2 + g]);
      }
      if (last_mine) {
        // ---- O of this tile: drain, normalise, write the bf16 output row slice and the log-sum-exp ----
        const uint32_t obuf = tcount % NOB;
        mbar_wait(&bar[bOFull + g * 2 + obuf], (tcount / NOB) & 1);
        tc_fence_after();
        WS_PROF(5);
        float o_run[DHP];
#pragma unroll
        for (int dq = 0; dq < DHP / 16; ++dq) {
          uint32_t o[16];
          tmem_ld16(trow + kNSB * kUK + obuf * DHP + dq * 16, o);
          tmem_wait_ld();
#pragma unroll
          for (int d = 0; d < 16; ++d) o_run[dq * 16 + d] = __uint_as_float(o[d]);
        }
        tc_fence_before();
        mbar_arrive(&bar[bOFree + g * 2 + obuf]);
        float l_run = o_run[DH];
        if (DROP) {
          mbar_wait(&bar[bLsum + ob * 2 + g], (it / OPB) & 1);
          l_run = part_s[rown] + part_s[kN + rown];
        }
        const float inv = (DROP ? p.inv_keep : 1.f) / l_run;
        T* og = (T*)p.out + ((size_t)bw * kN + rown) * p.C + head * DH;
        if constexpr (DH % 4 == 0) {
#pragma unroll
          for (int d = 0; d < DH; d += 4) {
            uint2 v;
            v.x = pack2t<T>(o_run[d] * inv, o_run[d + 1] * inv);
            v.y = pack2t<T>(o_run[d + 2] * inv, o_run[d + 3] * inv);
            *reinterpret_cast<uint2*>(og + d) = v;
          }
        } else {
#pragma unroll
          for (int d = 0; d < DH; ++d) og[d] = from_f32<T>(o_run[d] * inv);
        }
        p.lse[((size_t)bw * p.heads + head) * kN + rown] = (mb + __log2f(l_run)) * 0.6931471805599453f;
      }
      ++tcount;
      mbar_arrive(&bar[bOpFree + ob]);                              // this thread is done with the operand set
    }
    WS_PROF(6);
    if (tid == kSoft0 * 32) WS_PROF_OUT(0, 8);
    if (tid == (kSoft0 + 4) * 32) WS_PROF_OUT(8, 8);
  } else if (warp >= kStage0) {
    // =============================================================================================
    // staging warps: operand set of window `it` into buffer it % OPB
    // =============================================================================================
    // A (window, head) slice is 896 rows of DH bf16 at a row pitch of 3C elements.  One thread per ROW made every load
    // instruction touch 32 different 128-byte lines (L1 wavefronts, not DRAM, bound the staging: ~6 K clk per window, the
    // critical path of the whole kernel).  Here consecutive lanes take consecutive 8-byte PIECES of a row, so a warp-wide
    // load touches ~11 lines, and every piece goes straight to its place in the canonical layouts with one 8-byte store.
    // The columns beyond DH (one-hot / bias-table columns of Q' and K', the ones column of V, zero padding) do not depend
    // on the window: they are written once per operand buffer.  |q|^2 and max |k|^2 are computed from shared memory.
    const int st = tid - kStage0 * 32;
    const int sw = warp - kStage0;
    constexpr bool PIECES = DH % 4 == 0 && DH >= 12;
    constexpr int PPR = PIECES ? DH / 4 : 1;                        // 8-byte pieces per row
    if constexpr (PIECES) {
      for (int ob = 0; ob < OPB; ++ob) {
        uint8_t* opnd = smem + L.opnd0 + ob * L.opnd_bytes;
        for (int n = st; n < kN; n += kStageThreads) {
          const int id_ = n % p.wd;
          for (int e = DH; e < KS * 16; ++e)
            *reinterpret_cast<T*>(opnd + L.q + (e >> 3) * (kN * 16) + n * 16 + (e & 7) * 2) =
                (e - DH < p.wd && e - DH == id_) ? one : zero;
        }
        for (int j = st; j < NKT; j += kStageThreads) {
          const int jd = j % p.wd;
          for (int e = DH; e < KS * 16; ++e)
            *reinterpret_cast<T*>(opnd + L.k + (e >> 3) * (NKT * 16) + j * 16 + (e & 7) * 2) =
                (j < kN && e - DH < p.wd) ? from_f32<T>(td_s[(e - DH) * p.wd + jd] * inv_scale) : zero;
          for (int e = DH; e < DHP; ++e)
            *reinterpret_cast<T*>(opnd + L.v + (j >> 3) * (NDC * 128) + (e >> 3) * 128 + (j & 7) * 16 + (e & 7) * 2) =
                e == DH ? one : zero;
        }
      }
    }
    int bw = blockIdx.x / p.heads;
    WS_PROF_DECL(8);          // 0 wait free, 1 loads + layout stores, 2 barrier, 3 selectors + bound, 4 windows
    for (int it = 0;; ++it) {
      const int ob = it % OPB;
      uint8_t* opnd = smem + L.opnd0 + ob * L.opnd_bytes;
      uint8_t* Qs = opnd + L.q;
      uint8_t* Ks = opnd + L.k;
      uint8_t* Vs = opnd + L.v;
      uint32_t* sel_s = reinterpret_cast<uint32_t*>(opnd + L.sel);
      uint8_t* ids_s = opnd + L.ids;
      float* qn2_s = reinterpret_cast<float*>(opnd + L.qn2);
      WsHeader* hdr = reinterpret_cast<WsHeader*>(opnd + L.hdr);
      WS_PROF(3);
      if (it >= OPB) mbar_wait(&bar[bOpFree + ob], ((it / OPB) - 1) & 1);
      WS_PROF(0);
      const bool stop = bw >= n_pairs;
      if (st == 0) {
        hdr->bw = stop ? -1 : bw;
        hdr->exact = 0;
        // the window after this one: static for the first, then from this head's counter (CTAs do not progress evenly)
        hdr->next_bw = stop ? bw : (p.work ? stride + (int)atomicAdd(p.work + head, 1u) : bw + stride);
      }
      float qn2[2] = {0.f, 0.f};
      float kmax2 = 0.f;
      if (!stop) {
        const int b = bw / p.P, win = bw - b * p.P;
        if (MASKED) {
          if (p.sel != nullptr) {
            // selector table of this window precomputed per geometry (pwa_attn_sel_table): ONE bulk copy, completion
            // counted on the operand barrier (building it here cost the staging warps ~3 K clk per window)
            if (st == 0) {
              constexpr uint32_t kSelBytes = kIds * (kN / 4) * 4;
              mbar_expect_tx(&bar[bOpFull + ob], kSelBytes);
              bulk_g2s(sel_s, reinterpret_cast<const uint8_t*>(p.sel) + (size_t)win * kSelBytes, kSelBytes, &bar[bOpFull + ob]);
            }
          }
          if (st < kN / 4)
            reinterpret_cast<uint32_t*>(ids_s)[st] = reinterpret_cast<const uint32_t*>(p.ids + (size_t)win * kN)[st];
        }
        auto kv_off = [&](int j) {
          return j < kN ? ((size_t)bw * kN + j) * p.ldq + head * DH : ((size_t)b * p.I + (j - kN)) * p.ldp + head * DH;
        };
        if constexpr (PIECES) {
          // asynchronous 8-byte copies (LDGSTS): every piece of the window in flight at once, no register staging -- the
          // global round trip (~3 K clk under load) is paid once per window instead of once per register batch
          auto cp8 = [](uint8_t* dst, const T* src) {
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
          };
          const T* qb = (const T*)p.q + (size_t)bw * kN * p.ldq + head * DH;
          const T* kb = (const T*)p.k + (size_t)bw * kN * p.ldq + head * DH;
          const T* vb = (const T*)p.v + (size_t)bw * kN * p.ldq + head * DH;
          const T* kpb = (const T*)p.kp + (size_t)b * p.I * p.ldp + head * DH;
          const T* vpb = (const T*)p.vp + (size_t)b * p.I * p.ldp + head * DH;
          for (int i = st; i < kN * PPR; i += kStageThreads) {       // content rows: Q, K, V share the (row, part) decode
            const int row = i / PPR, part = i - row * PPR;
            const uint32_t so = (uint32_t)(row * p.ldq + part * 4);
            const uint32_t d16 = (uint32_t)(row * 16 + (part & 1) * 8);
            cp8(Qs + (part >> 1) * (kN * 16) + d16, qb + so);
            cp8(Ks + (part >> 1) * (NKT * 16) + d16, kb + so);
            cp8(Vs + (row >> 3) * (NDC * 128) + (part >> 1) * 128 + (row & 7) * 16 + (part & 1) * 8, vb + so);
          }
          for (int i = st; i < p.I * PPR; i += kStageThreads) {      // prompt rows of K and V
            const int r = i / PPR, part = i - r * PPR, row = kN + r;
            const uint32_t so = (uint32_t)(r * p.ldp + part * 4);
            cp8(Ks + (part >> 1) * (NKT * 16) + row * 16 + (part & 1) * 8, kpb + so);
            cp8(Vs + (row >> 3) * (NDC * 128) + (part >> 1) * 128 + (row & 7) * 16 + (part & 1) * 8, vpb + so);
          }
          asm volatile("cp.async.wait_all;" ::: "memory");
        } else {
          auto stage_q = [&](int t, const T (&row)[DH]) {
            const int n = t * 128 + st;
            qn2[t] = sumsq_w<DH>(row);
            qn2_s[n] = qn2[t];
            const int id_ = n % p.wd;
            T extra[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) extra[u] = (u == id_) ? one : zero;
            store_chunks_w<DH, KS>(Qs, kN * 16, n, row, extra, p.wd);
          };
          auto stage_k = [&](int j, const T (&row)[DH]) {
            const bool content = j < kN;
            kmax2 = fmaxf(kmax2, sumsq_w<DH>(row));
            const int jd = j % p.wd;
            T extra[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
              extra[u] = (content && u < p.wd) ? from_f32<T>(td_s[u * p.wd + jd] * inv_scale) : zero;
            store_chunks_w<DH, KS>(Ks, NKT * 16, j, row, extra, p.wd);
          };
          auto stage_v = [&](int j, const T (&row)[DH]) {
#pragma unroll
            for (int dc = 0; dc < NDC; ++dc) {
              __align__(16) T tmp[8];
#pragma unroll
              for (int e = 0; e < 8; ++e)
                tmp[e] = (dc * 8 + e < DH) ? row[dc * 8 + e < DH ? dc * 8 + e : 0] : (dc * 8 + e == DH ? one : zero);
              *reinterpret_cast<uint4*>(Vs + (j >> 3) * (NDC * 128) + dc * 128 + (j & 7) * 16) = *reinterpret_cast<const uint4*>(tmp);
            }
          };
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            T row[DH];
            load_row_w<DH>((const T*)p.q + ((size_t)bw * kN + t * 128 + st) * p.ldq + head * DH, row);
            stage_q(t, row);
          }
          for (int j = st; j < NKT; j += 128) {
            T row[DH], vrow[DH];
            load_row_w<DH>((const T*)(j < kN ? p.k : p.kp) + kv_off(j), row);
            load_row_w<DH>((const T*)(j < kN ? p.v : p.vp) + kv_off(j), vrow);
            stage_k(j, row);
            stage_v(j, vrow);
          }
        }
      }
      WS_PROF(1);
      stage_sync();                                               // pieces, ids, header of this operand set are in place
      WS_PROF(2);
      if (!stop) {
        if constexpr (PIECES) {
          // |q|^2 of this thread's two query rows and max |k|^2 over its key rows, from the staged copies
          auto row_sumsq = [&](const uint8_t* base, uint32_t chunk_stride, int row) {
            float a = 0.f;
#pragma unroll
            for (int part = 0; part < PPR; ++part) {
              const uint2 w = *reinterpret_cast<const uint2*>(base + (part >> 1) * chunk_stride + row * 16 + (part & 1) * 8);
              float f0, f1, f2, f3;
              unpack2t<T>(w.x, f0, f1);
              unpack2t<T>(w.y, f2, f3);
              a = fmaf(f0, f0, fmaf(f1, f1, fmaf(f2, f2, fmaf(f3, f3, a))));
            }
            return a;
          };
#pragma unroll
          for (int t = 0; t < 2; ++t) {
            qn2[t] = row_sumsq(Qs, kN * 16, t * 128 + st);
            qn2_s[t * 128 + st] = qn2[t];
          }
          for (int j = st; j < NKT; j += kStageThreads) kmax2 = fmaxf(kmax2, row_sumsq(Ks, NKT * 16, j));
        }
        kmax2 = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(kmax2)));   // non-negative floats order as uints
        if (lane == 0) kmax_w[ob][sw] = __float_as_uint(kmax2);
        if (MASKED && p.sel == nullptr) {
          // PRMT selectors: word w of row-id slot s covers keys 4w..4w+3 = packed pairs 2w (low half) and 2w+1 (high
          // half); a kept bf16 takes its own bytes (nibbles 1,0 / 3,2), a masked one those of the (e0,e0) operand
          for (int i = st; i < kIds * (kN / 4); i += kStageThreads) {
            const int s_ = i / (kN / 4), w = i - s_ * (kN / 4);
            const uint32_t idw = reinterpret_cast<const uint32_t*>(ids_s)[w];
            uint32_t sel = 0;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const bool keep = id_slot_w((idw >> (8 * e)) & 0xffu) == s_;
              const uint32_t nib = (e & 1) ? (keep ? 0x32u : 0x76u) : (keep ? 0x10u : 0x54u);
              sel |= nib << (((e & 1) ? 8 : 0) + ((e >> 1) ? 16 : 0));
            }
            sel_s[i] = sel;
          }
        }
      }
      stage_sync();                                               // partial key maxima
      const int next_bw = hdr->next_bw;
      if (!stop) {
        const float kmax = sqrtf(__uint_as_float(max(max(kmax_w[ob][0], kmax_w[ob][1]), max(kmax_w[ob][2], kmax_w[ob][3]))));
        if (st == 0) hdr->kmax = kmax;
        // stabiliser: upper bound of the row's logits; the row maximum is >= max_j bias - |q| max|k|, so the gap bounds how
        // far below the stabiliser the largest exponent argument can lie.  Too loose -> exact-max sweep for this window.
        bool loose = false;
#pragma unroll
        for (int t = 0; t < 2; ++t) {
          const float qk = sqrtf(qn2[t]) * kmax, rb = rowb_s[t * 128 + st];
          const float mbt = c2 * 1.01f * (qk + fmaxf(rb, 0.f));
          // (fp16: in a masked row the key that attains rb may be masked -- its logit is 0 -- so only min(rb - qk, 0) is a
          // lower bound of the row maximum there)
          const float lb = (MASKED && WsStab<T>::shift != 0.f) ? fminf(rb - qk, 0.f) : rb - qk;
          loose |= (mbt - c2 * lb) > WsStab<T>::max_gap;
        }
        if (loose) atomicOr(&hdr->exact, 1);
      }
      fence_proxy_async_smem();
      mbar_arrive(&bar[bOpFull + ob]);
      if (stop) break;
      bw = next_bw;
#ifdef PWA_TIMELINE_BUILD
      prof_[4] += 1;
#endif
    }
    WS_PROF(3);
    if (st == 0) WS_PROF_OUT(16, 8);
  } else if (warp >= kIssue0 && warp < kIssue0 + 2) {
    // =============================================================================================
    // MMA issuer of group g: S runs two units ahead of PV; tcgen05.mma executes in issue order per thread
    // =============================================================================================
    // The WHOLE warp runs the control flow with warp-uniform values (everything read from shared memory goes through a
    // shuffle broadcast), and only the tcgen05 instructions themselves sit under elect.sync: the MMA operands then live in
    // uniform registers.  With the loop inside `if (lane == 0)` every MMA was wrapped in an ELECT + 7 x R2UR.BROADCAST
    // waterfall loop and one thread issued an MMA only every ~170 clk -- the issuer was the kernel's critical path.
    {
      const int g = __shfl_sync(0xffffffffu, warp - kIssue0, 0);
      const uint32_t tg = __shfl_sync(0xffffffffu, tmem, 0) + (uint32_t)(g * GC);
      const uint32_t idescS64 = make_idesc<T>(128, 64, 0, 0), idescS32 = make_idesc<T>(128, 32, 0, 0);
      const uint32_t idescPV = make_idesc<T>(128, DHP, 0, 1);
      struct Cur {
        int it, pass, u, npass;
        bool stop, need_open;
        uint32_t opnd;
      };
      // blocking = false: only if the operand set is already there (the S look-ahead must not stall the PVs of the units
      // in flight behind a window that is still being staged)
      auto open_window = [&](Cur& c, bool blocking) -> bool {
        const int ob = c.it % OPB;
        if (blocking) mbar_wait(&bar[bOpFull + ob], (c.it / OPB) & 1);
        else if (!__any_sync(0xffffffffu, mbar_try_wait(&bar[bOpFull + ob], (c.it / OPB) & 1))) return false;   // (warp-uniform)
        const WsHeader* hdr = reinterpret_cast<const WsHeader*>(smem + L.opnd0 + ob * L.opnd_bytes + L.hdr);
        c.stop = __shfl_sync(0xffffffffu, hdr->bw, 0) < 0;
        c.npass = __shfl_sync(0xffffffffu, hdr->exact, 0) ? 2 : 1;
        c.pass = 0;
        c.u = 0;
        c.need_open = false;
        c.opnd = smem_u32(smem + L.opnd0 + ob * L.opnd_bytes);
        return true;
      };
      auto advance = [&](Cur& c) {
        if (++c.u == n_units) {
          c.u = 0;
          if (++c.pass == c.npass) {
            ++c.it;
            c.need_open = true;
          }
        }
      };
      Cur cs = {0, 0, 0, 1, false, true, 0u};
      open_window(cs, true);
      Cur cp = cs;
      uint32_t ns = 0, np = 0, tcount = 0, obuf = 0;
      WS_PROF_DECL(8);        // 0 issue S (+ operand waits), 1 wait P, 2 wait O free, 3 issue PV
      for (;;) {
        // ---- S of up to three units ahead (all S buffers: two being exponentiated by the two sets, one waiting) ----
        while (!cs.stop && ns < np + kNSB) {
          if (cs.need_open) {
            // with ONE operand buffer the next window is staged only after this one has retired completely: all of its
            // PVs must be issued before this thread may block on the next operand set
            if (OPB == 1 && np < ns) break;
            if (!open_window(cs, np == ns)) break;                  // block only when nothing else is left to do
            if (cs.stop) break;
          }
          const uint32_t buf = ns % kNSB;
          const int nk = cs.u == n_units - 1 ? last_nk : kUK;
          const uint32_t idesc = nk == kUK ? idescS64 : idescS32;
          const uint32_t koff = (uint32_t)(cs.u * kUK) * 16;
          tc_fence_after();
          if (elect_one_sync()) {
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
              const uint64_t da = make_smem_desc(cs.opnd + L.q + ks * 2 * (kN * 16) + g * (128 * 16), kN * 16, 128);
              const uint64_t db = make_smem_desc(cs.opnd + L.k + ks * 2 * (NKT * 16) + koff, NKT * 16, 128);
              mma_ss(tg + buf * kUK, da, db, idesc, ks > 0);
            }
            {
              const uint64_t da = make_smem_desc(smem_u32(Qa) + g * (128 * 16), kN * 16, 128);
              const uint64_t db = make_smem_desc(smem_u32(Ka) + koff, NKT * 16, 128);
              mma_ss(tg + buf * kUK, da, db, idesc, 1);
            }
            mma_commit(&bar[bSFull + g * 6 + ns % 6u]);
          }
          __syncwarp();
          ++ns;
          advance(cs);
        }
        if (np == ns) {
          if (cs.stop) break;                                       // everything issued and consumed
          continue;                                                 // (OPB == 1: the next window can be opened now)
        }
        // ---- PV of unit np ----
        if (cp.need_open) open_window(cp, true);
        const uint32_t buf = np % kNSB;
        WS_PROF(0);
        mbar_wait(&bar[bPReady + g * kNSB + buf], (np / kNSB) & 1);
        tc_fence_after();
        WS_PROF(1);
        const bool maxpass = cp.npass == 2 && cp.pass == 0;
        if (!maxpass) {
          if (cp.u == 0) {
            obuf = tcount % NOB;
            if (tcount >= (uint32_t)NOB) {                          // the accumulator's previous tile has been drained
              mbar_wait(&bar[bOFree + g * 2 + obuf], ((tcount / NOB) - 1) & 1);
              tc_fence_after();
            }
            WS_PROF(2);
          }
          const int nk = cp.u == n_units - 1 ? last_nk : kUK;
          if (elect_one_sync()) {
#pragma unroll
            for (int t = 0; t < kUK / 16; ++t) {
              if (t * 16 < nk) {
                const uint64_t dv = make_smem_desc(cp.opnd + L.v + ((cp.u * kUK + t * 16) >> 3) * (NDC * 128), NDC * 128, 128);
                mma_ts(tg + kNSB * kUK + obuf * DHP, tg + buf * kUK + t * 8, dv, idescPV, (cp.u > 0) | (t > 0));
              }
            }
            if (cp.u == n_units - 1) mma_commit(&bar[bOFull + g * 2 + obuf]);
          }
          __syncwarp();
          if (cp.u == n_units - 1) ++tcount;
        }
        ++np;
        advance(cp);
        WS_PROF(3);
      }
      if (g == 0 && lane == 0) WS_PROF_OUT(24, 8);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 512);
}

template <int DH, typename T>
int launch_ws(const AttnParams& p, cudaStream_t st) {
  constexpr int DHP = WCfg<DH>::DHP, KS = WCfg<DH>::KS;
  const int NKT = kN + p.I;
  const WsSmem L = ws_layout(KS, DHP, NKT, p.ids != nullptr);
  const size_t smem = L.total;
  int grid = 148;
  grid -= grid % p.heads;
  if (grid < p.heads) grid = p.heads;
  const int need = p.B * p.P * p.heads;
  if (grid > need) grid = need;
  auto kern = p.drop_thresh ? (p.ids ? attn_fwd_ws_kernel<DH, true, true, T> : attn_fwd_ws_kernel<DH, false, true, T>)
                            : (p.ids ? attn_fwd_ws_kernel<DH, true, false, T> : attn_fwd_ws_kernel<DH, false, false, T>);
  PWA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (p.work) PWA_CUDA_OK(cudaMemsetAsync(p.work, 0, sizeof(unsigned int) * p.heads, st));
  kern<<<grid, kThreadsW, smem, st>>>(p);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

}  // namespace

bool attn_ws_fits(const AttnParams& p) {
  const int dh = p.C / p.heads;
  return ws_layout((dh + 4 + 15) / 16, (dh + 1 + 15) / 16 * 16, kN + p.I, true).total <= 224u * 1024u;
}

template <typename T>
static int ws_forward_t(const AttnParams& p, cudaStream_t st) {
  switch (p.C / p.heads) {
    case 3: return launch_ws<3, T>(p, st);
    case 6: return launch_ws<6, T>(p, st);
    case 12: return launch_ws<12, T>(p, st);
    case 24: return launch_ws<24, T>(p, st);
    case 48: return launch_ws<48, T>(p, st);
  }
  set_error("tcgen05 attention: head_dim %d not instantiated", p.C / p.heads);
  return PWA_ERR_UNSUPPORTED;
}

int attn_ws_forward(const AttnParams& p, int dtype, cudaStream_t st) {
  return dtype == PWA_F16 ? ws_forward_t<__half>(p, st) : ws_forward_t<__nv_bfloat16>(p, st);
}

}  // namespace pwa
