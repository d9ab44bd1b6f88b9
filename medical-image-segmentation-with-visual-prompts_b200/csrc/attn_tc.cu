// (b) fused prompted window attention forward on the 5th-gen tensor cores (tcgen05 + TMEM), bf16 I/O.
//
// One CTA = 128 threads = one fixed head; it walks over (sample, window) pairs.  Per window the CTA stages
// this head's Q / K / V slices in shared memory in UMMA canonical (no-swizzle) layouts, then for each of the
// two 128-row query tiles and each key block (content 0-127, content 128-255, prompt 0-I):
//     S[128 x nk]  = Q'.K'^T            tcgen05.mma kind::f16, both operands from smem, fp32 accum in TMEM
//     P            = exp2(S*c - mb)     each thread owns one query row = one TMEM lane (tcgen05.ld 32x32b),
//                                       writes P back as packed bf16 over the consumed S columns (tcgen05.st)
//     O[128 x dh+1] = P.[V | 1]         tcgen05.mma with A = P straight from TMEM, B = V (MN-major) from smem;
//                                       the ones column of V yields the softmax denominator for free
// The softmax is bound by the MUFU pipe (one ex2 per logit; measured 28 ex2/clk/SM, csrc/ubench.cu), so the
// per-logit instruction stream is kept to FFMA + MUFU + 1/2 F2FP(pack):
//   * no row-max pass: the stabiliser mb of a row is the Cauchy-Schwarz bound c*(|q_i| max_j|k_j| + max bias),
//     known before the first MMA.  Softmax is shift invariant, so the result is identical as long as nothing
//     under/overflows; if a bound exceeds kMaxBound (never with LayerNorm-ed inputs) the CTA first makes an
//     exact-max sweep over the three key blocks (MMA + TMEM loads only) and uses that instead.
//   * no online rescaling: the same mb holds for all key blocks, partial O tiles are simply added.
//   * the shift mask is multiplicative and applied BEFORE softmax (window_attention.py:54-56): a masked logit
//     becomes 0, i.e. its probability is the row constant e0 = exp2(-mb).  It is applied on the PACKED bf16
//     pairs with one PRMT per pair, selecting between the computed pair and (e0,e0) with byte selectors that
//     depend only on (region id of the row, key pair): a [28 ids][128 pairs] table built once per window.
//
// Relative-position bias is folded INTO the QK^T MMA: bias[n][m] = Th[ih][jh] + Tw[iw][jw] + Td[id][jd] is a
// sum of three one-hot x table products, so Q' = [q | onehot_d(n) | 0 ;; onehot_h(n) | onehot_w(n)] and
// K' = [k | Td[.][jd]/scale | 0 ;; Th[.][jh]/scale | Tw[.][jw]/scale] give S = q.k + bias/scale.  Prompt keys use
// [tok/scale x wh | 0] so every query row picks up tok[i].  The one-hot / table halves do not depend on the
// window, so they are built once per CTA and stay resident in smem, as do the prompt-independent constants.
//
// Four CTAs are resident per SM (128 TMEM columns and ~54 KB smem each at head_dim 12): tcgen05.mma costs
// ~100 clk of latency per instruction but streams of different CTAs overlap (csrc/ubench.cu), so while one
// CTA waits for its MMAs or stages the next window, the others keep the MUFU pipe busy.
#include "attn.cuh"
#include "tc_common.cuh"

namespace pwa {
using namespace tc;

namespace {

constexpr int kRows = 128;        // query rows per tile = TMEM lanes = threads per CTA
constexpr int kN = 256;           // content tokens per window (two query tiles, two content key blocks)
constexpr int kTmemCols = 128;
constexpr int kOCol = 64;         // O accumulator lives in columns [64, 64 + DHP) of the S region
constexpr int kIds = 28;          // region ids 0..26 and 100 (-> 27), see pwa_region_ids
#ifndef PWA_BATCH_STAGING
#define PWA_BATCH_STAGING 0
#endif
constexpr bool kBatchStaging = PWA_BATCH_STAGING != 0;
constexpr float kMaxBound = 40.f; // log2 units: the largest exp2 argument of a row stays within [-2*kMaxBound, ~0]

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// exp2 on the FMA / ALU pipes (x <= 0): Cody-Waite split with round-to-nearest (magic-number add), degree-3 minimax
// polynomial of 2^f on [-0.5, 0.5] (max relative error 7.5e-5, far inside bf16's 2^-9), exponent patched in with one
// shift-add.  B200 has 16 ex2/clk/SM; four resident CTAs keep that pipe ~80 % busy in steady state (and it is the only
// pipe near its limit), so a fixed share of every row's logits -- kPolyPairs, a bit per packed pair of a 32-key chunk --
// can take this path instead: ~9 issue slots on pipes with headroom against 1/16 clk of MUFU.
// Measured at enc0: 4/16 of the pairs = no change (270 us), 6/16 +2 %, 8/16 +8 %: the kernel is not bound by the MUFU
// pipe alone, so the share is 0 by default (-DPWA_POLY_PAIRS=0x8888 etc. to re-measure).
#ifndef PWA_POLY_PAIRS
#define PWA_POLY_PAIRS 0x0u
#endif
constexpr uint32_t kPolyPairs = PWA_POLY_PAIRS;
__device__ __forceinline__ float poly_exp2(float x) {
  x = fmaxf(x, -125.f);
  const float t = x + 12582912.f;                  // 1.5 * 2^23: round(x) lands in the low mantissa bits
  const float f = x - (t - 12582912.f);            // [-0.5, 0.5]
  float q = fmaf(0.05517132f, f, 0.24261054f);
  q = fmaf(q, f, 0.69326097f);
  q = fmaf(q, f, 0.99992812f);
  return __int_as_float(__float_as_int(q) + (__float_as_int(t) << 23));
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}
__device__ __forceinline__ int id_slot(uint32_t id) { return id < (uint32_t)(kIds - 1) ? (int)id : kIds - 1; }
// packed fp32 pairs (sm_100 FFMA2 / FADD2): (d0, d1) = (a0, a1) * b + c ; (s0, s1) += (a0, a1)
__device__ __forceinline__ void ffma2(float& d0, float& d1, float a0, float a1, float b, float c) {
  unsigned long long a, bb, cc, d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %1};" : "=l"(bb) : "f"(b));
  asm("mov.b64 %0, {%1, %1};" : "=l"(cc) : "f"(c));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(bb), "l"(cc));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(d));
}
__device__ __forceinline__ void fadd2(float& s0, float& s1, float a0, float a1) {
  unsigned long long a, s, d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(s) : "f"(s0), "f"(s1));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(s), "l"(a));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(s0), "=f"(s1) : "l"(d));
}
// dropout on the 16 packed pairs of a 32-key chunk: row-sum of the undropped bf16 values, then one AND per pair
template <int G = 0>
__device__ __forceinline__ void drop_apply16(uint32_t (&pk)[16], uint32_t kw, float& s0, float& s1) {
  if constexpr (G < 16) {
    fadd2(s0, s1, __uint_as_float(pk[G] << 16), __uint_as_float(pk[G] & 0xffff0000u));
    pk[G] &= drop_pair_mask<G>(kw);
    drop_apply16<G + 1>(pk, kw, s0, s1);
  }
}

template <int DH> struct Cfg {
  static constexpr int DHP = (DH + 1 + 15) / 16 * 16;      // V / O width (PV MMA N) incl. the ones column at DH
  static constexpr int NDC = DHP / 8;                      // 16-byte chunks per V row
  static constexpr int KS = (DH + 4 + 15) / 16;            // k-steps of the staged [q | onehot_d] operand
  static constexpr int NACC = 64 / DHP;                    // independent O accumulators in TMEM columns [64, 128)
};

struct TcSmem {
  uint32_t q, k, v, qaug, kaug, sel, rowb, ids, total;     // byte offsets
};

__host__ __device__ inline TcSmem tc_layout(int KS, int DHP, int NKT, bool masked) {
  TcSmem s;
  uint32_t o = 0;
  s.q = o; o += KS * 2 * kN * 16;
  s.k = o; o += KS * 2 * NKT * 16;
  s.v = o; o += NKT * DHP * 2;
  s.qaug = o; o += 2 * kN * 16;
  s.kaug = o; o += 2 * NKT * 16;
  s.sel = o; o += masked ? kIds * (kN / 4) * 4 : 0;        // [id][pair of packed words] PRMT selectors
  s.rowb = o; o += kN * 4;
  s.ids = o; o += kN;
  s.total = o;
  return s;
}

template <int DH>
__device__ __forceinline__ void load_row(const __nv_bfloat16* src, __nv_bfloat16 (&dst)[DH]) {
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

template <int DH>
__device__ __forceinline__ float sumsq(const __nv_bfloat16 (&r)[DH]) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < DH; ++i) {
    const float v = __bfloat162float(r[i]);
    s = fmaf(v, v, s);
  }
  return s;
}

// staged K-dim layout of one head: [real DH | wd extra columns | zero pad] -> KS k-steps of 16
template <int DH, int KS>
__device__ __forceinline__ void store_chunks(uint8_t* base, uint32_t chunk_stride, int row, const __nv_bfloat16 (&real)[DH],
                                             const __nv_bfloat16* extra, int n_extra) {
#pragma unroll
  for (int c = 0; c < KS * 2; ++c) {
    __align__(16) __nv_bfloat16 tmp[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int col = c * 8 + e;
      const int x = col - DH;
      __nv_bfloat16 v = __float2bfloat16(0.f);
      if (col < DH) v = real[col < DH ? col : 0];
      else if (x < 4 && x < n_extra) v = extra[x & 3];
      tmp[e] = v;
    }
    *reinterpret_cast<uint4*>(base + c * chunk_stride + row * 16) = *reinterpret_cast<const uint4*>(tmp);
  }
}

// DROP: attention dropout (window_attention.py:57).  The keep mask (csrc/attn.cuh: 32 hash bits per 2x2 block of
// (query pair, key pair)) is applied to the PACKED bf16 probabilities with one AND per pair, after the shift mask;
// the softmax denominator, which the ones column of V can no longer deliver, is then summed in registers from the
// same bf16 values the MMA consumes, and the inverse keep rate is applied once in the epilogue.
template <int DH, bool MASKED, bool DROP>
__global__ void __launch_bounds__(kRows, (DH <= 12 ? 4 : (DH <= 24 ? 2 : 1))) attn_fwd_tc_kernel(AttnParams p) {
  constexpr int DHP = Cfg<DH>::DHP, NDC = Cfg<DH>::NDC, KS = Cfg<DH>::KS, NACC = Cfg<DH>::NACC;
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  __shared__ uint32_t kmax_s[4];

#ifdef PWA_TIMELINE_BUILD
  const long long t_kernel_start = clock64();
#endif
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NKT = kN + p.I;
  const TcSmem L = tc_layout(KS, DHP, NKT, MASKED);
  uint8_t* Qs = smem + L.q;
  uint8_t* Ks = smem + L.k;
  uint8_t* Vs = smem + L.v;
  uint8_t* Qa = smem + L.qaug;
  uint8_t* Ka = smem + L.kaug;
  uint32_t* sel_s = reinterpret_cast<uint32_t*>(smem + L.sel);
  float* rowb_s = reinterpret_cast<float*>(smem + L.rowb);
  uint8_t* ids_s = smem + L.ids;
  const int head = blockIdx.x % p.heads;
  const float inv_scale = 1.f / p.scale;
  const float c2 = p.scale * 1.4426950408889634f;          // logits -> log2 domain
  const uint32_t seed0 = DROP ? (p.drop_seed ? p.drop_seed[0] : p.seed_host[0]) : 0u;
  const uint32_t seed1 = DROP ? (p.drop_seed ? p.drop_seed[1] : p.seed_host[1]) : 0u;
  const DropThresh dth = drop_thresh_planes(DROP ? p.drop_thresh : 0u);
  const __nv_bfloat16 one = __float2bfloat16(1.f), zero = __float2bfloat16(0.f);

  // ---- once per CTA: window-independent halves of Q' and K', per-row upper bound of the bias ----
  // (the bias tables of this head go through shared memory first: the loops below read each entry many times, and
  //  chains of dependent global loads made this setup ~20 % of the kernel at the small stages)
  __shared__ float tab_s[16 * 16 + 4 * 4 + 128 + 4];            // th | tw (wh + ww <= 16) | td (wd <= 4) | tok (I <= 128) | max tok
  float* th_s = tab_s;
  float* tw_s = th_s + p.wh * p.wh;
  float* td_s = tw_s + p.ww * p.ww;
  float* tok_s = td_s + p.wd * p.wd;
  for (int i = tid; i < p.wh * p.wh; i += kRows) th_s[i] = p.th[head * p.wh * p.wh + i];
  for (int i = tid; i < p.ww * p.ww; i += kRows) tw_s[i] = p.tw[head * p.ww * p.ww + i];
  for (int i = tid; i < p.wd * p.wd; i += kRows) td_s[i] = p.td[head * p.wd * p.wd + i];
  for (int i = tid; i < p.I; i += kRows) tok_s[i] = p.tok[head * p.I + i];
  __syncthreads();
  if (warp == 0) {
    float bt = -1e30f;
    for (int j = lane; j < p.I; j += 32) bt = fmaxf(bt, tok_s[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) bt = fmaxf(bt, __shfl_xor_sync(0xffffffffu, bt, o));
    if (lane == 0) tok_s[p.I] = bt;
  }
  __syncthreads();
  for (int n = tid; n < kN; n += kRows) {
    const int id_ = n % p.wd, iw = (n / p.wd) % p.ww, ih = n / (p.wd * p.ww);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      __align__(16) __nv_bfloat16 tmp[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int col = c * 8 + e;
        tmp[e] = (col < p.wh) ? (col == ih ? one : zero) : ((col - p.wh < p.ww && col - p.wh == iw) ? one : zero);
      }
      *reinterpret_cast<uint4*>(Qa + c * (kN * 16) + n * 16) = *reinterpret_cast<const uint4*>(tmp);
    }
    float bh = -1e30f, bw = -1e30f, bd = -1e30f;
    const float bt = tok_s[p.I];
    for (int j = 0; j < p.wh; ++j) bh = fmaxf(bh, th_s[ih * p.wh + j]);
    for (int j = 0; j < p.ww; ++j) bw = fmaxf(bw, tw_s[iw * p.ww + j]);
    for (int j = 0; j < p.wd; ++j) bd = fmaxf(bd, td_s[id_ * p.wd + j]);
    rowb_s[n] = (p.I > 0 ? fmaxf(bh + bw + bd, bt) : bh + bw + bd) * inv_scale;   // max_j bias[n][j] / scale
  }
  for (int j = tid; j < NKT; j += kRows) {
    const bool content = j < kN;
    const int jw = (j / p.wd) % p.ww, jh = j / (p.wd * p.ww);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      __align__(16) __nv_bfloat16 tmp[8];
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
        tmp[e] = __float2bfloat16(v * inv_scale);
      }
      *reinterpret_cast<uint4*>(Ka + c * (NKT * 16) + j * 16) = *reinterpret_cast<const uint4*>(tmp);
    }
  }
  if (tid == 0) {
    mbar_init(&bar, 4);       // lane 0 of each of the four warps arrives (commit or plain arrive) per MMA group
    fence_mbar_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, kTmemCols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);   // this warp's 32 lanes
  uint32_t phase = 0;

  // One thread issues a tcgen05.mma every ~100 clk whatever its shape (csrc/ubench.cu), streams of different warps
  // overlap: every MMA group of a step is split over the four warps (lane 0 of each issues its share and commits;
  // the step's mbarrier expects four arrivals).  S: 32-key column slices; O: k-steps round-robin over NACC accumulators.
  const bool split_prompt = p.I > 0 && (p.I / 4) % 16 == 0;
  const uint32_t idescS32 = make_idesc_bf16(128, 32, 0, 0);
  const uint32_t idescSP = make_idesc_bf16(128, p.I > 0 ? (split_prompt ? p.I / 4 : p.I) : 16, 0, 0);
  const uint32_t idescPV = make_idesc_bf16(128, DHP, 0, 1);
  const int n_kb = p.I > 0 ? 3 : 2;
  const int n_pairs = p.B * p.P;
  const int stride = gridDim.x / p.heads;

  // clock64 timeline of thread 0 / CTA 0 (tools/timeline_fwd.py): compiled in only with -DPWA_TIMELINE_BUILD
#ifdef PWA_TIMELINE_BUILD
  long long* tl = reinterpret_cast<long long*>(p.delta);
  int tli = 0;
  const bool rec = p.debug && p.delta != nullptr && blockIdx.x == 0 && tid == 0;
#define STAMP(tag) do { if (rec && tli < 2000) { tl[2 * tli] = clock64(); tl[2 * tli + 1] = (tag); ++tli; } } while (0)
  if (rec) { tl[8000] = t_kernel_start; tl[8001] = clock64(); }     // kernel entry, end of the per-CTA setup
#else
#define STAMP(tag) do { } while (0)
#endif

  // S = Q'.K'^T for (query tile mt, key block kb); called by lane 0 of every warp
  auto issue_s = [&](int mt, int kb) {
    tc_fence_after();
    int k0;
    uint32_t idesc;
    if (kb < 2) { k0 = warp * 32; idesc = idescS32; }
    else if (split_prompt) { k0 = warp * (p.I / 4); idesc = idescSP; }
    else if (warp == 0) { k0 = 0; idesc = idescSP; }
    else { mbar_arrive(&bar); return; }
    const uint32_t koff = (uint32_t)(kb * 128 + k0) * 16;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      const uint64_t da = make_smem_desc(smem_u32(Qs) + ks * 2 * (kN * 16) + mt * (kRows * 16), kN * 16, 128);
      const uint64_t db = make_smem_desc(smem_u32(Ks) + ks * 2 * (NKT * 16) + koff, NKT * 16, 128);
      mma_ss(tmem + k0, da, db, idesc, ks > 0);
    }
    const uint64_t da = make_smem_desc(smem_u32(Qa) + mt * (kRows * 16), kN * 16, 128);
    const uint64_t db = make_smem_desc(smem_u32(Ka) + koff, NKT * 16, 128);
    mma_ss(tmem + k0, da, db, idesc, 1);
    mma_commit(&bar);
  };

  // Window distribution: the first one is static, every further one comes from this head's counter (p.work) -- CTAs
  // that share an SM do not progress at the same rate (warp scheduling is not fair between them), and with a static
  // split the slow ones ran on alone at the end with the SM's pipes mostly idle.  The counter is read one window ahead.
  __shared__ int next_s[2];
  for (int bw = blockIdx.x / p.heads, it = 0; bw < n_pairs; ++it) {
    const int b = bw / p.P, win = bw - b * p.P;
    if (tid == 0) next_s[it & 1] = p.work ? stride + (int)atomicAdd(p.work + head, 1u) : bw + stride;
    STAMP(1);
    // ---- stage this (window, head): Q, K (content + prompt rows), [V | 1], region ids ----
    __nv_bfloat16 extra[4];
    float qn2[2];
    float kmax2 = 0.f;
    // Global-load round trips are what staging costs (~1-2 K clk each while three other CTAs keep the SM busy).
    // kBatchStaging: two batches -- every Q and K row of this thread in flight at once, then every V row -- instead of
    // one round trip per row (all eight rows at once needs 48 live registers and spilled at the 128-register cap).
    // Measured: staging 9.8 K -> 7.1 K clk per window, kernel time unchanged to +4 % (the SM is bound by the MUFU pipe
    // shared by its four CTAs, not by one CTA's latency), so it stays off.
    auto stage_q = [&](int t, const __nv_bfloat16 (&row)[DH]) {
      const int n = t * kRows + tid;
      qn2[t] = sumsq<DH>(row);
      const int id_ = n % p.wd;
#pragma unroll
      for (int u = 0; u < 4; ++u) extra[u] = (u == id_) ? one : zero;
      store_chunks<DH, KS>(Qs, kN * 16, n, row, extra, p.wd);
    };
    auto kv_off = [&](int j) {
      return j < kN ? ((size_t)bw * kN + j) * p.ldq + head * DH : ((size_t)b * p.I + (j - kN)) * p.ldp + head * DH;
    };
    auto stage_k = [&](int j, const __nv_bfloat16 (&row)[DH]) {
      const bool content = j < kN;
      kmax2 = fmaxf(kmax2, sumsq<DH>(row));
      const int jd = j % p.wd;
#pragma unroll
      for (int u = 0; u < 4; ++u)
        extra[u] = (content && u < p.wd) ? __float2bfloat16(td_s[u * p.wd + jd] * inv_scale) : zero;
      store_chunks<DH, KS>(Ks, NKT * 16, j, row, extra, p.wd);
    };
    auto stage_v = [&](int j, const __nv_bfloat16 (&row)[DH]) {
#pragma unroll
      for (int dc = 0; dc < NDC; ++dc) {
        __align__(16) __nv_bfloat16 tmp[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) tmp[e] = (dc * 8 + e < DH) ? row[dc * 8 + e < DH ? dc * 8 + e : 0] : (dc * 8 + e == DH ? one : zero);
        *reinterpret_cast<uint4*>(Vs + (j >> 3) * (NDC * 128) + dc * 128 + (j & 7) * 16) =
            *reinterpret_cast<const uint4*>(tmp);
      }
    };
    if constexpr (kBatchStaging && DH <= 12) {
      constexpr int KR = 3;                                      // key rows per thread: NKT <= 384 (I <= 128)
      __nv_bfloat16 qrow[2][DH], krow[KR][DH];
#pragma unroll
      for (int t = 0; t < 2; ++t)
        load_row<DH>((const __nv_bfloat16*)p.q + ((size_t)bw * kN + t * kRows + tid) * p.ldq + head * DH, qrow[t]);
#pragma unroll
      for (int i = 0; i < KR; ++i) {
        const int j = i * kRows + tid;
        if (j < NKT) load_row<DH>((const __nv_bfloat16*)(j < kN ? p.k : p.kp) + kv_off(j), krow[i]);
      }
#pragma unroll
      for (int t = 0; t < 2; ++t) stage_q(t, qrow[t]);
#pragma unroll
      for (int i = 0; i < KR; ++i)
        if (i * kRows + tid < NKT) stage_k(i * kRows + tid, krow[i]);
#pragma unroll
      for (int i = 0; i < KR; ++i) {
        const int j = i * kRows + tid;
        if (j < NKT) load_row<DH>((const __nv_bfloat16*)(j < kN ? p.v : p.vp) + kv_off(j), krow[i]);
      }
#pragma unroll
      for (int i = 0; i < KR; ++i)
        if (i * kRows + tid < NKT) stage_v(i * kRows + tid, krow[i]);
    } else {
#pragma unroll
      for (int t = 0; t < 2; ++t) {
        __nv_bfloat16 row[DH];
        load_row<DH>((const __nv_bfloat16*)p.q + ((size_t)bw * kN + t * kRows + tid) * p.ldq + head * DH, row);
        stage_q(t, row);
      }
      for (int j = tid; j < NKT; j += kRows) {
        __nv_bfloat16 row[DH];
        load_row<DH>((const __nv_bfloat16*)(j < kN ? p.k : p.kp) + kv_off(j), row);
        stage_k(j, row);
        load_row<DH>((const __nv_bfloat16*)(j < kN ? p.v : p.vp) + kv_off(j), row);
        stage_v(j, row);
      }
    }
    if (MASKED) {
      for (int i = tid; i < kN / 4; i += kRows)
        reinterpret_cast<uint32_t*>(ids_s)[i] = reinterpret_cast<const uint32_t*>(p.ids + (size_t)win * kN)[i];
    }
    kmax2 = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(kmax2)));   // non-negative floats order as uints
    if (lane == 0) kmax_s[warp] = __float_as_uint(kmax2);
    fence_proxy_async_smem();
    __syncthreads();
    if (MASKED) {
      // (a table precomputed per geometry and loaded from L2 was measured slower than rebuilding it here)
      // PRMT selectors: word w of row-id slot s covers keys 4w..4w+3 = packed pairs 2w (low half) and 2w+1 (high half);
      // a kept bf16 takes its own bytes (nibbles 1,0 / 3,2), a masked one the bytes of the (e0,e0) operand (5,4 / 7,6)
      for (int i = tid; i < kIds * (kN / 4); i += kRows) {
        const int s = i / (kN / 4), w = i - s * (kN / 4);
        const uint32_t idw = reinterpret_cast<const uint32_t*>(ids_s)[w];
        uint32_t sel = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const bool keep = id_slot((idw >> (8 * e)) & 0xffu) == s;
          const uint32_t nib = (e & 1) ? (keep ? 0x32u : 0x76u) : (keep ? 0x10u : 0x54u);
          sel |= nib << (((e & 1) ? 8 : 0) + ((e >> 1) ? 16 : 0));
        }
        sel_s[i] = sel;
      }
    }
    const float kmax = sqrtf(__uint_as_float(max(max(kmax_s[0], kmax_s[1]), max(kmax_s[2], kmax_s[3]))));
    // stabiliser: upper bound of the row's logits; the row maximum itself is >= max_j bias - |q| max|k|, so
    // `gap` bounds how far below the stabiliser the largest exponent argument can lie
    float mb_t[2];
    bool loose = false;
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const float qk = sqrtf(qn2[t]) * kmax, rb = rowb_s[t * kRows + tid];
      mb_t[t] = c2 * 1.01f * (qk + fmaxf(rb, 0.f));
      loose |= (mb_t[t] - c2 * (rb - qk)) > 2.f * kMaxBound;
    }
    // (the __syncthreads_or also orders the selector table writes before their first use)
    const bool exact = __syncthreads_or(loose) != 0;
    STAMP(2);

    for (int mt = 0; mt < 2; ++mt) {
      const int rown = mt * kRows + tid;
      const uint32_t rid = MASKED ? ids_s[rown] : 0;
      float mb = mb_t[mt];
      if (exact) {
        // rare path: exact row maximum of the masked logits (masked entries count as 0, as in the reference)
        float mx = -1e30f;
        for (int kb = 0; kb < n_kb; ++kb) {
          const int nk = kb < 2 ? 128 : p.I;
          if (lane == 0) issue_s(mt, kb);
          __syncwarp();
          mbar_wait(&bar, phase);
          phase ^= 1;
          tc_fence_after();
          const bool do_mask = MASKED && kb < 2;
          for (int c = 0; c < nk / 32; ++c) {
            uint32_t r[32];
            tmem_ld32(trow + c * 32, r);
            tmem_wait_ld();
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              float s = __uint_as_float(r[e]);
              if (do_mask && ids_s[kb * 128 + c * 32 + e] != rid) s = 0.f;
              mx = fmaxf(mx, s);
            }
          }
          tc_fence_before();
          __syncthreads();
        }
        mb = mx * c2;
      }
      const uint32_t rhash = DROP ? drop_row_hash(seed0, seed1, (uint32_t)bw, (uint32_t)p.heads, (uint32_t)head, kN, (uint32_t)rown) : 0u;
      float lsum0 = 0.f, lsum1 = 0.f;
      const float e0 = fast_exp2(-mb);                           // weight of every masked (zeroed) logit
      const uint32_t e0pair = pack_bf16(e0, e0);
      const uint32_t* selrow = sel_s + id_slot(rid) * (kN / 4);
      float o_run[DH + 1];
#pragma unroll
      for (int d = 0; d <= DH; ++d) o_run[d] = 0.f;

      for (int kb = 0; kb < n_kb; ++kb) {
        const int nk = kb < 2 ? 128 : p.I;
        STAMP(10 + mt * 3 + kb);
        if (lane == 0) issue_s(mt, kb);
        __syncwarp();
        mbar_wait(&bar, phase);
        phase ^= 1;
        tc_fence_after();
        STAMP(100);

        // ---- P = exp2(S*c2 - mb), packed bf16 back into TMEM ----
        const bool do_mask = MASKED && kb < 2;
        for (int c = 0; c < nk / 32; ++c) {
          uint32_t r[32];
          tmem_ld32(trow + c * 32, r);
          tmem_wait_ld();
          uint32_t pk[16];
#pragma unroll
          for (int g = 0; g < 16; ++g) {
            float x0, x1;
            ffma2(x0, x1, __uint_as_float(r[2 * g]), __uint_as_float(r[2 * g + 1]), c2, -mb);   // one FFMA2 per pair
            const bool poly = (kPolyPairs >> g) & 1u;
            const float p0 = poly ? poly_exp2(x0) : fast_exp2(x0);
            const float p1 = poly ? poly_exp2(x1) : fast_exp2(x1);
            pk[g] = pack_bf16(p0, p1);
          }
          if (do_mask) {
            const uint4* sp = reinterpret_cast<const uint4*>(selrow + kb * 32 + c * 8);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const uint4 s4 = sp[h];
              const uint32_t sw[4] = {s4.x, s4.y, s4.z, s4.w};
#pragma unroll
              for (int w = 0; w < 4; ++w) {
                pk[h * 8 + w * 2] = prmt(pk[h * 8 + w * 2], e0pair, sw[w]);
                pk[h * 8 + w * 2 + 1] = prmt(pk[h * 8 + w * 2 + 1], e0pair, sw[w] >> 16);
              }
            }
          }
          if (DROP) {
            // keep bits of this row for the chunk's 32 keys (csrc/attn.cuh); the denominator is summed from the bf16
            // values the MMA would have consumed without dropout (after the shift mask)
            const uint32_t kw = drop_keep_word(rhash, (uint32_t)(kb * 4 + c), dth);
            drop_apply16(pk, kw, lsum0, lsum1);
          }
          tmem_st16(trow + c * 16, pk);
        }
        tmem_wait_st();
        STAMP(101);
        tc_fence_before();
        __syncthreads();
        STAMP(102);

        // ---- O_blk = P.[V | 1]: k-step t goes to accumulator t % NACC, issued by warp t % NACC ----
        const int nt = nk / 16;
        if (lane == 0) {
          if (warp < NACC && warp < nt) {
            tc_fence_after();
            for (int t = warp; t < nt; t += NACC) {
              const uint64_t dv = make_smem_desc(smem_u32(Vs) + ((kb * 128 + t * 16) >> 3) * (NDC * 128), NDC * 128, 128);
              mma_ts(tmem + kOCol + warp * DHP, tmem + t * 8, dv, idescPV, t >= NACC);
            }
            mma_commit(&bar);
          } else {
            mbar_arrive(&bar);
          }
        }
        __syncwarp();
        mbar_wait(&bar, phase);
        phase ^= 1;
        tc_fence_after();
        STAMP(103);
#pragma unroll
        for (int dq = 0; dq < DHP / 16; ++dq) {
          constexpr int AG = NACC >= 2 ? 2 : 1;                    // accumulators drained per tcgen05.wait::ld
#pragma unroll
          for (int a0 = 0; a0 < NACC; a0 += AG) {
            if (a0 < nt) {
              uint32_t o[AG][16];
#pragma unroll
              for (int a = 0; a < AG; ++a) tmem_ld16(trow + kOCol + (a0 + a) * DHP + dq * 16, o[a]);
              tmem_wait_ld();
#pragma unroll
              for (int a = 0; a < AG; ++a)
#pragma unroll
                for (int d = 0; d < 16; ++d)
                  if (dq * 16 + d <= DH) o_run[dq * 16 + d] += __uint_as_float(o[a][d]);
            }
          }
        }
        tc_fence_before();
        __syncthreads();   // everyone has drained O / P before the next S MMA overwrites the columns
        STAMP(104);
      }

      // ---- epilogue: normalise, write bf16 output row slice and log-sum-exp ----
      const float l_run = DROP ? lsum0 + lsum1 : o_run[DH];
      const float inv = (DROP ? p.inv_keep : 1.f) / l_run;
      __nv_bfloat16* og = (__nv_bfloat16*)p.out + ((size_t)bw * kN + rown) * p.C + head * DH;
      if constexpr (DH % 4 == 0) {
#pragma unroll
        for (int d = 0; d < DH; d += 4) {
          uint2 v;
          v.x = pack_bf16(o_run[d] * inv, o_run[d + 1] * inv);
          v.y = pack_bf16(o_run[d + 2] * inv, o_run[d + 3] * inv);
          *reinterpret_cast<uint2*>(og + d) = v;
        }
      } else {
#pragma unroll
        for (int d = 0; d < DH; ++d) og[d] = __float2bfloat16(o_run[d] * inv);
      }
      p.lse[((size_t)bw * p.heads + head) * kN + rown] = (mb + __log2f(l_run)) * 0.6931471805599453f;
    }
    bw = next_s[it & 1];   // written before this window's first block barrier, read after its last one; two slots, so
                           // that the next window's write cannot overtake a slow thread's read
  }
  STAMP(150);
#undef STAMP
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, kTmemCols);
}

template <int DH>
int launch_tc(const AttnParams& p, cudaStream_t st) {
  constexpr int DHP = Cfg<DH>::DHP, KS = Cfg<DH>::KS;
  const int NKT = kN + p.I;
  const TcSmem L = tc_layout(KS, DHP, NKT, p.ids != nullptr);
  const size_t smem = L.total;
  const int per_sm = (int)((227 * 1024) / (smem + 1024));
  int grid = 148 * (per_sm > 4 ? 4 : (per_sm < 1 ? 1 : per_sm));
  grid -= grid % p.heads;
  const int need = p.B * p.P * p.heads;
  if (grid > need) grid = need;
  if (grid < p.heads) grid = p.heads;
  auto kern = p.drop_thresh ? (p.ids ? attn_fwd_tc_kernel<DH, true, true> : attn_fwd_tc_kernel<DH, false, true>)
                            : (p.ids ? attn_fwd_tc_kernel<DH, true, false> : attn_fwd_tc_kernel<DH, false, false>);
  PWA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (p.work) PWA_CUDA_OK(cudaMemsetAsync(p.work, 0, sizeof(unsigned int) * p.heads, st));
  kern<<<grid, kRows, smem, st>>>(p);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

}  // namespace

bool attn_tc_supported(const AttnParams& p, int dtype) {
  if (dtype == PWA_F16) return attn_ws_supported(p, PWA_BF16) && attn_tc_bwd_supported(p, PWA_BF16);
  if (dtype != PWA_BF16) return false;
  if (p.N != kN) return false;                                   // two 128-row tiles / two 128-key content blocks
  if (p.wd > 4 || p.wh + p.ww > 16) return false;                // one-hot bias columns must fit the layout
  if (p.I % 32 != 0 || p.I > 128) return false;                  // prompt block = one MMA of N = I, read in 32-column chunks
  const int dh = p.C / p.heads;
  if (!(dh == 12 || dh == 24 || dh == 48 || dh == 6 || dh == 3)) return false;
  const TcSmem L = tc_layout((dh + 4 + 15) / 16, (dh + 1 + 15) / 16 * 16, kN + p.I, true);
  return L.total <= 200 * 1024;
}

int attn_tc_forward(const AttnParams& p, cudaStream_t st) {
  switch (p.C / p.heads) {
    case 3: return launch_tc<3>(p, st);
    case 6: return launch_tc<6>(p, st);
    case 12: return launch_tc<12>(p, st);
    case 24: return launch_tc<24>(p, st);
    case 48: return launch_tc<48>(p, st);
  }
  set_error("tcgen05 attention: head_dim %d not instantiated", p.C / p.heads);
  return PWA_ERR_UNSUPPORTED;
}

}  // namespace pwa
