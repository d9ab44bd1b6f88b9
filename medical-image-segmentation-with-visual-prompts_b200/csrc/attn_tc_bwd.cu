// (c) backward of the fused prompted window attention on tcgen05 tensor cores + TMEM, bf16 or fp16 I/O.
//
// One persistent CTA per SM (800 threads, all 512 TMEM columns) = one fixed head, walking over (sample, window)
// pairs.  Everything is computed in the TRANSPOSED orientation: the 128 TMEM lanes are KEYS (one key block:
// content 0-127, content 128-255, prompt tokens) and the TMEM columns are query rows, one UNIT = 64 rows:
//     S^T [128k x 64r] = K'.Q'^T      dP^T [128k x 64r] = V'.dO'^T        (SS MMAs, fp32 accum in TMEM)
//     P^T = exp2(S^T*c - lse)         g^T = P^T * dP^T                     (one thread per key, 32 rows each)
//     dV  [128k x dh] += P^T.dO       dK' [128k x dh'] += g^T.Q'           (TS MMAs: A = bf16 P^T / g^T in TMEM)
//     dKaug[128k x 16] += g^T.[onehot_h | onehot_w]                        (= relative-position-bias table
//                                                                           gradients, accumulated in TMEM over
//                                                                           ALL windows the CTA processes)
//     dQ' [128r x dh'] += g.K'                                             (A = g^T staged to smem as an MN-major
//                                                                           operand, B = K' MN-major)
// lse and delta = rowsum(dO*O) are known, so no row reduction is needed and there is exactly one exponential per
// (query, key) pair.  Per logit the CUDA cores issue FFMA + MUFU + FMUL + 2 x 1/2 F2FP: `- delta` rides in two
// spare K columns of the dP^T MMA (bf16 hi/lo split, V' columns = 1) and the multiplicative shift mask is applied
// on the PACKED bf16 pairs with one PRMT each (masked P^T -> exp(-lse) of that query, masked g^T -> 0).
//
// A tcgen05.mma costs ~100 clk of latency per dependent instruction and ~200 clk of issue time, but streams
// issued by different warps overlap (csrc/ubench.cu).  A clock64 timeline of the previous, barrier-synchronous
// version showed 500 clk of MUFU work per unit against 1700 clk of exposed MMA latency, so the CTA is
// warp-specialised and every hand-off is an mbarrier:
//     warps 0-15  compute, two groups of 8 that ping-pong over the units (group 0: even units, group 1: odd units;
//                 key = tid % 128, warpgroup = row half, two passes of 16 rows to stay within the register budget of an
//                 800-thread CTA): TMEM ld -> exp/mul/pack -> TMEM st + g^T to smem.  The
//                 waits / TMEM round trips / proxy fences of one group hide behind the exponentials of the other.
//     warp  16    issues S^T / dP^T of unit g as soon as the chains of unit g - NBUF have consumed that buffer
//     warps 17-19 issue the dV / dK' / dKaug chains of a unit when its packed operands are ready
//     warp  20    issues dQ' per (key block, query tile)
//     warps 21-24 service: stage the NEXT window's operands into the other half of a double buffer (global -> smem) and
//                 drain every accumulator of the current window (dV / dK' per key block, dQ' per window)
// Measured (tools/timeline.py, `make TIMELINE=1`): the kernel is now bound by the tensor pipe's per-instruction cost --
// 228 small MMAs per window at ~50 clk each whatever their N (csrc/ubench.cu), plus the stalls of five in-order
// streams with dependent accumulations -- not by the MUFU pipe; fewer, fatter MMAs (merged dK'/dKaug chains, 128-row
// units) are the next step.
// S^T / dP^T are NBUF-fold buffered in TMEM (3 x 128 columns at head_dim <= 12), so the compute warps run
// back to back on the MUFU pipe while the tensor pipe works 1-2 units behind / ahead.
// Semantics follow the reference autograd of window_attention.py:49-58 (mask multiplicative, pre-softmax:
// masked logits are 0, keep weight exp(-lse), and pass no gradient to q.k or the bias).
#include "attn.cuh"
#include "tc_common.cuh"

namespace pwa {
using namespace tc;

namespace {

constexpr int kN = 256;
constexpr int kThreadsB = 800;
constexpr int kCompute = 256;     // compute threads per group: group 0 = warps 0-7 (even units), group 1 = warps 8-15 (odd units)
constexpr int kGroups = 2;
constexpr int kIssue0 = kGroups * 8;   // first MMA-issuer warp (S, V, K, A, Q)
constexpr int kProd0 = kIssue0 + 5;    // first staging warp
constexpr int kProd = 128;        // service threads (4 warps, one per TMEM lane quadrant): staging + accumulator drains
constexpr int kIds = 28;          // region ids 0..26 and 100 (-> 27), see pwa_region_ids

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
}
__device__ __forceinline__ int id_slot(uint32_t id) { return id < (uint32_t)(kIds - 1) ? (int)id : kIds - 1; }

template <int DH> struct BCfg {
  static constexpr int DHP = (DH + 15) / 16 * 16;
  static constexpr int KS = (DH + 4 + 15) / 16;
  static constexpr int DKC = KS * 16;                            // staged K' / Q' width = dK' / dQ' accumulator width
  static constexpr bool FOLD = (DHP - DH) >= 2;                  // -delta rides in two spare K columns of the dP^T MMA
  static constexpr int ACC = DHP + DKC + 2 * DKC + 48;           // dV, dK', dQ'[2], dKaug[3]
  static constexpr int NBUF = (3 * 128 + ACC <= 512) ? 3 : ((2 * 128 + ACC <= 512) ? 2 : 1);
};

struct BwdSmem {
  // shared by all windows
  uint32_t qaug, kaug, g, gth, gtw, gtd, gtok;
  // per operand buffer (offsets relative to the buffer base)
  uint32_t q, k, v, dO, lse2, delta, wp, rs, sel, ids, opnd_bytes;
  uint32_t opnd0;        // base of operand buffer 0; buffer b at opnd0 + b * opnd_bytes
  int opb, gsb;          // number of operand / g^T buffers
  uint32_t total;
};

__host__ __device__ inline BwdSmem bwd_layout(int KS, int DHP, int NKT, int wh, int ww, int wd, int I, bool masked) {
  BwdSmem s;
  const int NKR = kN + 128;
  uint32_t o = 0;
  s.q = o; o += KS * 2 * kN * 16;
  s.k = o; o += KS * 2 * NKR * 16;               // key-side operands always hold 3 x 128 rows: the prompt block is issued as M = 128
  s.v = o; o += (DHP / 8) * NKR * 16;
  s.dO = o; o += (DHP / 8) * kN * 16;
  s.lse2 = o; o += kN * 4;
  s.delta = o; o += kN * 4;
  s.wp = o; o += kN * 2;                          // bf16 exp(-lse) per query (value of a masked P entry)
  s.rs = o; o += kN * 4;                          // dropout hash of every query row (csrc/attn.cuh: drop_row_hash)
  s.sel = o; o += masked ? kIds * (kN / 4) * 4 : 0;   // PRMT selectors [id slot][4 tokens], as in attn_tc.cu
  s.ids = o; o += kN;
  s.opnd_bytes = (o + 127) & ~127u;
  uint32_t sh = 0;
  s.qaug = sh; sh += 2 * kN * 16;
  s.kaug = sh; sh += 2 * NKR * 16;
  s.gth = sh; sh += wh * wh * 4;
  s.gtw = sh; sh += ww * ww * 4;
  s.gtd = sh; sh += wd * wd * 4;
  s.gtok = sh; sh += (I + 4) * 4;
  sh = (sh + 127) & ~127u;
  const uint32_t gbytes = 128 * 128 * 2;
  const uint32_t budget = 220 * 1024;
  s.gsb = (sh + 2 * gbytes + s.opnd_bytes <= budget) ? 2 : 1;
  s.g = sh; sh += s.gsb * gbytes;
  s.opb = (sh + 2 * s.opnd_bytes <= budget) ? 2 : 1;
  s.opnd0 = sh;
  s.total = sh + s.opb * s.opnd_bytes;
  return s;
}

template <int DH, typename E>
__device__ __forceinline__ void load_row_b(const E* src, E (&dst)[DH]) {
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

template <int DH, typename E>
__device__ __forceinline__ void store_row_b(E* dst, const float* v, float mul) {
  if constexpr (DH % 4 == 0) {
#pragma unroll
    for (int d = 0; d < DH; d += 4) {
      uint2 w;
      w.x = pack2t<E>(v[d] * mul, v[d + 1] * mul);
      w.y = pack2t<E>(v[d + 2] * mul, v[d + 3] * mul);
      *reinterpret_cast<uint2*>(dst + d) = w;
    }
  } else {
#pragma unroll
    for (int d = 0; d < DH; ++d) dst[d] = from_f32<E>(v[d] * mul);
  }
}

// [real DH | up to 4 extra columns | zero pad] -> NCH chunks of 8 columns, chunk c of row r at base + c*stride + r*16
template <int DH, int NCH, typename E>
__device__ __forceinline__ void store_chunks_b(uint8_t* base, uint32_t chunk_stride, int row, const E (&real)[DH],
                                               E x0, E x1, E x2, E x3) {
  const E zero = from_f32<E>(0.f);
#pragma unroll
  for (int c = 0; c < NCH; ++c) {
    __align__(16) E tmp[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int col = c * 8 + e;
      const int x = col - DH;
      E v = zero;
      if (col < DH) v = real[col < DH ? col : 0];
      else if (x == 0) v = x0;
      else if (x == 1) v = x1;
      else if (x == 2) v = x2;
      else if (x == 3) v = x3;
      tmp[e] = v;
    }
    *reinterpret_cast<uint4*>(base + c * chunk_stride + row * 16) = *reinterpret_cast<const uint4*>(tmp);
  }
}

// named barriers among the staging warps / the compute warps only
__device__ __forceinline__ void prod_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kProd) : "memory"); }
__device__ __forceinline__ void comp_sync() { asm volatile("bar.sync 2, %0;" ::"n"(kCompute) : "memory"); }

enum {
  bFullS = 0,      // [3] scores of a unit complete                 (tcgen05.commit, count 1)
  bDoneC = 3,      // [3] dV / dK' / dKaug chains of a unit retired (three commits) and its bReady phase consumed by the
                   //     dQ' issuer (one arrival): count 4
  bReady = 6,      // [3] packed P^T / g^T of a unit written        (256 compute threads)
  bDoneQ = 9,      // [2] dQ' chain of a query tile retired         (commit)
  bAccFree = 11,   // dV / dK' accumulators of a key block drained  (128 service threads)
  bDqFree = 12,    // dQ' accumulators of a window drained          (128)
  bOpFull = 13,    // [2] operand buffer staged                     (128)
  bKbDone = 15,    // all three accumulation chains of a key block retired (three commits, count 3)
  bWinQ = 16,      // every dQ' chain of a window retired            (commit)
  kNumBars = 17
};

// DROP: attention dropout (window_attention.py:57) with the mask of csrc/attn.cuh.  P^T feeds dV dropped (one AND on
// the packed pairs, after the shift mask; the inverse keep rate is applied when dV is drained), dP^T is masked and
// scaled before delta is subtracted (so delta cannot ride in the dP^T MMA: FOLD is off).
// E: element type of the token tensors and of the MMA operands (bf16 or fp16).  P^T uses the exact log-sum-exp (P <= 1), so
// fp16's range matters only for g = P (dP - delta), delta and the stored gradients: under a large loss scale they overflow to
// inf (NaN where inf meets inf), never to a finite value, and a non-finite dout stays non-finite -- GradScaler sees it.
template <int DH, bool MASKED, bool DROP, typename E>
// (72 registers is the hard cap: 25 warps spread 7/6/6/6 over the four sub-partitions of 16 384 registers each, and
//  7 warps x 32 x 80 does not fit -- a __maxnreg__(80) build fails to launch)
__global__ void __launch_bounds__(kThreadsB, 1) attn_bwd_tc_kernel(AttnParams p) {
  constexpr int DHP = BCfg<DH>::DHP, KS = BCfg<DH>::KS, DKC = BCfg<DH>::DKC, NBUF = BCfg<DH>::NBUF;
  constexpr bool FOLD = BCfg<DH>::FOLD && !DROP;
  // TMEM column map: NBUF x [S^T 64 | dP^T 64], then the accumulators
  constexpr uint32_t cACC = NBUF * 128, cDV = cACC, cDK = cDV + DHP, cDQ = cDK + DKC, cAUG = cDQ + 2 * DKC;
  static_assert(cAUG + 48 <= 512, "TMEM column budget");

  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar[kNumBars];
  __shared__ uint32_t tmem_base_s;

#ifdef PWA_TIMELINE_BUILD
  const long long t_kernel_start = clock64();
#endif
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NKT = kN + p.I;
  const int NKR = kN + 128;                        // rows allocated for key-side operands (prompt block issued as M = 128)
  const BwdSmem L = bwd_layout(KS, DHP, NKT, p.wh, p.ww, p.wd, p.I, MASKED);
  const int OPB = L.opb, GSB = L.gsb;
  // (GSB, OPB are 1 or 2, but `& (GSB - 1)` / a division-free form instead of `% GSB`, `/ GSB` in the unit loop were both
  //  measured SLOWER in the masked dropout variants, 708 -> 744-765 us at enc0: ptxas then spills 40 bytes more inside the
  //  unit loop at the 72-register cap; the divisions stay)
  uint8_t* Qa = smem + L.qaug;
  uint8_t* Ka = smem + L.kaug;
  float* gth_s = reinterpret_cast<float*>(smem + L.gth);
  float* gtw_s = reinterpret_cast<float*>(smem + L.gtw);
  float* gtd_s = reinterpret_cast<float*>(smem + L.gtd);
  float* gtok_s = reinterpret_cast<float*>(smem + L.gtok);

  const int head = blockIdx.x % p.heads;
  const float inv_scale = 1.f / p.scale;
  const float c2 = p.scale * 1.4426950408889634f;
  const uint32_t seed0 = DROP ? (p.drop_seed ? p.drop_seed[0] : p.seed_host[0]) : 0u;
  const uint32_t seed1 = DROP ? (p.drop_seed ? p.drop_seed[1] : p.seed_host[1]) : 0u;
  const DropThresh& dth = p.drop_planes;          // constant bank (filled by the dispatcher)
  const float keep_scale = DROP ? p.inv_keep : 1.f;
  const E one = from_f32<E>(1.f), zero = from_f32<E>(0.f);

  // ---- once per CTA: zero everything the MMAs may touch beyond the staged rows, window-independent operands ----
  for (uint32_t i = tid; i < L.total / 16; i += kThreadsB) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  for (int n = tid; n < kN; n += kThreadsB) {
    const int iw = (n / p.wd) % p.ww, ih = n / (p.wd * p.ww);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      __align__(16) E tmp[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int col = c * 8 + e;
        tmp[e] = (col < p.wh) ? (col == ih ? one : zero) : ((col - p.wh < p.ww && col - p.wh == iw) ? one : zero);
      }
      *reinterpret_cast<uint4*>(Qa + c * (kN * 16) + n * 16) = *reinterpret_cast<const uint4*>(tmp);
    }
  }
  // (bias tables of this head through shared memory: the gradient accumulators gth_s / gtw_s / gtok_s are free until the
  //  end of the kernel and are zeroed again below)
  for (int i = tid; i < p.wh * p.wh; i += kThreadsB) gth_s[i] = p.th[head * p.wh * p.wh + i];
  for (int i = tid; i < p.ww * p.ww; i += kThreadsB) gtw_s[i] = p.tw[head * p.ww * p.ww + i];
  for (int i = tid; i < p.I; i += kThreadsB) gtok_s[i] = p.tok[head * p.I + i];
  __syncthreads();
  for (int j = tid; j < NKT; j += kThreadsB) {
    const bool content = j < kN;
    const int jw = (j / p.wd) % p.ww, jh = j / (p.wd * p.ww);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      __align__(16) E tmp[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int col = c * 8 + e;
        float v = 0.f;
        if (content) {
          if (col < p.wh) v = gth_s[col * p.wh + jh];
          else if (col - p.wh < p.ww) v = gtw_s[(col - p.wh) * p.ww + jw];
        } else if (col < p.wh) {
          v = gtok_s[j - kN];
        }
        tmp[e] = from_f32<E>(v * inv_scale);
      }
      *reinterpret_cast<uint4*>(Ka + c * (NKR * 16) + j * 16) = *reinterpret_cast<const uint4*>(tmp);
    }
  }
  __syncthreads();
  for (int i = tid; i < p.wh * p.wh; i += kThreadsB) gth_s[i] = 0.f;
  for (int i = tid; i < p.ww * p.ww; i += kThreadsB) gtw_s[i] = 0.f;
  for (int i = tid; i < p.I + 4; i += kThreadsB) gtok_s[i] = 0.f;
  if (tid == 0) {
    for (int i = 0; i < 3; ++i) {
      mbar_init(&bar[bFullS + i], 1);
      mbar_init(&bar[bDoneC + i], 4);
      mbar_init(&bar[bReady + i], kCompute);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bar[bDoneQ + i], 1);
      mbar_init(&bar[bOpFull + i], kProd);
    }
    mbar_init(&bar[bAccFree], kProd);
    mbar_init(&bar[bDqFree], kProd);
    mbar_init(&bar[bKbDone], 3);
    mbar_init(&bar[bWinQ], 1);
    fence_mbar_init();
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (warp == 0) tmem_alloc(&tmem_base_s, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
#ifdef PWA_WATCHDOG
  if (tid == 0 && blockIdx.x == 0) printf("pwa watchdog: bwd mbarrier base smem 0x%x (index = (addr - base) / 8)\n", smem_u32(&bar[0]));
#endif

  const int n_kb = p.I > 0 ? 3 : 2;
  const int n_units = n_kb * 4;
  const int n_pairs = p.B * p.P;
  const int stride = gridDim.x / p.heads;
  const int bw0 = blockIdx.x / p.heads;

  // clock64 timelines of CTA 0 (tools/timeline.py): compiled in only with -DPWA_TIMELINE_BUILD
#ifdef PWA_TIMELINE_BUILD
#ifndef PWA_TL_SERVICE_WARP
#define PWA_TL_SERVICE_WARP 0      // which of the four service warps records its timeline
#endif
  long long* tl = reinterpret_cast<long long*>(p.delta);
  int tli = 0;
  const bool rec = p.debug && blockIdx.x == 0 &&
                   (tid == 0 || tid == kIssue0 * 32 || tid == (kIssue0 + 1) * 32 || tid == (kProd0 + PWA_TL_SERVICE_WARP) * 32 || tid == 256 ||
                    tid == (kIssue0 + 4) * 32);
  const int tlb = tid == 0 ? 0 : (tid == kIssue0 * 32 ? 2048 : (tid == (kIssue0 + 1) * 32 ? 4096 : (tid == 256 ? 8192 :
                  (tid == (kIssue0 + 4) * 32 ? 10240 : 6144))));
#define STAMP(tag) do { if (rec && tli < 1000) { tl[tlb + 2 * tli] = clock64(); tl[tlb + 2 * tli + 1] = (tag); ++tli; } } while (0)
  if (rec && tid == 0) { tl[16000] = t_kernel_start; tl[16001] = clock64(); }   // kernel entry, end of the per-CTA setup
#else
#define STAMP(tag) do { } while (0)
#endif

  if (warp < kIssue0) {
    // =============================================================================================
    // compute warps: two groups of 8 warps ping-pong over the units (group 0: even units = first 64-row half of a
    // query tile, group 1: odd units + every accumulator drain), so that the waits / TMEM round trips / proxy
    // fences of one group hide behind the exponentials of the other and 4 warps per scheduler feed the MUFU pipe
    // =============================================================================================
    const int grp = warp >> 3;
    const int n_groups = NBUF >= 2 ? kGroups : 1;                    // single S^T buffer: nothing to overlap
    const int wg = (warp >> 2) & 1;
    const int lane_row = tid & 127;                  // TMEM lane owned by this thread (key in S^T, row in dQ)
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    int it = 0;
    for (int bw = bw0; bw < n_pairs && grp < n_groups; bw += stride, ++it) {
      const int b = bw / p.P;
      const int ob = it % OPB;
      const uint8_t* opnd = smem + L.opnd0 + ob * L.opnd_bytes;
      const float* lse2_s = reinterpret_cast<const float*>(opnd + L.lse2);
      const float* delta_s = reinterpret_cast<const float*>(opnd + L.delta);
      const E* wp_s = reinterpret_cast<const E*>(opnd + L.wp);
      const uint32_t* rs_s = reinterpret_cast<const uint32_t*>(opnd + L.rs);
      const uint32_t* sel_s = reinterpret_cast<const uint32_t*>(opnd + L.sel);
      const uint8_t* ids_s = opnd + L.ids;
      STAMP(1);
      mbar_wait(&bar[bOpFull + ob], (it / OPB) & 1);
      STAMP(2);
      // (parity waits stay in step without awaiting the other group's phases: with NBUF = 3 a group has seen the S
      //  of unit g-2, which was committed after that of g-3 = the previous phase of its buffer; with NBUF = 2 each
      //  group owns one buffer; NBUF = 1 runs a single group.  Phases cannot run ahead of a waiter either: the next
      //  use of a buffer needs this group's own bReady arrival.)
      for (int unit = grp; unit < n_units; unit += n_groups) {
        const int g = it * n_units + unit, buf = g % NBUF, par = (g / NBUF) & 1;
        const int kb = unit >> 2, u = unit & 3, mt = u >> 1, hf = u & 1;
        const int nk = kb < 2 ? 128 : p.I;                         // valid keys in this block
        const bool warp_ok = (warp & 3) * 32 < nk;                 // (nk is a multiple of 32: whole warps are valid or not)
        const bool do_mask = MASKED && kb < 2;
        const int qt = it * n_kb * 2 + kb * 2 + mt, gs = qt % GSB;
        uint8_t* Gs = smem + L.g + gs * (128 * 128 * 2);
        const uint32_t cS = buf * 128, cP = cS + 64;
        STAMP(10 + unit);
        mbar_wait(&bar[bFullS + buf], par);
        tc_fence_after();
        STAMP(100);
        // dQ' of the query tile that used this g^T buffer before must have retired (both groups write row halves of it)
        if (qt >= GSB) mbar_wait(&bar[bDoneQ + gs], ((qt / GSB) - 1) & 1);
        if (warp_ok) {
          // ---- this thread: key = lane_row, rows r0 .. r0+31, in two passes of 16 (register budget: 768 threads) ----
          const int r0 = mt * 128 + hf * 64 + wg * 32;
          const uint32_t cid = do_mask ? ids_s[kb * 128 + lane_row] : 0;
          // dropout: this warp's tile is 32 keys (one key chunk) x 32 rows.  Lane l builds the keep word of row
          // r0 + drop_bitpos_inv(l), the 32x32 bit tile is transposed across the warp, and every lane fetches the word of
          // its key's bit position: bit drop_bitpos(i) of T = keep(row r0 + i, this thread's key), the same pair layout
          // as in the forward kernel, along rows.
          uint32_t T = 0u;
          if (DROP) {
            const uint32_t kwd = drop_keep_word(rs_s[r0 + drop_bitpos_inv(lane)], (uint32_t)(kb * 4 + (warp & 3)), dth);
            T = __shfl_sync(0xffffffffu, drop_transpose_tile(kwd, lane), drop_bitpos(lane));
          }
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            uint32_t s[16], dp[16];
            tmem_ld16(trow + cS + wg * 32 + h * 16, s);
            tmem_ld16(trow + cP + wg * 32 + h * 16, dp);
            tmem_wait_ld();
            uint32_t pk[8], gk[8];
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {
              const float4 l4 = *reinterpret_cast<const float4*>(lse2_s + r0 + h * 16 + q4 * 4);
              const float lv[4] = {l4.x, l4.y, l4.z, l4.w};
              float nd[4] = {0.f, 0.f, 0.f, 0.f};                 // -delta of the four rows (delta_s holds the negatives)
              if (!FOLD) {
                const float4 d4 = *reinterpret_cast<const float4*>(delta_s + r0 + h * 16 + q4 * 4);
                nd[0] = d4.x; nd[1] = d4.y; nd[2] = d4.z; nd[3] = d4.w;
              }
              float pv[4], gv[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int r = q4 * 4 + e;
                pv[e] = fast_exp2(fmaf(__uint_as_float(s[r]), c2, -lv[e]));
                if (DROP) {
                  // d P = keep * d P~ / keep_rate, then - delta: one bit test that predicates the multiply-add (the row's
                  // -delta is used by this thread exactly once, so it is updated in place)
                  float t = nd[e];
                  if (T & (1u << drop_bitpos(h * 16 + r))) t = fmaf(__uint_as_float(dp[r]), keep_scale, t);
                  gv[e] = pv[e] * t;
                } else {
                  const float dpe = __uint_as_float(dp[r]);
                  gv[e] = pv[e] * (FOLD ? dpe : dpe + nd[e]);
                }
              }
              pk[q4 * 2] = pack2t<E>(pv[0], pv[1]);
              pk[q4 * 2 + 1] = pack2t<E>(pv[2], pv[3]);
              gk[q4 * 2] = pack2t<E>(gv[0], gv[1]);
              gk[q4 * 2 + 1] = pack2t<E>(gv[2], gv[3]);
            }
            if (do_mask) {
              const uint4 s4 = *reinterpret_cast<const uint4*>(sel_s + id_slot(cid) * (kN / 4) + r0 / 4 + h * 4);
              const uint32_t sw[4] = {s4.x, s4.y, s4.z, s4.w};
              const uint4* wpp = reinterpret_cast<const uint4*>(wp_s + r0 + h * 16);
              const uint4 wa = wpp[0], wb = wpp[1];
              const uint32_t ww[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
              for (int w = 0; w < 4; ++w) {
                pk[w * 2] = prmt(pk[w * 2], ww[w * 2], sw[w]);
                pk[w * 2 + 1] = prmt(pk[w * 2 + 1], ww[w * 2 + 1], sw[w] >> 16);
                gk[w * 2] = prmt(gk[w * 2], 0u, sw[w]);
                gk[w * 2 + 1] = prmt(gk[w * 2 + 1], 0u, sw[w] >> 16);
              }
            }
            if (DROP) {
#pragma unroll
              for (int w = 0; w < 8; ++w)                          // dropped P^T entries do not reach dV (pair h * 8 + w of the tile)
                pk[w] &= drop_prmt(T << ((h * 8 + w) & 7), (h * 8 + w) < 8 ? 0xBBAAu : 0x9988u);
            }
            tmem_st8(trow + cS + wg * 32 + h * 8, pk);             // packed over this warpgroup's own consumed columns
            tmem_st8(trow + cP + wg * 32 + h * 8, gk);
            // g^T -> smem as the MN-major A operand of dQ = g.K : [row group of 8][key group of 8][key%8][16 B]
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              const int rg = (hf * 64 + wg * 32) / 8 + h * 2 + q;
              *reinterpret_cast<uint4*>(Gs + rg * 2048 + lane_row * 16) = make_uint4(gk[q * 4], gk[q * 4 + 1], gk[q * 4 + 2], gk[q * 4 + 3]);
            }
          }
          STAMP(102);
          tmem_wait_st();
        }
        fence_proxy_async_smem();
        tc_fence_before();
        mbar_arrive(&bar[bReady + buf]);
        STAMP(103);
      }
    }
  } else if (warp < kProd0) {
    // =============================================================================================
    // MMA issuers (one lane each)
    // =============================================================================================
    // The WHOLE warp runs the control flow with warp-uniform values and only the tcgen05 instructions sit under
    // elect.sync: the MMA operands then live in uniform registers.  With the loop inside `if (lane == 0)` ptxas wrapped
    // every MMA in an ELECT + R2UR.BROADCAST waterfall loop, ~170 clk per instruction and issuing thread (this is what
    // round 1 measured as "one thread issues a tcgen05.mma only every ~100-200 clk").
    {
      const uint32_t tmem = __shfl_sync(0xffffffffu, tmem_base_s, 0);
      const uint32_t idescT = make_idesc<E>(128, 64, 0, 0);       // S^T, dP^T : A K-major, B K-major, N = 64 rows
      const uint32_t idescDV = make_idesc<E>(128, DHP, 0, 1);     // dV  : A tmem, B = dO MN-major
      const uint32_t idescDK = make_idesc<E>(128, DKC, 0, 1);     // dK' : A tmem, B = Q' MN-major
      const uint32_t idescAUG = make_idesc<E>(128, 16, 0, 1);     // dKaug
      const uint32_t idescDQ = make_idesc<E>(128, DKC, 1, 1);     // dQ' : A = g smem MN-major, B = K' MN-major
      const int role = __shfl_sync(0xffffffffu, warp - kIssue0, 0); // 0 S, 1 V, 2 K, 3 A, 4 Q
      int it = 0;
      for (int bw = bw0; bw < n_pairs; bw += stride, ++it) {
        const int ob = it % OPB;
        const uint32_t opnd = smem_u32(smem + L.opnd0 + ob * L.opnd_bytes);
        const uint32_t Qs = opnd + L.q, Ks = opnd + L.k, Vs = opnd + L.v, dOs = opnd + L.dO;
        mbar_wait(&bar[bOpFull + ob], (it / OPB) & 1);
        for (int unit = 0; unit < n_units; ++unit) {
          const int g = it * n_units + unit, buf = g % NBUF, par = (g / NBUF) & 1;
          const int kb = unit >> 2, u = unit & 3, mt = u >> 1, hf = u & 1;
          const uint32_t qrow = (uint32_t)(mt * 128 + hf * 64);
          const uint32_t cS = buf * 128, cP = cS + 64;
          const uint32_t acc0 = u > 0;
          if (role == 0) {
            // the chains of the unit that used this buffer before must have consumed its packed P^T / g^T
            if (g >= NBUF) mbar_wait(&bar[bDoneC + buf], par ^ 1);
            tc_fence_after();
            STAMP(10 + unit);
            if (elect_one_sync()) {
#pragma unroll
              for (int ks = 0; ks < KS; ++ks) {
                const uint64_t da = make_smem_desc(Ks + ks * 2 * (NKR * 16) + kb * (128 * 16), NKR * 16, 128);
                const uint64_t db = make_smem_desc(Qs + ks * 2 * (kN * 16) + qrow * 16, kN * 16, 128);
                mma_ss(tmem + cS, da, db, idescT, ks > 0);
              }
              {
                const uint64_t da = make_smem_desc(smem_u32(Ka) + kb * (128 * 16), NKR * 16, 128);
                const uint64_t db = make_smem_desc(smem_u32(Qa) + qrow * 16, kN * 16, 128);
                mma_ss(tmem + cS, da, db, idescT, 1);
              }
#pragma unroll
              for (int ks = 0; ks < DHP / 16; ++ks) {
                const uint64_t da = make_smem_desc(Vs + ks * 2 * (NKR * 16) + kb * (128 * 16), NKR * 16, 128);
                const uint64_t db = make_smem_desc(dOs + ks * 2 * (kN * 16) + qrow * 16, kN * 16, 128);
                mma_ss(tmem + cP, da, db, idescT, ks > 0);
              }
              mma_commit(&bar[bFullS + buf]);
            }
            __syncwarp();
            STAMP(100);
          } else if (role <= 3) {
            mbar_wait(&bar[bReady + buf], par);
            if (role != 3 && u == 0) {
              // the previous key block's accumulators must have been drained before they are restarted
              const int tile = it * n_kb + kb;
              if (tile > 0) mbar_wait(&bar[bAccFree], (tile - 1) & 1);
            }
            tc_fence_after();
            STAMP(10 + unit);
            // K = 64 rows = 4 k-steps; A = packed bf16 in TMEM: rows 0-31 live at cols 0-15, rows 32-63 at cols 32-47
            if (elect_one_sync()) {
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const uint32_t acol = (t >> 1) * 32 + (t & 1) * 8;
              const uint32_t rows = qrow + t * 16;
              if (role == 1) {                                       // dV += P^T.dO
                const uint64_t bdo = make_smem_desc(dOs + rows * 16, 128, kN * 16);
                mma_ts(tmem + cDV, tmem + cS + acol, bdo, idescDV, acc0 | (t > 0));
              } else if (role == 2) {                                // dK' += g^T.Q'
                const uint64_t bq = make_smem_desc(Qs + rows * 16, 128, kN * 16);
                mma_ts(tmem + cDK, tmem + cP + acol, bq, idescDK, acc0 | (t > 0));
              } else {                                               // dKaug += g^T.Qaug   (accumulates over all windows)
                const uint64_t bqa = make_smem_desc(smem_u32(Qa) + rows * 16, 128, kN * 16);
                mma_ts(tmem + cAUG + kb * 16, tmem + cP + acol, bqa, idescAUG, (it > 0) | acc0 | (t > 0));
              }
            }
            mma_commit(&bar[bDoneC + buf]);
            if (u == 3) mma_commit(&bar[bKbDone]);                 // key block complete: the service warps drain dV / dK'
            }
            __syncwarp();
            STAMP(100);
          } else {
            // Every unit's phase is awaited in order, AND this issuer takes part in the recycling of the S^T ring: the dQ'
            // chains are not among the commits that free a buffer, so without the arrival below the compute groups could
            // run four units ahead of this warp (e.g. while it waits for bDqFree at a window start), bReady[buf] would
            // complete two phases, and a parity wait two phases behind never returns (observed as a rare hang).
            mbar_wait(&bar[bReady + buf], par);
            if (elect_one_sync()) mbar_arrive(&bar[bDoneC + buf]);
            __syncwarp();
            STAMP(10 + unit);
            if (hf == 0) continue;
            // dQ'[mt] += g[128 rows x nk keys] . K'[kb]
            const int nk = kb < 2 ? 128 : p.I;
            const int qt = it * n_kb * 2 + kb * 2 + mt, gs = qt % GSB;
            const uint32_t Gs = smem_u32(smem + L.g + gs * (128 * 128 * 2));
            if (kb == 0 && it > 0) mbar_wait(&bar[bDqFree], (it - 1) & 1);
            tc_fence_after();
            if (elect_one_sync()) {
#pragma unroll
              for (int t = 0; t < 8; ++t) {
                if (t * 16 < nk) {
                  const uint64_t da = make_smem_desc(Gs + t * 256, 128, 2048);
                  const uint64_t db = make_smem_desc(Ks + (kb * 128 + t * 16) * 16, 128, NKR * 16);
                  mma_ss(tmem + cDQ + mt * DKC, da, db, idescDQ, (kb > 0) | (t > 0));
                }
              }
              mma_commit(&bar[bDoneQ + gs]);
              if (kb == n_kb - 1 && mt == 1) mma_commit(&bar[bWinQ]);  // window complete: the service warps drain dQ'
            }
            __syncwarp();
            STAMP(100);
          }
        }
      }
    }
  } else {
    // =============================================================================================
    // service warps (4 warps = the four TMEM lane quadrants): stage the operands of the NEXT window (global -> smem,
    // in four parts) and, in between, drain the accumulators of the CURRENT window: dV / dK' after every key block,
    // dQ' at the end.  Neither compute group drains any more: the drains (~1 K clk each, after a ~1 K clk wait for the
    // accumulation chains) sat on the critical tail of one group and, through the 3-deep S^T ring, stalled the other.
    // =============================================================================================
    const int pt = tid - kProd0 * 32;
    const int lane_row = (warp & 3) * 32 + lane;                   // TMEM lane = key (dV, dK', dKaug) or query row (dQ')
    const uint32_t trow = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    float acc_d[2][4];                                             // dTd contributions of this thread's keys
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int u = 0; u < 4; ++u) acc_d[a][u] = 0.f;
    // Prompt dK / dV: for small heads this thread keeps the row of its prompt token in registers over all windows of a
    // sample and issues the global atomics once per sample instead of once per window (24 RED operations per key and
    // window were ~5 % of the kernel and sat on the window boundary)
    constexpr bool kRegPrompt = DH <= 12;
    float accp_k[kRegPrompt ? DH : 1], accp_v[kRegPrompt ? DH : 1];
#pragma unroll
    for (int d = 0; d < (kRegPrompt ? DH : 1); ++d) accp_k[d] = accp_v[d] = 0.f;
    int acc_b = -1;                                                // sample the register accumulators belong to
    auto flush_prompt = [&]() {
      if (!kRegPrompt || acc_b < 0 || lane_row >= p.I) return;
      float* gk = p.dkp + ((size_t)acc_b * p.I + lane_row) * p.C + head * DH;
      float* gv = p.dvp + ((size_t)acc_b * p.I + lane_row) * p.C + head * DH;
#pragma unroll
      for (int d = 0; d < (kRegPrompt ? DH : 1); ++d) {
        atomicAdd(gk + d, accp_k[d]);
        atomicAdd(gv + d, accp_v[d]);
        accp_k[d] = accp_v[d] = 0.f;
      }
    };

    // part 0 / 1: query rows pt / pt + 128 (+ ids, dropout row states); part 2: key rows pt, pt + 128; part 3: key rows
    // pt + 256 .. , selector table, hand-over; part < 0: everything
    auto stage = [&](int it, int bw, int part) {
      const int b = bw / p.P, win = bw - b * p.P;
      const int ob = it % OPB;
      uint8_t* opnd = smem + L.opnd0 + ob * L.opnd_bytes;
      uint8_t* Qs = opnd + L.q;
      uint8_t* Ks = opnd + L.k;
      uint8_t* Vs = opnd + L.v;
      uint8_t* dOs = opnd + L.dO;
      float* lse2_s = reinterpret_cast<float*>(opnd + L.lse2);
      float* delta_s = reinterpret_cast<float*>(opnd + L.delta);
      E* wp_s = reinterpret_cast<E*>(opnd + L.wp);
      uint32_t* rs_s = reinterpret_cast<uint32_t*>(opnd + L.rs);
      uint32_t* sel_s = reinterpret_cast<uint32_t*>(opnd + L.sel);
      uint8_t* ids_s = opnd + L.ids;
      const bool all = part < 0;
      if (all || part == 0) {
        STAMP(1);
        if (DROP)
          for (int m = pt; m < kN; m += kProd)
            rs_s[m] = drop_row_hash(seed0, seed1, (uint32_t)bw, (uint32_t)p.heads, (uint32_t)head, kN, (uint32_t)m);
        if (MASKED) {
          for (int i = pt; i < kN / 4; i += kProd)
            reinterpret_cast<uint32_t*>(ids_s)[i] = reinterpret_cast<const uint32_t*>(p.ids + (size_t)win * kN)[i];
          if (p.sel != nullptr && pt == 0) {
            // selector table of this window precomputed per geometry (pwa_attn_sel_table, the forward's table: the mask is
            // symmetric): ONE bulk copy whose bytes are counted on the operand barrier, instead of ~280 instructions per
            // service thread and window
            constexpr uint32_t kSelBytes = kIds * (kN / 4) * 4;
            mbar_expect_tx(&bar[bOpFull + ob], kSelBytes);
            bulk_g2s(sel_s, reinterpret_cast<const uint8_t*>(p.sel) + (size_t)win * kSelBytes, kSelBytes, &bar[bOpFull + ob]);
          }
        }
      }
      for (int qi = 0; qi < 2; ++qi) {                             // query rows: Q', dO' (+ delta, lse)
        if (!(all || part == qi)) continue;
        const int n = pt + qi * kProd;
        const size_t goff = ((size_t)bw * kN + n) * p.C + head * DH;
        E row[DH], drow[DH], orow[DH];
        load_row_b<DH>((const E*)p.q + ((size_t)bw * kN + n) * p.ldq + head * DH, row);
        load_row_b<DH>((const E*)p.dout + goff, drow);
        load_row_b<DH>((const E*)p.out + goff, orow);
        const float l2 = p.lse[((size_t)bw * p.heads + head) * kN + n] * 1.4426950408889634f;
        const int id_ = n % p.wd;
        store_chunks_b<DH, KS * 2>(Qs, kN * 16, n, row, id_ == 0 ? one : zero, id_ == 1 ? one : zero, id_ == 2 ? one : zero,
                                   id_ == 3 ? one : zero);
        float dl = 0.f;
#pragma unroll
        for (int d = 0; d < DH; ++d) dl = fmaf(to_f32(drow[d]), to_f32(orow[d]), dl);
        // dO' = [dO | -delta (hi, lo in E)]: with V' = [V | 1 1] the dP^T MMA yields dP - delta directly.  (fp16: a delta
        // beyond 65504 gives hi = +-inf, lo = -+inf and NaN in dP - delta: non-finite, as the fp32 value would make dq)
        const E dhi = from_f32<E>(-dl);
        const E dlo = from_f32<E>(-dl - to_f32(dhi));
        store_chunks_b<DH, DHP / 8>(dOs, kN * 16, n, drow, FOLD ? dhi : zero, FOLD ? dlo : zero, zero, zero);
        delta_s[n] = -dl;                                          // (the compute warps add it)
        lse2_s[n] = l2;
        wp_s[n] = from_f32<E>(fast_exp2(-l2));
      }
      for (int ki = 0; ki < 3; ++ki) {                             // key rows: K', V'
        if (!(all || (part == 2 && ki < 2) || (part == 3 && ki == 2))) continue;
        const int j = pt + ki * kProd;
        if (j >= NKT) continue;
        const bool content = j < kN;
        const size_t off = content ? ((size_t)bw * kN + j) * p.ldq + head * DH : ((size_t)b * p.I + (j - kN)) * p.ldp + head * DH;
        E row[DH], vrow[DH];
        load_row_b<DH>((const E*)(content ? p.k : p.kp) + off, row);
        load_row_b<DH>((const E*)(content ? p.v : p.vp) + off, vrow);
        const int jd = j % p.wd;
        E ex[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          ex[u] = (content && u < p.wd) ? from_f32<E>(__ldg(&p.td[(head * p.wd + u) * p.wd + jd]) * inv_scale) : zero;
        store_chunks_b<DH, KS * 2>(Ks, NKR * 16, j, row, ex[0], ex[1], ex[2], ex[3]);
        store_chunks_b<DH, DHP / 8>(Vs, NKR * 16, j, vrow, FOLD ? one : zero, FOLD ? one : zero, zero, zero);
      }
      if (all || part == 3) {
        if (MASKED && p.sel == nullptr) {
          prod_sync();                                             // ids of every service thread are in place
          // PRMT selectors: word w of id slot s covers tokens 4w..4w+3 = packed pairs 2w (low half) and 2w+1 (high half);
          // a kept bf16 takes its own bytes (nibbles 1,0 / 3,2), a masked one the bytes of the second operand (5,4 / 7,6)
          for (int i = pt; i < kIds * (kN / 4); i += kProd) {
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
        fence_proxy_async_smem();
        mbar_arrive(&bar[bOpFull + ob]);
        STAMP(2);
      }
    };

    // dV and dK' of key block kb (this thread: key = lane_row); both accumulators are free once they are in registers
    auto drain_kb = [&](int it, int bw, int kb) {
      const int b = bw / p.P;
      const int tile = it * n_kb + kb;
      mbar_wait(&bar[bKbDone], tile & 1);
      tc_fence_after();
      STAMP(108);
      const int nk = kb < 2 ? 128 : p.I;
      const int key = kb * 128 + lane_row;
      const bool key_ok = lane_row < nk;
      auto put_dv = [&](const float (&dv)[DHP]) {
        if (!key_ok) return;
        if (kb < 2) {
          store_row_b<DH>((E*)p.dv + ((size_t)bw * kN + key) * p.ldq + head * DH, dv, keep_scale);
        } else if constexpr (kRegPrompt) {
#pragma unroll
          for (int d = 0; d < DH; ++d) accp_v[d] = fmaf(dv[d], keep_scale, accp_v[d]);
        } else {
          float* gp = p.dvp + ((size_t)b * p.I + lane_row) * p.C + head * DH;
#pragma unroll
          for (int d = 0; d < DH; ++d) atomicAdd(gp + d, dv[d] * keep_scale);
        }
      };
      auto put_dk = [&](const float (&dk)[DKC]) {
        if (!key_ok) return;
        if (kb < 2) {
          store_row_b<DH>((E*)p.dk + ((size_t)bw * kN + key) * p.ldq + head * DH, dk, p.scale);
#pragma unroll
          for (int uu = 0; uu < 4; ++uu) acc_d[kb][uu] += dk[DH + uu];   // d K'[DH+u] = sum_rows(id==u) g = dTd[u][jd]
        } else if constexpr (kRegPrompt) {
#pragma unroll
          for (int d = 0; d < DH; ++d) accp_k[d] = fmaf(dk[d], p.scale, accp_k[d]);
        } else {
          float* gp = p.dkp + ((size_t)b * p.I + lane_row) * p.C + head * DH;
#pragma unroll
          for (int d = 0; d < DH; ++d) atomicAdd(gp + d, dk[d] * p.scale);
        }
      };
      float dv[DHP], dk[DKC];
#pragma unroll
      for (int dq = 0; dq < DHP / 16; ++dq) {
        uint32_t o[16];
        tmem_ld16(trow + cDV + dq * 16, o);
        tmem_wait_ld();
#pragma unroll
        for (int d = 0; d < 16; ++d) dv[dq * 16 + d] = __uint_as_float(o[d]);
      }
      // small heads: both accumulators into registers first, so that the next key block's chains can restart them
      // before any of the global stores / prompt atomics below is issued
      if constexpr (DHP + DKC > 64) put_dv(dv);
#pragma unroll
      for (int dq = 0; dq < DKC / 16; ++dq) {
        uint32_t o[16];
        tmem_ld16(trow + cDK + dq * 16, o);
        tmem_wait_ld();
#pragma unroll
        for (int d = 0; d < 16; ++d) dk[dq * 16 + d] = __uint_as_float(o[d]);
      }
      tc_fence_before();
      mbar_arrive(&bar[bAccFree]);
      if constexpr (DHP + DKC <= 64) put_dv(dv);
      put_dk(dk);
      STAMP(109);
    };

    // dQ' of the window (this thread: query rows lane_row and 128 + lane_row)
    auto drain_q = [&](int it, int bw) {
      mbar_wait(&bar[bWinQ], it & 1);
      tc_fence_after();
      float dq[2][DKC];
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
        for (int c = 0; c < DKC / 16; ++c) {
          uint32_t o[16];
          tmem_ld16(trow + cDQ + mt * DKC + c * 16, o);
          tmem_wait_ld();
#pragma unroll
          for (int d = 0; d < 16; ++d) dq[mt][c * 16 + d] = __uint_as_float(o[d]);
        }
        if constexpr (2 * DKC > 64)      // large heads: one tile at a time (registers)
          store_row_b<DH>((E*)p.dq + ((size_t)bw * kN + mt * 128 + lane_row) * p.ldq + head * DH, dq[mt], p.scale);
      }
      tc_fence_before();
      mbar_arrive(&bar[bDqFree]);
      if constexpr (2 * DKC <= 64) {
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
          store_row_b<DH>((E*)p.dq + ((size_t)bw * kN + mt * 128 + lane_row) * p.ldq + head * DH, dq[mt], p.scale);
      }
      STAMP(4);
    };

    const int n_win = (n_pairs - bw0 + stride - 1) / stride;
    stage(0, bw0, -1);
    for (int it = 0; it < n_win; ++it) {
      const int bw = bw0 + it * stride;
      if (bw / p.P != acc_b) {                                     // first window of another sample
        flush_prompt();
        acc_b = bw / p.P;
      }
      const bool has_next = it + 1 < n_win;
      // (with one operand buffer the next window can only be staged once this one is fully drained)
      const bool inter = has_next && OPB > 1;
      // the first key block retires about a third into the window, the second at two thirds: half of the staging fits
      // in front of each, and the next window's operands are complete well before this window ends
      if (inter) {
        stage(it + 1, bw + stride, 0);
        stage(it + 1, bw + stride, 1);
      }
      drain_kb(it, bw, 0);
      if (inter) {
        stage(it + 1, bw + stride, 2);
        stage(it + 1, bw + stride, 3);
      }
      drain_kb(it, bw, 1);
      if (n_kb == 3) drain_kb(it, bw, 2);
      drain_q(it, bw);
      if (has_next && !inter) stage(it + 1, bw + stride, -1);
    }

    flush_prompt();
    // ---- once per CTA: bias-table gradients ----
    // dKaug[key][u] = sum over all rows/windows of g * onehot: columns [0,wh) -> dTh[u][jh(key)], [wh,wh+ww) -> dTw[u][jw(key)];
    // for prompt keys the wh replicated columns sum to dtok[i].  The /scale of K'aug and the *scale of dS cancel.
    // (the last dKaug chain has retired: bKbDone counts all three chains of a key block)
    STAMP(150);
    // Shared-memory fp32 atomicAdd is a compare-and-swap loop (ATOMS.CAST.SPIN): ~60 of them per thread made this
    // epilogue 20 K clk per CTA.  With ww * wd == 32 (wd == 4) every table entry has ONE writer per (key block, warp):
    // a warp's keys share jh = 4 kb + warp, every 4 consecutive lanes share jw, lanes l, l+4, ... share jd.  So after the
    // shuffle reduction the values go to per-(kb, warp) slots with plain stores (the g^T staging buffers are free by
    // now) and are summed when the CTA's result is added to global memory.  Other window shapes keep the atomics.
    const bool fast = p.ww * p.wd == 32 && p.wd == 4;
    float* slot_w = reinterpret_cast<float*>(smem + L.g);            // [8][ww * ww]
    float* slot_d = slot_w + 8 * p.ww * p.ww;                        // [8][wd * wd]
    const int wq = warp & 3;
    for (int kb = 0; kb < n_kb; ++kb) {
      uint32_t o[16];
      tmem_ld16(trow + cAUG + kb * 16, o);
      tmem_wait_ld();
      const int key = kb * 128 + lane_row;
      if (kb < 2) {
        const int jw = (key / p.wd) % p.ww, jh = key / (p.wd * p.ww);
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          float v = __uint_as_float(o[c]);
          if (c < p.wh) {
            if (fast) {
              v = warp_sum(v);
              if (lane == 0) gth_s[c * p.wh + jh] = v;
            } else {
              atomicAdd(&gth_s[c * p.wh + jh], v);
            }
          } else if (c - p.wh < p.ww) {
            if (fast) {
              v += __shfl_xor_sync(0xffffffffu, v, 1);
              v += __shfl_xor_sync(0xffffffffu, v, 2);
              if ((lane & 3) == 0) slot_w[(kb * 4 + wq) * p.ww * p.ww + (c - p.wh) * p.ww + jw] = v;
            } else {
              atomicAdd(&gtw_s[(c - p.wh) * p.ww + jw], v);
            }
          }
        }
      } else if (lane_row < p.I) {
        float t = 0.f;
#pragma unroll
        for (int c = 0; c < 16; ++c)
          if (c < p.wh) t += __uint_as_float(o[c]);
        gtok_s[lane_row] = t;                                      // one key per thread
      }
    }
    STAMP(153);
#pragma unroll
    for (int kb = 0; kb < 2; ++kb) {
      const int jd = (kb * 128 + lane_row) % p.wd;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        float v = acc_d[kb][u];
        if (fast) {                                                // lanes l, l+4, l+8, ... share jd
          v += __shfl_xor_sync(0xffffffffu, v, 4);
          v += __shfl_xor_sync(0xffffffffu, v, 8);
          v += __shfl_xor_sync(0xffffffffu, v, 16);
          if (lane < 4) slot_d[(kb * 4 + wq) * 16 + u * 4 + jd] = v;
        } else if (u < p.wd) {
          atomicAdd(&gtd_s[u * p.wd + jd], v);
        }
      }
    }
    STAMP(154);
    prod_sync();
    STAMP(155);
    for (int i = pt; i < p.wh * p.wh; i += kProd) atomicAdd(&p.dth[head * p.wh * p.wh + i], gth_s[i]);
    for (int i = pt; i < p.ww * p.ww; i += kProd) {
      float v = gtw_s[i];
      if (fast) {
        v = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) v += slot_w[k * p.ww * p.ww + i];
      }
      atomicAdd(&p.dtw[head * p.ww * p.ww + i], v);
    }
    for (int i = pt; i < p.wd * p.wd; i += kProd) {
      float v = gtd_s[i];
      if (fast) {
        v = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) v += slot_d[k * 16 + i];
      }
      atomicAdd(&p.dtd[head * p.wd * p.wd + i], v);
    }
    for (int i = pt; i < p.I; i += kProd) atomicAdd(&p.dtok[head * p.I + i], gtok_s[i]);
  }
  STAMP(151);                                                      // role done
  tc_fence_before();
  __syncthreads();
  STAMP(152);                                                      // every role done
#undef STAMP
  if (warp == 0) tmem_dealloc(tmem, 512);
}

template <int DH, typename E>
int launch_bwd_tc(const AttnParams& p, cudaStream_t st) {
  constexpr int DHP = BCfg<DH>::DHP, KS = BCfg<DH>::KS;
  const int NKT = kN + p.I;
  const BwdSmem L = bwd_layout(KS, DHP, NKT, p.wh, p.ww, p.wd, p.I, p.ids != nullptr);
  const size_t smem = L.total;
  int grid = 148;
  grid -= grid % p.heads;
  if (grid < p.heads) grid = p.heads;
  const int need = p.B * p.P * p.heads;
  if (grid > need) grid = need;
  auto kern = p.drop_thresh ? (p.ids ? attn_bwd_tc_kernel<DH, true, true, E> : attn_bwd_tc_kernel<DH, false, true, E>)
                            : (p.ids ? attn_bwd_tc_kernel<DH, true, false, E> : attn_bwd_tc_kernel<DH, false, false, E>);
  PWA_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, kThreadsB, smem, st>>>(p);
  PWA_CUDA_OK(cudaGetLastError());
  return PWA_OK;
}

}  // namespace

bool attn_tc_bwd_supported(const AttnParams& p, int dtype) {
  if (!attn_tc_supported(p, dtype)) return false;
  const int dh = p.C / p.heads;
  const int KS = (dh + 4 + 15) / 16, DHP = (dh + 15) / 16 * 16;
  if (128 + DHP + 3 * KS * 16 + 48 > 512) return false;
  return bwd_layout(KS, DHP, kN + p.I, p.wh, p.ww, p.wd, p.I, true).total <= 224 * 1024;
}

template <typename E>
static int backward_t(const AttnParams& p, cudaStream_t st) {
  switch (p.C / p.heads) {
    case 3: return launch_bwd_tc<3, E>(p, st);
    case 6: return launch_bwd_tc<6, E>(p, st);
    case 12: return launch_bwd_tc<12, E>(p, st);
    case 24: return launch_bwd_tc<24, E>(p, st);
    case 48: return launch_bwd_tc<48, E>(p, st);
  }
  set_error("tcgen05 attention backward: head_dim %d not instantiated", p.C / p.heads);
  return PWA_ERR_UNSUPPORTED;
}

int attn_tc_backward(const AttnParams& p, int dtype, cudaStream_t st) {
  return dtype == PWA_F16 ? backward_t<__half>(p, st) : backward_t<__nv_bfloat16>(p, st);
}

}  // namespace pwa
