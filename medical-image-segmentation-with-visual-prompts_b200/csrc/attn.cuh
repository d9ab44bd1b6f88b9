// Parameter block shared by the attention kernels and the C-ABI dispatcher.
#pragma once
#include "common.cuh"

namespace pwa {

// dropout threshold as bit planes: tb[k] = all ones iff bit k of the threshold is set (see drop_keep_word below)
struct DropThresh {
  uint32_t tb[8];
};

struct AttnParams {
  const void *q, *k, *v, *kp, *vp;
  const float *th, *tw, *td, *tok;
  const uint8_t* ids;
  void* out;
  float* lse;
  const void* dout;
  void *dq, *dk, *dv;
  float *dkp, *dvp, *dth, *dtw, *dtd, *dtok, *delta;
  int B, P, C, heads, I, N, NK;
  int ldq, ldp;      // row strides (elements) of q/k/v (+ dq/dk/dv) and of kp/vp; out/dout/dkp/dvp use C
  int wh, ww, wd;
  float scale;
  // attention dropout (window_attention.py:57): 0 = off.  An element (query n, key j) is dropped iff its byte of a
  // counter-based hash is < drop_thresh (probability drop_thresh / 256); kept probabilities are scaled by inv_keep.
  uint32_t drop_thresh;
  DropThresh drop_planes;      // drop_thresh_planes(drop_thresh), filled by the dispatcher: read by the tcgen05 kernels straight
                               // from the constant bank (computed in the kernel, ptxas rebuilt the eight masks for every keep
                               // word under register pressure: 0.75 instructions per logit of the backward)
  float inv_keep;
  const uint32_t* drop_seed;   // DEVICE pointer to two 32-bit seed words (graph-replay safe), or null
  uint32_t seed_host[2];       // used when drop_seed is null
  const uint32_t* sel;         // forward: optional precomputed PRMT selector table [P][28][N/4] (pwa_attn_sel_table), or null
  unsigned int* work;          // forward: per-head window counters (zeroed by the launcher), or null = static round-robin
  int debug;         // PWA_TIMELINE=1: CTA 0 writes clock64 stamps into the (otherwise unused) delta buffer
};

// ---- dropout mask (v2): bit-sliced Bernoulli, 32 keys of one query row per call ----------------------------------
// The keep decisions of query row n for the 32 keys of key chunk c = j >> 5 (j = key index over content AND prompt
// keys) come out of ONE call: a per-row hash (full avalanche mix, once per row and window-head) is folded with the
// chunk index, eight 32-bit planes are derived from it (the upper halves of two products each), and the 8-bit numbers formed
// by the planes (plane k = bit k) are compared with the threshold bit-sliced: one 3-input logic op per plane for all 32
// keys at once.  Key j is kept iff its number is >= thresh (drop probability thresh / 256).  About 1.1 instructions
// per element instead of the ~5 (plus byte compares and selects) of one hash per 2x2 block.
// Key jj = j & 31 of the chunk sits at bit drop_bitpos(jj) of the word: the two keys of a packed bf16 pair g = jj >> 1
// are 8 bits apart, so that `word << (g & 7)` brings them to the sign bits of two bytes, which ONE sign-replicating
// PRMT turns into the 0xffff / 0 halves of the pair's AND mask (drop_pair_mask).
// The backward kernels walk along queries with one thread per key: there a warp generates the words of 32 rows (one
// per lane) and transposes the 32x32 bit tile with five shuffle steps (drop_transpose_tile).
__device__ __forceinline__ uint32_t drop_mix(uint32_t x) {
  x ^= x >> 16; x *= 0x21f0aaadu; x ^= x >> 15; x *= 0x735a2d97u; x ^= x >> 15;
  return x;
}
// hash of query row n of (sample * window, head); N = query rows per window
__device__ __forceinline__ uint32_t drop_row_hash(uint32_t s0, uint32_t s1, uint32_t bw, uint32_t heads, uint32_t head, uint32_t N,
                                                 uint32_t n) {
  return drop_mix(s0 + ((bw * heads + head) * N + n) * 0x85EBCA77u) ^ s1;
}
__host__ __device__ inline DropThresh drop_thresh_planes(uint32_t thresh) {
  DropThresh t;
  for (int k = 0; k < 8; ++k) t.tb[k] = ((thresh >> k) & 1u) ? 0xffffffffu : 0u;
  return t;
}
__host__ __device__ constexpr int drop_bitpos(int jj) {
  return ((jj >> 1) < 8 ? ((jj & 1) ? 31 : 23) : ((jj & 1) ? 15 : 7)) - ((jj >> 1) & 7);
}
__device__ __forceinline__ uint32_t drop_join_hi(uint32_t a, uint32_t b) {     // (a >> 16) | (b & 0xffff0000)
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, 0x7632;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
// keep bits of (row hash, key chunk): bit drop_bitpos(jj) = 1 iff key 32 * chunk + jj is kept
__device__ __forceinline__ uint32_t drop_keep_word(uint32_t row_hash, uint32_t chunk, const DropThresh& t) {
  uint32_t y = (row_hash ^ (chunk * 0x9E3779B1u)) * 0x2C1B3C6Du;
  y ^= y >> 15;
  // plane k = [high half of y * MB[k] : high half of y * MA[k]]: the well-mixed upper bits of two products, joined by ONE PRMT
  // (a single product folded with `w ^= w >> 16` cost a shift and two more logic ops per plane on the ALU pipe, the pipe
  // that binds the dropout variants, and left keys jj and jj + 16 of a chunk correlated at 0.06)
  constexpr uint32_t MA[8] = {0x9E3779B1u, 0x85EBCA77u, 0xC2B2AE3Du, 0x27D4EB2Fu, 0x165667B1u, 0xD3A2646Du, 0xFD7046C5u, 0xB55A4F09u};
  constexpr uint32_t MB[8] = {0x7FEB352Du, 0x846CA68Bu, 0x2C1B3C6Du, 0x297A2D39u, 0x9E485565u, 0xEF1D6B47u, 0x68E31DA5u, 0xB5297A4Du};
  uint32_t lt = 0u;                        // bit-sliced (number < thresh), planes from the least significant up
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const uint32_t w = drop_join_hi(y * MA[k], y * MB[k]);
    lt = (~w & (lt | t.tb[k])) | (lt & t.tb[k]);    // thresh bit 1: ~w | lt ; 0: ~w & lt   (majority of ~w, lt, tb)
  }
  return ~lt;
}
__device__ __forceinline__ bool drop_keep_elem(uint32_t keep_word, uint32_t j) { return (keep_word >> drop_bitpos((int)(j & 31u))) & 1u; }
// AND mask of packed pair g (keys 2g, 2g+1 of the chunk): 0xffff per kept half
__device__ __forceinline__ uint32_t drop_prmt(uint32_t a, uint32_t sel) {
  uint32_t d;
  asm("prmt.b32 %0, %1, %1, %2;" : "=r"(d) : "r"(a), "r"(sel));
  return d;
}
// inverse of drop_bitpos: which key of the chunk sits at bit p
__host__ __device__ constexpr int drop_bitpos_inv(int p) {
  return p >= 24 ? 2 * (31 - p) + 1 : (p >= 16 ? 2 * (23 - p) : (p >= 8 ? 2 * (8 + 15 - p) + 1 : 2 * (8 + 7 - p)));
}
template <int G> __device__ __forceinline__ uint32_t drop_pair_mask(uint32_t keep_word) {
  return drop_prmt(keep_word << (G & 7), G < 8 ? 0xBBAAu : 0x9988u);
}
// full 32-bit masks of the first / second element of pair g and the pair's packed mask (g: a constant after unrolling)
__device__ __forceinline__ void drop_elem_masks(uint32_t keep_word, int g, uint32_t& m0, uint32_t& m1, uint32_t& mpair) {
  const uint32_t x = keep_word << (g & 7);
  m0 = drop_prmt(x, g < 8 ? 0xAAAAu : 0x8888u);
  m1 = drop_prmt(x, g < 8 ? 0xBBBBu : 0x9999u);
  mpair = drop_prmt(x, g < 8 ? 0xBBAAu : 0x9988u);
}
// Transposition of a 32x32 bit tile held as one word per lane (whole warp): afterwards lane p holds bit p of every
// lane's input word, input lane l at bit l.
__device__ __forceinline__ uint32_t drop_transpose_tile(uint32_t x, int lane) {
#pragma unroll
  for (int d = 16; d >= 1; d >>= 1) {
    const uint32_t m = d == 16 ? 0x0000ffffu : (d == 8 ? 0x00ff00ffu : (d == 4 ? 0x0f0f0f0fu : (d == 2 ? 0x33333333u : 0x55555555u)));
    const uint32_t y = __shfl_xor_sync(0xffffffffu, x, d);
    const bool up = (lane & d) != 0;
    const uint32_t ys = up ? (y >> d) : (y << d);
    const uint32_t keep = up ? ~m : m;
    x = (x & keep) | (ys & ~keep);
  }
  return x;
}

// fp32-math CUDA-core kernels (attn_f32.cu)
int attn_f32_forward(const AttnParams& p, int dtype, cudaStream_t st);
int attn_f32_backward(const AttnParams& p, int dtype, cudaStream_t st);

// tcgen05 / TMEM kernels, bf16 or fp16.  attn_tc_supported (api.cu) is the one envelope that forward and backward dispatch
// on: the shapes the kernels are written for plus the budgets below.  The *_fits checks assume a shape inside that envelope.
bool attn_tc_supported(const AttnParams& p, int dtype);
bool attn_ws_fits(const AttnParams& p);                                   // attn_tc_ws.cu: shared memory of the forward
int attn_ws_forward(const AttnParams& p, int dtype, cudaStream_t st);
bool attn_tc_bwd_fits(const AttnParams& p);                               // attn_tc_bwd.cu: TMEM and shared memory of the backward
int attn_tc_backward(const AttnParams& p, int dtype, cudaStream_t st);
// deterministic tcgen05 backward (attn_tc_bwd.cu, Det<E> instantiations): p.dkp / p.dvp / p.dth / p.dtw / p.dtd / p.dtok are
// the workspace slot arrays of pwa_attn_bwd_det, attn_tc_bwd_slots(p) slots each
int attn_tc_backward_det(const AttnParams& p, int dtype, cudaStream_t st);
int attn_tc_bwd_slots(const AttnParams& p);

}  // namespace pwa
