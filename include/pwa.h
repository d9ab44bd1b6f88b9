/*
 * pwa.h -- C ABI of the B200-native prompted 3D shifted-window attention path.
 *
 * The reference (liamliaw/medical-image-segmentation-with-visual-prompts) is pure Python and
 * has no FFI of its own; its boundary for this path is the nn.Module API of
 *   src/modules/swin_transformer/swin_block.py      (SwinTransformerBlock, ConsecutiveSwinBlocks,
 *                                                     window_partition, window_reverse, get_attn_mask)
 *   src/modules/multi_head_attention/window_attention.py            (WindowAttention)
 *   src/modules/multi_head_attention/relative_positional_encoding.py (RelativePE)
 * The Python mirror of those classes in this repo calls the entry points below through ctypes
 * (see INTEGRATION.md for the binding a reference maintainer would add).  Each entry point names the
 * reference lines it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch types.
 *   - every device buffer is allocated by the caller; nothing here allocates, frees or synchronises.
 *   - every launch goes to the cudaStream_t passed in (void* so that C callers need no CUDA headers).
 *   - return 0 on success, <0 on error; pwa_last_error() returns a thread-local message.
 *   - the device is the caller's current device (one process per GPU).
 *   - debug-only entry points (clock64 timelines of the attention kernels) live in include/pwa_debug.h and exist only in
 *     libraries built with `make TIMELINE=1`.
 *   - re-entrant and thread-safe (no global mutable state besides one-time kernel attribute setup).
 *   - there is NO CPU fallback: device entry points fail with PWA_ERR_CUDA when no GPU is present.
 *   - `dtype` is PWA_F32, PWA_BF16 or PWA_F16 wherever an entry point takes one; the two 16-bit types take the same paths
 *     (tcgen05 kernels where the shape allows, the same envelope for both), fp32 runs on the CUDA-core kernels.
 */
#ifndef PWA_H_
#define PWA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PWA_VERSION 100

enum { PWA_OK = 0, PWA_ERR_ARG = -1, PWA_ERR_UNSUPPORTED = -2, PWA_ERR_CUDA = -3 };
/* Element type of the token tensors of an entry point's `dtype` argument.  Every kernel computes in fp32 (or accumulates in
 * fp32 on the tensor cores) whatever the storage type; PWA_F16 is IEEE binary16 (torch.float16, torch.autocast's default). */
enum { PWA_F32 = 0, PWA_BF16 = 1, PWA_F16 = 2 };

/* Window geometry of one block call.  Filled by pwa_geometry(); plain ints so that it can be
 * mirrored by a ctypes.Structure. */
typedef struct pwa_geom {
  int32_t dims[3];      /* H, W, D of the unpadded feature map                                      */
  int32_t ws[3];        /* window (wh, ww, wd)                                                      */
  int32_t shift[3];     /* effective shift, 0 where dims[a] <= ws[a]         (swin_block.py:265-270) */
  int32_t pads[6];      /* the reference's `paddings` (floor,ceil per axis)  (swin_block.py:150-161) */
  int32_t sp[3];        /* padded dims = dims + pads                                                */
  int32_t nwin[3];      /* P1,P2,P3 = sp / ws                                                       */
  int32_t data_lo[3];   /* low-side zero padding of the DATA = pads[2a+1] (F.pad(reversed), :163)    */
  int32_t crop_lo[3];   /* low-side offset of the output crop / mask box = pads[2a] (:247-253)       */
  int32_t P;            /* windows per sample                                                       */
  int32_t N;            /* tokens per window                                                        */
  int32_t masked;       /* 1 iff any shift > 0 (a shift mask exists, :173)                          */
  int32_t padded;       /* 1 iff any pad > 0                                                        */
} pwa_geom;

/* ---- host-only helpers (no GPU needed) ------------------------------------------------------ */

int pwa_version(void);
const char* pwa_last_error(void);

/* swin_block.py:146-164, 265-270: padding rule, effective shift, window counts. */
int pwa_geometry(const int32_t dims[3], const int32_t ws[3], const int32_t shift_cfg[3], pwa_geom* out);

/* swin_block.py:312-364 (get_attn_mask) in compressed form: one region id per (window, token),
 * uint8 [P][N] written to HOST memory; mask[p][i][j] == 1.0f iff ids[p][i] == ids[p][j].
 * ids are 9*rh+3*rw+rd (0..26) or 100 inside the un-padded box when the map is padded. */
int pwa_region_ids(const pwa_geom* g, uint8_t* ids_host);

/* PRMT selector table of the shift mask for the tcgen05 attention kernels: uint32 [P][28][N/4] to HOST memory, from
 * region ids uint8 [P][N] in HOST memory (see pwa_attn_shape.sel_table).  Depends only on the geometry. */
int pwa_attn_sel_table(const uint8_t* ids_host, int P, int N, uint32_t* table_host);

/* flat source index (into the unpadded H*W*D volume, -1 = zero padding) of every (window, token):
 * int32 [P][N] to HOST memory.  which = 0: input side (pad -> roll -> window_partition,
 * swin_block.py:163,174-178,292-299); which = 1: output side (window_reverse -> roll back -> crop,
 * swin_block.py:302-309,238-253). */
int pwa_index_map(const pwa_geom* g, int which, int32_t* map_host);

/* ---- (a) cyclic roll + pad + strided window partition / reverse ------------------------------ */

/* x [B][C][H][W][D] -> tokens [B][P][N][C].  lo = g->data_lo when (use_crop_lo & 1) == 0 (forward of the
 * block input), g->crop_lo when 1 (adjoint of pwa_reverse).  Replaces F.pad + torch.roll +
 * window_partition + rearrange (swin_block.py:163,174-178,205,209,214).
 * Bit 1 of use_crop_lo forces the element-wise generic kernel (checker for the staged fast kernel). */
int pwa_partition(const void* x, void* tokens, int B, int C, const pwa_geom* g, int use_crop_lo,
                  int dtype, void* stream);

/* tokens [B][P][N][C] -> x [B][C][H][W][D]; exact inverse index map incl. roll back and crop.
 * use_crop_lo == 1 for the block output (swin_block.py:228-253), 0 for the adjoint of
 * pwa_partition.  Token slots that map to padding are dropped. */
int pwa_reverse(const void* tokens, void* x, int B, int C, const pwa_geom* g, int use_crop_lo,
                int dtype, void* stream);

/* pwa_reverse of (tokens_a + tokens_b): fuses the last residual add of the block, `x + mlp(mlp_norm(x))`
 * (swin_block.py:227), into the window reverse.  The sum is formed in fp32 and rounded once to `dtype`. */
int pwa_reverse_add(const void* tokens_a, const void* tokens_b, void* x, int B, int C, const pwa_geom* g,
                    int use_crop_lo, int dtype, void* stream);

/* Row gather between channels-last arrangements: dst [B][rows_dst][C] <- src [B][rows_src][C] with
 * dst[b][j][:] = map[j] >= 0 ? src_a[b][map[j]][:] (+ src_b[b][map[j]][:] when src_b != NULL) : 0.
 * map: int32 [rows_dst] on the DEVICE, shared by all samples.  With maps composed on the host from
 * pwa_index_map() this is, without leaving the token layout, any chain of
 * window_reverse -> roll back -> crop -> pad -> roll -> window_partition between two blocks of a
 * ConsecutiveSwinBlocks pair (swin_block.py:66-71, 228-253, 150-214), the 2x2x2 strided slices + cat of
 * PatchMerging (down.py:21-47), and the partition of a channels-last feature map (the strides
 * down.py:48-53 leaves).  src_b fuses the block's last residual add (swin_block.py:227; fp32 sum, rounded once).
 * Every map is injective, so the adjoint is the same call with the inverse map. */
int pwa_gather_rows(const void* src_a, const void* src_b, void* dst, const int32_t* map, int B,
                    int64_t rows_src, int64_t rows_dst, int C, int dtype, void* stream);

/* dst[j] = sum over s < S of src[s][j]  (fp32, src [S][n] and dst [n] on the DEVICE).  Final reduction of the
 * token-split weight gradients of the block's Linear layers (swin_block.py:141-143, window_attention.py:28-32;
 * torch autograd in the reference): dW = dy^T x is computed as S batched slices of the token axis with fp32 partials. */
int pwa_colsum_f32(const float* src, float* dst, int S, int64_t n, void* stream);

/* dst[c] = sum over r < rows of x[r][c]: x [rows][C] bf16, fp16 or fp32 (dtype), dst [C] fp32, both on the
 * DEVICE; dst is zeroed by the call.  The bias gradient of the q|k|v projection (window_attention.py:28-30: nn.Linear with
 * bias; torch autograd sums the packed dq|dk|dv rows over all tokens there).  C must be a multiple of the elements per
 * 16 bytes (8 for bf16 / fp16, 4 for fp32) and at most 512 such vectors; x 16-byte aligned.  fp32 atomics: the sum order is not fixed
 * (pwa_colsum_rows_det fixes it). */
int pwa_colsum_rows(const void* x, float* dst, int64_t rows, int C, int dtype, void* stream);

/* y[i] = keep(i) ? x[i] / keep_rate : 0 for i < n, keep(i) a counter-based hash of the two uint32 words at seed_dev (DEVICE
 * memory) and i; rate in steps of 1/256.  Replaces nn.Dropout(proj_drop) after the attention output projection
 * (window_attention.py:33,60).  The same call on dy is the backward.  No generator state is involved, so an activation-
 * checkpointed block recomputes the same mask and a captured CUDA graph gets fresh masks whenever the seed words change.
 * The mask depends only on the seed words and i, not on dtype (fp32, bf16 or fp16 with fp32 math).
 * x == y is allowed; both 16-byte aligned. */
int pwa_dropout(const void* x, void* y, int64_t n, float p_drop, const void* seed_dev, int dtype, void* stream);

/* pwa_dropout over a [rows][C] tensor (C % 4 == 0, C <= 1024) that also emits colsum[c] = sum_rows y[r][c] (fp32 [C] on the
 * DEVICE, zeroed by this call).  Backward use: y = gradient of the Linear output in front of the dropout, colsum = gradient
 * of that Linear's bias (attn.proj.bias, window_attention.py:32,60) without a separate reduction pass. */
int pwa_dropout_colsum(const void* x, void* y, int64_t rows, int C, float p_drop, const void* seed_dev, float* colsum,
                       int dtype, void* stream);

/* ---- (b) fused prompted window attention, forward -------------------------------------------- */

typedef struct pwa_attn_shape {
  int32_t B, P, C, heads, I;   /* I = number of prompt tokens (0 = none)           */
  int32_t ws[3];               /* N = ws[0]*ws[1]*ws[2]                            */
  float scale;                 /* head_dim ** -0.5  (window_attention.py:25)       */
  float p_drop;                /* attention dropout probability (0 in eval), applied in steps of 1/256 after the
                                  softmax (window_attention.py:57); the forward and backward calls of one step must
                                  see the same seed words (all kernels: tcgen05 and fp32-math).                    */
  uint64_t seed, offset;       /* host seed words (e.g. torch's generator seed / offset)                          */
  int32_t ld_qkv;              /* row stride (elements) of q,k,v and dq,dk,dv; 0 = C.  3*C when q|k|v are the
                                  column blocks of ONE fused projection output [B][P][N][3C]            */
  int32_t ld_p;                /* row stride of kp, vp; 0 = C (2*C for a fused [B][I][2C] projection)  */
  const void* seed_dev;        /* optional DEVICE pointer to two uint32 seed words that replace seed/offset: the
                                  words can be refreshed by a device-side RNG op every step, which keeps a captured
                                  CUDA graph of the step valid (host scalars would be frozen into the graph)      */
  const void* sel_table;       /* optional DEVICE pointer to pwa_attn_sel_table() output [P][28][N/4] uint32 for `ids` (tcgen05
                                  forward and backward): fetched per window with one bulk copy instead of being rebuilt
                                  by every (window, head).  NULL = built in the kernel.                                */
  void* work;                  /* optional DEVICE scratch of >= 4*heads bytes (contents irrelevant, zeroed by the call on
                                  its stream): per-head work counters of the tcgen05 forward, which then hands windows
                                  to its CTAs dynamically instead of round-robin (CTAs sharing an SM do not progress
                                  at the same rate).  NULL = static distribution.                                  */
} pwa_attn_shape;

/* q,k,v [B][P][N][C]; kp,vp [B][I][C] (NULL when I == 0): keys/values of the prompt tokens,
 * shared by every window of a sample; th [h][wh][wh], tw [h][ww][ww], td [h][wd][wd], tok [h][I]:
 * fp32 bias tables INCLUDING the /3 and embed_dim**-0.5 factors
 * (relative_positional_encoding.py:116-123,136-138); ids uint8 [P][N] on the DEVICE or NULL (no
 * shift mask).  out [B][P][N][C]; lse fp32 [B][P][h][N] (natural-log sum-exp of the masked logits).
 * logits = (q.k^T*scale + bias) * mask ; softmax ; dropout ; @ v   (window_attention.py:49-58),
 * queries = the N content tokens only (prompt rows are cut by swin_block.py:222-225).
 * dtype PWA_F32 / PWA_BF16 / PWA_F16 for q, k, v, kp, vp, out.
 * impl: 0 = auto, 1 = fp32-math CUDA-core kernel (any dtype), 2 = tcgen05/TMEM kernel (bf16 or fp16; fp32 accumulation).
 * The fp16 tcgen05 forward keeps each row's largest probability a normal fp16 number (DESIGN.md §4(b)): it scales the
 * probabilities by 2^10 before rounding them and takes the exact-row-maximum sweep when the norm bound is loose by more
 * than 24 binades (bf16: 80). */
int pwa_attn_fwd(const void* q, const void* k, const void* v, const void* kp, const void* vp,
                 const float* th, const float* tw, const float* td, const float* tok,
                 const uint8_t* ids, void* out, float* lse, const pwa_attn_shape* s, int dtype,
                 int impl, void* stream);

/* ---- (c) backward ----------------------------------------------------------------------------- */

/* Inputs as pwa_attn_fwd plus out, lse, dout [B][P][N][C].  Outputs: dq,dk,dv [B][P][N][C] (dtype: fp32, bf16 or fp16;
 * in fp16 a gradient that overflows becomes inf, and a non-finite dout stays non-finite in every gradient it reaches);
 * dkp,dvp fp32 [B][I][C], summed over the P windows of each sample; dth,dtw,dtd,dtok fp32, summed
 * over batch and windows.  The fp32 accumulators are zeroed by this call (cudaMemsetAsync on
 * `stream`).  delta fp32 [B][P][h][N] is caller-provided scratch. */
int pwa_attn_bwd(const void* q, const void* k, const void* v, const void* kp, const void* vp,
                 const float* th, const float* tw, const float* td, const float* tok,
                 const uint8_t* ids, const void* out, const float* lse, const void* dout,
                 void* dq, void* dk, void* dv, float* dkp, float* dvp,
                 float* dth, float* dtw, float* dtd, float* dtok, float* delta,
                 const pwa_attn_shape* s, int dtype, int impl, void* stream);

/* ---- relative-position bias tables --------------------------------------------------------------- */

/* RelativePE.forward (relative_positional_encoding.py:99-142) in compact form.  enc_a [2*cap_a-1][E],
 * wc_a [heads][E] (a = h,w,d), enc_tok [I][E], w_tok [heads][E] (NULL when I == 0), all fp32.
 * Outputs th [heads][ws0][ws0], tw, td, tok [heads][I] INCLUDING the /3 and E^-0.5 factors (:116-123,136-138). */
int pwa_bias_tables_fwd(const float* enc_h, const float* enc_w, const float* enc_d, const float* wc_h,
                        const float* wc_w, const float* wc_d, const float* enc_tok, const float* w_tok,
                        float* th, float* tw, float* td, float* tok, int heads, int E, const int32_t ws[3],
                        const int32_t cap[3], int I, void* stream);

/* Gradients of the eight parameter tensors from the table gradients produced by pwa_attn_bwd. */
int pwa_bias_tables_bwd(const float* enc_h, const float* enc_w, const float* enc_d, const float* wc_h,
                        const float* wc_w, const float* wc_d, const float* enc_tok, const float* w_tok,
                        const float* dth, const float* dtw, const float* dtd, const float* dtok,
                        float* denc_h, float* denc_w, float* denc_d, float* dwc_h, float* dwc_w, float* dwc_d,
                        float* denc_tok, float* dw_tok, int heads, int E, const int32_t ws[3],
                        const int32_t cap[3], int I, void* stream);

/* ---- LayerNorm over the channel axis of window tokens, fused with the surrounding residual adds ----- */

/* s = x (+ res) ; y = LayerNorm(s) * gamma + beta over the last axis (C, C % 4 == 0, C <= 2048), rows x C
 * row-major.  Replaces nn.LayerNorm(eps=1e-6) at swin_block.py:216 (attn_norm) and :227 (mlp_norm) together
 * with the residual add of :222.  res / sum_out may be NULL (plain LayerNorm).  gamma, beta fp32.
 * mean, rstd: fp32 [rows], saved for the backward. */
int pwa_ln_fwd(const void* x, const void* res, const float* gamma, const float* beta, void* sum_out, void* y,
               float* mean, float* rstd, int64_t rows, int C, float eps, int dtype, void* stream);

/* dx = LayerNorm-backward(dy; x, gamma, mean, rstd) (+ dres) ; dgamma = sum_rows dy*xhat ; dbeta = sum_rows dy.
 * x is the tensor that was normalised (the sum when a residual was fused).  dres may be NULL.
 * dgamma/dbeta fp32 [C], zeroed by this call. */
int pwa_ln_bwd(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd,
               const void* dres, void* dx, float* dgamma, float* dbeta, int64_t rows, int C, int dtype, void* stream);

/* pwa_ln_bwd plus two optional fp32 [C] column sums over all rows (NULL = skip; zeroed by this call):
 * dres_colsum = sum_rows dres and dx_colsum = sum_rows dx.  In the block, dx is the gradient of `proj(o) + bias`
 * (window_attention.py:59) and dres that of `mlp(...) + bias` (swin_block.py:227), so these ARE the two Linear bias
 * gradients and come out of a pass that reads the tensors anyway. */
int pwa_ln_bwd2(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd,
                const void* dres, void* dx, float* dgamma, float* dbeta, float* dres_colsum, float* dx_colsum,
                int64_t rows, int C, int dtype, void* stream);

/* ---- token-domain GEMM with fused LayerNorm / residual / dropout prologue (tcgen05, bf16 or fp16) ---------------------- */

/* s = dropout(x) (+ res) ; z = LayerNorm(s) * gamma + beta (gamma == NULL: z = s) ; y = z @ W^T (+ bias).
 * x, res, sum_out, ln_out [T][C] bf16; W [Cout][C] bf16 row-major; bias [Cout] bf16 or NULL; y [T][Cout] bf16; mean, rstd fp32
 * [T] or NULL.  sum_out (s) and ln_out (z) are written when non-NULL.  p_drop > 0: the mask of pwa_dropout for the same seed
 * words (element index = row * C + column), so pwa_dropout / pwa_dropout_colsum on the upstream gradient is its backward.
 * One pass over the tokens for what the reference runs as LayerNorm + Linear (+ Dropout + add) modules: swin_block.py:216 +
 * window_attention.py:42-44 (attn_norm + to_q|to_k|to_v as one [C -> 3C] projection), window_attention.py:60 +
 * swin_block.py:222-227 (proj_drop, residual add, mlp_norm, the single-Linear MLP).  C % 16 == 0, 16 <= C <= 192,
 * Cout % 16 == 0 (pwa_token_gemm_supported).
 * pwa_token_gemm_fwd_dt takes the element type of x, res, sum_out, ln_out, W, bias and y: PWA_BF16 or PWA_F16 (fp32 LayerNorm
 * math and fp32 accumulation either way); pwa_token_gemm_fwd is its PWA_BF16 call. */
int pwa_token_gemm_supported(int C, int Cout);
int pwa_token_gemm_fwd(const void* x, const void* res, const float* gamma, const float* beta, const void* W, const void* bias,
                       void* sum_out, void* ln_out, void* y, float* mean, float* rstd, int64_t T, int C, int Cout, float eps,
                       float p_drop, const void* seed_dev, void* stream);
int pwa_token_gemm_fwd_dt(const void* x, const void* res, const float* gamma, const float* beta, const void* W, const void* bias,
                          void* sum_out, void* ln_out, void* y, float* mean, float* rstd, int64_t T, int C, int Cout, float eps,
                          float p_drop, const void* seed_dev, int dtype, void* stream);

/* 1 iff the tcgen05 kernels (forward and backward) support this shape and dtype (PWA_BF16 or PWA_F16: the same shapes for
 * both; else impl=0 runs the fp32-math kernel). */
int pwa_attn_tc_supported(const pwa_attn_shape* s, int dtype);

/* Window attention with DENSE position-bias / mask tensors: the literal argument form of the reference's
 * WindowAttention.forward(q, k, v, pos_bias, mask), multi_head_attention/window_attention.py:35-58 (after the three input
 * projections, before the output projection):
 *     logits[i][j] = (scale * q_i . k_j + bias[b,p,h,i,j]) * mask[b,p,h,i,j];   out = dropout(softmax_j(logits)) @ v
 * q rows [B*P*nq], k / v rows [B*P*nk] with row strides ld_* (elements) and head h at columns h*dh .. h*dh+dh-1; out /
 * dout rows are heads*dh wide and contiguous; lse / delta fp32 [B*P*heads*nq].  bias / mask: fp32 DEVICE tensors or NULL,
 * element (b,p,h,i,j) at b*stride[0] + p*stride[1] + h*stride[2] + i*stride[3] + j (j contiguous; stride 0 = broadcast).
 * dbias (or NULL): fp32 buffer with bias's strides, ZEROED by the caller; the gradient is accumulated with atomics.
 * p_drop in steps of 1/256 with the generator of pwa_attn_fwd (nq rows per window-head); seed_dev = two uint32 words on
 * the device.  fp32 arithmetic, fp32 / bf16 / fp16 I/O; head dims 3, 6, 8, 12, 16, 24, 32, 48. */
typedef struct pwa_dense_attn {
  int32_t B, P, heads, dh, nq, nk;
  int32_t ld_q, ld_k, ld_v;
  int64_t bias_stride[4];
  int64_t mask_stride[4];
  float scale, p_drop;
  const void* seed_dev;
} pwa_dense_attn;
int pwa_attn_dense_fwd(const void* q, const void* k, const void* v, const float* bias, const float* mask, void* out, float* lse,
                       const pwa_dense_attn* s, int dtype, void* stream);
int pwa_attn_dense_bwd(const void* q, const void* k, const void* v, const float* bias, const float* mask, const void* out,
                       const float* lse, const void* dout, void* dq, void* dk, void* dv, float* dbias, float* delta,
                       const pwa_dense_attn* s, int dtype, void* stream);

/* ---- deterministic reductions (torch.use_deterministic_algorithms) ----------------------------------------------------- */

/* The entry points above that return fp32 sums over CTAs (pwa_attn_bwd's dkp, dvp, dth, dtw, dtd, dtok; the column sums of
 * pwa_ln_bwd2, pwa_dropout_colsum and pwa_colsum_rows) add per-CTA partials with float atomics, so the last bits of those sums
 * depend on scheduling.  Each has a sibling, `<name>_det`, that returns the same sums bitwise reproducibly: every CTA writes
 * its partials in a fixed order to its own slot of a caller-provided DEVICE workspace, and a second pass (pwa_colsum_f32)
 * sums the slots in index order.  A result is reproduced for the same GPU model, library build and shape.
 *   - `<name>_det_workspace_size` returns the bytes the sibling needs (0 = none, NULL allowed) or a negative error code.  It
 *     needs no GPU.  A workspace smaller than that makes the sibling return PWA_ERR_ARG.
 *   - the siblings keep every other contract of their entry point: the same arguments and outputs, the caller's stream, no
 *     allocation and no synchronisation (they can be captured into a CUDA graph); the workspace contents on entry do not
 *     matter.
 *   - pwa_attn_bwd_det runs the tcgen05 kernel only (no `impl` argument): outside pwa_attn_tc_supported it returns
 *     PWA_ERR_UNSUPPORTED.  The fp32-math and dense-argument attention backwards have no deterministic form.
 *   - pwa_bias_tables_bwd has no cross-CTA sums; its sibling replaces the shared-memory atomics of the per-distance table
 *     gradient by fixed-order sums and needs no workspace. */
int64_t pwa_attn_bwd_det_workspace_size(const pwa_attn_shape* s, int dtype);
int pwa_attn_bwd_det(const void* q, const void* k, const void* v, const void* kp, const void* vp,
                     const float* th, const float* tw, const float* td, const float* tok,
                     const uint8_t* ids, const void* out, const float* lse, const void* dout,
                     void* dq, void* dk, void* dv, float* dkp, float* dvp,
                     float* dth, float* dtw, float* dtd, float* dtok, float* delta,
                     void* workspace, int64_t workspace_bytes, const pwa_attn_shape* s, int dtype, void* stream);

int64_t pwa_ln_bwd2_det_workspace_size(int64_t rows, int C, int dtype);
int pwa_ln_bwd2_det(const void* dy, const void* x, const float* gamma, const float* mean, const float* rstd,
                    const void* dres, void* dx, float* dgamma, float* dbeta, float* dres_colsum, float* dx_colsum,
                    int64_t rows, int C, int dtype, void* workspace, int64_t workspace_bytes, void* stream);

int64_t pwa_dropout_colsum_det_workspace_size(int64_t rows, int C, int dtype);
int pwa_dropout_colsum_det(const void* x, void* y, int64_t rows, int C, float p_drop, const void* seed_dev, float* colsum,
                           int dtype, void* workspace, int64_t workspace_bytes, void* stream);

int64_t pwa_colsum_rows_det_workspace_size(int64_t rows, int C, int dtype);
int pwa_colsum_rows_det(const void* x, float* dst, int64_t rows, int C, int dtype, void* workspace, int64_t workspace_bytes,
                        void* stream);

int64_t pwa_bias_tables_bwd_det_workspace_size(int heads, int E, const int32_t ws[3], const int32_t cap[3], int I);
int pwa_bias_tables_bwd_det(const float* enc_h, const float* enc_w, const float* enc_d, const float* wc_h,
                            const float* wc_w, const float* wc_d, const float* enc_tok, const float* w_tok,
                            const float* dth, const float* dtw, const float* dtd, const float* dtok,
                            float* denc_h, float* denc_w, float* denc_d, float* dwc_h, float* dwc_w, float* dwc_d,
                            float* denc_tok, float* dw_tok, int heads, int E, const int32_t ws[3],
                            const int32_t cap[3], int I, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- whole-volume sliding-window inference ----------------------------------------------------------------------------- */

/* The reference scores the downstream model on whole volumes by cutting them into roi-sized patches, running the model on
 * sub-batches of patches and adding the predictions back with overlap weights (SegmentationTrainer.test, SURVEY.md §3(4)).
 * These entry points are the GPU side of that loop (pwa_b200.inference builds the tiling on the host):
 *   - origins: int32 [n_total][4] table (b, x0, y0, z0) on the DEVICE, 16-byte aligned, in patch order (sample, then raster
 *     order over x, y, z).  Origins are >= 0; a patch may reach past the volume (an axis shorter than the roi).
 *   - cursor: int32 {first, count} on the DEVICE.  A call works on patches [first, first + count) of the table (count is
 *     clamped to [0, sw] and to the table).  pwa_tile_advance moves the cursor to the next sub-batch, so a captured CUDA
 *     graph of gather -> predictor -> stitch -> advance walks the whole table by replaying, with no host scalar in it.
 *   - dims = (X, Y, Z) of the volume, roi = (r0, r1, r2), 1 <= sw <= PWA_TILE_MAX_SW patches per sub-batch.
 *   - arguments are checked before any CUDA call (PWA_ERR_ARG without a GPU); nothing allocates or synchronises. */
#define PWA_TILE_MAX_SW 1024
/* Element types of label maps and target volumes. */
enum { PWA_LABEL_U8 = 0, PWA_LABEL_I32 = 1, PWA_LABEL_I64 = 2 };

/* patches [sw][Cin][r0][r1][r2] (dtype_out) <- image [B][Cin][X][Y][Z] (dtype_in): slot s < count holds the patch at
 * origins[first + s], voxels outside the volume read `cval` (rounded to dtype_in first, as F.pad does); slots >= count are all
 * `cval`.  Bit-exact against slicing + F.pad + .to(dtype_out).  16-byte vectors along z where roi[2] % 8 == 0 and the row is
 * aligned, elements otherwise. */
int pwa_tile_gather(const void* image, int dtype_in, int B, int Cin, const int32_t dims[3], const int32_t* origins,
                    int64_t n_total, const int32_t* cursor, const int32_t roi[3], int sw, float cval, void* patches,
                    int dtype_out, void* stream);

/* acc fp32 [B][K][X][Y][Z] += weight * pred and wsum fp32 [B][X][Y][Z] += weight for the `count` patches of this call, with
 * pred [sw][K][r0][r1][r2] (fp32, bf16 or fp16) and the importance map weight fp32 [r0][r1][r2].  No float atomics: each
 * covered voxel is read once, gets the terms of the covering patches added one after the other in patch order (fused
 * multiply-add, fp32) and is written once, so the sums are bitwise independent of sw and reproducible from run to run. */
int pwa_tile_stitch(const void* pred, int dtype_pred, const float* weight, int B, int K, const int32_t dims[3],
                    const int32_t* origins, int64_t n_total, const int32_t* cursor, const int32_t roi[3], int sw,
                    float* acc, float* wsum, void* stream);

/* cursor {first, count} <- {first + count, min(sw, n_total - first - count)}: one single-thread kernel. */
int pwa_tile_advance(int32_t* cursor, int sw, int64_t n_total, void* stream);

/* One pass over acc [B][K][X][Y][Z] and wsum [B][X][Y][Z]; each output is optional (NULL = skip):
 *   - out [B][K][X][Y][Z] = acc / wsum in dtype_out (fp32 division, rounded once);
 *   - labels [B][X][Y][Z] = argmax over K of the fp32 acc / wsum, the lowest class on ties (torch.argmax), uint8 for K <= 256
 *     and int32 otherwise;
 *   - tp, fp, fn int64 [B][K] (zeroed by the call, exact integer atomics) against target [B][X][Y][Z] of type target_dtype
 *     (PWA_LABEL_*); voxels whose target is outside [0, K) are not counted.  Counting needs K <= 1024. */
int pwa_tile_finalize(const float* acc, const float* wsum, int B, int K, const int32_t dims[3], void* out, int dtype_out,
                      void* labels, const void* target, int target_dtype, int64_t* tp, int64_t* fp, int64_t* fn, void* stream);

/* tp, fp, fn int64 [B][K] (zeroed by the call) of a label map against a target, both [B][nvox] of types PWA_LABEL_*; voxels
 * whose label or target is outside [0, K) are not counted.  K <= 1024. */
int pwa_seg_counts(const void* labels, int label_dtype, const void* target, int target_dtype, int B, int64_t nvox, int K,
                   int64_t* tp, int64_t* fp, int64_t* fn, void* stream);

/* ---- segmentation losses ----------------------------------------------------------------------------------------------- */

/* The per-(sample, class) sums behind MONAI's DiceLoss / FocalLoss / DiceFocalLoss with integer label maps (pwa_b200.trainer
 * builds the losses from them).  logits and dlogits: contiguous [B][K][nvox] (PWA_F32 / PWA_BF16 / PWA_F16); labels: [B][nvox]
 * of type PWA_LABEL_*; one-hot y_k = [label == k], a label outside [0, K) is an all-zero row.  Per voxel:
 *   p_k = x_k (PWA_ACT_NONE), sigmoid(x_k) (PWA_ACT_SIGMOID) or softmax over the K channels (PWA_ACT_SOFTMAX);
 *   sums [4][B][K] fp32: I = sum p_k y_k, P = sum p_k (p_k^2 with squared_pred), G = sum y_k, F = sum focal_k;
 *   focal_k, PWA_FOCAL_SIGMOID: (x - x y - log sigmoid(x)) exp(gamma log sigmoid(-x (2y - 1))), times (alpha y + (1 - alpha)(1 - y));
 *   focal_k, PWA_FOCAL_SOFTMAX: -(1 - q_k)^gamma log(q_k) y_k, q = softmax over channels c0 .. K-1 (c0 = focal_skip_bg), 0 for
 *     k < c0, times (1 - alpha) for k = 0 and alpha otherwise;  F = 0 with PWA_FOCAL_OFF.
 *   alpha = NaN: no alpha factor.  focal_skip_bg needs PWA_FOCAL_SOFTMAX; alpha needs a focal form and focal_skip_bg = 0.
 * pwa_segloss_bwd: dlogits = d(sum_{q,b,k} dsums[q][b][k] sums[q][b][k]) / dlogits (the G row has no gradient), computed in
 * fp32 and rounded once to the logits' dtype.
 * The forward's CTAs store their partial sums to their own slots of the DEVICE workspace (pwa_segloss_workspace_size bytes, a
 * function of B, K and nvox; needs no GPU) and pwa_colsum_f32 sums the slots in index order: no float atomics, the sums are
 * bitwise reproducible for a given GPU model, build and shape.  Arguments are checked before any CUDA call (PWA_ERR_ARG
 * without a GPU); nothing allocates or synchronises, everything runs on `stream`. */
#define PWA_SEGLOSS_MAX_K 32
enum { PWA_ACT_NONE = 0, PWA_ACT_SIGMOID = 1, PWA_ACT_SOFTMAX = 2 };
enum { PWA_FOCAL_OFF = 0, PWA_FOCAL_SIGMOID = 1, PWA_FOCAL_SOFTMAX = 2 };
typedef struct pwa_segloss {
  int32_t B, K;              /* 1 <= B <= 65535, 2 <= K <= PWA_SEGLOSS_MAX_K */
  int64_t nvox;              /* voxels per sample and class, >= 1 */
  int32_t act, squared_pred, focal, focal_skip_bg;
  float gamma, alpha;        /* gamma >= 0; alpha NaN = none */
} pwa_segloss;

int64_t pwa_segloss_workspace_size(const pwa_segloss* s);
int pwa_segloss_fwd(const void* logits, int dtype, const void* labels, int label_dtype, const pwa_segloss* s, float* sums,
                    void* workspace, int64_t workspace_bytes, void* stream);
int pwa_segloss_bwd(const void* logits, int dtype, const void* labels, int label_dtype, const pwa_segloss* s,
                    const float* dsums, void* dlogits, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* PWA_H_ */
