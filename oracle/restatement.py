"""CPU restatement of the reference's prompted 3D shifted-window attention block.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Written from the behaviour of the
reference (file:line citations are into /root/reference/src/modules/), not from its
code structure: windows are described by explicit index maps, the shift mask by
per-axis region ids, the position bias by three small per-axis tables, and only the
N content tokens of a window are used as queries (the reference also runs the I prompt
rows as queries and then cuts them, `swin_transformer/swin_block.py:222-225`).

Parity pinning: the reference has no tests/goldens of its own; this file is pinned by
`tests/golden/*.npz`, produced by `oracle/gen_golden.py` from the live reference
(`tests/test_oracle_golden.py` holds this file to those vectors).

Everything is plain torch, differentiable, dtype-agnostic (fp32/fp64) and device-agnostic: the CPU is where
it is pinned against the goldens; the BASELINE-size parity tests (`tests/test_gpu_multiwindow.py`) let torch
execute the SAME functions in float64 on the GPU, because a 2.8 GB logit tensor per block takes minutes on
host cores.  None of the repo's kernels is involved either way.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F


# --------------------------------------------------------------------------------------
# geometry
# --------------------------------------------------------------------------------------
def pad_amounts(dims: Sequence[int], ws: Sequence[int]) -> Tuple[int, ...]:
    """The reference's `paddings` list (floor_h, ceil_h, floor_w, ceil_w, floor_d, ceil_d).
    swin_block.py:150-161: if ANY axis is not divisible by its window, EVERY axis gets
    floor/ceil((ws - dim % ws)/2) -- an axis that is already divisible therefore grows by a
    whole window.  NOTE the reference then calls F.pad(x, reversed(paddings)) (:163), and
    reversing the flat list also swaps each (lo, hi) pair: the DATA is padded by ceil on the
    low side and floor on the high side, while the mask box (:345-350) and the final crop
    (:247-253) use floor low / ceil high.  With an odd remainder the block output is therefore
    displaced by one voxel along that axis.  We reproduce this: see `data_lo` / `crop_lo`."""
    if all(d % w == 0 for d, w in zip(dims, ws)):
        return (0, 0, 0, 0, 0, 0)
    out = []
    for d, w in zip(dims, ws):
        r = w - d % w
        out += [r // 2, r - r // 2]
    return tuple(out)


def data_lo(pads) -> Tuple[int, int, int]:
    """Low-side zero padding actually applied to the data (F.pad with reversed list, :163)."""
    return (pads[1], pads[3], pads[5])


def crop_lo(pads) -> Tuple[int, int, int]:
    """Low-side offset used by the output crop (:247-253) and the mask's interior box (:345-350)."""
    return (pads[0], pads[2], pads[4])


def effective_shift(dims: Sequence[int], ws: Sequence[int], shift: Sequence[int]) -> Tuple[int, ...]:
    """swin_block.py:265-270: shift forced to 0 on axes whose UNPADDED size <= window."""
    return tuple(0 if d <= w else s for d, w, s in zip(dims, ws, shift))


def padded_dims(dims, pads):
    return tuple(d + pads[2 * a] + pads[2 * a + 1] for a, d in enumerate(dims))


def _axis_coords(sp: int, w: int) -> np.ndarray:
    """coords[p, t] = rolled-frame coordinate of token index t in window index p along
    one axis.  einops '(h p1)' makes the window-token index the OUTER factor
    (swin_block.py:292-299), i.e. windows are strided: coord = t * (sp // w) + p."""
    n_win = sp // w
    p = np.arange(n_win)[:, None]
    t = np.arange(w)[None, :]
    return t * n_win + p


def gather_index(dims, ws, shift, pads, lo=None) -> np.ndarray:
    """int64 [P, N]: flat index into the UNPADDED volume (h*W*D + w*D + d) of the voxel
    that lands at (window, token) after pad -> roll(-shift) -> strided partition, or -1
    where the voxel is zero padding.  swin_block.py:163,174-178,205,209.  `lo` is the low-side
    offset between padded and unpadded coordinates: data_lo(pads) for the input side (default),
    crop_lo(pads) for the output side."""
    H, W, D = dims
    sp = padded_dims(dims, pads)
    lo = data_lo(pads) if lo is None else lo
    per_axis = []
    for a in range(3):
        r = _axis_coords(sp[a], ws[a])                     # rolled-frame coordinate
        src = (r + shift[a]) % sp[a] - lo[a]               # torch.roll(-s): out[i] = in[(i+s) % S]
        src = np.where((src >= 0) & (src < dims[a]), src, -1)
        per_axis.append(src)
    ah, aw, ad = per_axis                                   # [P_a, w_a]
    # window order (p1 p2 p3) row-major, token order (h w d) row-major
    h = ah[:, None, None, :, None, None]
    w = aw[None, :, None, None, :, None]
    d = ad[None, None, :, None, None, :]
    valid = (h >= 0) & (w >= 0) & (d >= 0)
    flat = np.where(valid, (h * W + w) * D + d, -1)
    P = ah.shape[0] * aw.shape[0] * ad.shape[0]
    N = ws[0] * ws[1] * ws[2]
    return flat.reshape(P, N).astype(np.int64)


def partition_tokens(x: torch.Tensor, ws, shift, pads) -> torch.Tensor:
    """[B,C,H,W,D] -> [B,P,N,C] (zero where padding)."""
    B, C = x.shape[:2]
    dims = tuple(x.shape[2:])
    idx = torch.from_numpy(gather_index(dims, ws, shift, pads)).to(x.device)
    P, N = idx.shape
    flat = x.reshape(B, C, -1)
    flat = torch.cat([flat, flat.new_zeros(B, C, 1)], dim=2)      # slot -1 -> zeros
    g = flat[:, :, idx.reshape(-1)]                                # [B,C,P*N]
    return g.reshape(B, C, P, N).permute(0, 2, 3, 1).contiguous()


def reverse_tokens(y: torch.Tensor, dims, ws, shift, pads) -> torch.Tensor:
    """[B,P,N,C] -> [B,C,H,W,D]: window_reverse + roll back + crop (swin_block.py:228-253).
    Uses the CROP offsets, which differ from the data offsets for odd remainders (see
    pad_amounts).  Every output voxel is hit exactly once."""
    B, P, N, C = y.shape
    idx = torch.from_numpy(gather_index(dims, ws, shift, pads, crop_lo(pads))).reshape(-1).to(y.device)
    keep = idx >= 0
    src = y.permute(0, 3, 1, 2).reshape(B, C, P * N)[:, :, keep]
    out = y.new_zeros(B, C, dims[0] * dims[1] * dims[2])
    out = out.index_copy(2, idx[keep], src)
    return out.reshape(B, C, *dims)


def _axis_region(sp: int, w: int, s: int) -> np.ndarray:
    """Per-axis region index in the rolled frame.  swin_block.py:320-334 fills three Python
    slices in order (later fills overwrite): [0,-w), [-w,-s), [-s,None).  With s == 0 the
    last slice is the whole axis, so everything becomes region 2."""
    reg = np.zeros(sp, dtype=np.int64)
    for k, sl in enumerate((slice(0, -w), slice(-w, -s), slice(-s, None))):
        reg[sl] = k
    return reg


def region_ids(dims, ws, shift, pads) -> np.ndarray:
    """int64 [P, N] region id per (window, token): 9*rh + 3*rw + rd, overwritten by 100
    inside the box [lo, Sp-hi) when any padding exists (swin_block.py:336-350), laid out
    by the same strided partition as the data (:352-356)."""
    sp = padded_dims(dims, pads)
    any_pad = any(p > 0 for p in pads)
    regs, inside, coords = [], [], []
    for a in range(3):
        regs.append(_axis_region(sp[a], ws[a], shift[a]))
        c = np.arange(sp[a])
        inside.append((c >= pads[2 * a]) & (c < sp[a] - pads[2 * a + 1]))
        coords.append(_axis_coords(sp[a], ws[a]))
    ch = coords[0][:, None, None, :, None, None]
    cw = coords[1][None, :, None, None, :, None]
    cd = coords[2][None, None, :, None, None, :]
    ids = 9 * regs[0][ch] + 3 * regs[1][cw] + regs[2][cd]
    if any_pad:
        box = inside[0][ch] & inside[1][cw] & inside[2][cd]
        ids = np.where(box, 100, ids)
    P = coords[0].shape[0] * coords[1].shape[0] * coords[2].shape[0]
    return ids.reshape(P, ws[0] * ws[1] * ws[2])


def attn_mask_from_ids(ids: np.ndarray) -> torch.Tensor:
    """float32 [1,P,N,N], 1.0 where region ids agree (swin_block.py:358-360)."""
    t = torch.from_numpy(ids)
    return (t[:, :, None] == t[:, None, :]).to(torch.float32).unsqueeze(0)


# --------------------------------------------------------------------------------------
# relative position bias
# --------------------------------------------------------------------------------------
def bias_tables(pe: Dict[str, torch.Tensor], ws, embed_dim: int, num_prompt_tokens: int):
    """Per-axis tables T_a[h,i,j] and prompt-token bias tok[h,i], already carrying the
    /3 and embed_dim**-0.5 factors of relative_positional_encoding.py:116-123,136-138.
    R_a[h,i,j] = sum_c weights_content_a[h,c] * enc_content_a[clamp(j-i+w_a-1), c] (:101-115,
    index buffers :40-62 with max_abs_pos = max_cap_dist = window, swin_block.py:118-126)."""
    scale = embed_dim ** -0.5
    tabs = []
    for a, name in enumerate("hwd"):
        w = ws[a]
        enc = pe[f"enc_content_{name}"]
        wt = pe[f"weights_content_{name}"]
        cap = (enc.shape[0] + 1) // 2
        i = torch.arange(w, device=enc.device).reshape(-1, 1)
        j = torch.arange(w, device=enc.device).reshape(1, -1)
        rel = torch.clamp(j - i + cap - 1, 0, 2 * (cap - 1))
        tabs.append(torch.einsum("hc,nmc->hnm", wt, enc[rel]) * (scale / 3.0))
    tok = None
    if num_prompt_tokens > 0:
        enc_tok = torch.cat([pe[k] for k in sorted(k for k in pe if k.startswith("enc_token."))], dim=0)
        assert enc_tok.shape[0] == num_prompt_tokens, "dim_i must equal max_prompts*tokens_per_prompt"
        tok = torch.einsum("hc,ic->hi", pe["weights_token"], enc_tok) * scale
    return tabs[0], tabs[1], tabs[2], tok


def dense_bias(th, tw, td, tok) -> torch.Tensor:
    """[h, N, N+I]; content token n = (ih, iw, id) row-major."""
    h, wh, _ = th.shape
    ww, wd = tw.shape[1], td.shape[1]
    b = (th[:, :, None, None, :, None, None]
         + tw[:, None, :, None, None, :, None]
         + td[:, None, None, :, None, None, :])
    N = wh * ww * wd
    b = b.reshape(h, N, N)
    if tok is not None:
        b = torch.cat([b, tok[:, None, :].expand(-1, N, -1).to(b.dtype)], dim=2)
    return b


# --------------------------------------------------------------------------------------
# attention + block
# --------------------------------------------------------------------------------------
_DROP_PLANE_MUL = (0x9E3779B1, 0x85EBCA77, 0xC2B2AE3D, 0x27D4EB2F, 0x165667B1, 0xD3A2646D, 0xFD7046C5, 0xB55A4F09)
_DROP_PLANE_MUL_B = (0x7FEB352D, 0x846CA68B, 0x2C1B3C6D, 0x297A2D39, 0x9E485565, 0xEF1D6B47, 0x68E31DA5, 0xB5297A4D)


def _drop_bitpos(jj):
    """Bit of a 32-key keep word that holds key jj of the chunk (csrc/attn.cuh: drop_bitpos)."""
    g, odd = jj >> 1, jj & 1
    return ((31 if odd else 23) if g < 8 else (15 if odd else 7)) - (g & 7)


def _drop_threshold(p_drop):
    t = min(int(p_drop * 256.0 + 0.5), 255)
    return 1 if (p_drop > 0 and t == 0) else t


def dropout_keep_factor(seed_words, B, P, num_heads, N, NK, p_drop):
    """The attention-dropout mask of the B200 kernels (csrc/attn.cuh: drop_row_hash / drop_keep_word), restated with
    numpy: float64 [B,P,h,N,NK] holding 0 for dropped and 1/keep_rate for kept entries.  The reference applies
    nn.Dropout to the dense probabilities (window_attention.py:57); the kernels cannot reproduce torch's Philox stream
    over a tensor they never materialise, so parity is: same distribution (Bernoulli, rate in steps of 1/256,
    inverse-keep-rate scaling) and exact agreement with THIS mask for given seed words.
    Per (sample*window, head, query row) one avalanche hash; per 32-key chunk a folded value y; eight planes
    [hi16(y * MB_k) : hi16(y * MA_k)]; key jj of the chunk reads bit drop_bitpos(jj) of every plane, plane k = bit k of an 8-bit number,
    kept iff number >= round(256 p)."""
    M = np.uint64(0xFFFFFFFF)
    u = np.uint64

    def mix(x):
        x = x & M
        x ^= x >> u(16); x = (x * u(0x21f0aaad)) & M
        x ^= x >> u(15); x = (x * u(0x735a2d97)) & M
        x ^= x >> u(15)
        return x

    t = _drop_threshold(p_drop)
    s0, s1 = (u(int(w) & 0xFFFFFFFF) for w in seed_words)
    bw = np.arange(B * P, dtype=np.uint64)[:, None, None, None]
    hd = np.arange(num_heads, dtype=np.uint64)[None, :, None, None]
    n = np.arange(N, dtype=np.uint64)[None, None, :, None]
    j = np.arange(NK, dtype=np.uint64)[None, None, None, :]
    row = mix(s0 + ((((bw * u(num_heads) + hd) * u(N) + n) * u(0x85EBCA77)) & M)) ^ s1
    y = ((row ^ (((j >> u(5)) * u(0x9E3779B1)) & M)) * u(0x2C1B3C6D)) & M
    y ^= y >> u(15)
    pos = np.array([_drop_bitpos(int(v) & 31) for v in range(NK)], dtype=np.uint64)[None, None, None, :]
    num = np.zeros(y.shape, dtype=np.uint64)
    for k, (ma, mb) in enumerate(zip(_DROP_PLANE_MUL, _DROP_PLANE_MUL_B)):
        w = (((y * u(ma)) & M) >> u(16)) | ((y * u(mb)) & u(0xFFFF0000))
        num |= ((w >> pos) & u(1)) << u(k)
    keep = num >= u(t)
    return torch.from_numpy(keep.astype(np.float64) * (256.0 / (256 - t))).reshape(B, P, num_heads, N, NK)


def dropout_keep_factor_torch(seed_words, bw0, n_bw, num_heads, N, NK, p_drop, device="cpu"):
    """dropout_keep_factor for the (sample, window) pairs bw0 .. bw0+n_bw-1 only, as torch int64 arithmetic on
    `device`: float64 [n_bw, h, N, NK].  Same hash, same bit selection (tests/test_host_cpu.py compares the two)."""
    M = 0xFFFFFFFF

    def mix(x):
        x = x & M
        x = x ^ (x >> 16); x = (x * 0x21f0aaad) & M
        x = x ^ (x >> 15); x = (x * 0x735a2d97) & M
        x = x ^ (x >> 15)
        return x

    t = _drop_threshold(p_drop)
    s0, s1 = (int(w) & M for w in seed_words)
    ar = lambda n, shape: torch.arange(n, dtype=torch.int64, device=device).reshape(shape)
    bw = ar(n_bw, (-1, 1, 1, 1)) + bw0
    hd, n, j = ar(num_heads, (1, -1, 1, 1)), ar(N, (1, 1, -1, 1)), ar(NK, (1, 1, 1, -1))
    row = mix(s0 + ((((bw * num_heads + hd) * N + n) * 0x85EBCA77) & M)) ^ s1
    y = ((row ^ (((j >> 5) * 0x9E3779B1) & M)) * 0x2C1B3C6D) & M
    y = y ^ (y >> 15)
    pos = torch.tensor([_drop_bitpos(v & 31) for v in range(NK)], dtype=torch.int64, device=device).reshape(1, 1, 1, -1)
    num = torch.zeros_like(y)
    for k, (ma, mb) in enumerate(zip(_DROP_PLANE_MUL, _DROP_PLANE_MUL_B)):
        w = (((y * ma) & M) >> 16) | ((y * mb) & 0xFFFF0000)
        num = num | (((w >> pos) & 1) << k)
    return (num >= t).to(torch.float64) * (256.0 / (256 - t))


def elementwise_dropout_keep_factor(seed_words, n, p_drop):
    """The projection-dropout mask of csrc/dropout.cu (pwa_dropout) restated: float64 [n] of 0 / (1/keep_rate).  One
    32-bit hash per 4 consecutive elements (two avalanche mixes of seed and quad index), one byte per element, kept iff
    byte >= round(256 p).  Stands for nn.Dropout(proj_drop) (window_attention.py:60): same distribution, different
    stream (torch's Philox)."""
    M = np.uint64(0xFFFFFFFF)
    u = np.uint64

    def mix(x):
        x = x & M
        x ^= x >> u(16); x = (x * u(0x21f0aaad)) & M
        x ^= x >> u(15); x = (x * u(0x735a2d97)) & M
        x ^= x >> u(15)
        return x

    t = _drop_threshold(p_drop)
    s0, s1 = (u(int(w) & 0xFFFFFFFF) for w in seed_words)
    i = np.arange(n, dtype=np.uint64)
    q = i >> u(2)
    h = mix(s0 + ((q & M) * u(0x9E3779B1) & M) + (((q >> u(32)) * u(0x85EBCA77)) & M)) ^ s1
    bits = mix(h)
    byte = (bits >> (u(8) * (i & u(3)))) & u(0xFF)
    return torch.from_numpy((byte >= u(t)).astype(np.float64) * (256.0 / (256 - t)))


def elementwise_dropout_keep_factor_torch(seed_words, n0, n, p_drop, device="cpu"):
    """elementwise_dropout_keep_factor for the elements n0 .. n0+n-1 only, as torch int64 arithmetic on `device`:
    float64 [n].  Same hash, same byte selection (tests/test_oracle_dropout_cpu.py compares the two); a whole-stage mask
    (tens of millions of elements) is then a few device passes instead of a host loop."""
    M = 0xFFFFFFFF

    def mix(x):
        x = x & M
        x = x ^ (x >> 16); x = (x * 0x21f0aaad) & M
        x = x ^ (x >> 15); x = (x * 0x735a2d97) & M
        x = x ^ (x >> 15)
        return x

    t = _drop_threshold(p_drop)
    s0, s1 = (int(w) & M for w in seed_words)
    i = torch.arange(n, dtype=torch.int64, device=device) + int(n0)
    q = i >> 2
    h = mix(s0 + (((q & M) * 0x9E3779B1) & M) + (((q >> 32) * 0x85EBCA77) & M)) ^ s1
    byte = (mix(h) >> (8 * (i & 3))) & 0xFF
    return (byte >= t).to(torch.float64) * (256.0 / (256 - t))


def block_keep_factors(seed_words, x_shape, ws, num_heads, num_prompt_tokens, attn_drop, proj_drop, device="cpu"):
    """The two dropout masks one block of the B200 kernels applies, from the block's four seed words (what
    SwinTransformerBlock draws per forward): words 0-1 seed the attention mask, float64 [B,P,h,N,N+I] over the
    (sample * window) index b*P + p; words 2-3 seed the projection mask, float64 [B,P,N,C] over the block's window-token
    tensor in row-major order (the element index of pwa_dropout and of the fused dropout + residual + LayerNorm GEMM).
    x_shape: the block input [B,C,H,W,D].  A site with rate 0 gets None.  Returns (attn_keep, proj_keep) for
    block_forward."""
    B, C = x_shape[:2]
    ws = tuple(ws)
    sp = padded_dims(tuple(x_shape[2:]), pad_amounts(tuple(x_shape[2:]), ws))
    P = math.prod(s // w for s, w in zip(sp, ws))
    N = math.prod(ws)
    w = [int(v) for v in seed_words]
    attn = proj = None
    if attn_drop > 0:
        attn = dropout_keep_factor_torch(w[0:2], 0, B * P, num_heads, N, N + num_prompt_tokens, attn_drop, device)
        attn = attn.reshape(B, P, num_heads, N, N + num_prompt_tokens)
    if proj_drop > 0:
        proj = elementwise_dropout_keep_factor_torch(w[2:4], 0, B * P * N * C, proj_drop, device).reshape(B, P, N, C)
    return attn, proj


def prompted_window_attention(q, k, v, kp, vp, bias, ids, scale, num_heads, drop=None):
    """q,k,v [B,P,N,C]; kp,vp [B,I,C] or None; bias [h,N,N+I]; ids int [P,N] or None.
    window_attention.py:45-59: logits = (q.k^T*scale + bias) * mask, softmax over keys, [dropout,] @ v.
    Prompt columns are never masked (swin_block.py:187-196).  drop: optional [B,P,h,N,N+I] keep factors
    (0 or 1/keep_rate) applied to the probabilities (window_attention.py:57)."""
    B, P, N, C = q.shape
    dh = C // num_heads

    def split(t):
        return t.reshape(*t.shape[:-1], num_heads, dh)

    qh = split(q).permute(0, 1, 3, 2, 4)                     # [B,P,h,N,dh]
    kh = split(k).permute(0, 1, 3, 2, 4)
    vh = split(v).permute(0, 1, 3, 2, 4)
    if kp is not None:
        kph = split(kp).permute(0, 2, 1, 3)[:, None].expand(-1, P, -1, -1, -1)   # [B,P,h,I,dh]
        vph = split(vp).permute(0, 2, 1, 3)[:, None].expand(-1, P, -1, -1, -1)
        kh = torch.cat([kh, kph], dim=3)
        vh = torch.cat([vh, vph], dim=3)
    s = torch.matmul(qh, kh.transpose(-1, -2)) * scale + bias.to(qh.dtype)[None, None]
    if ids is not None:
        t = torch.as_tensor(ids).to(s.device)
        m = (t[:, :, None] == t[:, None, :]).to(s.dtype)                       # [P,N,N]
        if kp is not None:
            m = torch.cat([m, m.new_ones(P, N, kp.shape[1])], dim=2)
        s = s * m[None, :, None]
    a = torch.softmax(s, dim=-1)
    if drop is not None:
        a = a * drop.to(a.dtype)
    o = torch.matmul(a, vh)                                                    # [B,P,h,N,dh]
    return o.permute(0, 1, 3, 2, 4).reshape(B, P, N, C)


def window_attention_module(sd: Dict[str, torch.Tensor], q, k, v, pos_bias, mask, num_heads: int, drop=None):
    """The whole reference module with its literal arguments (window_attention.py:35-61): to_q / to_k / to_v (no bias),
    head split c = head * dh + d, logits = (q k^T * scale + pos_bias) * mask with pos_bias / mask any tensors (or None)
    that broadcast against [b,p,h,n_q,n_k], softmax over keys, optional keep factors `drop` [b,p,h,n_q,n_k], @ v, proj.
    sd: to_q.weight, to_k.weight, to_v.weight, proj.weight, proj.bias.  q [b,p,n_q,C]; k, v [b,p,n_k,C]."""
    b, p, nq, C = q.shape
    dh = C // num_heads
    scale = dh ** -0.5

    def heads(t):
        return t.reshape(*t.shape[:-1], num_heads, dh).permute(0, 1, 3, 2, 4)     # [b,p,h,n,dh]

    qh = heads(q @ sd["to_q.weight"].t())
    kh = heads(k @ sd["to_k.weight"].t())
    vh = heads(v @ sd["to_v.weight"].t())
    s = torch.matmul(qh, kh.transpose(-1, -2)) * scale
    if pos_bias is not None:
        s = s + pos_bias
    if mask is not None:
        s = s * mask
    a = torch.softmax(s, dim=-1)
    if drop is not None:
        a = a * drop.to(a.dtype)
    o = torch.matmul(a, vh).permute(0, 1, 3, 2, 4).reshape(b, p, nq, C)
    return o @ sd["proj.weight"].t() + sd["proj.bias"]


def split_block_params(sd: Dict[str, torch.Tensor]):
    pe = {k[3:]: v for k, v in sd.items() if k.startswith("pe.")}
    return pe


def block_forward(sd: Dict[str, torch.Tensor], x: torch.Tensor, p: Optional[torch.Tensor],
                  ws, shift_cfg, num_heads: int, attn_drop: float = 0.0, proj_drop: float = 0.0,
                  attn_keep: Optional[torch.Tensor] = None, proj_keep: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One SwinTransformerBlock.forward_attn_mlp (swin_block.py:145-255) from a state dict
    with the reference's key names.  attn_drop / proj_drop > 0: torch's own dropout on the attention probabilities and
    on the projection output, as the reference applies it (window_attention.py:57,60) -- used by the CPU timing arm.
    attn_keep [B,P,h,N,N+I] / proj_keep [B,P,N,C]: explicit keep factors (0 or 1/keep_rate, see block_keep_factors) that
    take the place of the dropout at that site whatever its rate: attn_keep multiplies the attention probabilities,
    proj_keep the projection output o @ Wproj^T + bproj before the residual add."""
    ws = tuple(ws)
    dims = tuple(x.shape[2:])
    C = x.shape[1]
    pads = pad_amounts(dims, ws)
    shift = effective_shift(dims, ws, shift_cfg)
    masked = any(s > 0 for s in shift)
    I = 0 if p is None else p.shape[1]
    pe = split_block_params(sd)
    E = pe["enc_content_h"].shape[1]
    th, tw, td, tok = bias_tables(pe, ws, E, I)
    bias = dense_bias(th, tw, td, tok)
    ids = region_ids(dims, ws, shift, pads) if masked else None

    xw = partition_tokens(x, ws, shift, pads)                                  # [B,P,N,C]
    ln = F.layer_norm(xw, (C,), sd["attn_norm.weight"], sd["attn_norm.bias"], 1e-6)
    q = ln @ sd["attn.to_q.weight"].t()
    k = ln @ sd["attn.to_k.weight"].t()
    v = ln @ sd["attn.to_v.weight"].t()
    kp = vp = None
    if p is not None:
        lp = F.layer_norm(p, (C,), sd["attn_norm.weight"], sd["attn_norm.bias"], 1e-6)
        kp = lp @ sd["attn.to_k.weight"].t()
        vp = lp @ sd["attn.to_v.weight"].t()
    dh = C // num_heads
    drop = attn_keep
    if attn_drop > 0 and attn_keep is None:
        B_, P_, N_ = q.shape[:3]
        drop = F.dropout(torch.ones(B_, P_, num_heads, N_, N_ + I, dtype=q.dtype, device=q.device), attn_drop, True)
    o = prompted_window_attention(q, k, v, kp, vp, bias, ids, dh ** -0.5, num_heads, drop=drop)
    a = o @ sd["attn.proj.weight"].t() + sd["attn.proj.bias"]                  # :60
    if proj_keep is not None:
        a = a * proj_keep.to(a.dtype)
    elif proj_drop > 0:
        a = F.dropout(a, proj_drop, True)
    y = a + xw                                                                  # :222
    z = F.layer_norm(y, (C,), sd["mlp_norm.weight"], sd["mlp_norm.bias"], 1e-6)
    y = y + z @ sd["mlp.weight"].t() + sd["mlp.bias"]                          # :227 single Linear
    return reverse_tokens(y, dims, ws, shift, pads)


def patch_merging_forward(sd: Dict[str, torch.Tensor], x: torch.Tensor, merge_last_dim: bool) -> torch.Tensor:
    """down.py:21-53.  Channel-block order of the 2x2x2 neighbourhood is
    (dh,dw,dd) = 000,100,010,001,110,101,011,111 (:31-39); 2x2x1 is 00,10,01,11 (:41-45)."""
    B, C, H, W, D = x.shape
    # odd axes get one zero plane on the LOW side: the reference reverses the flat list
    # (0,pad_h,0,pad_w,0,pad_d) before F.pad (down.py:26-28), which swaps each (lo,hi) pair.
    x = F.pad(x, (D % 2, 0, W % 2, 0, H % 2, 0))
    H, W, D = x.shape[2:]
    if merge_last_dim:
        offs = [(0, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1), (1, 1, 0), (1, 0, 1), (0, 1, 1), (1, 1, 1)]
        parts = [x[:, :, a::2, b::2, c::2] for a, b, c in offs]
        Do = D // 2
    else:
        offs = [(0, 0), (1, 0), (0, 1), (1, 1)]
        parts = [x[:, :, a::2, b::2, :] for a, b in offs]
        Do = D
    t = torch.cat(parts, dim=1).permute(0, 2, 3, 4, 1)                          # [B,H/2,W/2,Do,kC]
    kc = t.shape[-1]
    t = F.layer_norm(t, (kc,), sd["norm.weight"], sd["norm.bias"], 1e-6)
    t = t @ sd["reduction.weight"].t()
    return t.permute(0, 4, 1, 2, 3).contiguous()


def pair_forward(sd: Dict[str, torch.Tensor], x, p_pair, ws, num_heads, down: bool, merge_last_dim: bool = True,
                 attn_drop: float = 0.0, proj_drop: float = 0.0, keep=None):
    """ConsecutiveSwinBlocks.forward (swin_block.py:66-71): unshifted block, then block
    shifted by ws//2, then optional PatchMerging.  keep: None, or per block the (attn_keep, proj_keep) pair of
    block_forward (block_keep_factors of that block's seed words)."""
    ws = tuple(ws)
    shift = tuple(w // 2 for w in ws)
    for i, sh in enumerate(((0, 0, 0), shift)):
        sub = {k[len(f"swin_blocks.{i}."):]: v for k, v in sd.items() if k.startswith(f"swin_blocks.{i}.")}
        ak, pk = (None, None) if keep is None else keep[i]
        x = block_forward(sub, x, p_pair[i], ws, sh, num_heads, attn_drop, proj_drop, attn_keep=ak, proj_keep=pk)
    if down:
        sub = {k[len("merge."):]: v for k, v in sd.items() if k.startswith("merge.")}
        x = patch_merging_forward(sub, x, merge_last_dim)
    return x
