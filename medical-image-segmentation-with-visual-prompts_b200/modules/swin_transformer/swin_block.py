"""Prompted 3D shifted-window transformer block on hand-written sm_100a kernels.

Drop-in for the reference's swin_transformer/swin_block.py: `ConsecutiveSwinBlocks` (:16-95),
`SwinTransformerBlock` (:98-289) and the free functions `window_partition` (:292), `window_reverse`
(:302), `get_attn_mask` (:312) keep their constructor arguments, forward(x, p) signatures, parameter
names/shapes (state-dict compatible) and parameter-group accessors.

What differs is HOW one block runs (reference forward_attn_mlp, :145-255):
  reference: F.pad -> RelativePE dense bias -> torch.roll -> dense float mask [1,P,N',N'] -> rearrange ->
             cat(prompts) per window -> LN -> 3 Linear -> bmm/softmax/bmm over [B,P,h,N',N'] -> ...
  here:      ONE partition kernel (pad + roll + strided window gather + channels-last, csrc/partition.cu)
             -> LN -> Linear -> ONE fused attention kernel (bias tables + uint8 region ids + softmax + PV,
             prompt K/V computed once per sample instead of once per window, csrc/attn_*.cu)
             -> proj/residual/LN/Linear -> ONE reverse kernel (window reverse + roll back + crop).
Only the N content tokens are queries: the reference also pushes the I prompt rows of every window
through attention and cuts them afterwards (:222-225), which cannot influence the output.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F
import torch.utils.checkpoint as checkpoint

from ... import functional as PF
from ...geometry import get_geometry, rowmap_from_voxels, rowmap_regroup
from ..multi_head_attention import BiasTables, RelativePE, WindowAttention
from .down import PatchMerging


import os as _os
_NO_TOKEN_GEMM = _os.environ.get("PWA_NO_TOKEN_GEMM", "0") == "1"      # (A/B measurements: separate LayerNorm kernels + cuBLAS)
_CKPT_POLICY = _os.environ.get("PWA_CHECKPOINT", "selective")           # 'selective' | 'full' (see _tokens_forward_ckpt)
_FORCE_TOKEN_GEMM = _os.environ.get("PWA_FORCE_TOKEN_GEMM", "0") == "1"  # (tests: the fused kernels at every supported shape)


def _is_channels_last(x):
    """[B,C,H,W,D] tensor whose memory is [B,H,W,D,C]-contiguous (what PatchMerging's final rearrange leaves,
    reference down.py:48-53)."""
    return x.dim() == 5 and x.shape[1] > 1 and x.permute(0, 2, 3, 4, 1).is_contiguous()


def _partition_any(x, geom):
    """pad + roll + strided window partition -> [B,P,N,C]: a row gather for channels-last memory, the transposing
    partition kernel (csrc/partition.cu) for the reference's channels-first layout."""
    if _is_channels_last(x):
        b, c = x.shape[:2]
        rows = x.permute(0, 2, 3, 4, 1).reshape(b, -1, c)
        return PF.gather_rows(rows, None, rowmap_from_voxels(geom)).view(b, geom.P, geom.N, c)
    return PF.partition_tokens(x, geom)


class _SideInputs:
    """What one block's forward needs that does NOT depend on the feature map: the relative-position bias tables, the
    five Linear weights packed in the compute dtype, and the K|V projection of the LayerNorm-ed prompt tokens.  About ten
    launches of 2-10 us per block (and as many again in backward) that would otherwise sit serially between the big
    kernels; `ConsecutiveSwinBlocks` computes them for both blocks on a side stream, where they overlap the partition /
    LayerNorm / projection kernels of the main chain (a captured step keeps them as a parallel graph branch, and
    autograd runs their backward on the same side stream).  `ready` is recorded on that stream after the last of them."""
    __slots__ = ("tables", "lowp", "kvp", "seed", "ready")

    def __init__(self, tables, lowp, kvp, seed=None, ready=None):
        self.tables, self.lowp, self.kvp, self.seed, self.ready = tables, lowp, kvp, seed, ready

    def tensors(self):
        out = [t for t in self.tables if t is not None] + [self.lowp['qkv']._base]
        if self.kvp is not None:
            out.append(self.kvp)
        if self.seed is not None:
            out.append(self.seed)
        return out


_SIDE_STREAMS = {}


def _side_stream(device):
    key = torch.device(device).index if torch.device(device).index is not None else torch.cuda.current_device()
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=key)
    return _SIDE_STREAMS[key]


class ConsecutiveSwinBlocks(nn.Module):
    """Unshifted block, block shifted by window//2, optional PatchMerging (reference :16-71)."""

    def __init__(self, hidden_channels: int, num_heads: int, pos_bias_embed_dim: int, max_prompts: int,
                 tokens_per_prompt: int, window_size: Sequence[int], use_token_params: bool = True,
                 shift_size: Sequence[int] = None, down: bool = True, merge_last_dim: bool = True,
                 use_checkpoint: bool = False, out_channels: int = None, proj_drop: float = 0.0,
                 attn_drop: float = 0.0):
        super().__init__()
        self.window_size = window_size
        self.shift_size = tuple(s // 2 for s in window_size) if shift_size is None else shift_size
        self.no_shift = tuple(0 for _ in window_size)
        self.down = down
        self.use_checkpoint = use_checkpoint
        self.checkpoint_policy = _CKPT_POLICY
        self.swin_blocks = nn.ModuleList([
            SwinTransformerBlock(hidden_channels=hidden_channels, window_size=self.window_size,
                                 pos_bias_embed_dim=pos_bias_embed_dim, num_heads=num_heads, max_prompts=max_prompts,
                                 tokens_per_prompt=tokens_per_prompt, use_token_params=use_token_params,
                                 shift_size=shift, attn_drop=attn_drop, proj_drop=proj_drop,
                                 use_checkpoint=use_checkpoint)
            for shift in (self.no_shift, self.shift_size)])
        if down:
            self.merge = PatchMerging(in_channels=hidden_channels,
                                      out_channels=2 * hidden_channels if out_channels is None else out_channels,
                                      merge_last_dim=merge_last_dim)

    def _token_pipeline_ok(self, x):
        if not x.is_cuda or x.dim() != 5:
            return False
        # block-level hooks must keep firing: fall back to calling the blocks one by one
        mods = list(self.swin_blocks) + ([self.merge] if self.down else [])
        return not any(m._forward_hooks or m._forward_pre_hooks or m._backward_hooks for m in mods)

    def forward(self, x, p=(None, None)):
        if not self._token_pipeline_ok(x):
            for blk, prompt in zip(self.swin_blocks, p):
                x = blk(x, prompt)
            return self.merge(x) if self.down else x
        # Token pipeline: between the two blocks (and into PatchMerging) the feature map never leaves the
        # channels-last token layout.  The reference's window_reverse -> roll back -> crop -> pad -> roll ->
        # window_partition chain (:228-253 then :150-214) is ONE row gather (csrc/gather.cu) with a host-composed
        # index map, fused with the block's last residual add.
        blk0, blk1 = self.swin_blocks
        g0, g1 = blk0._geometry(x.shape[2:]), blk1._geometry(x.shape[2:])
        cdt, in_dtype = blk0._compute_dtype(x), x.dtype
        with torch.autocast('cuda', enabled=False):
            side = self._take_prefetched(x, p, cdt) or self._side_inputs_async(x, p, cdt)
            tok = _partition_any(x.to(cdt), g0)
            y, m = blk0._tokens_forward_ckpt(tok, p[0], g0, cdt, side[0])
            tok = PF.gather_rows(y, m, rowmap_regroup(g0, g1)).view(x.shape[0], g1.P, g1.N, x.shape[1])
            y, m = blk1._tokens_forward_ckpt(tok, p[1], g1, cdt, side[1])
            if self.down:
                out = self.merge.forward_tokens(y, m, g1)
            else:
                out = PF.reverse_add_tokens(y, m, g1)
        return out.to(in_dtype)

    def prefetch_side_inputs(self, p, like: torch.Tensor):
        """Start computing what the two blocks need besides the feature map (bias tables, packed weights, prompt K|V: see
        _SideInputs) NOW, on the side stream, for a forward(x, p) that comes later with the same prompt tensors.  A model
        calls this for ALL of its stages at the top of its forward: their ~14 tiny launches per stage then run under the
        first stage's long kernels instead of in front of each stage's first GEMM (the parameters and prompts they depend
        on are known from the start).  `like`: any tensor with the device and dtype the stage's input will have.  Only
        acts under CUDA-graph capture (launched eagerly the step is host-bound and a second stream costs more than it hides);
        results that no forward claims are dropped by the next call."""
        self._prefetched = None
        if not (like.is_cuda and torch.cuda.is_current_stream_capturing()):
            return
        cdt = self.swin_blocks[0]._compute_dtype(like)
        c = self.swin_blocks[0].mlp.weight.shape[0]
        with torch.autocast('cuda', enabled=False):
            side = self._side_inputs_async(like, p, cdt, channels=c)
        self._prefetched = (tuple(p), cdt, side)

    def _take_prefetched(self, x, p, cdt):
        pre, self._prefetched = getattr(self, "_prefetched", None), None
        if pre is None or pre[1] != cdt or len(pre[0]) != len(p) or any(a is not b for a, b in zip(pre[0], p)):
            return None
        return pre[2]

    def _side_inputs_async(self, x, p, cdt, channels=None):
        """_SideInputs of both blocks; under CUDA-graph capture they are enqueued on the device's side stream (forked
        from the capturing stream here, joined by each block right before its first use of them)."""
        main = torch.cuda.current_stream(x.device)
        side = _side_stream(x.device)
        channels = x.shape[1] if channels is None else channels
        if not torch.cuda.is_current_stream_capturing():
            # launched eagerly the step is bound by the host, not by the device: a second stream only adds event and
            # stream-switch calls (measured: 10.7 -> 13.0 ms per step); the branch pays off as a parallel graph branch
            return [blk._side_inputs(prompt, cdt, channels) for blk, prompt in zip(self.swin_blocks, p)]
        side.wait_stream(main)
        out = []
        with torch.cuda.stream(side):
            for blk, prompt in zip(self.swin_blocks, p):
                si = blk._side_inputs(prompt, cdt, channels)
                si.ready = torch.cuda.Event()
                si.ready.record(side)
                for t in si.tensors():
                    t.record_stream(main)          # allocated on the side stream, consumed on the main one
                out.append(si)
        return out

    def named_parameters_body(self):
        out = [kv for blk in self.swin_blocks for kv in blk.named_parameters_body()]
        if self.down:
            out.extend(self.merge.named_parameters())
        return out

    def named_parameters_bias_content(self):
        return [kv for blk in self.swin_blocks for kv in blk.named_parameters_bias_content()]

    def named_parameters_bias_prompt_tokens(self):
        return [kv for blk in self.swin_blocks for kv in blk.named_parameters_bias_prompt_tokens()]


class SwinTransformerBlock(nn.Module):
    def __init__(self, hidden_channels: int, window_size: Sequence[int], pos_bias_embed_dim: int, num_heads: int,
                 max_prompts: int, tokens_per_prompt: int, use_token_params: bool = True,
                 shift_size: Optional[Sequence[int]] = None, attn_drop: float = 0.0, proj_drop: float = 0.0,
                 use_checkpoint: bool = False):
        super().__init__()
        self.num_heads = num_heads
        self.window_size = window_size
        self.shift_size = shift_size
        self.use_checkpoint = use_checkpoint
        self.checkpoint_policy = _CKPT_POLICY
        # submodule creation order = reference order (:118-143), so seeded init is bit-identical
        self.pe = RelativePE(embed_dim=pos_bias_embed_dim, num_heads=num_heads, max_abs_pos=window_size,
                             max_cap_dist=window_size, max_prompts=max_prompts, tokens_per_prompt=tokens_per_prompt,
                             use_token_params=use_token_params)
        self.attn_norm = nn.LayerNorm(hidden_channels, eps=1e-6)
        self.attn = WindowAttention(dim=hidden_channels, num_heads=num_heads, attn_drop=attn_drop, proj_drop=proj_drop)
        self.mlp_norm = nn.LayerNorm(hidden_channels, eps=1e-6)
        self.mlp = nn.Linear(hidden_channels, hidden_channels)    # the reference "MLP" is ONE Linear (:141-143)

    def _compute_dtype(self, x):
        """bf16 for a bf16 input or under autocast(bfloat16); fp16 for an fp16 input or under autocast(float16) (torch's
        default autocast dtype); else fp32.  The 16-bit types run on the tcgen05 kernels, fp32 on the CUDA-core ones."""
        if x.dtype == torch.bfloat16:
            return torch.bfloat16
        autocast = torch.get_autocast_dtype('cuda') if torch.is_autocast_enabled() else None
        if autocast == torch.bfloat16:
            return torch.bfloat16
        if x.dtype == torch.float16 or autocast == torch.float16:
            return torch.float16
        return torch.float32

    def _lowp_weights(self, cdt):
        """The five Linear weights and the two Linear biases of the block concatenated and cast to the compute dtype
        with ONE cat + ONE cast (instead of a cast per Linear and call); slices: qkv [3C,C], kv [2C,C], proj [C,C],
        mlp [C,C], proj_b [C], mlp_b [C]."""
        with torch.no_grad():
            a = self.attn
            c = self.mlp.weight.shape[0]
            w = torch.cat([a.to_q.weight, a.to_k.weight, a.to_v.weight, a.proj.weight, self.mlp.weight,
                           a.proj.bias[None], self.mlp.bias[None]], dim=0).to(cdt)
        return {'qkv': w[:3 * c], 'kv': w[c:3 * c], 'proj': w[3 * c:4 * c], 'mlp': w[4 * c:5 * c],
                'proj_b': w[5 * c], 'mlp_b': w[5 * c + 1]}

    def _side_inputs(self, p, cdt, c):
        """Bias tables, packed low-precision weights and the prompt K|V projection (see _SideInputs)."""
        ws = tuple(self.window_size)
        n_prompt = 0 if p is None else p.size(1)
        tables = self.pe.tables(ws[0], ws[1], ws[2], n_prompt)
        lowp = self._lowp_weights(cdt)
        kvp = None
        if p is not None:
            if p.dim() != 3 or p.shape[-1] != c:
                raise ValueError(f"SwinTransformerBlock: prompt tokens must be [B, I, {c}], got {tuple(p.shape)}")
            prompts = PF.layer_norm(p.to(cdt), self.attn_norm.weight, self.attn_norm.bias, 1e-6)
            kvp = self.attn.project_prompts(prompts, lowp)
        # the four dropout seed words of this forward (attention, projection): one tiny RNG launch that belongs on the side
        # branch as well, and outside every checkpointed region
        seed = None
        if self.training and (self.attn.attn_drop.p > 0 or self.attn.proj_drop.p > 0):
            seed = PF.new_dropout_seed(tables[0].device, 4)
        return _SideInputs(tables, lowp, kvp, seed)

    def _use_token_gemm(self, c, rows, dtype):
        return (PF.layer_norm_supported(c) and PF.token_gemm_supported(c, 3 * c, dtype) and not _NO_TOKEN_GEMM
                and (_FORCE_TOKEN_GEMM or PF.token_gemm_profitable(c, rows)))

    # The token-domain work of a block (reference :215-227) in three pieces, so that activation checkpointing can wrap
    # the two cheap ones and leave the attention kernel's results saved (see _tokens_forward):
    def _seg_pre(self, xw, cdt, side):
        """attn_norm + q|k|v projection: window tokens [B,P,N,C] -> (alias of xw for the shortcut, q|k|v [B,P,N,3C])."""
        c = xw.shape[-1]
        a_ = self.attn
        if side.ready is not None:
            torch.cuda.current_stream(xw.device).wait_event(side.ready)
        if self._use_token_gemm(c, xw.numel() // c, xw.dtype):
            # SURVEY 8f-1: LayerNorm-1 + q|k|v projection in ONE tcgen05 kernel (csrc/token_gemm.cu)
            return PF.ln_linear_pass(xw, self.attn_norm.weight, self.attn_norm.bias, 1e-6, side.lowp['qkv'],
                                     a_.to_q.weight, a_.to_k.weight, a_.to_v.weight)
        # pwa LayerNorm kernels (csrc/ln.cu).  xw is needed again as the shortcut: its second use goes through the alias, so
        # that both of its gradients are summed inside the LayerNorm-backward kernel
        xw, tokens = PF.layer_norm_with_passthrough(xw, self.attn_norm.weight, self.attn_norm.bias, 1e-6)
        return xw, PF.multi_linear(tokens, None, a_.to_q.weight, a_.to_k.weight, a_.to_v.weight, lowp=side.lowp['qkv'])

    def _seg_post(self, o, xw, cdt, side, drop_seed):
        """Output projection, projection dropout, `+ shortcut`, mlp_norm, MLP Linear: (attention output, shortcut) ->
        (y, m) with block output tokens = y + m."""
        c = xw.shape[-1]
        a_ = self.attn
        lowp = side.lowp
        _, p_proj = a_._drop_rates()
        if self._use_token_gemm(c, xw.numel() // c, xw.dtype):
            # projection dropout + residual add + LayerNorm-2 + MLP Linear in ONE kernel; its backward also yields the
            # gradients of proj.bias and mlp.bias
            a = a_.project_out(o, lowp, dropout=False)
            return PF.drop_add_ln_linear(a, xw, self.mlp_norm.weight, self.mlp_norm.bias, 1e-6, lowp['mlp'], lowp['mlp_b'],
                                         p_proj, None if drop_seed is None else drop_seed[2:4], self.mlp.weight, self.mlp.bias,
                                         bias_of_a=a_.proj.bias)
        # the gradients of proj.bias and mlp.bias are column sums of tensors the mlp_norm backward streams anyway (d of the
        # attention branch, and d of y which equals d of m: both only meet in y + m); the two Linears skip their own bias
        # reductions.  mlp.bias: always.  proj.bias: only without projection dropout between proj and the add (with it,
        # d(proj output) = mask * d(attention branch), a different column sum).
        fuse_db = p_proj == 0
        a = a_.project_out(o, lowp, proj_bias_grad=not fuse_db, drop_seed=drop_seed)
        y, z = PF.add_layer_norm(a, xw, self.mlp_norm.weight, self.mlp_norm.bias, 1e-6,
                                 bias_of_x=a_.proj.bias if fuse_db else None, bias_of_res=self.mlp.bias)
        m = PF.multi_linear(z, self.mlp.bias, self.mlp.weight, lowp=lowp['mlp'], bias_grad=False, lowp_bias=lowp['mlp_b'])
        return y, m

    def _tokens_forward(self, xw, p, geom, cdt, drop_seed=None, side=None, ckpt=False):
        """Window tokens [B,P,N,C] (= shortcut) -> (y, m) with block output tokens = y + m  (reference :215-227);
        the last add is left to the consumer (window reverse / regroup / PatchMerging gather fuse it).
        ckpt: the two token segments around the attention kernel run under activation checkpointing; the kernel's own
        saved tensors (q|k|v, its output, the log-sum-exp) stay, so the backward recomputes two LayerNorms and two small
        GEMMs per block but never the attention.  The [B,P,h,N',N'] logits -- what checkpointing is there to avoid in the
        reference -- never exist here in either mode."""
        ws = tuple(self.window_size)
        ids = geom.region_ids(xw.device) if geom.masked else None
        c = xw.shape[-1]
        if not PF.layer_norm_supported(c):
            raise NotImplementedError(f"SwinTransformerBlock: hidden_channels = {c} (the LayerNorm kernels need a multiple of "
                                      "4, at most 2048); there is no torch fallback")
        if side is None:
            side = self._side_inputs(p, cdt, c)
        if drop_seed is None:
            drop_seed = side.seed
        run = ((lambda fn, *a: checkpoint.checkpoint(fn, *a, use_reentrant=False, preserve_rng_state=False)) if ckpt
               else (lambda fn, *a: fn(*a)))
        xw, qkv = run(self._seg_pre, xw, cdt, side)
        th, tw, td, tok = side.tables
        o = self.attn.attend_packed(qkv, BiasTables(th, tw, td, tok, ws), ids, side.kvp, drop_seed)
        return run(self._seg_post, o, xw, cdt, side, drop_seed)

    def _tokens_forward_ckpt(self, xw, p, geom, cdt, side=None):
        """_tokens_forward, under activation checkpointing when `use_checkpoint` is set (reference :257-260).  The
        seed words of the attention dropout AND of the projection dropout (both seeded kernels, csrc/attn.cuh and
        csrc/dropout.cu) are drawn OUTSIDE the checkpointed regions and passed in, so the recomputation sees the same masks
        without saving / restoring the CUDA generator state -- which a graph capture cannot do.  The reference's example
        config (use_checkpoint, attn_drop = proj_drop = 0.1) therefore runs inside a captured step.
        `checkpoint_policy`: 'selective' (default) keeps the attention kernel's results and recomputes only the token
        segments around it; 'full' recomputes the whole token pipeline of the block, attention included."""
        if not (self.use_checkpoint and torch.is_grad_enabled()):
            return self._tokens_forward(xw, p, geom, cdt, None, side)
        if side is None:
            side = self._side_inputs(p, cdt, xw.shape[-1])
        seed = side.seed
        if self.checkpoint_policy == 'selective':
            return self._tokens_forward(xw, p, geom, cdt, seed, side, True)
        return checkpoint.checkpoint(self._tokens_forward, xw, p, geom, cdt, seed, side, use_reentrant=False,
                                     preserve_rng_state=False)

    def _geometry(self, dims):
        shift_cfg = tuple(self.shift_size) if self.shift_size is not None else (0, 0, 0)
        return get_geometry(tuple(int(d) for d in dims), tuple(self.window_size), shift_cfg)

    def forward_attn_mlp(self, x, p=None):
        if not x.is_cuda:
            raise RuntimeError("pwa_b200.SwinTransformerBlock runs on CUDA (sm_100a) only; there is no CPU path")
        geom = self._geometry(x.shape[2:])
        cdt = self._compute_dtype(x)
        in_dtype = x.dtype
        with torch.autocast('cuda', enabled=False):
            xw = _partition_any(x.to(cdt), geom)                            # [B,P,N,C] = shortcut
            y, m = self._tokens_forward(xw, p, geom, cdt)
            out = PF.reverse_add_tokens(y, m, geom)                         # reverse(y + mlp(LN2(y))) -> [B,C,H,W,D]
        return out.to(in_dtype)

    def forward(self, x, p=None):
        if self.use_checkpoint:
            return checkpoint.checkpoint(self.forward_attn_mlp, x, p, use_reentrant=False)
        return self.forward_attn_mlp(x, p)

    def get_shift_size(self, shape_x):
        return tuple(0 if d <= w else s for d, w, s in zip(shape_x, self.window_size, self.shift_size))

    def named_parameters_body(self):
        return [*self.attn_norm.named_parameters(), *self.attn.named_parameters(),
                *self.mlp_norm.named_parameters(), *self.mlp.named_parameters()]

    def named_parameters_bias_content(self):
        return [*self.pe.named_parameters_bias_content()]

    def named_parameters_bias_prompt_tokens(self):
        return [*self.pe.named_parameters_bias_prompt_tokens()]


# --------------------------------------------------------------------------------------------------
# free functions with the reference's signatures
# --------------------------------------------------------------------------------------------------
def window_partition(x, window_size):
    """[b,c,H,W,D] -> [b,P,c,wh,ww,wd], strided windows (reference :292-299).  Dims must be divisible."""
    ws = tuple(window_size)
    geom = get_geometry(tuple(x.shape[2:]), ws, (0, 0, 0))
    if geom.padded:
        raise RuntimeError("window_partition: feature map not divisible by the window")
    tok = PF.partition_tokens(x, geom)                                      # [b,P,N,c]
    return tok.permute(0, 1, 3, 2).reshape(x.shape[0], geom.P, x.shape[1], *ws)


def window_reverse(x, window_size, shape_x):
    """[b,P,c,wh,ww,wd] -> [b,c,H,W,D] (reference :302-309)."""
    ws = tuple(window_size)
    geom = get_geometry(tuple(shape_x), ws, (0, 0, 0))
    b, P, c = x.shape[:3]
    tok = x.reshape(b, P, c, geom.N).permute(0, 1, 3, 2).contiguous()
    return PF.reverse_tokens(tok, geom)


def get_attn_mask(shape_x: Sequence[int], window_size: Sequence[int], shift_size: Sequence[int],
                  paddings: Sequence[int], device: Optional[torch.device] = None):
    """float32 [1,P,N,N] multiplicative shift mask (reference :312-364), expanded from the uint8 region
    ids the kernels use.  `shape_x` is the PADDED shape and `paddings` the reference's floor/ceil list."""
    from ... import _lib
    import ctypes as C
    import numpy as np
    g = _lib.PwaGeom()
    for a in range(3):
        g.ws[a], g.shift[a], g.sp[a] = window_size[a], shift_size[a], shape_x[a]
        g.pads[2 * a], g.pads[2 * a + 1] = paddings[2 * a], paddings[2 * a + 1]
        g.nwin[a] = shape_x[a] // window_size[a]
    g.P = g.nwin[0] * g.nwin[1] * g.nwin[2]
    g.N = window_size[0] * window_size[1] * window_size[2]
    g.padded = int(any(v > 0 for v in paddings))
    ids = np.empty((g.P, g.N), dtype=np.uint8)
    _lib.check(_lib.lib.pwa_region_ids(C.byref(g), ids.ctypes.data), "pwa_region_ids")
    t = torch.from_numpy(ids).to(device if device is not None else 'cpu')
    return (t[:, :, None] == t[:, None, :]).to(torch.float32).unsqueeze(0)
