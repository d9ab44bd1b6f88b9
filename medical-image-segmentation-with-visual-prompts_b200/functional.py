"""torch.autograd glue around the C-ABI kernels.  PyTorch is plumbing here (device memory, streams,
autograd graph); all work is done by the sm_100a kernels in libpwa_b200.so.  CUDA tensors only."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import functools

import torch

from . import _lib
from .geometry import Geometry

_DT = {torch.float32: _lib.PWA_F32, torch.bfloat16: _lib.PWA_BF16, torch.float16: _lib.PWA_F16}
_LOWP = (torch.bfloat16, torch.float16)          # the 16-bit compute types: tcgen05 kernels where the shape allows


class KernelStats:
    """Launch accounting for bench.py: how many of OUR kernels were launched, and (optionally) CUDA-event
    timings around each C-ABI call on the launching stream.  Off by default (zero overhead)."""
    enabled = False
    timing = False
    launches = 0
    records = []          # (name, start_event, end_event, work) ; work = algorithmic FLOPs or bytes

    @classmethod
    def reset(cls, enabled=True, timing=False):
        cls.enabled, cls.timing, cls.launches, cls.records = enabled, timing, 0, []

    @classmethod
    def summary(cls):
        """name -> (calls, total_ms, total_work).  Call after torch.cuda.synchronize()."""
        out = {}
        for name, e0, e1, work in cls.records:
            c, ms, w = out.get(name, (0, 0.0, 0.0))
            out[name] = (c + 1, ms + e0.elapsed_time(e1), w + work)
        return out


class _timed:
    def __init__(self, name, n_kernels, work, t):
        self.name, self.n, self.work, self.t = name, n_kernels, work, t

    def __enter__(self):
        if KernelStats.enabled:
            KernelStats.launches += self.n
            if KernelStats.timing:
                self.e0 = torch.cuda.Event(enable_timing=True)
                self.e1 = torch.cuda.Event(enable_timing=True)
                self.e0.record(torch.cuda.current_stream(self.t.device))
        return self

    def __exit__(self, *exc):
        if KernelStats.enabled and KernelStats.timing:
            self.e1.record(torch.cuda.current_stream(self.t.device))
            KernelStats.records.append((self.name, self.e0, self.e1, self.work))
        return False


def _dtype_code(t: torch.Tensor) -> int:
    if t.dtype not in _DT:
        raise TypeError(f"pwa kernels support float32, bfloat16 and float16, got {t.dtype}")
    return _DT[t.dtype]


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("pwa_b200 has no CPU path: tensors must live on a CUDA device (sm_100a)")


def _stream(t: torch.Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(0 if t is None else t.data_ptr())


# ------------------------------------------------------------------------------------------------
# (a) partition / reverse
# ------------------------------------------------------------------------------------------------
def _force_bits(force_generic, force_word, force_vec):
    """Kernel selection bits of pwa_partition / pwa_reverse (tests cross-check the paths): default = TMA-staged kernel
    when the shape is inside its envelope, else vector -> word -> generic."""
    return (2 if force_generic else 0) | (4 if force_word else 0) | (8 if force_vec else 0)


def _partition_raw(x: torch.Tensor, geom: Geometry, crop_lo: int, force_generic: bool = False,
                   force_word: bool = False, force_vec: bool = False) -> torch.Tensor:
    B, Cc = x.shape[:2]
    out = torch.empty((B, geom.P, geom.N, Cc), dtype=x.dtype, device=x.device)
    with torch.cuda.device(x.device), _timed("partition", 1, 2.0 * out.numel() * out.element_size(), x):
        rc = _lib.lib.pwa_partition(_ptr(x), _ptr(out), B, Cc, geom.ref(), crop_lo | _force_bits(force_generic, force_word, force_vec),
                                    _dtype_code(x), _stream(x))
    _lib.check(rc, "pwa_partition")
    return out


def _reverse_raw(tok: torch.Tensor, geom: Geometry, crop_lo: int, force_generic: bool = False,
                 force_word: bool = False, force_vec: bool = False) -> torch.Tensor:
    B, _, _, Cc = tok.shape
    out = torch.empty((B, Cc, *geom.dims), dtype=tok.dtype, device=tok.device)
    with torch.cuda.device(tok.device), _timed("reverse", 1, 2.0 * tok.numel() * tok.element_size(), tok):
        rc = _lib.lib.pwa_reverse(_ptr(tok), _ptr(out), B, Cc, geom.ref(), crop_lo | _force_bits(force_generic, force_word, force_vec),
                                  _dtype_code(tok), _stream(tok))
    _lib.check(rc, "pwa_reverse")
    return out


class _Partition(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, geom):
        ctx.geom = geom
        return _partition_raw(x.contiguous(), geom, 0)

    @staticmethod
    def backward(ctx, g):
        # adjoint of a gather = scatter with the same (data-side) index map; padding slots drop out
        return _reverse_raw(g.contiguous(), ctx.geom, 0), None


class _Reverse(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tok, geom):
        ctx.geom = geom
        return _reverse_raw(tok.contiguous(), geom, 1)

    @staticmethod
    def backward(ctx, g):
        return _partition_raw(g.contiguous(), ctx.geom, 1), None


class _ReverseAdd(torch.autograd.Function):
    @staticmethod
    def forward(ctx, tok_a, tok_b, geom):
        ctx.geom = geom
        tok_a, tok_b = tok_a.contiguous(), tok_b.contiguous()
        B, _, _, Cc = tok_a.shape
        out = torch.empty((B, Cc, *geom.dims), dtype=tok_a.dtype, device=tok_a.device)
        with torch.cuda.device(tok_a.device), _timed("reverse", 1, 3.0 * tok_a.numel() * tok_a.element_size(), tok_a):
            rc = _lib.lib.pwa_reverse_add(_ptr(tok_a), _ptr(tok_b), _ptr(out), B, Cc, geom.ref(), 1, _dtype_code(tok_a),
                                          _stream(tok_a))
        _lib.check(rc, "pwa_reverse_add")
        return out

    @staticmethod
    def backward(ctx, g):
        d = _partition_raw(g.contiguous(), ctx.geom, 1)
        return d, d, None


def reverse_add_tokens(tok_a: torch.Tensor, tok_b: torch.Tensor, geom: Geometry) -> torch.Tensor:
    """reverse_tokens(tok_a + tok_b) in one kernel (the block's last residual add, swin_block.py:227)."""
    _require_cuda(tok_a, tok_b)
    if tok_a.shape != tok_b.shape or tok_a.dtype != tok_b.dtype or tuple(tok_a.shape[1:3]) != (geom.P, geom.N):
        raise ValueError("reverse_add_tokens: mismatching token tensors")
    return _ReverseAdd.apply(tok_a, tok_b, geom)


def partition_tokens(x: torch.Tensor, geom: Geometry) -> torch.Tensor:
    """[B,C,H,W,D] -> [B,P,N,C]: zero-pad, roll by -shift, strided window partition, channels last."""
    _require_cuda(x)
    if tuple(x.shape[2:]) != geom.dims:
        raise ValueError(f"feature map {tuple(x.shape[2:])} does not match geometry {geom.dims}")
    return _Partition.apply(x, geom)


def reverse_tokens(tok: torch.Tensor, geom: Geometry) -> torch.Tensor:
    """[B,P,N,C] -> [B,C,H,W,D]: window reverse, roll back, crop."""
    _require_cuda(tok)
    if tuple(tok.shape[1:3]) != (geom.P, geom.N):
        raise ValueError(f"token tensor {tuple(tok.shape)} does not match geometry P={geom.P} N={geom.N}")
    return _Reverse.apply(tok, geom)


# ------------------------------------------------------------------------------------------------
# row gather between channels-last arrangements (csrc/gather.cu)
# ------------------------------------------------------------------------------------------------
def _gather_rows_raw(a: torch.Tensor, b: Optional[torch.Tensor], idx: torch.Tensor, rows_src: int, rows_dst: int):
    B, Cc = a.shape[0], a.shape[-1]
    out = torch.empty((B, rows_dst, Cc), dtype=a.dtype, device=a.device)
    nbytes = ((2 if b is None else 3) * min(rows_src, rows_dst) * B * Cc) * a.element_size()
    with torch.cuda.device(a.device), _timed("gather_rows", 1, float(nbytes), a):
        rc = _lib.lib.pwa_gather_rows(_ptr(a), _ptr(b), _ptr(out), _ptr(idx), B, rows_src, rows_dst, Cc, _dtype_code(a),
                                      _stream(a))
    _lib.check(rc, "pwa_gather_rows")
    return out


class _GatherRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, rowmap):
        fwd, bwd = rowmap.on(a.device)
        a = a.contiguous()
        b = b.contiguous() if b is not None else None
        ctx.rowmap, ctx.has_b, ctx.in_shape = rowmap, b is not None, a.shape
        ctx.save_for_backward(bwd)
        return _gather_rows_raw(a, b, fwd, rowmap.rows_src, rowmap.rows_dst)

    @staticmethod
    def backward(ctx, g):
        (bwd,) = ctx.saved_tensors
        rm = ctx.rowmap
        d = _gather_rows_raw(g.contiguous(), None, bwd, rm.rows_dst, rm.rows_src).view(ctx.in_shape)
        return d, (d if ctx.has_b else None), None


def gather_rows(a: torch.Tensor, b: Optional[torch.Tensor], rowmap) -> torch.Tensor:
    """out[B, rows_dst, C] with out[:, j] = a[:, map[j]] (+ b[:, map[j]]) or 0 where map[j] < 0.  a (and b) hold
    rowmap.rows_src rows of C contiguous elements per sample (any leading shape)."""
    _require_cuda(a, b)
    if a.numel() != a.shape[0] * rowmap.rows_src * a.shape[-1] or (b is not None and (b.shape != a.shape or b.dtype != a.dtype)):
        raise ValueError(f"gather_rows: source {tuple(a.shape)} does not hold {rowmap.rows_src} rows per sample")
    return _GatherRows.apply(a, b, rowmap)


# ------------------------------------------------------------------------------------------------
# (b)/(c) fused prompted window attention
# ------------------------------------------------------------------------------------------------
IMPL_AUTO, IMPL_F32, IMPL_TC = 0, 1, 2
# per-head work counters of the tcgen05 forward (pwa_attn_shape.work): True = windows are handed to the CTAs dynamically,
# False = static round-robin.  Both distributions are parity-tested (tests/test_gpu_multiwindow.py).
DYNAMIC_WORK = True


_SEL_TABLES = {}


def sel_table_for(ids: Optional[torch.Tensor]):
    """Device copy of pwa_attn_sel_table(ids) (PRMT selectors of the shift mask, [P,28,N/4] int32), cached per ids tensor:
    region ids are cached per geometry (Geometry.region_ids), so this is built once per geometry and device.  Returns None
    when it cannot be built right now (first use inside a CUDA-graph capture): the kernel then builds its own."""
    if ids is None or ids.dim() != 2 or ids.shape[1] % 4 != 0:
        return None
    key = (ids.data_ptr(), tuple(ids.shape), ids.device)
    hit = _SEL_TABLES.get(key)
    if hit is not None and hit[0] is ids:
        return hit[1]
    if torch.cuda.is_current_stream_capturing():
        return None
    import numpy as np
    host = np.ascontiguousarray(ids.detach().cpu().numpy())
    P, N = host.shape
    tab = np.empty((P, 28, N // 4), dtype=np.uint32)
    _lib.check(_lib.lib.pwa_attn_sel_table(host.ctypes.data, P, N, tab.ctypes.data), "pwa_attn_sel_table")
    dev = torch.from_numpy(tab.view(np.int32)).to(ids.device)
    _SEL_TABLES[key] = (ids, dev)          # (holding `ids` keeps its data_ptr from being recycled under the key)
    return dev


def _shape_struct(B, P, Cc, heads, I, ws, scale, p_drop=0.0, seed=0, offset=0, ld_qkv=0, ld_p=0, seed_dev=None, work=None,
                  sel=None):
    s = _lib.PwaAttnShape()
    s.B, s.P, s.C, s.heads, s.I = B, P, Cc, heads, I
    s.ld_qkv, s.ld_p = ld_qkv, ld_p
    s.ws[0], s.ws[1], s.ws[2] = ws
    s.scale, s.p_drop, s.seed, s.offset = float(scale), float(p_drop), int(seed), int(offset)
    s.seed_dev = None if seed_dev is None else seed_dev.data_ptr()
    s.work = None if work is None else work.data_ptr()      # forward only: per-head window counters
    s.sel_table = None if sel is None else sel.data_ptr()   # precomputed shift-mask selectors (tcgen05 kernels)
    return s


def _check_attn_side_inputs(B, P, N, Cc, dtype, kp, vp, kp_width, th, tw, td, tok, ids, heads, ws):
    """The kernels index these tensors with raw pointers: every shape / dtype the reference would reject (at its
    torch.cat / broadcast) is rejected here, before a launch could read out of bounds."""
    ws = tuple(int(w) for w in ws)
    if len(ws) != 3 or ws[0] * ws[1] * ws[2] != N:
        raise ValueError(f"window {ws} does not hold N = {N} tokens")
    for name, t, w in (("th", th, ws[0]), ("tw", tw, ws[1]), ("td", td, ws[2])):
        if tuple(t.shape) != (heads, w, w):
            raise ValueError(f"bias table {name} must be [{heads},{w},{w}], got {tuple(t.shape)}")
    I = 0
    if kp is not None:
        if kp.dim() != 3 or kp.shape[0] != B or kp.shape[2] != kp_width * Cc or kp.dtype != dtype:
            raise ValueError(f"prompt keys/values must be [{B}, I, {kp_width * Cc}] {dtype}, got {tuple(kp.shape)} {kp.dtype} "
                             "(one row set per sample)")
        I = kp.shape[1]
        if vp is not None and (vp.shape != kp.shape or vp.dtype != dtype):
            raise ValueError(f"vp {tuple(vp.shape)} does not match kp {tuple(kp.shape)}")
        if kp_width == 1 and vp is None:
            raise ValueError("vp missing")
        if tok is None or tuple(tok.shape) != (heads, I):
            raise ValueError(f"prompt-token bias must be [{heads},{I}]")
    elif vp is not None:
        raise ValueError("vp given without kp")
    if ids is not None and (ids.dtype != torch.uint8 or tuple(ids.shape) != (P, N)):
        raise ValueError(f"region ids must be uint8 [{P},{N}], got {ids.dtype} {tuple(ids.shape)}")


class _WindowAttention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, kp, vp, th, tw, td, tok, ids, heads, ws, scale, impl, p_drop=0.0, seed=None):
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        B, P, N, Cc = q.shape
        I = 0 if kp is None else kp.shape[1]
        if kp is not None:
            kp, vp, tok = kp.contiguous(), vp.contiguous(), tok.contiguous().float()
        th, tw, td = th.contiguous().float(), tw.contiguous().float(), td.contiguous().float()
        out = torch.empty_like(q)
        lse = torch.empty((B, P, heads, N), dtype=torch.float32, device=q.device)
        work = torch.empty(heads, dtype=torch.int32, device=q.device) if DYNAMIC_WORK else None
        s = _shape_struct(B, P, Cc, heads, I, ws, scale, p_drop=p_drop, seed_dev=seed, work=work,
                          sel=sel_table_for(ids) if q.dtype in _LOWP and impl != IMPL_F32 else None)
        with torch.cuda.device(q.device), _timed("attn_fwd", 1, 4.0 * B * P * N * (N + I) * Cc, q):
            rc = _lib.lib.pwa_attn_fwd(_ptr(q), _ptr(k), _ptr(v), _ptr(kp), _ptr(vp), _ptr(th), _ptr(tw), _ptr(td),
                                       _ptr(tok), _ptr(ids), _ptr(out), _ptr(lse), C.byref(s), _dtype_code(q), impl,
                                       _stream(q))
        _lib.check(rc, "pwa_attn_fwd")
        ctx.save_for_backward(q, k, v, kp, vp, th, tw, td, tok, ids, out, lse, seed)
        ctx.meta = (heads, tuple(ws), scale, impl, I, p_drop)
        return out

    @staticmethod
    def backward(ctx, dout):
        q, k, v, kp, vp, th, tw, td, tok, ids, out, lse, seed = ctx.saved_tensors
        heads, ws, scale, impl, I, p_drop = ctx.meta
        B, P, N, Cc = q.shape
        dout = dout.contiguous()
        dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        f32 = dict(dtype=torch.float32, device=q.device)
        dkp = torch.empty((B, I, Cc), **f32) if I else None
        dvp = torch.empty((B, I, Cc), **f32) if I else None
        dth, dtw, dtd = torch.empty_like(th), torch.empty_like(tw), torch.empty_like(td)
        dtok = torch.empty_like(tok) if I else None
        delta = torch.empty_like(lse)
        s = _shape_struct(B, P, Cc, heads, I, ws, scale, p_drop=p_drop, seed_dev=seed,
                          sel=sel_table_for(ids) if q.dtype in _LOWP and impl != IMPL_F32 else None)
        with torch.cuda.device(q.device), _timed("attn_bwd", 2, 8.0 * B * P * N * (N + I) * Cc, q):
            rc = _lib.lib.pwa_attn_bwd(_ptr(q), _ptr(k), _ptr(v), _ptr(kp), _ptr(vp), _ptr(th), _ptr(tw), _ptr(td),
                                       _ptr(tok), _ptr(ids), _ptr(out), _ptr(lse), _ptr(dout), _ptr(dq), _ptr(dk),
                                       _ptr(dv), _ptr(dkp), _ptr(dvp), _ptr(dth), _ptr(dtw), _ptr(dtd), _ptr(dtok),
                                       _ptr(delta), C.byref(s), _dtype_code(q), impl, _stream(q))
        _lib.check(rc, "pwa_attn_bwd")
        if I:
            dkp, dvp = dkp.to(q.dtype), dvp.to(q.dtype)
        return dq, dk, dv, dkp, dvp, dth, dtw, dtd, dtok, None, None, None, None, None, None, None


# ------------------------------------------------------------------------------------------------
# dense-argument attention (csrc/attn_dense.cu): WindowAttention.forward(q, k, v, pos_bias, mask) as the reference takes it
# ------------------------------------------------------------------------------------------------
def _dense_operand(t, shape5, name):
    """A bias / mask tensor broadcastable to [b,p,h,nq,nk] -> (fp32 tensor with a contiguous last axis, strides over
    (b,p,h,i) with 0 for broadcast axes, the 5-d shape it was materialised in)."""
    if t is None:
        return None, (0, 0, 0, 0), None
    if t.dim() > 5:
        raise ValueError(f"WindowAttention: {name} has {t.dim()} dimensions, at most 5 ([b,p,h,n_q,n_k]) expected")
    t5 = t.reshape((1,) * (5 - t.dim()) + tuple(t.shape))
    for have, want in zip(t5.shape, shape5):
        if have != 1 and have != want:
            raise ValueError(f"WindowAttention: {name} of shape {tuple(t.shape)} does not broadcast to {tuple(shape5)}")
    if t5.shape[-1] != shape5[-1]:
        t5 = t5.expand(*t5.shape[:-1], shape5[-1])
    t5 = t5.to(torch.float32).contiguous()
    strides = tuple(0 if t5.shape[i] == 1 else t5.stride(i) for i in range(4))
    return t5, strides, tuple(t5.shape)


class _DenseWindowAttention(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, k, v, bias, mask, heads, scale, p_drop, seed):
        b, p, nq, Cc = q.shape
        nk = k.shape[2]
        dh = Cc // heads
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        shape5 = (b, p, heads, nq, nk)
        bias5, bst, _ = _dense_operand(None if bias is None else bias.detach(), shape5, "pos_bias")
        mask5, mst, _ = _dense_operand(None if mask is None else mask.detach(), shape5, "mask")
        s = _lib.PwaDenseAttn()
        s.B, s.P, s.heads, s.dh, s.nq, s.nk = b, p, heads, dh, nq, nk
        s.ld_q = s.ld_k = s.ld_v = Cc
        for i in range(4):
            s.bias_stride[i], s.mask_stride[i] = bst[i], mst[i]
        s.scale, s.p_drop = float(scale), float(p_drop)
        s.seed_dev = None if seed is None else seed.data_ptr()
        out = torch.empty_like(q)
        lse = torch.empty((b, p, heads, nq), dtype=torch.float32, device=q.device)
        with torch.cuda.device(q.device):
            rc = _lib.lib.pwa_attn_dense_fwd(_ptr(q), _ptr(k), _ptr(v), _ptr(bias5), _ptr(mask5), _ptr(out), _ptr(lse), s,
                                             _dtype_code(q), _stream(q))
        _lib.check(rc, "pwa_attn_dense_fwd")
        ctx.save_for_backward(q, k, v, bias5, mask5, out, lse, seed)
        ctx.shape_struct = s
        ctx.bias_meta = None if bias is None else (tuple(bias.shape), bias.dtype)
        return out

    @staticmethod
    def backward(ctx, dout):
        q, k, v, bias5, mask5, out, lse, seed = ctx.saved_tensors
        s = ctx.shape_struct
        dout = dout.contiguous()
        dq, dk, dv = torch.empty_like(q), torch.empty_like(k), torch.empty_like(v)
        want_db = bias5 is not None and ctx.needs_input_grad[3]
        dbias = torch.zeros_like(bias5) if want_db else None
        delta = torch.empty_like(lse)
        with torch.cuda.device(q.device):
            rc = _lib.lib.pwa_attn_dense_bwd(_ptr(q), _ptr(k), _ptr(v), _ptr(bias5), _ptr(mask5), _ptr(out), _ptr(lse), _ptr(dout),
                                             _ptr(dq), _ptr(dk), _ptr(dv), _ptr(dbias), _ptr(delta), s, _dtype_code(q), _stream(q))
        _lib.check(rc, "pwa_attn_dense_bwd")
        db = None
        if want_db:
            shape, dt = ctx.bias_meta
            db = dbias.sum_to_size((1,) * (5 - len(shape)) + shape).reshape(shape).to(dt)
        return dq, dk, dv, db, None, None, None, None, None


def dense_window_attention(q, k, v, pos_bias, mask, heads: int, scale: float, p_drop: float = 0.0,
                           seed: Optional[torch.Tensor] = None) -> torch.Tensor:
    """softmax((scale q k^T + pos_bias) * mask) v per (sample, window, head), with the reference's literal argument form
    (window_attention.py:45-58): q [b,p,n_q,C], k / v [b,p,n_k,C] already projected, `pos_bias` / `mask` dense tensors (or
    None) that broadcast against [b,p,h,n_q,n_k].  Differentiable in q, k, v and pos_bias.  Returns [b,p,n_q,C]."""
    _require_cuda(q, k, v, pos_bias, mask, seed)
    if q.dim() != 4 or k.shape != v.shape or k.shape[:2] != q.shape[:2] or k.shape[-1] != q.shape[-1]:
        raise ValueError(f"WindowAttention: q {tuple(q.shape)}, k {tuple(k.shape)}, v {tuple(v.shape)} are not [b,p,n,C] tensors of one window set")
    if q.shape[-1] % heads != 0:
        raise ValueError('WindowAttention: The dimension is not compatible with the number of heads!')
    if not (q.dtype == k.dtype == v.dtype):
        raise TypeError("WindowAttention: q, k, v must share a dtype")
    if p_drop > 0 and seed is None:
        seed = new_dropout_seed(q.device)
    return _DenseWindowAttention.apply(q, k, v, pos_bias, mask, int(heads), float(scale), float(p_drop), seed if p_drop > 0 else None)


def prompted_window_attention(q, k, v, kp, vp, th, tw, td, tok, ids, heads: int, ws: Sequence[int], scale: float,
                              impl: int = IMPL_AUTO, p_drop: float = 0.0, seed: Optional[torch.Tensor] = None) -> torch.Tensor:
    """q,k,v [B,P,N,C]; kp,vp [B,I,C] or None; th/tw/td [h,w,w] + tok [h,I] fp32 bias tables;
    ids uint8 [P,N] or None.  Returns [B,P,N,C].  See include/pwa.h: pwa_attn_fwd."""
    _require_cuda(q, k, v, kp, vp, th, tw, td, tok, ids)
    if q.shape[-1] % heads != 0:
        raise ValueError('WindowAttention: The dimension is not compatible with the number of heads!')
    if q.dim() != 4 or k.shape != q.shape or v.shape != q.shape or k.dtype != q.dtype or v.dtype != q.dtype:
        raise ValueError(f"prompted_window_attention: q, k, v must be equal-shaped [B,P,N,C], got {tuple(q.shape)}, "
                         f"{tuple(k.shape)}, {tuple(v.shape)}")
    _check_attn_side_inputs(q.shape[0], q.shape[1], q.shape[2], q.shape[3], q.dtype, kp, vp, 1, th, tw, td, tok, ids, heads, ws)
    if p_drop > 0 and seed is None:
        seed = new_dropout_seed(q.device)
    return _WindowAttention.apply(q, k, v, kp, vp, th, tw, td, tok, ids, heads, tuple(ws), scale, impl, float(p_drop), seed)


# ------------------------------------------------------------------------------------------------
# LayerNorm over channels (+ fused residual add)
# ------------------------------------------------------------------------------------------------
class _AddLayerNorm(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, res, gamma, beta, eps, bias_of_x=None, bias_of_res=None):
        x = x.contiguous()
        Cc = x.shape[-1]
        rows = x.numel() // Cc
        y = torch.empty_like(x)
        mean = torch.empty(rows, dtype=torch.float32, device=x.device)
        rstd = torch.empty(rows, dtype=torch.float32, device=x.device)
        g32, b32 = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        s = None
        if res is not None:
            res = res.contiguous()
            s = torch.empty_like(x)
        nbytes = (2 if res is None else 4) * x.numel() * x.element_size()
        with torch.cuda.device(x.device), _timed("ln_fwd", 1, float(nbytes), x):
            rc = _lib.lib.pwa_ln_fwd(_ptr(x), _ptr(res), _ptr(g32), _ptr(b32), _ptr(s), _ptr(y), _ptr(mean), _ptr(rstd),
                                     rows, Cc, float(eps), _dtype_code(x), _stream(x))
        _lib.check(rc, "pwa_ln_fwd")
        normed = x if res is None else s
        ctx.save_for_backward(normed, g32, mean, rstd)
        ctx.has_res = res is not None
        ctx.param_dtypes = (gamma.dtype, beta.dtype)
        # bias parameters whose gradients are column sums this backward produces anyway (see include/pwa.h: pwa_ln_bwd2)
        ctx.bias_dtypes = (None if bias_of_x is None else bias_of_x.dtype, None if bias_of_res is None else bias_of_res.dtype)
        if res is None:
            return y
        return s, y

    @staticmethod
    def backward(ctx, *grads):
        normed, g32, mean, rstd = ctx.saved_tensors
        if ctx.has_res:
            ds, dy = grads
        else:
            (dy,), ds = grads, None
        Cc = normed.shape[-1]
        rows = normed.numel() // Cc
        dy = dy.contiguous() if dy is not None else torch.zeros_like(normed)
        ds = ds.contiguous() if ds is not None else None
        dx = torch.empty_like(normed)
        dg = torch.empty(Cc, dtype=torch.float32, device=normed.device)
        db = torch.empty(Cc, dtype=torch.float32, device=normed.device)
        bx_dt, br_dt = ctx.bias_dtypes
        dbx = torch.empty(Cc, dtype=torch.float32, device=normed.device) if bx_dt is not None else None
        dbr = torch.empty(Cc, dtype=torch.float32, device=normed.device) if br_dt is not None and ds is not None else None
        nbytes = (3 if ds is None else 4) * normed.numel() * normed.element_size()
        with torch.cuda.device(normed.device), _timed("ln_bwd", 1, float(nbytes), normed):
            rc = _lib.lib.pwa_ln_bwd2(_ptr(dy), _ptr(normed), _ptr(g32), _ptr(mean), _ptr(rstd), _ptr(ds), _ptr(dx), _ptr(dg),
                                      _ptr(db), _ptr(dbr), _ptr(dbx), rows, Cc, _dtype_code(normed), _stream(normed))
        _lib.check(rc, "pwa_ln_bwd")
        gd, bd = ctx.param_dtypes
        return (dx, (dx if ctx.has_res else None), dg.to(gd), db.to(bd), None,
                None if dbx is None else dbx.to(bx_dt), None if dbr is None else dbr.to(br_dt))


class _LayerNormPass(torch.autograd.Function):
    """(x_alias, y) with y = LayerNorm(x) and x_alias = x (same storage): for an x that is ALSO consumed as a residual
    further down (the block's shortcut, swin_block.py:215-222).  Routing that second use through x_alias lets the backward
    add its gradient inside the LayerNorm-backward kernel (`dres`) instead of a separate full-size add pass."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps):
        x = x.contiguous()
        Cc = x.shape[-1]
        rows = x.numel() // Cc
        y = torch.empty_like(x)
        mean = torch.empty(rows, dtype=torch.float32, device=x.device)
        rstd = torch.empty(rows, dtype=torch.float32, device=x.device)
        g32, b32 = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        with torch.cuda.device(x.device), _timed("ln_fwd", 1, 2.0 * x.numel() * x.element_size(), x):
            rc = _lib.lib.pwa_ln_fwd(_ptr(x), None, _ptr(g32), _ptr(b32), None, _ptr(y), _ptr(mean), _ptr(rstd), rows, Cc, float(eps),
                                     _dtype_code(x), _stream(x))
        _lib.check(rc, "pwa_ln_fwd")
        ctx.save_for_backward(x, g32, mean, rstd)
        ctx.param_dtypes = (gamma.dtype, beta.dtype)
        return x.view_as(x), y

    @staticmethod
    def backward(ctx, dalias, dy):
        x, g32, mean, rstd = ctx.saved_tensors
        Cc = x.shape[-1]
        rows = x.numel() // Cc
        if dy is None:
            return dalias, None, None, None
        dy = dy.contiguous()
        dalias = dalias.contiguous() if dalias is not None else None
        dx = torch.empty_like(x)
        dg = torch.empty(Cc, dtype=torch.float32, device=x.device)
        db = torch.empty(Cc, dtype=torch.float32, device=x.device)
        nbytes = (3 if dalias is None else 4) * x.numel() * x.element_size()
        with torch.cuda.device(x.device), _timed("ln_bwd", 1, float(nbytes), x):
            rc = _lib.lib.pwa_ln_bwd2(_ptr(dy), _ptr(x), _ptr(g32), _ptr(mean), _ptr(rstd), _ptr(dalias), _ptr(dx), _ptr(dg), _ptr(db),
                                      None, None, rows, Cc, _dtype_code(x), _stream(x))
        _lib.check(rc, "pwa_ln_bwd")
        gd, bd = ctx.param_dtypes
        return dx, dg.to(gd), db.to(bd), None


def layer_norm_with_passthrough(x, gamma, beta, eps: float = 1e-6):
    """(x_alias, LayerNorm(x)); use x_alias wherever x is needed again (see _LayerNormPass)."""
    _require_cuda(x, gamma, beta)
    return _LayerNormPass.apply(x, gamma, beta, eps)


def layer_norm(x, gamma, beta, eps: float = 1e-6):
    """LayerNorm over the last axis on the pwa kernel (C % 4 == 0, C <= 2048)."""
    _require_cuda(x, gamma, beta)
    return _AddLayerNorm.apply(x, None, gamma, beta, eps)


def add_layer_norm(x, res, gamma, beta, eps: float = 1e-6, bias_of_x=None, bias_of_res=None):
    """(s, y) with s = x + res and y = LayerNorm(s): the residual add of swin_block.py:222 fused into mlp_norm.
    bias_of_x / bias_of_res: optional Linear bias parameters whose gradients equal the column sums of d(x) and of
    d(s) respectively (x = Linear(..) + bias_of_x; s is only ever added to Linear(..) + bias_of_res downstream): the
    backward kernel produces them on the fly, and the Linears are then called with bias_grad=False."""
    _require_cuda(x, res, gamma, beta)
    return _AddLayerNorm.apply(x, res, gamma, beta, eps, bias_of_x, bias_of_res)


def layer_norm_supported(C: int) -> bool:
    return C % 4 == 0 and C <= 2048


# ------------------------------------------------------------------------------------------------
# relative-position bias tables
# ------------------------------------------------------------------------------------------------
class _BiasTables(torch.autograd.Function):
    @staticmethod
    def forward(ctx, enc_h, enc_w, enc_d, wc_h, wc_w, wc_d, enc_tok, w_tok, ws):
        ten = [t.detach().float().contiguous() for t in (enc_h, enc_w, enc_d, wc_h, wc_w, wc_d)]
        has_tok = enc_tok is not None
        tk = [t.detach().float().contiguous() for t in (enc_tok, w_tok)] if has_tok else [None, None]
        heads, E = ten[3].shape
        I = tk[0].shape[0] if has_tok else 0
        dev = ten[0].device
        f32 = dict(dtype=torch.float32, device=dev)
        th, tw, td = (torch.empty((heads, w, w), **f32) for w in ws)
        tok = torch.empty((heads, I), **f32) if has_tok else None
        a3 = C.c_int32 * 3
        cap = a3(*[(t.shape[0] + 1) // 2 for t in ten[:3]])
        wsa = a3(*ws)
        with torch.cuda.device(dev), _timed("bias_tables_fwd", 1, 0.0, ten[0]):
            rc = _lib.lib.pwa_bias_tables_fwd(*[_ptr(t) for t in ten], _ptr(tk[0]), _ptr(tk[1]), _ptr(th), _ptr(tw),
                                              _ptr(td), _ptr(tok), heads, E, wsa, cap, I, _stream(ten[0]))
        _lib.check(rc, "pwa_bias_tables_fwd")
        ctx.save_for_backward(*ten, *([tk[0], tk[1]] if has_tok else []))
        ctx.meta = (tuple(ws), has_tok, [t.dtype for t in (enc_h, enc_w, enc_d, wc_h, wc_w, wc_d)])
        if not has_tok:
            ctx.mark_non_differentiable()
            return th, tw, td
        return th, tw, td, tok

    @staticmethod
    def backward(ctx, *g):
        ws, has_tok, dts = ctx.meta
        saved = ctx.saved_tensors
        ten, tk = list(saved[:6]), (list(saved[6:8]) if has_tok else [None, None])
        heads, E = ten[3].shape
        I = tk[0].shape[0] if has_tok else 0
        grads = [None if x is None else x.contiguous().float() for x in g]
        shapes = [(heads, w, w) for w in ws]
        for i in range(3):
            if grads[i] is None:
                grads[i] = torch.zeros(shapes[i], dtype=torch.float32, device=ten[0].device)
        dtok = None
        if has_tok:
            dtok = grads[3] if grads[3] is not None else torch.zeros((heads, I), dtype=torch.float32, device=ten[0].device)
        outs = [torch.empty_like(t) for t in ten]
        dtk = [torch.empty_like(t) for t in tk] if has_tok else [None, None]
        a3 = C.c_int32 * 3
        cap = a3(*[(t.shape[0] + 1) // 2 for t in ten[:3]])
        with torch.cuda.device(ten[0].device), _timed("bias_tables_bwd", 1, 0.0, ten[0]):
            rc = _lib.lib.pwa_bias_tables_bwd(*[_ptr(t) for t in ten], _ptr(tk[0]), _ptr(tk[1]), _ptr(grads[0]),
                                              _ptr(grads[1]), _ptr(grads[2]), _ptr(dtok), *[_ptr(t) for t in outs],
                                              _ptr(dtk[0]), _ptr(dtk[1]), heads, E, a3(*ws), cap, I, _stream(ten[0]))
        _lib.check(rc, "pwa_bias_tables_bwd")
        outs = [o.to(d) for o, d in zip(outs, dts)]
        return (*outs, dtk[0], dtk[1], None)


def bias_tables(enc_h, enc_w, enc_d, wc_h, wc_w, wc_d, enc_tok, w_tok, ws):
    """Compact relative-position bias (th, tw, td, tok|None) on the pwa kernel; see include/pwa.h."""
    _require_cuda(enc_h, enc_w, enc_d, wc_h, wc_w, wc_d, enc_tok, w_tok)
    out = _BiasTables.apply(enc_h, enc_w, enc_d, wc_h, wc_w, wc_d, enc_tok, w_tok, tuple(int(w) for w in ws))
    return out if len(out) == 4 else (*out, None)


# ------------------------------------------------------------------------------------------------
# packed variant: q|k|v are the column blocks of one fused projection output
# ------------------------------------------------------------------------------------------------
class _WindowAttentionPacked(torch.autograd.Function):
    @staticmethod
    def forward(ctx, qkv, kvp, th, tw, td, tok, ids, heads, ws, scale, impl, p_drop=0.0, seed=None):
        qkv = qkv.contiguous()
        B, P, N, C3 = qkv.shape
        Cc = C3 // 3
        I = 0 if kvp is None else kvp.shape[1]
        es = qkv.element_size()
        if kvp is not None:
            kvp, tok = kvp.contiguous(), tok.contiguous().float()
        th, tw, td = th.contiguous().float(), tw.contiguous().float(), td.contiguous().float()
        out = torch.empty((B, P, N, Cc), dtype=qkv.dtype, device=qkv.device)
        lse = torch.empty((B, P, heads, N), dtype=torch.float32, device=qkv.device)
        work = torch.empty(heads, dtype=torch.int32, device=qkv.device) if DYNAMIC_WORK else None
        s = _shape_struct(B, P, Cc, heads, I, ws, scale, p_drop=p_drop, ld_qkv=C3, ld_p=2 * Cc, seed_dev=seed, work=work,
                          sel=sel_table_for(ids) if qkv.dtype in _LOWP and impl != IMPL_F32 else None)
        q0 = qkv.data_ptr()
        p0 = 0 if kvp is None else kvp.data_ptr()
        vpp = C.c_void_p
        with torch.cuda.device(qkv.device), _timed("attn_fwd", 1, 4.0 * B * P * N * (N + I) * Cc, qkv):
            rc = _lib.lib.pwa_attn_fwd(vpp(q0), vpp(q0 + Cc * es), vpp(q0 + 2 * Cc * es), vpp(p0), vpp(p0 + Cc * es if p0 else 0),
                                       _ptr(th), _ptr(tw), _ptr(td), _ptr(tok), _ptr(ids), _ptr(out), _ptr(lse), C.byref(s),
                                       _dtype_code(qkv), impl, _stream(qkv))
        _lib.check(rc, "pwa_attn_fwd")
        ctx.save_for_backward(qkv, kvp, th, tw, td, tok, ids, out, lse, seed)
        ctx.meta = (heads, tuple(ws), scale, impl, I, p_drop)
        return out

    @staticmethod
    def backward(ctx, dout):
        qkv, kvp, th, tw, td, tok, ids, out, lse, seed = ctx.saved_tensors
        heads, ws, scale, impl, I, p_drop = ctx.meta
        B, P, N, C3 = qkv.shape
        Cc = C3 // 3
        es = qkv.element_size()
        dout = dout.contiguous()
        dqkv = torch.empty_like(qkv)
        f32 = dict(dtype=torch.float32, device=qkv.device)
        dkvp32 = torch.empty((2, B, I, Cc), **f32) if I else None
        dth, dtw, dtd = torch.empty_like(th), torch.empty_like(tw), torch.empty_like(td)
        dtok = torch.empty_like(tok) if I else None
        delta = torch.empty_like(lse)
        s = _shape_struct(B, P, Cc, heads, I, ws, scale, p_drop=p_drop, ld_qkv=C3, ld_p=2 * Cc, seed_dev=seed,
                          sel=sel_table_for(ids) if qkv.dtype in _LOWP and impl != IMPL_F32 else None)
        q0, d0 = qkv.data_ptr(), dqkv.data_ptr()
        p0 = 0 if kvp is None else kvp.data_ptr()
        vpp = C.c_void_p
        with torch.cuda.device(qkv.device), _timed("attn_bwd", 2, 8.0 * B * P * N * (N + I) * Cc, qkv):
            rc = _lib.lib.pwa_attn_bwd(vpp(q0), vpp(q0 + Cc * es), vpp(q0 + 2 * Cc * es), vpp(p0), vpp(p0 + Cc * es if p0 else 0),
                                       _ptr(th), _ptr(tw), _ptr(td), _ptr(tok), _ptr(ids), _ptr(out), _ptr(lse), _ptr(dout),
                                       vpp(d0), vpp(d0 + Cc * es), vpp(d0 + 2 * Cc * es),
                                       _ptr(dkvp32[0] if I else None), _ptr(dkvp32[1] if I else None),
                                       _ptr(dth), _ptr(dtw), _ptr(dtd), _ptr(dtok), _ptr(delta), C.byref(s),
                                       _dtype_code(qkv), impl, _stream(qkv))
        _lib.check(rc, "pwa_attn_bwd")
        dkvp = None
        if I:
            dkvp = torch.cat([dkvp32[0], dkvp32[1]], dim=-1).to(qkv.dtype)          # [B,I,2C]
        return dqkv, dkvp, dth, dtw, dtd, dtok, None, None, None, None, None, None, None


def new_dropout_seed(device, words: int = 2) -> torch.Tensor:
    """32-bit seed words ON THE DEVICE (two per dropout site: forward and backward share them).  Drawn with a CUDA RNG op,
    so torch.manual_seed governs it and a captured CUDA graph gets fresh words on every replay."""
    return torch.randint(0, 2 ** 31 - 1, (words,), dtype=torch.int32, device=device)


class _SeededDropout(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, p_drop, seed, bias_of_x=None):
        # bias_of_x: the bias parameter of the Linear that produced x -- its gradient (column sums of dx) comes out of
        # the backward's masking pass (pwa_dropout_colsum); that Linear is then called with bias_grad=False
        x = x.contiguous()
        ctx.bias_dtype = None if bias_of_x is None else bias_of_x.dtype
        y = torch.empty_like(x)
        with torch.cuda.device(x.device), _timed("dropout", 1, 2.0 * x.numel() * x.element_size(), x):
            rc = _lib.lib.pwa_dropout(_ptr(x), _ptr(y), x.numel(), float(p_drop), _ptr(seed), _dtype_code(x), _stream(x))
        _lib.check(rc, "pwa_dropout")
        ctx.save_for_backward(seed)
        ctx.p_drop = float(p_drop)
        return y

    @staticmethod
    def backward(ctx, dy):
        (seed,) = ctx.saved_tensors
        dy = dy.contiguous()
        dx = torch.empty_like(dy)
        Cc = dy.shape[-1]
        db = None
        with torch.cuda.device(dy.device), _timed("dropout", 1, 2.0 * dy.numel() * dy.element_size(), dy):
            if ctx.bias_dtype is not None:
                db = torch.empty(Cc, dtype=torch.float32, device=dy.device)
                rc = _lib.lib.pwa_dropout_colsum(_ptr(dy), _ptr(dx), dy.numel() // Cc, Cc, ctx.p_drop, _ptr(seed), _ptr(db),
                                                 _dtype_code(dy), _stream(dy))
            else:
                rc = _lib.lib.pwa_dropout(_ptr(dy), _ptr(dx), dy.numel(), ctx.p_drop, _ptr(seed), _dtype_code(dy), _stream(dy))
        _lib.check(rc, "pwa_dropout")
        return dx, None, None, (None if db is None else db.to(ctx.bias_dtype))


def dropout_colsum_supported(C: int) -> bool:
    return C % 4 == 0 and C <= 1024


def seeded_dropout(x: torch.Tensor, p_drop: float, seed: Optional[torch.Tensor] = None, bias_of_x=None) -> torch.Tensor:
    """Dropout whose mask is a pure function of two device seed words and the element index (csrc/dropout.cu): the
    reference's nn.Dropout(proj_drop) (window_attention.py:60), safe under activation checkpointing inside a CUDA graph."""
    _require_cuda(x, seed)
    if p_drop <= 0.0:
        return x
    if seed is None:
        seed = new_dropout_seed(x.device)
    if seed.dtype != torch.int32 or seed.numel() < 2:
        raise ValueError("seeded_dropout: seed must be an int32 tensor with two words")
    return _SeededDropout.apply(x, float(p_drop), seed, bias_of_x)


def prompted_window_attention_packed(qkv, kvp, th, tw, td, tok, ids, heads: int, ws: Sequence[int], scale: float,
                                     impl: int = IMPL_AUTO, p_drop: float = 0.0, seed: Optional[torch.Tensor] = None) -> torch.Tensor:
    """qkv [B,P,N,3C] = [q | k | v] of one fused projection; kvp [B,I,2C] = [kp | vp] or None.
    p_drop > 0: attention dropout after the softmax (window_attention.py:57) with the mask derived from `seed`
    (int32 [2] on the device, default: new_dropout_seed)."""
    _require_cuda(qkv, kvp, th, tw, td, tok, ids)
    if qkv.shape[-1] % (3 * heads) != 0:
        raise ValueError('WindowAttention: The dimension is not compatible with the number of heads!')
    if qkv.dim() != 4:
        raise ValueError(f"prompted_window_attention_packed: qkv must be [B,P,N,3C], got {tuple(qkv.shape)}")
    _check_attn_side_inputs(qkv.shape[0], qkv.shape[1], qkv.shape[2], qkv.shape[3] // 3, qkv.dtype, kvp, None, 2, th, tw, td, tok,
                            ids, heads, ws)
    if p_drop > 0 and seed is None:
        seed = new_dropout_seed(qkv.device)
    return _WindowAttentionPacked.apply(qkv, kvp, th, tw, td, tok, ids, heads, tuple(ws), scale, impl, float(p_drop), seed)


# ------------------------------------------------------------------------------------------------
# Linear layers with fp32 master weights and bf16/fp32 activations (cuBLAS GEMMs; plain library calls)
# ------------------------------------------------------------------------------------------------
def _mm_f32(a, b):
    """a @ b accumulated and returned in fp32 (no bf16 round trip of weight gradients)."""
    if a.dtype == torch.float32:
        return torch.mm(a, b)
    try:
        return torch.mm(a, b, out_dtype=torch.float32)
    except (TypeError, RuntimeError):
        if a.dtype == torch.float16:          # an fp16 result would overflow / round the fp32 sums: upcast instead
            return torch.mm(a.float(), b.float())
        return torch.mm(a, b).float()


@functools.lru_cache(maxsize=None)
def _token_split(T):
    """Number of slices of the token axis for the batched weight-gradient GEMM: the divisor of T closest to 72 within
    [32, 160] (0 = none)."""
    cands = [d for d in range(32, 161) if T % d == 0]
    return min(cands, key=lambda d: abs(d - 72)) if cands else 0


def colsum_f32(part):
    """[S, ...] fp32 -> [...]: sum over the leading axis on the pwa kernel (csrc/reduce.cu)."""
    _require_cuda(part)
    part = part.contiguous()
    out = torch.empty(part.shape[1:], dtype=torch.float32, device=part.device)
    with torch.cuda.device(part.device), _timed("colsum", 1, 4.0 * part.numel(), part):
        rc = _lib.lib.pwa_colsum_f32(_ptr(part), _ptr(out), part.shape[0], out.numel(), _stream(part))
    _lib.check(rc, "pwa_colsum_f32")
    return out


def colsum_rows(x2):
    """[T, C] bf16 / fp16 / fp32 -> fp32 [C] column sums on the pwa kernel (csrc/reduce.cu: pwa_colsum_rows): the bias gradient of a
    Linear whose output gradient is x2 (window_attention.py:28-30).  torch's generic reduction for shapes outside the
    kernel's envelope (C not a multiple of 16 bytes, strided rows)."""
    _require_cuda(x2)
    T, Cc = x2.shape
    e = 16 // x2.element_size()
    if x2.dtype not in _DT or not x2.is_contiguous() or Cc % e or Cc // e > 512 or x2.data_ptr() % 16:
        return x2.sum(dim=0, dtype=torch.float32)
    if T == 0:
        return torch.zeros(Cc, dtype=torch.float32, device=x2.device)
    out = torch.empty(Cc, dtype=torch.float32, device=x2.device)
    with torch.cuda.device(x2.device), _timed("colsum_rows", 1, float(x2.numel() * x2.element_size()), x2):
        rc = _lib.lib.pwa_colsum_rows(_ptr(x2), _ptr(out), T, Cc, _dtype_code(x2), _stream(x2))
    _lib.check(rc, "pwa_colsum_rows")
    return out


def _wgrad(dy2, x2):
    """dW = dy^T x in fp32, dy [T,Cout], x [T,Cin].  For the block's Linears the output is tiny (48x48 .. 288x96) and
    T is 10^4..10^6 tokens: cuBLAS picks a split-K kernel that takes ~50 us at enc0 whatever Cout is (1.7-3.3 TB/s).
    Slicing the token axis into ~72 batches (torch.bmm, fp32 partials, one sum) streams the operands at 4-4.8 TB/s:
    51.7 -> 21.5 us for 48x48, 51.6 -> 35.4 us for 144x48, 16.7 -> 9.6 us for 96x96 (tools/wgrad_probe.py)."""
    T, co = dy2.shape
    ci = x2.shape[1]
    if dy2.dtype != torch.float32 and dy2.is_contiguous() and x2.is_contiguous():
        S = 0
        if T >= 16384 and co * ci <= 40960:
            S = _token_split(T)
        elif T >= 8192 and T % 8 == 0 and co * ci <= 131072:
            S = 8          # larger outputs (576x192, 192x384): few slices, 23.6 -> 16.2 us and 13.7 -> 9.4 us (tools/wgrad_probe2.py)
        if S:
            try:
                part = torch.bmm(dy2.view(S, T // S, co).transpose(1, 2), x2.view(S, T // S, ci), out_dtype=torch.float32)
            except (TypeError, RuntimeError):
                part = None
            if part is not None:
                return colsum_f32(part)
    return _mm_f32(dy2.t(), x2)


class _MultiLinear(torch.autograd.Function):
    """y = x @ cat(weights)^T (+ bias): several nn.Linear weights that share an input, as ONE GEMM."""

    @staticmethod
    def forward(ctx, x, bias, lowp, bias_grad, lowp_bias, *weights):
        # `lowp`: the same weights already concatenated and cast to x.dtype (one cat + one cast per block instead
        # of two kernels per Linear); the fp32 master weights stay the autograd inputs
        w = lowp if lowp is not None else (weights[0] if len(weights) == 1 else torch.cat(weights, dim=0)).detach().to(x.dtype)
        x2 = x.reshape(-1, x.shape[-1])
        if bias is not None:
            y = torch.addmm(lowp_bias if lowp_bias is not None else bias.detach().to(x.dtype), x2, w.t())
        else:
            y = torch.mm(x2, w.t())
        ctx.save_for_backward(x2, w)
        ctx.meta = (x.shape, [wt.shape[0] for wt in weights], [wt.dtype for wt in weights],
                    None if (bias is None or not bias_grad) else bias.dtype)
        return y.reshape(*x.shape[:-1], w.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x2, w = ctx.saved_tensors
        xshape, rows, wdts, bdt = ctx.meta
        dy2 = dy.reshape(-1, dy.shape[-1])
        dx = torch.mm(dy2, w).reshape(xshape) if ctx.needs_input_grad[0] else None
        db = colsum_rows(dy2).to(bdt) if bdt is not None and ctx.needs_input_grad[1] else None
        dws = [None] * len(rows)
        if any(ctx.needs_input_grad[5:]):
            dw = _wgrad(dy2, x2)
            o = 0
            for i, r in enumerate(rows):
                if ctx.needs_input_grad[5 + i]:
                    dws[i] = dw[o:o + r].to(wdts[i])
                o += r
        return (dx, db, None, None, None, *dws)


def multi_linear(x, bias, *weights, lowp=None, bias_grad=True, lowp_bias=None):
    """bias_grad=False: the bias gradient is produced elsewhere (add_layer_norm's fused column sums); lowp / lowp_bias:
    the weights (concatenated) and the bias already cast to x.dtype."""
    return _MultiLinear.apply(x, bias, lowp, bias_grad, lowp_bias, *weights)


# ------------------------------------------------------------------------------------------------
# token-domain GEMMs with fused LayerNorm / residual / dropout prologue (csrc/token_gemm.cu, tcgen05)
# ------------------------------------------------------------------------------------------------
def token_gemm_supported(C: int, Cout: int, dtype) -> bool:
    return dtype in _LOWP and bool(_lib.lib.pwa_token_gemm_supported(int(C), int(Cout)))


def token_gemm_profitable(C: int, rows: int) -> bool:
    """Where the fused kernel beats separate LayerNorm kernels + cuBLAS today (tools/bench_token_gemm.py): the narrow,
    token-rich stages (C = 48: 442 K tokens at 96^3).  At C >= 96 its tile phases run serially on one CTA per SM and the
    separate kernels win; those stages keep them."""
    return C <= 48 and rows >= 32768


def _token_gemm_raw(x2, res2, g32, b32, w, bias, want_sum, want_ln, want_stats, eps, p_drop, seed):
    rows, Cc = x2.shape
    Cout = w.shape[0]
    dev = x2.device
    y = torch.empty((rows, Cout), dtype=x2.dtype, device=dev)
    s = torch.empty_like(x2) if want_sum else None
    z = torch.empty_like(x2) if want_ln else None
    mean = torch.empty(rows, dtype=torch.float32, device=dev) if want_stats else None
    rstd = torch.empty(rows, dtype=torch.float32, device=dev) if want_stats else None
    nbytes = ((1 if res2 is None else 2) + (1 if want_sum else 0) + (1 if want_ln else 0)) * x2.numel() * 2 + y.numel() * 2
    with torch.cuda.device(dev), _timed("token_gemm", 1, float(nbytes), x2):
        rc = _lib.lib.pwa_token_gemm_fwd_dt(_ptr(x2), _ptr(res2), _ptr(g32), _ptr(b32), _ptr(w), _ptr(bias), _ptr(s), _ptr(z),
                                            _ptr(y), _ptr(mean), _ptr(rstd), rows, Cc, Cout, float(eps), float(p_drop), _ptr(seed),
                                            _dtype_code(x2), _stream(x2))
    _lib.check(rc, "pwa_token_gemm_fwd")
    return y, s, z, mean, rstd


def _ln_backward_raw(dy, x, g32, mean, rstd, dres, want_res_colsum, want_x_colsum):
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    dx = torch.empty_like(x)
    f32 = dict(dtype=torch.float32, device=x.device)
    dg, db = torch.empty(Cc, **f32), torch.empty(Cc, **f32)
    dbr = torch.empty(Cc, **f32) if want_res_colsum and dres is not None else None
    dbx = torch.empty(Cc, **f32) if want_x_colsum else None
    nbytes = (3 if dres is None else 4) * x.numel() * x.element_size()
    with torch.cuda.device(x.device), _timed("ln_bwd", 1, float(nbytes), x):
        rc = _lib.lib.pwa_ln_bwd2(_ptr(dy), _ptr(x), _ptr(g32), _ptr(mean), _ptr(rstd), _ptr(dres), _ptr(dx), _ptr(dg), _ptr(db),
                                  _ptr(dbr), _ptr(dbx), rows, Cc, _dtype_code(x), _stream(x))
    _lib.check(rc, "pwa_ln_bwd")
    return dx, dg, db, dbr, dbx


class _LnLinearPass(torch.autograd.Function):
    """(x_alias, y) with y = LayerNorm(x) @ cat(weights)^T in ONE kernel (attn_norm + to_q|to_k|to_v, swin_block.py:216 +
    window_attention.py:42-44); x_alias = x for the block's shortcut, whose gradient the LayerNorm backward sums in."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps, lowp_w, *weights):
        x = x.contiguous()
        Cc = x.shape[-1]
        g32, b32 = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        w = lowp_w if lowp_w is not None else (weights[0] if len(weights) == 1 else torch.cat(weights, dim=0)).detach().to(x.dtype)
        w = w.contiguous()
        y, _, tokens, mean, rstd = _token_gemm_raw(x.view(-1, Cc), None, g32, b32, w, None, False, True, True, eps, 0.0, None)
        ctx.save_for_backward(x, g32, mean, rstd, tokens, w)
        ctx.meta = ([wt.shape[0] for wt in weights], [wt.dtype for wt in weights], (gamma.dtype, beta.dtype))
        return x.view_as(x), y.view(*x.shape[:-1], w.shape[0])

    @staticmethod
    def backward(ctx, dalias, dy):
        x, g32, mean, rstd, tokens, w = ctx.saved_tensors
        rows_w, wdts, (gd, bd) = ctx.meta
        dy2 = dy.reshape(-1, dy.shape[-1])
        dtok = torch.mm(dy2, w)
        dws = [None] * len(rows_w)
        if any(ctx.needs_input_grad[5:]):
            dw = _wgrad(dy2.contiguous(), tokens)
            o = 0
            for i, r in enumerate(rows_w):
                if ctx.needs_input_grad[5 + i]:
                    dws[i] = dw[o:o + r].to(wdts[i])
                o += r
        dres = dalias.contiguous().view(-1, x.shape[-1]) if dalias is not None else None
        dx, dg, db, _, _ = _ln_backward_raw(dtok, x.view(-1, x.shape[-1]), g32, mean, rstd, dres, False, False)
        return (dx.view_as(x), dg.to(gd), db.to(bd), None, None, *dws)


def ln_linear_pass(x, gamma, beta, eps, lowp_w, *weights):
    _require_cuda(x, gamma, beta, lowp_w)
    return _LnLinearPass.apply(x, gamma, beta, eps, lowp_w, *weights)


class _DropAddLnLinear(torch.autograd.Function):
    """(s, m) with s = dropout(a) + res and m = LayerNorm(s) @ W^T + bias in ONE kernel: projection dropout, the residual add,
    mlp_norm and the single-Linear MLP of the block (window_attention.py:60, swin_block.py:222-227).  `bias_of_a` is the
    bias of the Linear that produced `a` (attn.proj.bias): its gradient is the column sum of d(a), a by-product of the
    backward passes here, as is the gradient of `bias` (column sum of the gradient that reaches s directly)."""

    @staticmethod
    def forward(ctx, a, res, gamma, beta, eps, lowp_w, lowp_b, p_drop, seed, weight, bias, bias_of_a):
        a, res = a.contiguous(), res.contiguous()
        Cc = a.shape[-1]
        g32, b32 = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        w = (lowp_w if lowp_w is not None else weight.detach().to(a.dtype)).contiguous()
        bb = (lowp_b if lowp_b is not None else bias.detach().to(a.dtype)).contiguous() if bias is not None else None
        m, s, z, mean, rstd = _token_gemm_raw(a.view(-1, Cc), res.view(-1, Cc), g32, b32, w, bb, True, True, True, eps, p_drop, seed)
        ctx.save_for_backward(s, g32, mean, rstd, z, w, seed)
        ctx.meta = (float(p_drop), weight.dtype, None if bias is None else bias.dtype, None if bias_of_a is None else bias_of_a.dtype,
                    (gamma.dtype, beta.dtype), a.shape)
        return s.view_as(a), m.view(*a.shape[:-1], w.shape[0])

    @staticmethod
    def backward(ctx, ds, dm):
        s, g32, mean, rstd, z, w, seed = ctx.saved_tensors
        p_drop, wdt, bdt, badt, (gd, bd), ashape = ctx.meta
        Cc = s.shape[-1]
        dm2 = dm.reshape(-1, dm.shape[-1]).contiguous()
        dz = torch.mm(dm2, w)
        dw = _wgrad(dm2, z).to(wdt) if ctx.needs_input_grad[9] else None
        ds2 = ds.contiguous().view(-1, Cc) if ds is not None else None
        want_b = bdt is not None and ctx.needs_input_grad[10] and ds2 is not None
        want_ba = badt is not None and ctx.needs_input_grad[11]
        dx, dg, db, dbr, dbx = _ln_backward_raw(dz, s, g32, mean, rstd, ds2, want_b, want_ba and p_drop == 0.0)
        dbias = dbr.to(bdt) if dbr is not None else (colsum_rows(dm2).to(bdt) if bdt is not None and ctx.needs_input_grad[10] else None)
        if p_drop > 0.0:
            da = torch.empty_like(dx)
            dba = None
            with torch.cuda.device(dx.device), _timed("dropout", 1, 2.0 * dx.numel() * dx.element_size(), dx):
                if want_ba and dropout_colsum_supported(Cc):
                    dba = torch.empty(Cc, dtype=torch.float32, device=dx.device)
                    rc = _lib.lib.pwa_dropout_colsum(_ptr(dx), _ptr(da), dx.numel() // Cc, Cc, p_drop, _ptr(seed), _ptr(dba),
                                                     _dtype_code(dx), _stream(dx))
                else:
                    rc = _lib.lib.pwa_dropout(_ptr(dx), _ptr(da), dx.numel(), p_drop, _ptr(seed), _dtype_code(dx), _stream(dx))
            _lib.check(rc, "pwa_dropout")
            if want_ba and dba is None:
                dba = colsum_rows(da)
        else:
            da, dba = dx, dbx
        return (da.view(ashape), dx.view(ashape), dg.to(gd), db.to(bd), None, None, None, None, None, dw, dbias,
                None if dba is None else dba.to(badt))


def drop_add_ln_linear(a, res, gamma, beta, eps, lowp_w, lowp_b, p_drop, seed, weight, bias, bias_of_a=None):
    _require_cuda(a, res, gamma, beta, weight, seed)
    if a.shape != res.shape or a.dtype != res.dtype:
        raise ValueError("drop_add_ln_linear: a and res must match")
    if p_drop > 0 and seed is None:
        seed = new_dropout_seed(a.device)
    return _DropAddLnLinear.apply(a, res, gamma, beta, eps, lowp_w, lowp_b, float(p_drop), seed, weight, bias, bias_of_a)
