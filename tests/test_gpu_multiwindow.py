"""Parity of the PERSISTENT tcgen05 attention kernels in the regime the benchmark runs them in.

Both kernels walk many (sample, window, head) units per CTA (forward: grid = min(B*P*h, 148*k) with per-head work
counters; backward: grid = min(B*P*h, 148), double-buffered next-window staging, S^T ring recycled across windows, dKaug
accumulated in TMEM over ALL windows of a CTA, prompt dK/dV kept in registers across the windows of a sample).  The cases
of tests/test_gpu_parity.py give every CTA exactly ONE window; here B*P*h is 448 ... 6912, i.e. BASELINE.json's stage
shapes (SURVEY.md §8: enc0/enc1/enc2/dec0/dec1 at 96^3, enc0 at 128^3), and the forward AND all nine gradients are
compared with the oracle (oracle/restatement.py: prompted_window_attention, float64).

Who executes the oracle: the 2.8 GB (fp32) logit tensor of one enc0 call makes the float64 restatement take minutes on
host cores, so torch executes the SAME restatement functions on the GPU (float64 torch ops; none of this repo's kernels),
window-chunked; one enc0 case per direction is ALSO run on the host CPU so that the device execution of the oracle is
itself pinned.  Tolerance: BASELINE.json north_star, bf16 rtol 2e-2 / fp32 rtol 1e-4 with atol = rtol * max|ref|."""
import numpy as np
import pytest
import torch

import pwa_b200
from pwa_b200 import functional as PF
from oracle import restatement as R
from tests.util import rel_linf

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL_F32 = 1e-4
RTOL_BF16 = 2e-2
RTOL_F16 = 5e-3            # tests/test_gpu_fp16.py (that module imports this one, so the value is restated here)
WS = (8, 8, 4)
N = 256
NAMES = ["q", "k", "v", "kp", "vp", "th", "tw", "td", "tok"]

# name -> (B, dims of the feature map, C, heads, I)       stage table of SURVEY.md §8
STAGES = {
    "enc0":      (4, (48, 48, 48), 48, 4, 64),        # P = 432, dh 12: 6912 window-heads
    "enc0_nop":  (2, (48, 48, 48), 48, 4, 0),         # no prompt tokens
    "enc0_i32":  (2, (48, 48, 48), 48, 4, 32),
    "enc1":      (4, (24, 24, 24), 96, 8, 64),        # P = 54: 1728
    "enc1_i128": (2, (24, 24, 24), 96, 8, 128),       # the widest prompt block the tcgen05 kernels take
    "enc1_i96":  (2, (24, 24, 24), 96, 8, 96),
    "enc2":      (4, (12, 12, 24), 192, 16, 64),      # padded to 16x16x28, P = 28: 1792
    "dec0":      (8, (12, 12, 24), 192, 4, 64),       # dh 48: 896
    "dec1":      (4, (24, 24, 24), 96, 4, 64),        # dh 24: 864
    "enc0_128":  (1, (64, 64, 64), 48, 4, 64),        # 128^3 patches: P = 1024
    "fs12_enc0": (4, (32, 32, 32), 12, 4, 64),        # cfg1 (feature_size 12): dh 3, P = 128: 2048
    "fs12_dec1": (8, (16, 16, 16), 24, 4, 64),        # dh 6, P = 16: 512
}


def _inputs(stage, shifted, seed, dtype):
    B, dims, C, heads, I = STAGES[stage]
    shift_cfg = (4, 4, 2) if shifted else (0, 0, 0)
    geom = pwa_b200.get_geometry(dims, WS, shift_cfg)
    pads, shift = R.pad_amounts(dims, WS), R.effective_shift(dims, WS, shift_cfg)
    ids = R.region_ids(dims, WS, shift, pads).astype(np.uint8) if geom.masked else None      # oracle's own ids
    if ids is not None:
        assert torch.equal(geom.region_ids(DEV).cpu(), torch.from_numpy(ids))                 # bit-exact (a4)
    P = geom.P
    gen = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=gen)
    q, k, v = r(B, P, N, C), r(B, P, N, C), r(B, P, N, C)
    kp, vp = (r(B, I, C), r(B, I, C)) if I else (None, None)
    th, tw, td = 0.5 * r(heads, 8, 8), 0.5 * r(heads, 8, 8), 0.5 * r(heads, 4, 4)
    tok = 0.5 * r(heads, I) if I else None
    go = r(B, P, N, C)
    io = [None if t is None else t.to(dtype) for t in (q, k, v, kp, vp)]
    return io + [th, tw, td, tok], ids, go.to(dtype), heads, P


def _oracle(ten, ids, go, heads, device, p_drop=0.0, seed_words=None, win_chunk=108):
    """float64 oracle, one sample and `win_chunk` windows at a time (per-window independence; the reductions over
    windows / samples happen in the autograd accumulation of the leaves)."""
    f64 = [None if t is None else t.to(device, torch.float64).requires_grad_(True) for t in ten]
    q, k, v, kp, vp, th, tw, td, tok = f64
    B, P, _, C = q.shape
    I = 0 if kp is None else kp.shape[1]
    scale = (C // heads) ** -0.5
    gof = go.to(device, torch.float64)
    out = torch.empty(q.shape, dtype=torch.float64, device=device)
    for b in range(B):
        for p0 in range(0, P, win_chunk):
            p1 = min(P, p0 + win_chunk)
            bias = R.dense_bias(th, tw, td, tok)
            drop = None
            if p_drop > 0:
                drop = R.dropout_keep_factor_torch(seed_words, b * P + p0, p1 - p0, heads, N, N + I, p_drop, device)[None]
            o = R.prompted_window_attention(q[b:b + 1, p0:p1], k[b:b + 1, p0:p1], v[b:b + 1, p0:p1],
                                            None if kp is None else kp[b:b + 1], None if vp is None else vp[b:b + 1],
                                            bias, None if ids is None else ids[p0:p1], scale, heads, drop=drop)
            (o * gof[b:b + 1, p0:p1]).sum().backward()
            out[b, p0:p1] = o.detach()[0]
    return out, [None if t is None else t.grad for t in f64]


def _run_kernel(ten, ids, go, heads, impl, p_drop=0.0, seed=None):
    dev = [None if t is None else t.to(DEV).requires_grad_(True) for t in ten]
    ids_d = None if ids is None else torch.from_numpy(ids).to(DEV)
    scale = (ten[0].shape[-1] // heads) ** -0.5
    out = PF.prompted_window_attention(*dev, ids_d, heads, WS, scale, impl, p_drop=p_drop, seed=seed)
    out.backward(go.to(DEV))
    return out.detach(), [None if t is None else t.grad for t in dev]


def _compare(got, ref, rtol, tag):
    out, grads = got
    ref_out, ref_grads = ref
    errs = {"out": rel_linf(out, ref_out)}
    for n, g, r in zip(NAMES, grads, ref_grads):
        if r is not None:
            errs["d" + n] = rel_linf(g, r)
    bad = {k: v for k, v in errs.items() if not v < rtol}
    print(tag, {k: f"{v:.2e}" for k, v in errs.items()})
    assert not bad, (tag, bad)


CASES = [(s, sh) for s in STAGES for sh in (False, True)]


@pytest.mark.parametrize("stage,shifted", CASES)
def test_tcgen05_persistent_fwd_bwd_vs_oracle(stage, shifted):
    """IMPL_TC forward + all nine gradients against the float64 oracle at BASELINE stage shapes (many windows per CTA)."""
    B, dims, C, heads, I = STAGES[stage]
    ten, ids, go, heads, P = _inputs(stage, shifted, seed=41, dtype=torch.bfloat16)
    s = PF._shape_struct(B, P, C, heads, I, WS, (C // heads) ** -0.5)
    assert pwa_b200._lib.lib.pwa_attn_tc_supported(s, pwa_b200._lib.PWA_BF16) == 1, "stage must run on the tcgen05 kernels"
    assert B * P * heads >= 3 * 148
    ref = _oracle(ten, ids, go, heads, DEV)
    _compare(_run_kernel(ten, ids, go, heads, PF.IMPL_TC), ref, RTOL_BF16, f"{stage} shifted={shifted}")


@pytest.mark.parametrize("shifted", [False, True])
def test_tcgen05_static_window_distribution(shifted):
    """pwa_attn_shape.work == NULL (static round-robin over CTAs) must give the same results as the per-head counters."""
    stage = "enc0"
    ten, ids, go, heads, P = _inputs(stage, shifted, seed=43, dtype=torch.bfloat16)
    ref = _oracle(ten, ids, go, heads, DEV)
    dyn = _run_kernel(ten, ids, go, heads, PF.IMPL_TC)
    PF.DYNAMIC_WORK = False
    try:
        sta = _run_kernel(ten, ids, go, heads, PF.IMPL_TC)
    finally:
        PF.DYNAMIC_WORK = True
    _compare(sta, ref, RTOL_BF16, f"static shifted={shifted}")
    assert torch.equal(sta[0], dyn[0])          # the forward is deterministic whichever CTA takes a window


@pytest.mark.parametrize("stage,shifted", [("enc0", True), ("enc0", False), ("enc1", True), ("enc2", True), ("dec0", True),
                                           ("dec1", False), ("enc0_nop", True)])
def test_tcgen05_persistent_dropout_vs_oracle(stage, shifted):
    """attn_drop = 0.1 (the reference's example config) in the persistent regime: same hash mask as the oracle restates."""
    B, dims, C, heads, I = STAGES[stage]
    ten, ids, go, heads, P = _inputs(stage, shifted, seed=47, dtype=torch.bfloat16)
    words = [20261018, 777777]
    seed = torch.tensor(words, dtype=torch.int32, device=DEV)
    ref = _oracle(ten, ids, go, heads, DEV, p_drop=0.1, seed_words=words)
    _compare(_run_kernel(ten, ids, go, heads, PF.IMPL_TC, p_drop=0.1, seed=seed), ref, RTOL_BF16,
             f"dropout {stage} shifted={shifted}")


@pytest.mark.parametrize("shifted", [False, True])
def test_oracle_on_host_cpu_pins_device_execution(shifted):
    """One enc0 case (B = 1, 1728 window-heads) with the oracle executed on the HOST CPU in float64: the kernel must pass
    against it, and the GPU-executed oracle must agree with it to float64 round-off."""
    B, dims, C, heads, I = STAGES["enc0"]
    ten, ids, go, heads, P = _inputs("enc0", shifted, seed=53, dtype=torch.bfloat16)
    ten = [None if t is None else (t[:1] if i < 5 else t) for i, t in enumerate(ten)]
    go = go[:1]
    ref_cpu = _oracle(ten, ids, go, heads, "cpu")
    ref_dev = _oracle(ten, ids, go, heads, DEV)
    assert rel_linf(ref_dev[0], ref_cpu[0]) < 1e-12
    for a, b in zip(ref_dev[1], ref_cpu[1]):
        assert rel_linf(a, b) < 1e-11
    _compare(_run_kernel(ten, ids, go, heads, PF.IMPL_TC), ref_cpu, RTOL_BF16, f"cpu-oracle shifted={shifted}")


@pytest.mark.parametrize("stage,shifted", [("enc0_i32", True), ("enc1", False), ("dec0", True)])
def test_f32_kernels_at_stage_shapes_vs_oracle(stage, shifted):
    """The fp32-math kernels (the reference's own arithmetic, rtol 1e-4) at stage shapes."""
    B, dims, C, heads, I = STAGES[stage]
    ten, ids, go, heads, P = _inputs(stage, shifted, seed=59, dtype=torch.float32)
    ref = _oracle(ten, ids, go, heads, DEV)
    _compare(_run_kernel(ten, ids, go, heads, PF.IMPL_F32), ref, RTOL_F32, f"f32 {stage} shifted={shifted}")


def _block_oracle(blk, x, p, go, heads, shift_cfg):
    sd = {k: v.detach().to(DEV, torch.float64).requires_grad_(True) for k, v in blk.state_dict().items()
          if v.is_floating_point()}
    x64 = x.to(DEV, torch.float64).requires_grad_(True)
    p64 = p.to(DEV, torch.float64).requires_grad_(True)
    y = R.block_forward(sd, x64, p64, WS, shift_cfg, heads)
    (y * go.to(DEV, torch.float64)).sum().backward()
    return y.detach(), x64.grad, p64.grad, {k: v.grad for k, v in sd.items()}


@pytest.mark.parametrize("stage,shifted,dtype,rtol", [
    ("enc0", True, torch.bfloat16, RTOL_BF16), ("enc0", False, torch.bfloat16, RTOL_BF16),
    ("enc2", True, torch.bfloat16, RTOL_BF16), ("dec0", True, torch.bfloat16, RTOL_BF16),
    ("enc1", True, torch.float32, RTOL_F32), ("enc0", True, torch.float32, RTOL_F32),
    ("enc0", True, torch.float16, RTOL_F16), ("enc2", True, torch.float16, RTOL_F16)])
def test_block_full_size_vs_oracle(stage, shifted, dtype, rtol):
    """Whole SwinTransformerBlock (partition, LayerNorms, projections, attention, reverse; all 21 gradient tensors) at a
    BASELINE stage shape against R.block_forward in float64."""
    B, dims, C, heads, I = STAGES[stage]
    B = min(B, 2)
    shift_cfg = (4, 4, 2) if shifted else (0, 0, 0)
    torch.manual_seed(61)
    blk = pwa_b200.SwinTransformerBlock(hidden_channels=C, window_size=WS, pos_bias_embed_dim=64, num_heads=heads,
                                        max_prompts=1, tokens_per_prompt=I, shift_size=shift_cfg).to(DEV)
    with torch.no_grad():
        for n, prm in blk.named_parameters():
            if n.startswith("pe."):
                prm.mul_(3.0)
            elif n.endswith("norm.weight"):
                prm.add_(0.2 * torch.randn_like(prm))
            elif n.endswith("bias"):
                prm.add_(0.1 * torch.randn_like(prm))
    x = torch.randn(B, C, *dims, device=DEV).to(dtype)
    p = (0.5 * torch.randn(B, I, C, device=DEV)).to(dtype)
    go = torch.randn(B, C, *dims, device=DEV).to(dtype)
    ref_y, ref_dx, ref_dp, ref_g = _block_oracle(blk, x, p, go, heads, shift_cfg)
    xd, pd = x.clone().requires_grad_(True), p.clone().requires_grad_(True)
    y = blk(xd, pd)
    y.backward(go)
    errs = {"out": rel_linf(y, ref_y), "dx": rel_linf(xd.grad, ref_dx), "dp": rel_linf(pd.grad, ref_dp)}
    for n, prm in blk.named_parameters():
        errs[n] = rel_linf(prm.grad if prm.grad is not None else torch.zeros_like(prm), ref_g[n])
    print(stage, shifted, dtype, {k: f"{v:.1e}" for k, v in errs.items()})
    bad = {k: v for k, v in errs.items() if not v < rtol}
    assert not bad, bad
