"""float16 compute path: fp16 tensors and torch.autocast(float16) on the tcgen05 kernels (and the fp32-math kernels outside
their envelope), with GradScaler.

Tolerance: rtol 5e-3 (normalised L-inf, atol = rtol * max|ref|) against the float64 oracle fed the fp16-rounded inputs.
Where it comes from: the bf16 bound of 2e-2 scaled by fp16's finer rounding (unit roundoff 2^-11 against bf16's 2^-8: 8x),
2.5e-3, with 2x headroom for the terms that do not shrink with the storage type (fp32 ex2.approx, fp32 accumulation
order).  The accuracy claim of the path is checked separately: on the same inputs the worst fp16 error over the output and
the nine gradients is at most half the worst bf16 error."""
import types

import numpy as np
import pytest
import torch

import pwa_b200
from pwa_b200 import functional as PF
from pwa_b200 import _lib
from oracle import restatement as R
from tests.util import golden_names, load_block_case, load_npz, rel_linf
from tests.test_gpu_multiwindow import STAGES, WS, _compare, _inputs, _oracle, _run_kernel, NAMES
from tests.test_gpu_parity import ATTN_CASES, TC_CASES, _attn_inputs, _oracle_attn

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL_F16 = 5e-3
H = torch.float16


def _errs(got, ref):
    out, grads = got
    e = {"out": rel_linf(out, ref[0])}
    for n, g, r in zip(NAMES, grads, ref[1]):
        if r is not None:
            e["d" + n] = rel_linf(g, r)
    return e


# ---- 1. data movement is exact ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("force", [(False, False, False), (True, False, False), (False, True, False), (False, False, True)])
@pytest.mark.parametrize("dims,shift", [((16, 16, 8), (4, 4, 2)), ((12, 20, 6), (4, 4, 2)), ((16, 16, 8), (0, 0, 0))])
def test_fp16_partition_reverse_exact(dims, shift, force):
    g = pwa_b200.get_geometry(dims, WS, shift)
    B, C = 2, 24
    x = torch.randn(B, C, *dims, device=DEV).to(H)
    tok = PF._partition_raw(x, g, 0, *force)
    idx = torch.from_numpy(g.index_map_host(0).astype(np.int64)).to(DEV).reshape(-1)
    flat = torch.cat([x.reshape(B, C, -1), x.new_zeros(B, C, 1)], dim=2)
    assert torch.equal(tok, flat[:, :, idx].reshape(B, C, g.P, g.N).permute(0, 2, 3, 1))
    # reverse_add: (a + b) in fp32, rounded once to fp16
    a, b = torch.randn(B, g.P, g.N, C, device=DEV).to(H), torch.randn(B, g.P, g.N, C, device=DEV).to(H)
    ref = PF.reverse_tokens((a.float() + b.float()).half(), g)
    got = PF.reverse_add_tokens(a, b, g)
    assert got.dtype == H and torch.equal(got, ref)


def test_fp16_gather_rows_exact():
    B, rows, C = 3, 1000, 40
    a, b = torch.randn(B, rows, C, device=DEV).to(H), torch.randn(B, rows, C, device=DEV).to(H)
    perm = torch.randperm(rows, device=DEV)
    m = torch.where(torch.rand(rows, device=DEV) < 0.1, torch.full_like(perm, -1), perm).to(torch.int32)
    for bb, ref_src in ((None, a), (b, (a.float() + b.float()).half())):
        out = PF._gather_rows_raw(a, bb, m, rows, rows)
        ref = torch.where((m >= 0)[None, :, None], ref_src[:, m.clamp(min=0).long()], torch.zeros((), dtype=H, device=DEV))
        assert torch.equal(out, ref)
    # odd channel count: 2-byte vectors
    a3, b3 = a[..., :3].contiguous(), b[..., :3].contiguous()
    out = PF._gather_rows_raw(a3, b3, m, rows, rows)
    ref = torch.where((m >= 0)[None, :, None], (a3.float() + b3.float()).half()[:, m.clamp(min=0).long()],
                      torch.zeros((), dtype=H, device=DEV))
    assert torch.equal(out, ref)


# ---- 2. attention vs the float64 oracle at the stage shapes --------------------------------------------------------------
@pytest.mark.parametrize("stage,shifted", [(s, sh) for s in STAGES for sh in (False, True)])
def test_fp16_tcgen05_stages_vs_oracle(stage, shifted):
    """fp16 tcgen05 forward + nine gradients within 5e-3, and at most half the worst bf16 error on the same inputs."""
    B, dims, C, heads, I = STAGES[stage]
    ten16, ids, go16, heads, P = _inputs(stage, shifted, seed=41, dtype=H)
    s = PF._shape_struct(B, P, C, heads, I, WS, (C // heads) ** -0.5)
    assert _lib.lib.pwa_attn_tc_supported(s, _lib.PWA_F16) == 1
    e16 = _errs(_run_kernel(ten16, ids, go16, heads, PF.IMPL_TC), _oracle(ten16, ids, go16, heads, DEV))
    ten_b, ids, go_b, heads, P = _inputs(stage, shifted, seed=41, dtype=torch.bfloat16)
    eb = _errs(_run_kernel(ten_b, ids, go_b, heads, PF.IMPL_TC), _oracle(ten_b, ids, go_b, heads, DEV))
    print(stage, shifted, "fp16", max(e16.values()), "bf16", max(eb.values()))
    bad = {k: v for k, v in e16.items() if not v < RTOL_F16}
    assert not bad, bad
    assert max(e16.values()) <= 0.5 * max(eb.values())


# ---- 3. loose stabiliser -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("masked", [False, True])
def test_fp16_loose_norm_bound(masked):
    """One key ~5x longer than the others and orthogonal to every query: the norm bound |q| max|k| sits ~45 binades
    above the true row maximum -- below the bf16 sweep threshold (80), far outside fp16's normal range.  Without the fp16
    stabiliser rule the probabilities flush to zero (O = 0/0)."""
    B, P, ws, C, heads, I = 1, 2, (8, 8, 4), 48, 4, 64
    ten, ids, go = _attn_inputs(B, P, ws, C, heads, I, masked, seed=13)
    dh = C // heads
    q, k = ten[0], ten[1]
    for h in range(heads):                     # query and key slices of each head: key 7 along a direction no query has
        sl = slice(h * dh, (h + 1) * dh)
        q[..., sl.start] = 0.0
        k[:, :, 7, sl] = 0.0
        k[:, :, 7, sl.start] = 16.0
    scale = dh ** -0.5
    ten_r = [None if t is None else (t.to(H).double() if i < 5 else t.float().double()) for i, t in enumerate(ten)]
    ref_out, ref_grads = _oracle_attn(ten_r, ids, go.to(H).double(), heads, ws, scale)
    dev = [None if t is None else (t.to(DEV, H) if i < 5 else t.to(DEV, torch.float32)).requires_grad_(True)
           for i, t in enumerate(ten)]
    out = PF.prompted_window_attention(*dev, None if ids is None else ids.to(DEV), heads, ws, scale, PF.IMPL_TC)
    assert torch.isfinite(out.float()).all()
    assert rel_linf(out, ref_out) < RTOL_F16
    out.backward(go.to(DEV, H))
    for n, t, g in zip(NAMES, dev, ref_grads):
        if t is not None:
            assert torch.isfinite(t.grad.float()).all(), n
            assert rel_linf(t.grad, g) < RTOL_F16, n


@pytest.mark.parametrize("case", [(1, 2, (8, 8, 4), 48, 4, 64, True), (1, 2, (8, 8, 4), 48, 4, 64, False),
                                  (1, 1, (8, 8, 4), 96, 4, 32, True)])
def test_fp16_large_logits_exact_max_path(case):
    B, P, ws, C, heads, I, masked = case
    ten, ids, go = _attn_inputs(B, P, ws, C, heads, I, masked, seed=11, qk_gain=5.0)
    scale = (C // heads) ** -0.5
    ten_r = [None if t is None else (t.to(H).double() if i < 5 else t.float().double()) for i, t in enumerate(ten)]
    ref_out, _ = _oracle_attn(ten_r, ids, go.to(H).double(), heads, ws, scale)
    dev = [None if t is None else (t.to(DEV, H) if i < 5 else t.to(DEV, torch.float32)) for i, t in enumerate(ten)]
    out = PF.prompted_window_attention(*dev, None if ids is None else ids.to(DEV), heads, ws, scale, PF.IMPL_TC)
    assert torch.isfinite(out.float()).all()
    assert rel_linf(out, ref_out) < RTOL_F16


# ---- 4. dropout ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("stage,shifted", [("enc0", True), ("enc1", False), ("dec0", True), ("enc0_nop", True)])
def test_fp16_attention_dropout_vs_oracle(stage, shifted):
    ten, ids, go, heads, P = _inputs(stage, shifted, seed=47, dtype=H)
    words = [20261018, 777777]
    seed = torch.tensor(words, dtype=torch.int32, device=DEV)
    ref = _oracle(ten, ids, go, heads, DEV, p_drop=0.1, seed_words=words)
    _compare(_run_kernel(ten, ids, go, heads, PF.IMPL_TC, p_drop=0.1, seed=seed), ref, RTOL_F16, f"fp16 dropout {stage}")


def test_fp16_dropout_mask_matches_bf16():
    x = torch.randn(4099 * 8, device=DEV) + 3.0                  # no zeros in the input
    seed = torch.tensor([123, 456], dtype=torch.int32, device=DEV)
    yh = PF.seeded_dropout(x.half(), 0.3, seed)
    yb = PF.seeded_dropout(x.bfloat16(), 0.3, seed)
    assert torch.equal(yh == 0, yb == 0)
    assert 0.2 < (yh == 0).float().mean().item() < 0.4


def test_fp16_checkpointed_pair_with_dropout_matches_plain():
    torch.manual_seed(17)
    pair = pwa_b200.ConsecutiveSwinBlocks(hidden_channels=48, num_heads=4, pos_bias_embed_dim=64, max_prompts=1,
                                          tokens_per_prompt=64, window_size=(8, 8, 4), down=True, attn_drop=0.1,
                                          proj_drop=0.1).to(DEV).train()
    x0 = torch.randn(2, 48, 16, 16, 8, device=DEV).half()
    ps = [(0.2 * torch.randn(2, 64, 48, device=DEV)).half() for _ in range(2)]
    res = []
    for ckpt in (False, True):
        pair.use_checkpoint = ckpt
        for blk in pair.swin_blocks:
            blk.use_checkpoint = ckpt
        for p in pair.parameters():
            p.grad = None
        x = x0.clone().requires_grad_(True)
        torch.manual_seed(11)
        y = pair(x, tuple(ps))
        assert y.dtype == H
        y.float().square().mean().backward()
        res.append((y.detach(), x.grad.clone(), [p.grad.clone() for p in pair.parameters() if p.grad is not None]))
    assert torch.equal(res[0][0], res[1][0])
    assert rel_linf(res[1][1], res[0][1]) < 5e-3
    for a, b in zip(res[0][2], res[1][2]):
        assert rel_linf(b, a) < 5e-3


# ---- 5. token GEMM -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,Cout", [(48, 144), (48, 48), (96, 288), (192, 576), (192, 192), (16, 48)])
@pytest.mark.parametrize("mode", ["ln", "res_ln_bias", "drop_res_ln_bias", "plain_bias"])
def test_fp16_token_gemm_vs_float64(C, Cout, mode):
    torch.manual_seed(C * 7 + Cout)
    rows = 128 * 9 + 37
    x = torch.randn(rows, C, device=DEV).half()
    res = torch.randn(rows, C, device=DEV).half() if "res" in mode else None
    W = (torch.randn(Cout, C, device=DEV) / C ** 0.5).half()
    bias = (0.1 * torch.randn(Cout, device=DEV)).half() if "bias" in mode else None
    ln = "ln" in mode
    gamma = (1 + 0.2 * torch.randn(C, device=DEV)) if ln else None
    beta = 0.1 * torch.randn(C, device=DEV) if ln else None
    p_drop = 0.1 if "drop" in mode else 0.0
    words = [77, 88]
    seed = torch.tensor(words, dtype=torch.int32, device=DEV) if p_drop else None
    y, s, z, mean, rstd = PF._token_gemm_raw(x, res, gamma, beta, W, bias, res is not None or p_drop > 0, ln, ln, 1e-6, p_drop, seed)
    assert y.dtype == H
    s64 = x.double()
    if p_drop:
        keep = R.elementwise_dropout_keep_factor(words, rows * C, p_drop).to(DEV).reshape(rows, C)
        s64 = (s64 * keep).to(H).double()
    if res is not None:
        s64 = (s64 + res.double()).to(H).double()
    if s is not None:
        assert torch.equal(s.double(), s64)
    z64 = s64
    if ln:
        m64 = s64.mean(dim=1, keepdim=True)
        r64 = (s64.var(dim=1, unbiased=False, keepdim=True) + 1e-6).rsqrt()
        z64 = (s64 - m64) * r64 * gamma.double() + beta.double()
        assert rel_linf(z, z64) < RTOL_F16
        z64 = z.double()
    y64 = z64 @ W.double().t() + (bias.double() if bias is not None else 0.0)
    assert rel_linf(y, y64) < RTOL_F16


# ---- 6. outside the tcgen05 envelope -------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ATTN_CASES)
@pytest.mark.parametrize("impl", ["f32", "auto"])
def test_fp16_fp32_math_kernels_vs_oracle(case, impl):
    B, P, ws, C, heads, I, masked = case
    ten, ids, go = _attn_inputs(B, P, ws, C, heads, I, masked, seed=3)
    scale = (C // heads) ** -0.5
    s = PF._shape_struct(B, P, C, heads, I, ws, scale)
    if impl == "auto" and _lib.lib.pwa_attn_tc_supported(s, _lib.PWA_F16):
        pytest.skip("inside the tcgen05 envelope (held by the stage tests)")
    ten_r = [None if t is None else (t.to(H).double() if i < 5 else t.float().double()) for i, t in enumerate(ten)]
    ref_out, ref_grads = _oracle_attn(ten_r, ids, go.to(H).double(), heads, ws, scale)
    dev = [None if t is None else (t.to(DEV, H) if i < 5 else t.to(DEV, torch.float32)).requires_grad_(True)
           for i, t in enumerate(ten)]
    out = PF.prompted_window_attention(*dev, None if ids is None else ids.to(DEV), heads, ws, scale,
                                       PF.IMPL_F32 if impl == "f32" else 0)
    assert out.dtype == H and rel_linf(out, ref_out) < RTOL_F16
    out.backward(go.to(DEV, H))
    for n, t, g in zip(NAMES, dev, ref_grads):
        if t is not None:
            assert rel_linf(t.grad, g) < RTOL_F16, n


def test_fp16_tc_supported_equals_bf16():
    for B, dims, C, heads, I in STAGES.values():
        P = pwa_b200.get_geometry(dims, WS, (4, 4, 2)).P
        s = PF._shape_struct(B, P, C, heads, I, WS, (C // heads) ** -0.5)
        assert _lib.lib.pwa_attn_tc_supported(s, _lib.PWA_F16) == _lib.lib.pwa_attn_tc_supported(s, _lib.PWA_BF16) == 1
    for B, P, ws, C, heads, I, masked in TC_CASES + ATTN_CASES:
        s = PF._shape_struct(B, P, C, heads, I, ws, (C // heads) ** -0.5)
        assert _lib.lib.pwa_attn_tc_supported(s, _lib.PWA_F16) == _lib.lib.pwa_attn_tc_supported(s, _lib.PWA_BF16)


# ---- 7. blocks and models ------------------------------------------------------------------------------------------------
def _block_tol(n, ws):
    return 1.5 * RTOL_F16 if ("pe." in n and tuple(ws) == (4, 4, 2)) else RTOL_F16


@pytest.mark.parametrize("name", golden_names("blk_"))
def test_fp16_block_vs_reference_golden(name):
    from tests.test_gpu_parity import _make_block
    meta, sd, x, p, go, out, grads = load_block_case(name, torch.float32)
    blk = _make_block(meta, sd)
    xd = x.to(DEV, H).requires_grad_(True)
    pd = p.to(DEV, H).requires_grad_(True) if p is not None else None
    y = blk(xd, pd)
    assert y.dtype == H
    assert rel_linf(y, out) < RTOL_F16
    y.backward(go.to(DEV, H))
    assert rel_linf(xd.grad, grads["x"]) < RTOL_F16
    if p is not None:
        assert rel_linf(pd.grad, grads["p"]) < RTOL_F16
    for n, prm in blk.named_parameters():
        g = prm.grad if prm.grad is not None else torch.zeros_like(prm)
        assert rel_linf(g, grads[n]) < _block_tol(n, meta["ws"]), n


@pytest.mark.parametrize("tag,mld", [("mld1", True), ("mld0", False), ("odd1", True)])
def test_fp16_pair_merge_vs_reference_golden(tag, mld):
    d = load_npz("pair_merge")
    sd = {k[len(tag) + 4:]: torch.from_numpy(v) for k, v in d.items() if k.startswith(tag + ".sd.")}
    pair = pwa_b200.ConsecutiveSwinBlocks(hidden_channels=12, num_heads=2, pos_bias_embed_dim=16, max_prompts=1,
                                          tokens_per_prompt=8, window_size=(4, 4, 2), down=True, merge_last_dim=mld)
    pair.load_state_dict(sd)
    pair.to(DEV)
    t = lambda k: torch.from_numpy(d[f"{tag}.{k}"])
    x = t("x").to(DEV, H).requires_grad_(True)
    p0, p1 = t("p0").to(DEV, H).requires_grad_(True), t("p1").to(DEV, H).requires_grad_(True)
    y = pair(x, (p0, p1))
    assert rel_linf(y, t("out")) < RTOL_F16
    y.backward(t("go").to(DEV, H))
    for nm, g in (("x", x.grad), ("p0", p0.grad), ("p1", p1.grad)):
        assert rel_linf(g, t("grad." + nm)) < RTOL_F16, nm
    for n, prm in pair.named_parameters():
        g = prm.grad if prm.grad is not None else torch.zeros_like(prm)
        assert rel_linf(g, t("grad." + n)) < _block_tol(n, (4, 4, 2)), n


def test_autocast_float16_selects_fp16_compute():
    blk = pwa_b200.SwinTransformerBlock(hidden_channels=48, window_size=(8, 8, 4), pos_bias_embed_dim=64, num_heads=4,
                                        max_prompts=1, tokens_per_prompt=64)
    x32 = torch.randn(1, 48, 8, 8, 4, device=DEV)
    with torch.autocast("cuda"):
        assert blk._compute_dtype(x32) == H
    with torch.autocast("cuda", dtype=torch.bfloat16):
        assert blk._compute_dtype(x32) == torch.bfloat16
        assert blk._compute_dtype(x32.half()) == torch.bfloat16
    assert blk._compute_dtype(x32) == torch.float32
    assert blk._compute_dtype(x32.half()) == H
    assert blk._compute_dtype(x32.bfloat16()) == torch.bfloat16


def test_fp16_swin_unetr_autocast_vs_reference_golden():
    """SwinUnetR under the default torch.autocast('cuda') (float16) within the bound of the bf16 model test, and with a worst
    error below the bf16 run's."""
    from oracle import gen_golden_model as G
    from tests.test_gpu_model import _build
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for name, mode, dims, batch, dec_prompt in G.CASES:
            d = load_npz(name)
            worst = {}
            for ac in (torch.float16, torch.bfloat16):
                model = _build(name, mode, dec_prompt)
                x = G.case_inputs(name, batch, dims).to(DEV)
                with torch.autocast("cuda", dtype=ac):
                    out = model(x)
                loss, errs = 0.0, {}
                for k, t in G.output_items(out):
                    errs["out." + k] = rel_linf(G.subsample(t.float()), torch.from_numpy(d["out." + k]))
                    loss = loss + (t.float() * G.upstream_grad(name, k, t.shape).to(DEV)).sum()
                loss.backward()
                prm = dict(model.named_parameters())
                gmax = max(float(np.abs(ref).max()) for k, ref in d.items() if k.startswith("grad."))
                for k, ref in d.items():
                    if k.startswith("grad."):
                        p = prm[k[5:]]
                        errs[k] = G.grad_error(p.grad if p.grad is not None else torch.zeros_like(p), ref, gmax)
                worst_ref = max(float(d["bf16ref." + k]) for k in errs if k.startswith("grad."))
                tol = {k: (4e-2 if k.startswith("out.") else max(4e-2, 1.5 * worst_ref)) for k in errs}
                bad = {k: (v, tol[k]) for k, v in errs.items() if not v < tol[k]}
                assert not bad, (name, ac, bad)
                worst[ac] = max(errs.values())
            print(name, {str(k): f"{v:.2e}" for k, v in worst.items()})
            assert worst[torch.float16] < worst[torch.bfloat16], (name, worst)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


# ---- 8. GradScaler -------------------------------------------------------------------------------------------------------
def test_fp16_nonfinite_dout_propagates():
    B, P, ws, C, heads, I, masked = 1, 2, (8, 8, 4), 48, 4, 64, True
    ten, ids, go = _attn_inputs(B, P, ws, C, heads, I, masked, seed=5)
    dev = [None if t is None else (t.to(DEV, H) if i < 5 else t.to(DEV, torch.float32)).requires_grad_(True)
           for i, t in enumerate(ten)]
    out = PF.prompted_window_attention(*dev, ids.to(DEV), heads, ws, (C // heads) ** -0.5, PF.IMPL_TC)
    g = go.to(DEV, H)
    g[0, 1, 5, 3] = float("inf")                  # window 1, query 5, head 0
    out.backward(g)
    q, k, v = dev[0].grad, dev[1].grad, dev[2].grad
    assert not torch.isfinite(q[0, 1, 5, :12].float()).all()
    assert not torch.isfinite(k[0, 1, :, :12].float()).all()
    assert not torch.isfinite(v[0, 1, :, 3].float()).all()
    assert torch.isfinite(q[0, 0].float()).all() and torch.isfinite(q[0, 1, :, 12:].float()).all()   # other windows / heads
    scaler = torch.amp.GradScaler("cuda")
    scaler.scale(torch.ones((), device=DEV))          # (creates the scale tensor, as the scaled backward of a step would)
    prm = torch.nn.Parameter(torch.zeros(q.shape, device=DEV))
    prm.grad = q.float()
    opt = torch.optim.SGD([prm], lr=1.0)
    scaler.unscale_(opt)
    assert sum(v.item() for v in scaler._found_inf_per_device(opt).values()) > 0


def test_fp16_gradscaler_inside_graphed_step():
    """scaler.scale(loss).backward() captured in a GraphedStep: the scale tensor is read by the replay, scaler.update()
    changes it in place.  Starting at 2^32 the first replays overflow: their steps are skipped (parameters unchanged) and the
    scale halves; a later replay steps, with unscaled gradients matching an eager fp16 step at the same scale."""
    import bench
    from pwa_b200.graphs import GraphedStep
    args = types.SimpleNamespace(patch=64, batch=1, dropout=0.0, frozen=False)
    wl = bench.EncoderWorkload(torch.device(DEV), args, use_checkpoint=False)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 32)
    opt = torch.optim.SGD(wl.params, lr=1e-3)

    def step(x):
        b = x.shape[0]
        ps = [wl.prompts[j].to(x.dtype).unsqueeze(0).expand(b, -1, -1) for j in range(2 * len(wl.model))]
        loss = 0.0
        for j, st in enumerate(wl.model):
            x = st(x, (ps[2 * j], ps[2 * j + 1]))
            loss = loss + x.float().square().mean()
        scaler.scale(loss).backward()
        return loss.detach()

    gen = torch.Generator().manual_seed(3)
    x = wl.host_batch(gen, H).to(DEV)
    g = GraphedStep(step, [x], wl.params, warmup=1)
    stepped = False
    for it in range(40):
        before = [p.detach().clone() for p in wl.params]
        scale0 = scaler.get_scale()
        g(x)
        g.bind_grads()
        grads = [None if p.grad is None else p.grad.clone() for p in wl.params]
        scaler.step(opt)
        scaler.update()
        changed = any(not torch.equal(a, p.detach()) for a, p in zip(before, wl.params))
        if scaler.get_scale() < scale0:                  # overflow: skipped and halved
            assert not changed and scaler.get_scale() == scale0 / 2
            assert it < 39
            continue
        assert changed
        stepped = True
        # eager reference at the same scale, from the same parameters (restore them)
        with torch.no_grad():
            for p, a in zip(wl.params, before):
                p.copy_(a)
        for p in wl.params:
            p.grad = None
        b = x.shape[0]
        ps = [wl.prompts[j].to(H).unsqueeze(0).expand(b, -1, -1) for j in range(2 * len(wl.model))]
        xx, loss = x, 0.0
        for j, st in enumerate(wl.model):
            xx = st(xx, (ps[2 * j], ps[2 * j + 1]))
            loss = loss + xx.float().square().mean()
        (loss * scale0).backward()
        for gr, p in zip(grads, wl.params):
            if gr is not None:
                assert rel_linf(gr.float() / scale0, p.grad.float() / scale0) < RTOL_F16
        break
    assert stepped
