"""Deterministic mode: torch.use_deterministic_algorithms(True) runs the `_det` siblings of the entry points whose cross-CTA sums
are float atomics (include/pwa.h), and their results are bitwise reproducible.

1. Each sibling, called three times on the same inputs, gives torch.equal results; one of the three calls runs while GEMMs
   on a second stream occupy SMs, so the CTAs are scheduled differently.  Each result is also held to float64 with the
   tolerance the tests of the atomic kernels use: 1e-5 * sum |term| per column sum, 2e-2 (bf16) / 5e-3 (fp16) for attention.
2. Through the modules: a ConsecutiveSwinBlocks pair (with each checkpoint policy), the frozen-backbone prompt gradients, a
   GraphedStep captured under the flag, and bench.py started twice in fresh processes.
3. The fp32-math and dense-argument attention backwards have no deterministic form: they raise, or warn with warn_only=True.
"""
import contextlib
import glob
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

# cuBLAS needs this before its first handle is created to be deterministic (torch raises without it under the flag)
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

import pwa_b200
from pwa_b200 import functional as PF
from oracle import restatement as R
from tests.util import rel_linf
from tests.test_gpu_multiwindow import RTOL_BF16, RTOL_F16, WS, _compare, _inputs, _oracle, _run_kernel
from tests.test_gpu_token_reductions import LOOP_CASES, _check_colsum, _ln_bwd_ref, _rows_input

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F16, BF16, F32 = torch.float16, torch.bfloat16, torch.float32
RTOL = {BF16: RTOL_BF16, F16: RTOL_F16}


@pytest.fixture
def deterministic():
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    yield
    torch.use_deterministic_algorithms(prev, warn_only=prev_warn)


@contextlib.contextmanager
def _busy_side_stream():
    """GEMMs on a second stream that hold SMs while the body's kernels launch: their CTAs start on the SMs left free and in
    another order than on an idle GPU."""
    side = torch.cuda.Stream()
    a = torch.randn(8192, 8192, device=DEV, dtype=BF16)
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        for _ in range(8):
            a = a @ a.T * 1e-4
    yield
    torch.cuda.synchronize()


def _three_runs(fn):
    """fn() three times (the second under a busy side stream); asserts the results are torch.equal; returns the first."""
    outs = [fn()]
    with _busy_side_stream():
        outs.append(fn())
    outs.append(fn())
    torch.cuda.synchronize()
    for o in outs[1:]:
        for a, b in zip(outs[0], o):
            assert (a is None and b is None) or torch.equal(a, b)
    return outs[0]


def _ws(nbytes):
    assert nbytes >= 0, nbytes
    return torch.empty(max(nbytes, 1), dtype=torch.uint8, device=DEV)


# ---- 1a. token-domain siblings at row counts where every CTA loops -------------------------------------------------------
@pytest.mark.parametrize("dtype", [BF16, F16, F32])
@pytest.mark.parametrize("C,rows", LOOP_CASES)
def test_ln_bwd2_det(dtype, C, rows):
    gen = torch.Generator(device=DEV).manual_seed(C + rows)
    gamma = (1 + 0.2 * torch.randn(C, generator=gen, device=DEV)).float()
    x, dy, dres = (_rows_input(rows, C, dtype, gen) for _ in range(3))
    xd = x.double()
    mean = xd.mean(1).float()
    rstd = ((xd - xd.mean(1, keepdim=True)).square().mean(1) + 1e-6).rsqrt().float()
    code = PF._dtype_code(x)
    ws = _ws(PF._lib.lib.pwa_ln_bwd2_det_workspace_size(rows, C, code))

    def run():
        dx = torch.empty_like(x)
        sums = [torch.full((C,), float("nan"), device=DEV) for _ in range(4)]
        PF._lib.check(PF._lib.lib.pwa_ln_bwd2_det(PF._ptr(dy), PF._ptr(x), PF._ptr(gamma), PF._ptr(mean), PF._ptr(rstd),
                                                  PF._ptr(dres), PF._ptr(dx), *[PF._ptr(t) for t in sums], rows, C, code,
                                                  PF._ptr(ws), ws.numel(), PF._stream(x)), "pwa_ln_bwd2_det")
        return [dx, *sums]

    dx, dg, db, dbr, dbx = _three_runs(run)
    _, terms = _ln_bwd_ref(dy, x, gamma, mean, rstd, dres)
    for name, got in (("dgamma", dg), ("dbeta", db), ("dres_colsum", dbr), ("dx_colsum", dbx)):
        t, mag = terms[name]
        _check_colsum(got, t.sum(0), mag.sum(0), name)


@pytest.mark.parametrize("dtype", [BF16, F16, F32])
@pytest.mark.parametrize("C,rows", LOOP_CASES)
def test_dropout_colsum_det(dtype, C, rows):
    gen = torch.Generator(device=DEV).manual_seed(3 * C + rows)
    dy = _rows_input(rows, C, dtype, gen)
    words = [20261021, -5]
    seed = torch.tensor(words, dtype=torch.int32, device=DEV)
    code = PF._dtype_code(dy)
    ws = _ws(PF._lib.lib.pwa_dropout_colsum_det_workspace_size(rows, C, code))

    def run():
        dx, cs = torch.empty_like(dy), torch.full((C,), float("nan"), device=DEV)
        PF._lib.check(PF._lib.lib.pwa_dropout_colsum_det(PF._ptr(dy), PF._ptr(dx), rows, C, 0.1, PF._ptr(seed), PF._ptr(cs), code,
                                                         PF._ptr(ws), ws.numel(), PF._stream(dy)), "pwa_dropout_colsum_det")
        return [dx, cs]

    dx, cs = _three_runs(run)
    keep = R.elementwise_dropout_keep_factor(words, rows * C, 0.1).to(DEV).reshape(rows, C)
    term = dy.double() * keep
    assert torch.equal(dx == 0, (keep == 0) | (dy == 0))
    _check_colsum(cs, term.sum(0), term.abs().sum(0), "dropout colsum")


@pytest.mark.parametrize("dtype", [BF16, F16, F32])
@pytest.mark.parametrize("C,rows", LOOP_CASES)
def test_colsum_rows_det(dtype, C, rows, deterministic):
    gen = torch.Generator(device=DEV).manual_seed(5 * C + rows)
    x = _rows_input(rows, C, dtype, gen)
    (out,) = _three_runs(lambda: [PF.colsum_rows(x)])          # the flag routes colsum_rows to pwa_colsum_rows_det
    _check_colsum(out, x.double().sum(0), x.double().abs().sum(0), "colsum_rows")


# ---- 1b. attention: enc0 with dropout, and every head dim with I = 0 and I = 128 ----------------------------------------
def _attn_case(C, heads, I, seed, dtype, B=2, dims=(32, 32, 32)):
    """Shifted window attention inputs at dims (8x8x4 windows: P = 128 at 32^3, so every CTA of the backward takes several
    windows); returns (ten, ids, go, heads) in the format of tests/test_gpu_multiwindow.py."""
    geom = pwa_b200.get_geometry(dims, WS, (4, 4, 2))
    ids = R.region_ids(dims, WS, R.effective_shift(dims, WS, (4, 4, 2)), R.pad_amounts(dims, WS)).astype(np.uint8)
    gen = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=gen)
    P, N = geom.P, 256
    ten = [r(B, P, N, C), r(B, P, N, C), r(B, P, N, C), r(B, I, C) if I else None, r(B, I, C) if I else None,
           0.5 * r(heads, 8, 8), 0.5 * r(heads, 8, 8), 0.5 * r(heads, 4, 4), 0.5 * r(heads, I) if I else None]
    ten = [None if t is None else (t.to(dtype) if i < 5 else t.float()) for i, t in enumerate(ten)]
    return ten, ids, r(B, P, N, C).to(dtype), heads


ATTN_DET_CASES = [("enc0", None)] + [(dh, I) for dh in (3, 6, 12, 24, 48) for I in (0, 128)]


@pytest.mark.parametrize("dtype", [BF16, F16])
@pytest.mark.parametrize("case", ATTN_DET_CASES, ids=lambda c: f"{c[0]}" if c[1] is None else f"dh{c[0]}_I{c[1]}")
def test_attn_bwd_det(case, dtype, deterministic):
    if case[0] == "enc0":                                        # B = 4, P = 432, I = 64, shifted
        ten, ids, go, heads, _ = _inputs("enc0", True, seed=11, dtype=dtype)
    else:
        dh, I = case
        ten, ids, go, heads = _attn_case(4 * dh, 4, I, seed=13 + dh + I, dtype=dtype)
    words = [20261021, 4242]
    seed = torch.tensor(words, dtype=torch.int32, device=DEV)

    def run():
        out, grads = _run_kernel(ten, ids, go, heads, PF.IMPL_AUTO, p_drop=0.1, seed=seed)
        return [out, *grads]

    got = _three_runs(run)
    ref = _oracle(ten, ids, go, heads, DEV, p_drop=0.1, seed_words=words)
    _compare((got[0], got[1:]), ref, RTOL[dtype], f"det {case} {dtype}")


# ---- 2. through the modules ------------------------------------------------------------------------------------------------
def _pair(dtype, policy):
    torch.manual_seed(0)
    m = pwa_b200.ConsecutiveSwinBlocks(hidden_channels=48, num_heads=4, pos_bias_embed_dim=64, max_prompts=1, tokens_per_prompt=64,
                                       window_size=WS, use_token_params=True, down=True, merge_last_dim=True,
                                       use_checkpoint=policy is not None, attn_drop=0.1, proj_drop=0.1).to(DEV).train()
    if policy is not None:
        for mod in m.modules():
            if hasattr(mod, "checkpoint_policy"):
                mod.checkpoint_policy = policy
    return m


@pytest.mark.parametrize("dtype", [BF16, F16])
@pytest.mark.parametrize("policy", [None, "selective", "full"])
def test_pair_gradients_bitwise(dtype, policy, deterministic):
    m = _pair(dtype, policy)
    gen = torch.Generator().manual_seed(7)
    x0 = torch.randn(4, 48, 48, 48, 48, generator=gen).to(DEV, dtype)
    p0 = [torch.randn(1, 64, 48, generator=gen).to(DEV, dtype).expand(4, -1, -1) for _ in range(2)]

    def run():
        torch.manual_seed(123)                                   # dropout seed words come from the CUDA generator
        m.zero_grad(set_to_none=True)
        x = x0.clone().requires_grad_(True)
        ps = [p.clone().requires_grad_(True) for p in p0]
        y = m(x, tuple(ps))
        y.float().square().mean().backward()
        return [x.grad, ps[0].grad, ps[1].grad] + [p.grad for p in m.parameters()]

    a, b = run(), run()
    assert len(a) > 3 and all(g is not None for g in a[:3])
    for ga, gb in zip(a, b):
        assert (ga is None and gb is None) or torch.equal(ga, gb)


def _workload(batch, dropout, frozen):
    sys.path.insert(0, ROOT)
    import bench
    args = types.SimpleNamespace(patch=96, dropout=dropout, frozen=frozen, batch=batch)
    return bench.EncoderWorkload(torch.device(DEV), args, use_checkpoint=False)


def test_frozen_backbone_prompt_gradients_bitwise(deterministic):
    """Config 4 (frozen backbone: prompt tokens and their bias parameters train) on the encoder at batch 1."""
    wl = _workload(1, 0.1, True)
    x0 = torch.randn(wl.in_shape, generator=torch.Generator().manual_seed(5)).to(DEV, BF16)

    def run():
        torch.manual_seed(321)
        for p in wl.params:
            p.grad = None
        wl.step(x0.clone())
        return [p.grad.clone() for p in wl.params]

    a, b = run(), run()
    assert any("prompts" in n for n, _ in wl.named_params)
    for ga, gb in zip(a, b):
        assert torch.equal(ga, gb)


def test_graphed_step_captured_under_the_flag(deterministic):
    from pwa_b200.graphs import GraphedStep
    wl = _workload(1, 0.0, False)
    x0 = torch.randn(wl.in_shape, generator=torch.Generator().manual_seed(6)).to(DEV, BF16)
    g = GraphedStep(wl.step, [x0.clone().requires_grad_(True)], wl.params)
    runs = []
    for _ in range(2):
        loss = g(x0)
        torch.cuda.synchronize()
        runs.append([loss.clone(), g.input_grads[0].clone()] + [p.grad.clone() for p in wl.params])
    for a, b in zip(*runs):
        assert torch.equal(a, b)


def test_bench_outputs_bitwise_in_fresh_processes(tmp_path):
    code = ("import runpy, sys, torch; torch.use_deterministic_algorithms(True); sys.argv = sys.argv[1:]; "
            "runpy.run_path(sys.argv[0], run_name='__main__')")
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    dirs = []
    for i in range(2):
        d = tmp_path / f"run{i}"
        cmd = [sys.executable, "-c", code, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
               "--no-cpu-baseline", "--no-variants", "--no-kernels", "--dump-outputs", str(d)]
        subprocess.run(cmd, check=True, env=env, cwd=str(tmp_path), timeout=1800)
        dirs.append(d)
    names = sorted(os.path.basename(f) for f in glob.glob(str(dirs[0] / "*.npy")))
    assert names and names == sorted(os.path.basename(f) for f in glob.glob(str(dirs[1] / "*.npy")))
    for n in names:
        assert np.array_equal(np.load(dirs[0] / n), np.load(dirs[1] / n)), n


# ---- 3. no deterministic form --------------------------------------------------------------------------------------------
def _fp32_attention_loss():
    ten, ids, go, heads = _attn_case(48, 4, 64, seed=3, dtype=F32, B=1, dims=(16, 16, 8))
    dev = [None if t is None else t.to(DEV).requires_grad_(True) for t in ten]
    out = PF.prompted_window_attention(*dev, torch.from_numpy(ids).to(DEV), heads, WS, 12 ** -0.5)
    return (out * go.to(DEV)).sum(), dev[0]


def _dense_attention_loss():
    q, k, v = (torch.randn(1, 2, 64, 48, device=DEV, requires_grad=True) for _ in range(3))
    bias = torch.randn(4, 64, 64, device=DEV, requires_grad=True)
    return PF.dense_window_attention(q, k, v, bias, None, 4, 12 ** -0.5).sum(), q


@pytest.mark.parametrize("make", [_fp32_attention_loss, _dense_attention_loss], ids=["fp32_math", "dense"])
def test_no_deterministic_form_raises_or_warns(make):
    prev = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(True)
        loss, _ = make()
        with pytest.raises(RuntimeError, match="deterministic"):
            loss.backward()
        torch.use_deterministic_algorithms(True, warn_only=True)
        loss, leaf = make()
        with pytest.warns(UserWarning, match="deterministic"):
            loss.backward()
        assert leaf.grad is not None and torch.isfinite(leaf.grad).all()
    finally:
        torch.use_deterministic_algorithms(prev)
