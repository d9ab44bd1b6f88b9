"""The token-domain kernels (csrc/ln.cu, csrc/dropout.cu, csrc/reduce.cu) against float64 torch on the same stored inputs.

Three things the block-level tests cannot see:
- every LayerNorm dispatch branch of `ln_dispatch` / `ln_dispatch_v`, forward and backward, with and without the residual
  and each combination of the two bias column sums of `pwa_ln_bwd2`, including rows = 1 and rows = 0;
- the column reductions (dgamma, dbeta, dres_colsum, dx_colsum, pwa_dropout_colsum, pwa_colsum_rows) at row counts where
  every CTA of the default launch runs several tiles of its persistent loop, so that the bulk-copy ring is refilled and its
  parity flips.  Each reduced column is held to a bound that one CTA's partial, dropped or added twice, exceeds 4x;
- the column-sum contracts of the fused autograd Functions add_layer_norm and drop_add_ln_linear.
The float64 references run as torch ops on the GPU (none of this repository's kernels)."""
import pytest
import torch

from pwa_b200 import functional as PF
from oracle import restatement as R
from tests.util import rel_linf

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F16, BF16, F32 = torch.float16, torch.bfloat16, torch.float32
DTYPES = [BF16, F16, F32]
EPS = 1e-6
# per-element outputs (y, s, dx, dropout): fp32 math, ONE rounding to the I/O type (2^-9 bf16, 2^-11 fp16 relative);
# the bound is normalised L-inf (tests.util.rel_linf) with 2x headroom over that rounding
RTOL = {F32: 1e-5, BF16: 4e-3, F16: 1e-3}
# column sums: |got_c - ref_c| <= K_SUM * sum_rows |term_rc| (fp32 accumulation in registers, shared memory and atomics)
K_SUM = 1e-5
MAX_GRID = 148 * 8          # the largest grid any of these kernels launches (dropout_launch, ln_launch forward)


def _offset(C, lo=0.5, hi=1.0):
    """Per-column offsets of alternating sign and magnitude in [lo, hi]: never zero, so every column total grows linearly
    with the rows (a missing tile or CTA partial is then a fixed fraction of it, not lost in sqrt(rows) noise)."""
    c = torch.arange(C, device=DEV, dtype=torch.float64)
    return ((-1.0) ** c) * (lo + (hi - lo) * (c % 7) / 6)


def _rows_input(rows, C, dtype, gen, offset=True):
    x = torch.randn(rows, C, generator=gen, device=DEV, dtype=torch.float64)
    return (x + _offset(C) if offset else x).to(dtype)


def _check_colsum(got, ref, mag, what, detect=False):
    """got / ref / mag: [C]; mag = sum over rows of |term|.  detect: the bound must also be 4x below one CTA's share of
    every column total, so that a dropped or doubled CTA partial cannot pass."""
    got, ref, mag = got.double(), ref.double(), mag.double()
    tol = K_SUM * mag + 1e-30
    err = (got - ref).abs()
    assert bool((err <= tol).all()), (what, float((err / tol).max()))
    if detect:
        assert bool((tol < ref.abs() / (4 * MAX_GRID)).all()), (what, "bound too loose to see one CTA",
                                                                 float((tol * 4 * MAX_GRID / ref.abs()).max()))


# ---------------------------------------------------------------------------------------------------------------------
# float64 LayerNorm references
# ---------------------------------------------------------------------------------------------------------------------
def _ln_fwd_ref(x, res, gamma, beta, dtype):
    s = x.double() if res is None else (x.double() + res.double()).to(dtype).double()     # the kernel normalises the STORED sum
    mean = s.mean(1)
    rstd = ((s - mean[:, None]).square().mean(1) + EPS).rsqrt()
    y = (s - mean[:, None]) * rstd[:, None] * gamma.double() + beta.double()
    return s, y, mean, rstd


def _ln_bwd_ref(dy, x, gamma, mean, rstd, dres):
    """dx, and {name: (terms, magnitudes)} of the column sums dgamma, dbeta, dres_colsum, dx_colsum (mean / rstd: the fp32
    values the kernel is given).  A term's magnitude bounds its own fp32 rounding error as well: for dx that is the sum of
    the absolute values of the parts it is computed from (they cancel, |dx| alone can be far smaller)."""
    dy, x, gamma, rstd = dy.double(), x.double(), gamma.double(), rstd.double()[:, None]
    mean = mean.double()[:, None]
    xh = (x - mean) * rstd
    xh_mag = (x.abs() + mean.abs()) * rstd                # (x - mean also cancels)
    g = dy * gamma
    s1, s2 = g.mean(1, keepdim=True), (g * xh).mean(1, keepdim=True)
    dx = rstd * (g - s1 - xh * s2)
    dx_mag = rstd * (g.abs() + s1.abs()) + xh_mag * s2.abs()
    if dres is not None:
        dx, dx_mag = dx + dres.double(), dx_mag + dres.double().abs()
    terms = {"dgamma": (dy * xh, dy.abs() * xh_mag), "dbeta": (dy, dy.abs()), "dx_colsum": (dx, dx_mag),
             "dres_colsum": None if dres is None else (dres.double(), dres.double().abs())}
    return dx, terms


def _run_ln(x, res, gamma, beta, dy, dres, want_rs, want_xs, dtype, detect=False):
    """pwa_ln_fwd then pwa_ln_bwd2 (on the forward's stored sum and statistics), every output against float64."""
    rows, C = x.shape
    if res is None:
        y = PF.layer_norm(x, gamma, beta, EPS)
        s = x
    else:
        s, y = PF.add_layer_norm(x, res, gamma, beta, EPS)
    # the statistics the backward consumes: run the forward kernel through the raw entry point (the autograd wrapper keeps
    # them in its context)
    mean = torch.full((rows,), float("nan"), device=DEV)
    rstd = torch.full((rows,), float("nan"), device=DEV)
    y2 = torch.empty_like(x)
    s2 = torch.empty_like(x) if res is not None else None
    rc = PF._lib.lib.pwa_ln_fwd(PF._ptr(x), PF._ptr(res), PF._ptr(gamma), PF._ptr(beta), PF._ptr(s2), PF._ptr(y2),
                                PF._ptr(mean), PF._ptr(rstd), rows, C, EPS, PF._dtype_code(x), PF._stream(x))
    PF._lib.check(rc, "pwa_ln_fwd")
    s64, y64, m64, r64 = _ln_fwd_ref(x, res, gamma, beta, dtype)
    assert torch.equal(y, y2) and (res is None or torch.equal(s, s2))          # the wrapper is the same kernel
    if res is not None:
        assert torch.equal(s.double(), s64)                                      # one fp32 add, one rounding
    assert rel_linf(y, y64) < RTOL[dtype], ("y", rel_linf(y, y64))
    assert rel_linf(mean, m64) < 1e-5 and rel_linf(rstd, r64) < 1e-5
    dx, dg, db, drs, dxs = PF._ln_backward_raw(dy, s, gamma, mean, rstd, dres, want_rs, want_xs)
    assert (drs is not None) == (want_rs and dres is not None) and (dxs is not None) == want_xs
    dx64, terms = _ln_bwd_ref(dy, s, gamma, mean, rstd, dres)
    assert rel_linf(dx, dx64) < RTOL[dtype], ("dx", rel_linf(dx, dx64))
    for name, got in (("dgamma", dg), ("dbeta", db), ("dres_colsum", drs), ("dx_colsum", dxs)):
        if got is not None:
            t, mag = terms[name]
            _check_colsum(got, t.sum(0), mag.sum(0), name, detect)


# ---------------------------------------------------------------------------------------------------------------------
# B. the LayerNorm branch table
# ---------------------------------------------------------------------------------------------------------------------
# C -> kernel under the default environment (ln_dispatch / ln_dispatch_v in csrc/ln.cu are the source of truth).
# 16-bit rows with C % 8 == 0 and 16-byte aligned pointers take EPV = 8 (nvec = C / 8):
#   nvec <= 32  -> bulk-copy kernels ln_{fwd,bwd}_bulk_kernel, G = 4 (C <= 32), 8 (C <= 64), 16 (C <= 128), 32 (C <= 256)
#   nvec > 32   -> register kernels, G = 32: NV = 2 (C <= 512), 4 (C <= 1024), 8 (C <= 2048)
# 16-bit rows with C % 8 != 0 (or a misaligned pointer) and all fp32 rows take EPV = 4 (nvec = C / 4), register kernels:
#   G = 4 (C <= 16), 8 (C <= 32), 16 (C <= 64), 32 (C <= 128); NV = 2 (C <= 256), 4 (C <= 512), 8 (C <= 1024), 16 (C <= 2048)
# The backward of a register kernel with NV >= 2 and no residual / no column sums is the PLAIN specialisation
# (ln_bwd_kernel<..., true>).
LN_TABLE = [
    # (dtype, C, misaligned)
    *[(t, C, False) for t in (BF16, F16) for C in (8, 24, 32)],     # bulk, G = 4
    *[(t, 48, False) for t in (BF16, F16)],                         # bulk, G = 8
    *[(t, 128, False) for t in (BF16, F16)],                        # bulk, G = 16
    *[(t, 256, False) for t in (BF16, F16)],                        # bulk, G = 32
    *[(t, C, False) for t in (BF16, F16) for C in (384, 1024, 2048)],   # register EPV 8: NV = 2, 4, 8
    *[(t, C, False) for t in (BF16, F16) for C in (12, 36)],        # register EPV 4: G = 4, 16
    *[(t, 48, True) for t in (BF16, F16)],                          # register EPV 4 (not 16-byte aligned), G = 16
    *[(F32, C, False) for C in (12, 48, 128, 192, 384, 1024, 2048)],    # G = 4, 16, 32; NV = 2, 4, 8, 16
]
COLSUMS = [(False, False), (True, False), (False, True), (True, True)]      # (dres_colsum, dx_colsum)


def _operand(rows, C, dtype, gen, misaligned):
    """[rows, C] of dtype; misaligned: a view 4 elements (8 bytes) into a larger buffer, so not 16-byte aligned."""
    t = _rows_input(rows, C, dtype, gen)
    if not misaligned:
        return t
    buf = torch.empty(rows * C + 4, dtype=dtype, device=DEV)
    v = buf[4:].view(rows, C)
    v.copy_(t)
    assert v.data_ptr() % 16 != 0
    return v


@pytest.mark.parametrize("dtype,C,misaligned", LN_TABLE, ids=lambda v: str(v).replace("torch.", ""))
@pytest.mark.parametrize("rows", [1, 2999])
def test_layer_norm_branch_table(dtype, C, misaligned, rows):
    """Each dispatch branch, without and with the residual, and its backward with none, either and both column sums:
    y, s, mean, rstd, dx, dgamma, dbeta, dres_colsum, dx_colsum against float64.  2999 rows: not a multiple of any
    kernel's tile; 1 row: a single, partial tile."""
    gen = torch.Generator(device=DEV).manual_seed(C * 131 + rows)
    gamma = (1 + 0.3 * torch.randn(C, generator=gen, device=DEV)).float()
    beta = (0.2 * torch.randn(C, generator=gen, device=DEV)).float()
    x = _operand(rows, C, dtype, gen, misaligned)
    res = _operand(rows, C, dtype, gen, misaligned)
    dy = _operand(rows, C, dtype, gen, misaligned)
    dres = _operand(rows, C, dtype, gen, misaligned)
    for with_res in (False, True):
        for want_rs, want_xs in COLSUMS:
            _run_ln(x, res if with_res else None, gamma, beta, dy, dres if with_res else None, want_rs, want_xs, dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C", [48, 384])
def test_layer_norm_zero_rows(dtype, C):
    """rows = 0 (valid, non-null row buffers): the forward succeeds and writes nothing; the backward still zeroes dgamma,
    dbeta and both column sums, which start out NaN."""
    f32 = dict(dtype=torch.float32, device=DEV)
    rowbuf = [torch.full((1, C), float("nan"), dtype=dtype, device=DEV) for _ in range(6)]
    g = torch.ones(C, **f32)
    stats = [torch.full((1,), float("nan"), **f32) for _ in range(2)]
    out = [torch.full((C,), float("nan"), **f32) for _ in range(4)]
    lib, p, dt, st = PF._lib.lib, PF._ptr, PF._dtype_code(rowbuf[0]), PF._stream(rowbuf[0])
    x, res, sm, y, dy, dx = rowbuf
    PF._lib.check(lib.pwa_ln_fwd(p(x), p(res), p(g), p(g), p(sm), p(y), p(stats[0]), p(stats[1]), 0, C, EPS, dt, st),
                  "pwa_ln_fwd")
    PF._lib.check(lib.pwa_ln_bwd2(p(dy), p(x), p(g), p(stats[0]), p(stats[1]), p(res), p(dx), *[p(t) for t in out], 0, C,
                                  dt, st), "pwa_ln_bwd2")
    for t in rowbuf + stats:
        assert bool(t.isnan().all())                      # untouched
    for t in out:
        assert torch.equal(t, torch.zeros_like(t))


# ---------------------------------------------------------------------------------------------------------------------
# C. column reductions where every CTA loops
# ---------------------------------------------------------------------------------------------------------------------
def _ln_tiles(dtype, C, rows, fwd, with_res):
    """(tiles, CTAs, ring stages) of the default LayerNorm launch; restates ln_dispatch / ln_launch_bulk_r / ln_launch in
    csrc/ln.cu with no PWA_LN_* variable set (register kernels have no ring: stages = 1)."""
    if dtype != F32 and C % 8 == 0 and C <= 256:          # bulk-copy kernels: PWA_LN_BULK_RF = 1, PWA_LN_BULK_RB = 2
        nvec = C // 8
        G = 4 if nvec <= 4 else 8 if nvec <= 8 else 16 if nvec <= 16 else 32
        R_ = 1 if fwd else 2
        nop = (2 if with_res else 1) if fwd else (3 if with_res else 2)
        tiles = -(-rows // (256 // G * R_))
        cap = 148 * ((4 if R_ == 1 else 3) if fwd else (3 if R_ == 1 else 2))
        return tiles, max(1, min(tiles, cap)), 12 // nop // R_
    nvec = C // (8 if dtype != F32 and C % 8 == 0 else 4)
    G = 4 if nvec <= 4 else 8 if nvec <= 8 else 16 if nvec <= 16 else 32
    tiles = -(-rows // (256 // G))                        # PWA_LN_RF = PWA_LN_RB = 1
    cap = 148 * (8 if fwd else 4)
    if not fwd:
        few = tiles // 6 if tiles // 6 > 148 else min(tiles, 148)
        cap = min(cap, few)
    return tiles, max(1, min(tiles, cap)), 1


def _dropout_tiles(C, rows):
    """dropout_launch (csrc/dropout.cu) with a column sum: blocks of a multiple of C / 4 threads, one quad per thread and
    iteration, at most 148 * 8 CTAs."""
    threads = 256 // (C // 4) * (C // 4)
    tiles = -(-(rows * C // 4) // threads)
    return tiles, max(1, min(tiles, 148 * 8)), 1


def _colsum_rows_tiles(dtype, C, rows):
    """pwa_colsum_rows (csrc/reduce.cu): 16-byte vectors, four per thread and main-loop iteration, at most 148 * 2 CTAs."""
    vpr = C // (16 // torch.empty(0, dtype=dtype).element_size())
    threads = 512 // vpr * vpr
    nvec = rows * vpr
    blocks = max(1, min(-(-nvec // (threads * 4)), 148 * 2))
    return nvec // (threads * 4), blocks, 1


def _assert_loops(tiles_blocks_stages, what):
    tiles, blocks, stages = tiles_blocks_stages
    assert tiles // blocks >= 2 * stages + 1, (what, tiles, blocks, stages)        # every CTA wraps its ring twice


# C = 48: enc0 at 96^3 (B = 4: 442 368 tokens); C = 96: enc1 (B = 4: 55 296 tokens) x 3, which the 16-bit forward needs to
# give each of its 592 CTAs 13 tiles; C = 384: the PatchMerging norm after enc0 (55 296 tokens).  + 37: a ragged last tile.
LOOP_CASES = [(48, 442368 + 37), (96, 3 * 55296 + 37), (384, 55296 + 37)]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C,rows", LOOP_CASES)
def test_layer_norm_reductions_where_every_cta_loops(dtype, C, rows):
    """LayerNorm forward with a residual, and backward with a residual and both column sums, at row counts where every
    CTA runs >= 2 * stages + 1 tiles: dgamma, dbeta, dres_colsum and dx_colsum column by column against float64."""
    _assert_loops(_ln_tiles(dtype, C, rows, True, True), "ln fwd")
    _assert_loops(_ln_tiles(dtype, C, rows, False, True), "ln bwd")
    gen = torch.Generator(device=DEV).manual_seed(C + rows)
    gamma = (1 + 0.2 * torch.randn(C, generator=gen, device=DEV)).float()
    beta = (0.1 * torch.randn(C, generator=gen, device=DEV)).float()
    x, res, dy, dres = (_rows_input(rows, C, dtype, gen) for _ in range(4))
    _run_ln(x, res, gamma, beta, dy, dres, True, True, dtype, detect=True)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C,rows", LOOP_CASES)
def test_dropout_colsum_where_every_cta_loops(dtype, C, rows):
    """pwa_dropout_colsum: the masked tensor and its column sums (fp32 products, before rounding) against float64."""
    _assert_loops(_dropout_tiles(C, rows), "dropout")
    gen = torch.Generator(device=DEV).manual_seed(3 * C + rows)
    dy = _rows_input(rows, C, dtype, gen)
    words = [20261021, -5]
    seed = torch.tensor(words, dtype=torch.int32, device=DEV)
    dx = torch.empty_like(dy)
    cs = torch.full((C,), float("nan"), device=DEV)
    PF._lib.check(PF._lib.lib.pwa_dropout_colsum(PF._ptr(dy), PF._ptr(dx), rows, C, 0.1, PF._ptr(seed), PF._ptr(cs),
                                                 PF._dtype_code(dy), PF._stream(dy)), "pwa_dropout_colsum")
    keep = R.elementwise_dropout_keep_factor(words, rows * C, 0.1).to(DEV).reshape(rows, C)
    term = dy.double() * keep
    assert torch.equal(dx == 0, (keep == 0) | (dy == 0))
    assert rel_linf(dx, term) < RTOL[dtype]
    _check_colsum(cs, term.sum(0), term.abs().sum(0), "dropout colsum", detect=True)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C,rows", LOOP_CASES)
def test_colsum_rows_where_every_cta_loops(dtype, C, rows):
    """pwa_colsum_rows with every CTA running >= 3 iterations of its four-vector main loop."""
    _assert_loops(_colsum_rows_tiles(dtype, C, rows), "colsum_rows")
    gen = torch.Generator(device=DEV).manual_seed(5 * C + rows)
    x = _rows_input(rows, C, dtype, gen)
    out = PF.colsum_rows(x)
    _check_colsum(out, x.double().sum(0), x.double().abs().sum(0), "colsum_rows", detect=True)


# ---------------------------------------------------------------------------------------------------------------------
# D. the fused autograd Functions whose bias gradients are these column sums
# ---------------------------------------------------------------------------------------------------------------------
ENC0_ROWS, ENC0_C = 442368, 48


def _stored(t64, dtype):
    """t64 with the value rounded to dtype (as the kernel stores it) and the gradient of t64 passed straight through."""
    return t64 + (t64.detach().to(dtype).double() - t64.detach())


def _ln64(s, gamma, beta):
    return torch.nn.functional.layer_norm(s, (s.shape[-1],), gamma, beta, EPS)


def _fused_inputs(dtype, seed):
    gen = torch.Generator(device=DEV).manual_seed(seed)
    rows, C = ENC0_ROWS, ENC0_C
    r = lambda *s: torch.randn(*s, generator=gen, device=DEV)
    prm = dict(gamma=1 + 0.2 * r(C), beta=0.1 * r(C), w=r(C, C) / C ** 0.5, b_mlp=0.1 * r(C), b_proj=0.1 * r(C))
    prm = {k: torch.nn.Parameter(v) for k, v in prm.items()}
    a, res, g = (_rows_input(rows, C, dtype, gen) for _ in range(3))
    return prm, a, res, g


def _linear64(z64, w, b, dtype):
    """z64 @ W^T + b as the kernels compute it: the weight and bias stored in dtype, W's gradient g^T z of the stored z."""
    w_st = w.detach().to(dtype).double()
    return z64 @ w_st.t() + z64.detach() @ (w - w.detach()).t() + _stored(b, dtype)


def _compare_grads(got, ref, dtype):
    for name in got:
        tol = 1e-3 if name.startswith("b_") else 2 * RTOL[dtype]      # bias gradients: fp32 column sums
        e = rel_linf(got[name], ref[name])
        assert e < tol, (name, e)


@pytest.mark.parametrize("dtype", [BF16, F16])
def test_add_layer_norm_bias_gradients(dtype):
    """add_layer_norm(x, res, ..., bias_of_x, bias_of_res) wired as the block wires it (swin_block.py, _seg_post):
    x = proj output (its bias: bias_of_x), s = x + res, m = mlp(LayerNorm(s)) (its bias: bias_of_res), output s + m.
    bias_of_res receives the column sum of the gradient that reaches s directly; that equals the column sum of dm (the
    mlp bias gradient) only because s and m meet in s + m, so the upstream gradients here are ds = dm = g, as in the block."""
    prm, a, res, g = _fused_inputs(dtype, 71)
    x = a.clone().requires_grad_(True)
    rd = res.clone().requires_grad_(True)
    s, z = PF.add_layer_norm(x, rd, prm["gamma"], prm["beta"], EPS, bias_of_x=prm["b_proj"], bias_of_res=prm["b_mlp"])
    m = PF.multi_linear(z, prm["b_mlp"], prm["w"], bias_grad=False)
    (s + m).backward(g)
    got = {"dx": x.grad, "dres": rd.grad, **{k: v.grad for k, v in prm.items()}}
    # float64 autograd of the unfused formulas on the same stored values; the proj bias is already inside x (value + 0)
    p64 = {k: v.detach().double().requires_grad_(True) for k, v in prm.items()}
    x64, r64 = a.double().requires_grad_(True), res.double().requires_grad_(True)
    s64 = _stored(x64 + (p64["b_proj"] - p64["b_proj"].detach()) + r64, dtype)
    z64 = _stored(_ln64(s64, p64["gamma"], p64["beta"]), dtype)
    m64 = _linear64(z64, p64["w"], p64["b_mlp"], dtype)
    ((s64 + m64) * g.double()).sum().backward()
    ref = {"dx": x64.grad, "dres": r64.grad, **{k: v.grad for k, v in p64.items()}}
    assert torch.equal(s.double(), s64.detach())
    _compare_grads(got, ref, dtype)


@pytest.mark.parametrize("dtype", [BF16, F16])
@pytest.mark.parametrize("p_drop", [0.0, 0.1])
def test_drop_add_ln_linear_bias_gradients(dtype, p_drop):
    """drop_add_ln_linear(a, res, ..., weight, bias, bias_of_a): s = dropout(a) + res, m = LayerNorm(s) @ W^T + bias in
    the fused token GEMM, output s + m as in the block.  bias receives the column sum of ds, which is the mlp bias gradient
    only because the block adds s + m (ds = dm = g here); bias_of_a (attn.proj.bias) receives the column sum of da,
    through pwa_ln_bwd2 (p_drop = 0) or pwa_dropout_colsum (p_drop > 0)."""
    prm, a, res, g = _fused_inputs(dtype, 73)
    words = [1234567, 7654321]
    seed = torch.tensor(words, dtype=torch.int32, device=DEV)
    ad, rd = a.clone().requires_grad_(True), res.clone().requires_grad_(True)
    s, m = PF.drop_add_ln_linear(ad, rd, prm["gamma"], prm["beta"], EPS, None, None, p_drop, seed, prm["w"], prm["b_mlp"],
                                 bias_of_a=prm["b_proj"])
    (s + m).backward(g)
    got = {"da": ad.grad, "dres": rd.grad, **{k: v.grad for k, v in prm.items()}}
    p64 = {k: v.detach().double().requires_grad_(True) for k, v in prm.items()}
    a64, r64 = a.double().requires_grad_(True), res.double().requires_grad_(True)
    d64 = a64 + (p64["b_proj"] - p64["b_proj"].detach())
    if p_drop:
        keep = R.elementwise_dropout_keep_factor(words, ENC0_ROWS * ENC0_C, p_drop).to(DEV).reshape(ENC0_ROWS, ENC0_C)
        d64 = _stored(d64 * keep, dtype)                  # the kernel rounds the dropped value, then the sum
    s64 = _stored(d64 + r64, dtype)
    z64 = _stored(_ln64(s64, p64["gamma"], p64["beta"]), dtype)
    m64 = _linear64(z64, p64["w"], p64["b_mlp"], dtype)
    ((s64 + m64) * g.double()).sum().backward()
    ref = {"da": a64.grad, "dres": r64.grad, **{k: v.grad for k, v in p64.items()}}
    assert torch.equal(s.double(), s64.detach())
    assert rel_linf(m, m64) < 2 * RTOL[dtype], rel_linf(m, m64)
    _compare_grads(got, ref, dtype)
