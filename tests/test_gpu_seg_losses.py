"""Segmentation losses on the GPU (pwa_b200.trainer.seg_losses, csrc/segloss.cu) against the float64 restatement of MONAI's
formulas (oracle/seg_losses.py), evaluated on the STORED logits upcast:
  1. a grid over K, activation, include_background, squared_pred, jaccard, batch, reductions, both focal forms, gamma, alpha,
     Dice-focal weights, logits and label dtypes, batch sizes, aligned and odd volumes and a logits view offset by one element
     (the scalar path): each sum within 1e-5 of the sum of its terms' magnitudes, the loss within 1e-5 relative, dlogits within
     the project's normalised L-inf bounds;
  2. the production shapes [8, 2, 96^3] (config 4 head) and [4, 5, 96^3] (phase-2 seg_pred head) in bf16 with int64 labels;
  3. edge values: out-of-range labels, logits of +-60 (fp32) and +-1e4 (fp16), a class absent from prediction and target;
  4. reproducibility: bitwise-equal sums, loss and dlogits over three calls (one next to GEMMs on a second stream) and between
     eager and a captured replay; no host synchronisation; no error or warning under torch.use_deterministic_algorithms(True);
  5. end to end: a small downstream SwinUnetR trained with DiceFocalLoss inside a GraphedStep."""
import contextlib
import math
import warnings

import pytest
import torch

import pwa_b200
from pwa_b200 import _lib
from pwa_b200.graphs import GraphedStep
from pwa_b200.trainer import DiceFocalLoss, DiceLoss, FocalLoss, synthetic_loader_downstream
from pwa_b200.trainer import seg_losses as S
from oracle import seg_losses as O
from tests.util import rel_linf

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16
GRAD_RTOL = {F32: 1e-4, BF16: 2e-2, F16: 5e-3}
# upstream gradient of the loss, as GradScaler would scale it: a mean over B*K*nvox terms puts unscaled fp16 gradients near the
# subnormal range, where their rounding is absolute rather than relative (both sides get the same factor)
SCALE = 1024.0
THREADS, GRID_UNIT = 256, 8      # csrc/segloss.cu: threads per CTA, voxels per thread-run in the grid rule

MODULES = {"dice": DiceLoss, "focal": FocalLoss, "dicefocal": DiceFocalLoss}
ORACLES = {"dice": O.dice_loss, "focal": O.focal_loss, "dicefocal": O.dice_focal_loss}

CONFIGS = [
    ("dice", dict(softmax=True)),
    ("dice", dict(sigmoid=True, include_background=False)),
    ("dice", dict()),
    ("dice", dict(softmax=True, squared_pred=True, reduction="sum")),
    ("dice", dict(sigmoid=True, jaccard=True, batch=True)),
    ("dice", dict(softmax=True, include_background=False, jaccard=True, reduction="none")),
    ("dice", dict(squared_pred=True, batch=True, reduction="none")),
    ("dice", dict(softmax=True, batch=True, include_background=False, smooth_nr=0.0, smooth_dr=1e-6)),
    ("focal", dict(gamma=2.0)),
    ("focal", dict(gamma=0.0, alpha=0.25, reduction="sum")),
    ("focal", dict(gamma=1.5, include_background=False)),
    ("focal", dict(gamma=2.0, use_softmax=True)),
    ("focal", dict(gamma=0.0, use_softmax=True, include_background=False)),
    ("focal", dict(gamma=1.5, use_softmax=True, alpha=0.25, reduction="sum")),
    ("focal", dict(gamma=2.0, use_softmax=True, include_background=False, reduction="sum")),
    ("focal", dict(gamma=1.5, alpha=0.25, include_background=False)),
    ("dicefocal", dict(softmax=True, lambda_dice=0.7, lambda_focal=1.3)),
    ("dicefocal", dict(softmax=True, use_softmax=True, gamma=1.5, lambda_focal=0.5)),
    ("dicefocal", dict(sigmoid=True, alpha=0.25, gamma=0.0, include_background=False, squared_pred=True)),
    ("dicefocal", dict(softmax=True, use_softmax=True, include_background=False, jaccard=True, batch=True, reduction="sum")),
    ("dicefocal", dict(gamma=2.0, lambda_dice=2.0, lambda_focal=0.25)),
    ("dicefocal", dict(softmax=True, use_softmax=True, alpha=0.25, gamma=0.0, lambda_dice=1.5)),
]
KS, DTYPES = (2, 3, 5, 14, 32), (F32, BF16, F16)
LABEL_DTYPES = (torch.uint8, torch.int32, torch.int64, torch.float32)
SPATIAL = ((8, 8, 8), (7, 9, 11))      # nvox a multiple of 8 (vector path) and odd


def _grid():
    cases = []
    for c, (kind, kw) in enumerate(CONFIGS):
        for r in range(3):
            i = 3 * c + r
            cases.append(pytest.param(kind, kw, KS[i % 5], DTYPES[i % 3], LABEL_DTYPES[i % 4], (1, 3)[(i // 2) % 2],
                                      SPATIAL[(i // 3) % 2], i % 7 == 0, i % 2 == 0, id=f"{kind}{c}-{i}"))
    return cases


def _logits(shape, dtype, act_none, offset, seed, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(shape, generator=g) if act_none else torch.randn(shape, generator=g) * scale
    if not offset:
        return x.to(DEV, dtype)
    buf = torch.zeros(x.numel() + 1, dtype=dtype, device=DEV)
    buf[1:] = x.flatten().to(DEV, dtype)
    return buf[1:].view(shape)                       # 2 or 4 bytes past an aligned address: the scalar path


def _labels(B, K, spatial, ldtype, with_channel, seed):
    g = torch.Generator().manual_seed(seed + 1)
    lab = torch.randint(0, K, (B, 1) + spatial if with_channel else (B,) + spatial, generator=g)
    return lab.to(ldtype).to(DEV)


def _cfg_flags(cfg):
    act, sq, focal, skip, gamma, alpha = cfg
    return dict(sigmoid=act == _lib.PWA_ACT_SIGMOID, softmax=act == _lib.PWA_ACT_SOFTMAX, squared_pred=bool(sq),
                focal={0: None, 1: "sigmoid", 2: "softmax"}[focal], gamma=gamma, alpha=None if math.isnan(alpha) else alpha,
                include_background=not skip)


def _kernel_sums(mod, x, lab):
    xf, yf, _ = S._prepare(x, lab, "test")
    with torch.no_grad():
        return S._SegLossSums.apply(xf, yf, mod.cfg)


def _check_sums(mod, x, lab):
    sums = _kernel_sums(mod, x, lab)
    ref, mag = O.seg_sums(x.detach().double(), lab, **_cfg_flags(mod.cfg))
    err = (sums.double() - ref).abs()
    bad = err > 1e-5 * mag
    assert not bool(bad.any()), (err[bad][:8].tolist(), mag[bad][:8].tolist())
    return sums


def _check_loss_and_grad(kind, kw, x, lab, dtype, seed=0):
    mod = MODULES[kind](to_onehot_y=True, **kw)
    xg = x.detach().requires_grad_(True)                  # shares x's storage: an offset view keeps its offset
    out = mod(xg, lab)
    assert out.dtype == F32
    x64 = x.detach().double().requires_grad_(True)
    ref = ORACLES[kind](x64, lab, **kw)
    assert out.shape == ref.shape
    tol = 1e-5 * ref.detach().abs().max().item()
    assert (out.detach().double() - ref.detach()).abs().max().item() <= tol, (out, ref)
    w = torch.randn(out.shape, generator=torch.Generator().manual_seed(seed + 7)).to(DEV) if out.dim() else 1.0
    ((out * w).sum() * SCALE).backward()
    ((ref * w).sum() * SCALE).backward()
    assert xg.grad.dtype == dtype and xg.grad.shape == x.shape
    assert bool(torch.isfinite(xg.grad).all())
    err = rel_linf(xg.grad, x64.grad)
    assert err <= GRAD_RTOL[dtype], err
    return mod, out, xg.grad


@pytest.mark.parametrize("kind,kw,K,dtype,ldtype,B,spatial,offset,with_channel", _grid())
def test_grid_against_float64_oracle(kind, kw, K, dtype, ldtype, B, spatial, offset, with_channel):
    act_none = kind != "focal" and not kw.get("sigmoid") and not kw.get("softmax")
    seed = 17 * K + 5 * B + sum(spatial)
    x = _logits((B, K) + spatial, dtype, act_none, offset, seed)
    lab = _labels(B, K, spatial, ldtype, with_channel, seed)
    mod, _, _ = _check_loss_and_grad(kind, kw, x, lab, dtype, seed)
    _check_sums(mod, x, lab)


@pytest.mark.parametrize("B,K,kw", [(8, 2, dict(softmax=True)),
                                    (4, 5, dict(softmax=True, use_softmax=True, include_background=False, gamma=2.0))])
def test_production_shapes(B, K, kw):
    spatial = (96, 96, 96)
    nvox = 96 ** 3
    x = _logits((B, K) + spatial, BF16, False, False, 11 + K)
    lab = _labels(B, K, spatial, torch.int64, True, 11 + K)
    mod, _, _ = _check_loss_and_grad("dicefocal", kw, x, lab, BF16)
    sums = _check_sums(mod, x, lab)
    assert sums[2].sum().item() == B * nvox                 # G counts every voxel once
    # every thread of every CTA of the forward loops over more than one run of voxels
    slots = S.segloss_workspace_size(B, K, nvox) // (16 * B * K)
    assert nvox // GRID_UNIT >= 2 * THREADS * slots, slots


def test_out_of_range_labels_are_zero_rows():
    for ldtype, bad in ((torch.uint8, 255), (torch.int64, -1), (torch.int32, 7)):
        x = _logits((2, 3, 6, 5, 4), F32, False, False, 3)
        lab = _labels(2, 3, (6, 5, 4), ldtype, True, 3)
        lab.view(-1)[::5] = bad
        for kind, kw in (("dicefocal", dict(softmax=True)), ("dicefocal", dict(sigmoid=True, use_softmax=False, gamma=1.5)),
                         ("focal", dict(use_softmax=True, alpha=0.25))):
            mod, _, _ = _check_loss_and_grad(kind, kw, x, lab, F32)
            sums = _check_sums(mod, x, lab)
            assert sums[2].sum().item() == (lab.view(-1) != bad).sum().item()


@pytest.mark.parametrize("dtype,mag", [(F32, 60.0), (F16, 1e4)])
def test_extreme_logits(dtype, mag):
    g = torch.Generator().manual_seed(4)
    shape = (2, 4, 8, 8, 8)
    x = (torch.randint(0, 2, shape, generator=g).float() * 2 - 1) * mag
    x = x * torch.rand(shape, generator=g).gt(0.3).float()         # some zeros among the +-mag values
    x = x.to(DEV, dtype)
    lab = _labels(2, 4, (8, 8, 8), torch.int64, True, 4)
    for kind, kw in (("dicefocal", dict(softmax=True, gamma=2.0)), ("dicefocal", dict(softmax=True, use_softmax=True, gamma=1.5)),
                     ("dicefocal", dict(sigmoid=True, gamma=0.0, alpha=0.25)),
                     ("focal", dict(use_softmax=True, include_background=False, gamma=2.0)),
                     ("dice", dict(sigmoid=True, squared_pred=True))):
        mod, out, grad = _check_loss_and_grad(kind, kw, x, lab, dtype)
        assert bool(torch.isfinite(out).all())
        _check_sums(mod, x, lab)


def test_absent_class_gives_zero_dice():
    B, K, spatial = 2, 3, (8, 8, 8)
    lab = _labels(B, 2, spatial, torch.int64, True, 5)                 # class 2 never in the target
    x = _logits((B, K) + spatial, F32, True, False, 5)
    x[:, 2] = 0.0                                                      # nor in the prediction (act none)
    f = DiceLoss(to_onehot_y=True, reduction="none")(x, lab)
    assert tuple(f.shape) == (B, K, 1, 1, 1)
    assert torch.all(f[:, 2] == 0.0)
    x2 = _logits((B, K) + spatial, F32, False, False, 5)
    x2[:, 2] = -60.0                                                   # softmax: p ~ 1e-26
    f2 = DiceLoss(to_onehot_y=True, softmax=True, reduction="none")(x2, lab)
    assert float(f2[:, 2].abs().max()) < 1e-6


@contextlib.contextmanager
def _busy_side_stream():
    """Matrix products on a second stream that hold SMs while the body's kernels launch."""
    side = torch.cuda.Stream()
    a = torch.randn(4096, 4096, device=DEV, dtype=BF16)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(8):
            a = (a @ a).clamp_(-1, 1)
    yield
    torch.cuda.current_stream().wait_stream(side)


def _run_once(mod, x, lab):
    xg = x.detach().clone().requires_grad_(True)
    sums = _kernel_sums(mod, xg, lab)
    loss = mod(xg, lab)
    loss.backward()
    return [sums, loss.detach(), xg.grad]


@pytest.mark.parametrize("K,dtype", [(2, BF16), (5, F16), (14, F32)])
def test_bitwise_reproducible(K, dtype):
    B, spatial = 3, (32, 32, 24)
    x = _logits((B, K) + spatial, dtype, False, False, 9)
    lab = _labels(B, K, spatial, torch.int64, True, 9)
    mod = DiceFocalLoss(to_onehot_y=True, softmax=True, use_softmax=K > 2, gamma=1.5)
    runs = [_run_once(mod, x, lab)]
    with _busy_side_stream():
        runs.append(_run_once(mod, x, lab))
    runs.append(_run_once(mod, x, lab))
    torch.cuda.synchronize()
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert torch.equal(a, b)
    # eager == a captured replay of the loss alone (forward and backward)

    def step(xx, ll):
        loss = mod(xx, ll)
        loss.backward()
        return loss.detach()
    gs = GraphedStep(step, [x.detach().clone().requires_grad_(True), lab], [], warmup=2)
    loss = gs(x, lab)
    torch.cuda.synchronize()
    assert torch.equal(loss, runs[0][1])
    assert torch.equal(gs.input_grads[0], runs[0][2])


def test_no_host_sync_and_deterministic_mode():
    B, K, spatial = 2, 5, (16, 16, 16)
    x = _logits((B, K) + spatial, BF16, False, False, 10)
    lab = _labels(B, K, spatial, torch.float32, True, 10)              # float labels: the .long() conversion is in the path
    mod = DiceFocalLoss(to_onehot_y=True, softmax=True, include_background=False, use_softmax=True, gamma=2.0)
    xg = x.detach().clone().requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        loss = mod(xg, lab)
        loss.backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        with warnings.catch_warnings():
            warnings.simplefilter("error")
            torch.use_deterministic_algorithms(True)
            xd = x.detach().clone().requires_grad_(True)
            loss_d = mod(xd, lab)
            loss_d.backward()
            torch.cuda.synchronize()
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
    assert torch.equal(loss_d, loss.detach()) and torch.equal(xd.grad, xg.grad)


def test_autocast_and_grad_scaler():
    B, K, spatial = 2, 2, (16, 16, 8)
    g = torch.Generator().manual_seed(12)
    conv = torch.nn.Conv3d(1, K, 3, padding=1).to(DEV)
    img = torch.rand((B, 1) + spatial, generator=g).to(DEV)
    lab = _labels(B, K, spatial, torch.int64, True, 12)
    mod = DiceFocalLoss(to_onehot_y=True, softmax=True)
    for dtype in (BF16, F16):
        conv.zero_grad(set_to_none=True)
        opt = torch.optim.SGD(conv.parameters(), lr=0.0)
        scaler = torch.amp.GradScaler("cuda", enabled=dtype == F16)
        with torch.autocast("cuda", dtype=dtype):
            logits = conv(img)
            logits.retain_grad()
            loss = mod(logits, lab)
        assert logits.dtype == dtype and loss.dtype == F32
        scaler.scale(loss).backward()
        scaler.unscale_(opt)
        assert bool(torch.isfinite(conv.weight.grad).all())
        scaler.step(opt)
        scaler.update()
        # reference: the same autocast logits, upcast, through the oracle
        lg = logits.detach().double().requires_grad_(True)
        ref = O.dice_focal_loss(lg, lab, softmax=True)
        ref.backward()
        assert abs(loss.item() - ref.item()) <= 1e-5 * abs(ref.item())
        scale = scaler.get_scale() if dtype == F16 else 1.0
        assert rel_linf(logits.grad.double() / scale, lg.grad) < GRAD_RTOL[dtype]


def test_downstream_swin_unetr_in_graphed_step():
    """config 4 reduced (tests/test_gpu_model.py model_cfg4_small): downstream mode, frozen backbone, dropout 0, bf16 autocast,
    DiceFocalLoss(to_onehot_y=True, softmax=True) on the `downstream` head against synthetic masks, captured in a GraphedStep."""
    from oracle import gen_golden_model as G
    conf = G.model_conf("downstream", dec_prompt=True)
    assert conf.attn_drop == 0.0 and conf.proj_drop == 0.0
    model = pwa_b200.SwinUnetR(conf).double().train()
    G.fill_params_deterministic(model)
    model = model.float().to(DEV)
    named = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
    names = [n for n, _ in named]
    assert any("prompt" in n for n in names) and any("downstream" in n for n in names)
    params = [p for _, p in named]
    batch = next(iter(synthetic_loader_downstream(1, 2, patch=(32, 32, 32), classes=conf.output_channels_downstream, seed=3)))
    img, mask = batch["image"].to(DEV), batch["mask"].to(DEV)
    loss_fn = DiceFocalLoss(to_onehot_y=True, softmax=True)

    def step(x, m):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = model(x)["downstream"]
        loss = loss_fn(out, m)
        loss.backward()
        return loss.detach()

    for p in params:
        p.grad = None
    eager_loss = step(img, mask)
    eager_grads = [None if p.grad is None else p.grad.clone() for p in params]
    gs = GraphedStep(step, [img, mask], params, warmup=2)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        l1 = gs(img, mask).clone()
        g1 = [None if g is None else g.clone() for g in gs.static_grads]
        l2 = gs(img, mask).clone()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert torch.equal(l1, l2)
    assert abs(l1.item() - eager_loss.item()) <= 1e-5 * abs(eager_loss.item())
    n_checked = 0
    for n, ge, gg in zip(names, eager_grads, g1):
        assert (ge is None) == (gg is None), n
        if ge is None:
            continue
        assert rel_linf(gg, ge) < 4e-2, n
        n_checked += 1
    assert n_checked >= 3
