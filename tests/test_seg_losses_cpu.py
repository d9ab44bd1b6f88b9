"""CPU-only checks of the segmentation losses (pwa_b200.trainer.seg_losses, csrc/segloss.cu): the workspace query answers
without a GPU, malformed calls of the C ABI return PWA_ERR_ARG before any CUDA call, the Python layer raises
NotImplementedError / ValueError for what it does not support, and the float64 oracle (oracle/seg_losses.py) agrees with values
worked out by hand on a 2-class, 8-voxel case."""
import ctypes
import math

import pytest
import torch

import pwa_b200
from pwa_b200 import _lib
from pwa_b200.trainer import DiceFocalLoss, DiceLoss, FocalLoss
from pwa_b200.trainer.seg_losses import segloss_workspace_size
from oracle import seg_losses as O

L = _lib.lib
NAN = float("nan")


def _shape(B=2, K=3, nvox=1000, act=_lib.PWA_ACT_SOFTMAX, sq=0, focal=_lib.PWA_FOCAL_OFF, skip=0, gamma=2.0, alpha=NAN):
    return _lib.PwaSegLoss(B, K, nvox, act, sq, focal, skip, gamma, alpha)


def test_exports_and_constants():
    for sym in _lib.SEGLOSS_SYMBOLS:
        assert sym in _lib.EXPORTED_SYMBOLS and hasattr(L, sym)
    assert pwa_b200.trainer.DiceFocalLoss is DiceFocalLoss
    assert _lib.PWA_SEGLOSS_MAX_K == 32


def test_workspace_size_needs_no_gpu():
    for B, K, nvox in [(1, 2, 1), (8, 2, 96 ** 3), (4, 5, 96 ** 3), (3, 32, 7 * 9 * 11), (65535, 2, 8)]:
        n = L.pwa_segloss_workspace_size(ctypes.byref(_shape(B, K, nvox)))
        assert n > 0 and n % (16 * B * K) == 0, (B, K, nvox, n)
        assert n == segloss_workspace_size(B, K, nvox)
        # the slot count is a function of (B, nvox): the same for every K, activation and focal form
        assert n // (16 * B * K) == L.pwa_segloss_workspace_size(ctypes.byref(_shape(B, 7, nvox, focal=1))) // (16 * B * 7)
    # a larger volume never needs fewer slots
    assert segloss_workspace_size(1, 2, 96 ** 3) >= segloss_workspace_size(1, 2, 32 ** 3)
    for bad in (_shape(B=0), _shape(K=1), _shape(K=33), _shape(nvox=0), _shape(B=65536)):
        assert L.pwa_segloss_workspace_size(ctypes.byref(bad)) == -1
    assert L.pwa_segloss_workspace_size(None) == -1


# fake device addresses: every call below is malformed, so the library returns before it touches them
P = ctypes.c_void_p(1 << 20)
F32P = ctypes.c_void_p(1 << 21)
WS = ctypes.c_void_p(1 << 22)
BIG = 1 << 30


def _fwd(shape, logits=P, dtype=_lib.PWA_BF16, labels=P, ldt=_lib.PWA_LABEL_I64, sums=F32P, ws=WS, nbytes=BIG):
    return L.pwa_segloss_fwd(logits, dtype, labels, ldt, None if shape is None else ctypes.byref(shape), sums, ws, nbytes, None)


def _bwd(shape, logits=P, dtype=_lib.PWA_BF16, labels=P, ldt=_lib.PWA_LABEL_I64, dsums=F32P, dlogits=P):
    return L.pwa_segloss_bwd(logits, dtype, labels, ldt, None if shape is None else ctypes.byref(shape), dsums, dlogits, None)


SIG, SMX = _lib.PWA_FOCAL_SIGMOID, _lib.PWA_FOCAL_SOFTMAX
BAD_SHAPES = [  # (shape, text in the error message)
    (_shape(K=1), "K=1"), (_shape(K=33), "K=33"), (_shape(B=0), "B=0"), (_shape(B=65536), "B=65536"),
    (_shape(nvox=0), "nvox=0"), (_shape(nvox=-5), "nvox=-5"), (_shape(act=3), "act=3"), (_shape(sq=2), "squared_pred=2"),
    (_shape(focal=3), "focal=3"),
    (_shape(focal=SIG, skip=1), "focal_skip_bg"), (_shape(focal=_lib.PWA_FOCAL_OFF, skip=1), "focal_skip_bg"),
    (_shape(focal=SMX, skip=2), "focal_skip_bg"),
    (_shape(focal=SMX, skip=1, alpha=0.25), "alpha"), (_shape(focal=_lib.PWA_FOCAL_OFF, alpha=0.25), "alpha"),
    (_shape(focal=SIG, alpha=float("inf")), "alpha"),
    (_shape(focal=SIG, gamma=-1.0), "gamma"), (_shape(focal=SMX, gamma=NAN), "gamma"),
]


def _err(rc, needle):
    assert rc == -1, rc                                   # PWA_ERR_ARG
    assert needle in L.pwa_last_error().decode(), (needle, L.pwa_last_error().decode())


@pytest.mark.parametrize("shape,needle", BAD_SHAPES)
def test_bad_shape_is_err_arg(shape, needle):
    _err(_fwd(shape), needle)
    _err(_bwd(shape), needle)


def test_bad_pointers_dtypes_and_workspace_are_err_arg():
    ok = _shape(B=2, K=3, nvox=1000)
    _err(_fwd(None), "null shape")
    _err(_bwd(None), "null shape")
    _err(_fwd(ok, logits=None), "null logits")
    _err(_fwd(ok, labels=None), "null logits")
    _err(_fwd(ok, sums=None), "null sums")
    _err(_fwd(ok, ws=None), "workspace")
    _err(_fwd(ok, dtype=3), "bad logits dtype")
    _err(_fwd(ok, ldt=3), "bad label dtype")
    need = L.pwa_segloss_workspace_size(ctypes.byref(ok))
    _err(_fwd(ok, nbytes=need - 4), "workspace of")
    _err(_bwd(ok, logits=None), "null logits")
    _err(_bwd(ok, labels=None), "null logits")
    _err(_bwd(ok, dsums=None), "null dsums")
    _err(_bwd(ok, dlogits=None), "null dsums")
    _err(_bwd(ok, dtype=-1), "bad logits dtype")
    _err(_bwd(ok, ldt=7), "bad label dtype")


def test_not_implemented_options():
    with pytest.raises(NotImplementedError, match="to_onehot_y"):
        DiceLoss(softmax=True)
    with pytest.raises(NotImplementedError, match="to_onehot_y"):
        FocalLoss()
    with pytest.raises(NotImplementedError, match="to_onehot_y"):
        DiceFocalLoss(softmax=True)
    with pytest.raises(NotImplementedError, match="other_act"):
        DiceLoss(to_onehot_y=True, other_act=torch.tanh)
    with pytest.raises(NotImplementedError, match="other_act"):
        DiceFocalLoss(to_onehot_y=True, other_act=torch.tanh)
    with pytest.raises(NotImplementedError, match="weight"):
        DiceLoss(to_onehot_y=True, weight=[1.0, 2.0])
    with pytest.raises(NotImplementedError, match="weight"):
        FocalLoss(to_onehot_y=True, weight=[1.0, 2.0])
    with pytest.raises(NotImplementedError, match="focal_weight"):
        DiceFocalLoss(to_onehot_y=True, focal_weight=[1.0, 2.0])
    with pytest.raises(NotImplementedError, match="weight"):
        DiceFocalLoss(to_onehot_y=True, weight=[1.0, 2.0])
    with pytest.raises(NotImplementedError, match="reduction='none'"):
        FocalLoss(to_onehot_y=True, reduction="none")
    with pytest.raises(NotImplementedError, match="reduction='none'"):
        DiceFocalLoss(to_onehot_y=True, reduction="none")
    with pytest.raises(NotImplementedError, match="alpha"):
        FocalLoss(to_onehot_y=True, use_softmax=True, include_background=False, alpha=0.25)
    with pytest.raises(NotImplementedError, match="alpha"):
        DiceFocalLoss(to_onehot_y=True, use_softmax=True, include_background=False, alpha=0.25)
    x = torch.zeros(2, 33, 4, 4, 4)
    with pytest.raises(NotImplementedError, match="K=33"):
        DiceLoss(to_onehot_y=True, softmax=True)(x, torch.zeros(2, 1, 4, 4, 4, dtype=torch.long))
    # what IS supported constructs without a GPU
    DiceLoss(to_onehot_y=True, reduction="none")
    FocalLoss(to_onehot_y=True, use_softmax=True, include_background=False)
    FocalLoss(to_onehot_y=True, use_softmax=True, alpha=0.25)
    DiceFocalLoss(to_onehot_y=True, sigmoid=True, alpha=0.25)


def test_value_errors():
    with pytest.raises(ValueError, match="mutually exclusive"):
        DiceLoss(to_onehot_y=True, sigmoid=True, softmax=True)
    with pytest.raises(ValueError, match="mutually exclusive"):
        DiceFocalLoss(to_onehot_y=True, sigmoid=True, softmax=True)
    with pytest.raises(ValueError, match="reduction"):
        DiceLoss(to_onehot_y=True, reduction="max")
    with pytest.raises(ValueError, match="gamma"):
        FocalLoss(to_onehot_y=True, gamma=-1.0)
    with pytest.raises(ValueError, match="lambda"):
        DiceFocalLoss(to_onehot_y=True, lambda_dice=-1.0)
    loss = DiceFocalLoss(to_onehot_y=True, softmax=True)
    with pytest.raises(ValueError, match="K >= 2"):
        loss(torch.zeros(2, 1, 4, 4, 4), torch.zeros(2, 1, 4, 4, 4))
    for tgt in ((2, 2, 4, 4, 4), (2, 1, 4, 4, 5), (1, 1, 4, 4, 4), (2, 4, 4), (2, 1, 1, 4, 4, 4)):
        with pytest.raises(ValueError, match="target must be"):
            loss(torch.zeros(2, 3, 4, 4, 4), torch.zeros(tgt))
    # a well-formed call on CPU tensors: there is no CPU path
    with pytest.raises(RuntimeError, match="no CPU path"):
        loss(torch.zeros(2, 3, 4, 4, 4), torch.zeros(2, 4, 4, 4, dtype=torch.long))


# ------------------------------------------------------------------------------------------------------------------------
# the oracle against hand-worked values: K = 2, 8 voxels ([1, 2, 2, 2, 2]), labels 0 0 0 1 1 1 1 0
# ------------------------------------------------------------------------------------------------------------------------
LAB = [0, 0, 0, 1, 1, 1, 1, 0]
P1 = [0.1, 0.2, 0.3, 0.9, 0.8, 0.7, 0.6, 0.4]          # p of class 1; class 0 gets 1 - p1 (act none)
EPS = 1e-5


def _x_prob():
    x = torch.tensor([[1 - p for p in P1], P1], dtype=torch.float64)
    return x.view(1, 2, 2, 2, 2), torch.tensor(LAB).view(1, 1, 2, 2, 2)


def test_oracle_dice_by_hand():
    x, lab = _x_prob()
    # both classes: I = 0.9 + 0.8 + 0.7 + 0.6 = 3, P = 4, G = 4
    assert O.dice_loss(x, lab).item() == pytest.approx(1 - (6 + EPS) / (8 + EPS), abs=1e-12)
    assert O.dice_loss(x, lab, jaccard=True).item() == pytest.approx(1 - (6 + EPS) / (2 * (8 - 3) + EPS), abs=1e-12)
    # squared_pred: P = .81 + .64 + .49 + .36 + .01 + .04 + .09 + .16 = 2.6 for both classes
    assert O.dice_loss(x, lab, squared_pred=True).item() == pytest.approx(1 - (6 + EPS) / (6.6 + EPS), abs=1e-12)
    assert O.dice_loss(x, lab, include_background=False, reduction="sum").item() == pytest.approx(1 - (6 + EPS) / (8 + EPS), abs=1e-12)
    none = O.dice_loss(x, lab, reduction="none")
    assert tuple(none.shape) == (1, 2, 1, 1, 1)
    assert tuple(O.dice_loss(x, lab, reduction="none", batch=True).shape) == (2, 1, 1, 1)
    # a third class absent from both the prediction (p = 0) and the target: its Dice is 1 - eps / eps = 0
    x3 = torch.cat([x, torch.zeros_like(x[:, :1])], 1)
    f = O.dice_loss(x3, lab, reduction="none").flatten()
    assert f[2].item() == 0.0
    assert f[0].item() == pytest.approx(1 - (6 + EPS) / (8 + EPS), abs=1e-12)
    sums, _ = O.seg_sums(x3, lab)
    ref = torch.tensor([[3, 3, 0], [4, 4, 0], [4, 4, 0], [0, 0, 0]], dtype=torch.float64)
    assert torch.allclose(sums[:, 0], ref, rtol=0, atol=1e-12)


LOGITS = [[0.5, -1.0, 2.0, 0.0, -0.5, 1.5, -2.0, 0.25], [-0.5, 1.0, 0.0, 3.0, 0.5, -1.0, 1.0, -0.75]]


def _x_logits():
    return torch.tensor(LOGITS, dtype=torch.float64).view(1, 2, 2, 2, 2), torch.tensor(LAB).view(1, 2, 2, 2)


def _sig(v):
    return 1 / (1 + math.exp(-v))


@pytest.mark.parametrize("gamma", [0.0, 2.0])
def test_oracle_sigmoid_focal_by_hand(gamma):
    x, lab = _x_logits()
    terms = []
    for k in range(2):
        for v in range(8):
            xv, y = LOGITS[k][v], 1.0 if LAB[v] == k else 0.0
            pt = _sig(xv) if y else 1 - _sig(xv)              # probability of the true side
            terms.append(-math.log(pt) * (1 - pt) ** gamma)   # BCE weighted by (1 - pt)^gamma
    assert O.focal_loss(x, lab, gamma=gamma).item() == pytest.approx(sum(terms) / 16, rel=1e-12)
    assert O.focal_loss(x, lab, gamma=gamma, reduction="sum").item() == pytest.approx(sum(terms) / 8, rel=1e-12)
    assert O.focal_loss(x, lab, gamma=gamma, include_background=False).item() == pytest.approx(sum(terms[8:]) / 8, rel=1e-12)
    a = 0.25
    wt = [(a if LAB[v] == k else 1 - a) for k in range(2) for v in range(8)]
    assert O.focal_loss(x, lab, gamma=gamma, alpha=a).item() == pytest.approx(sum(w * t for w, t in zip(wt, terms)) / 16, rel=1e-12)
    sums, _ = O.seg_sums(x, lab, focal="sigmoid", gamma=gamma)
    assert sums[3, 0].tolist() == pytest.approx([sum(terms[:8]), sum(terms[8:])], rel=1e-12)


@pytest.mark.parametrize("gamma", [0.0, 2.0])
def test_oracle_softmax_focal_by_hand(gamma):
    x, lab = _x_logits()
    terms = [0.0] * 16
    for v in range(8):
        t = LAB[v]
        z = [LOGITS[0][v], LOGITS[1][v]]
        q = math.exp(z[t]) / (math.exp(z[0]) + math.exp(z[1]))
        terms[t * 8 + v] = -((1 - q) ** gamma) * math.log(q)
    assert O.focal_loss(x, lab, gamma=gamma, use_softmax=True).item() == pytest.approx(sum(terms) / 16, rel=1e-12)
    # include_background=False: channel 0 is dropped BEFORE the softmax, so the one remaining channel has q = 1 and log q = 0
    assert O.focal_loss(x, lab, gamma=gamma, use_softmax=True, include_background=False).item() == 0.0
    sums, _ = O.seg_sums(x, lab, focal="softmax", gamma=gamma)
    assert sums[3, 0].tolist() == pytest.approx([sum(terms[:8]), sum(terms[8:])], rel=1e-12)
    # DiceFocal = lambda_dice * Dice + lambda_focal * Focal
    df = O.dice_focal_loss(x, lab, softmax=True, gamma=gamma, lambda_dice=0.7, lambda_focal=1.3, use_softmax=True)
    ref = 0.7 * O.dice_loss(x, lab, softmax=True) + 1.3 * sum(terms) / 16
    assert df.item() == pytest.approx(ref.item(), rel=1e-12)


def test_oracle_out_of_range_labels_are_zero_rows():
    y = O.one_hot(torch.tensor([[0, 1, 2, -1, 255]]), 2, 1)
    assert y[0].tolist() == [[1, 0, 0, 0, 0], [0, 1, 0, 0, 0]]
    y = O.one_hot(torch.tensor([[0.0, 1.7, 1.0]]), 2, 1)           # float labels: .long() truncation
    assert y[0].tolist() == [[1, 0, 0], [0, 1, 1]]
