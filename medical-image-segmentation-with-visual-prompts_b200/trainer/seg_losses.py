"""Segmentation losses on the sm_100a kernels: `DiceLoss`, `FocalLoss` and `DiceFocalLoss` with MONAI's constructor arguments
(1.3-series semantics), for integer label maps (`to_onehot_y=True`).  A user of the reference swaps
`from monai.losses import DiceFocalLoss` for `from pwa_b200.trainer import DiceFocalLoss`.

One kernel pass (`pwa_segloss_fwd`, include/pwa.h) reads the logits x [B, K, *S] and the labels once and returns four sums per
(sample, class), fp32 [4, B, K]; with one-hot y_k = [label == k] (a label outside [0, K) is an all-zero row) and the Dice
activation p (x as given, sigmoid(x), or softmax over the K channels):
    I = sum_v p_k y_k,   P = sum_v p_k (p_k^2 with squared_pred),   G = sum_v y_k,   F = sum_v focal_k
    focal_k, sigmoid form:  (x_k - x_k y_k - log sigmoid(x_k)) * exp(gamma * log sigmoid(-x_k (2 y_k - 1)))
                            [* (alpha y_k + (1 - alpha)(1 - y_k))]
    focal_k, softmax form:  -(1 - q_k)^gamma log(q_k) y_k for k >= c0, 0 below; q = softmax over channels c0 .. K-1, where
                            c0 = 1 with include_background=False (MONAI drops channel 0 before this softmax), else 0
                            [* (1 - alpha) for k = 0, alpha otherwise]
The losses are torch arithmetic on those sums; channel 0 is dropped after the activation when include_background=False
(K' = K - 1), and nvox is the number of voxels per sample:
    Dice:  with batch=True, I, P, G are first summed over the batch;  den = G + P  (jaccard: 2 (den - I));
           f = 1 - (2 I + smooth_nr) / (den + smooth_dr);  reduction mean / sum / none ([B, K', 1, ...], [K', 1, ...] with batch)
    Focal: mean = sum F / (B K' nvox);  sum = sum_{b,k} F / nvox  (MONAI averages over space first)
    DiceFocal = lambda_dice * Dice + lambda_focal * Focal, both with the same activation flags, include_background and reduction;
           its focal part takes the sigmoid form unless use_softmax=True, also when softmax=True drives the Dice part.
The backward kernel (`pwa_segloss_bwd`) recomputes the activation per voxel and writes the exact derivative of the sums'
contribution in fp32, rounded once to the logits' dtype.  No option reaches the kernel except the activation, squared_pred and
the focal form, gamma and alpha.

Not supported (NotImplementedError): to_onehot_y=False (one-hot or soft targets), other_act, class weights (weight /
focal_weight), the focal terms with reduction="none", alpha with the softmax focal form and include_background=False (MONAI
ignores alpha there), K > 32.  ValueError: K < 2, sigmoid and softmax both set, a target that is not [B, 1, *S] or [B, *S].

Inputs: logits fp32 / bf16 / fp16 on a CUDA device (under torch.autocast the model's bf16 / fp16 output goes in as it is; the
loss is fp32).  Non-contiguous logits (e.g. a channels-last conv output) are copied once with .contiguous().  Labels uint8,
int32 or int64 are read as they are; any other dtype (e.g. float labels holding integers) is converted once with .long()
(truncation, as MONAI's one_hot does).
The sums are bitwise reproducible (no float atomics), nothing synchronises with the host and nothing allocates outside torch's
caching allocator: the losses run under torch.use_deterministic_algorithms(True), inside a captured GraphedStep and with
GradScaler.
"""
from __future__ import annotations

import math
from typing import Optional

import torch
import torch.nn as nn

from .. import _lib
from ..functional import _dtype_code, _ptr, _stream
from ..inference import _LABEL_DT

_REDUCTIONS = ("mean", "sum", "none")


def _cfg(act: int, squared_pred: bool, focal: int, skip_bg: bool, gamma: float, alpha: Optional[float]) -> tuple:
    return (act, int(squared_pred), focal, int(skip_bg), float(gamma), float("nan") if alpha is None else float(alpha))


def _shape(B: int, K: int, nvox: int, cfg: tuple) -> _lib.PwaSegLoss:
    act, squared, focal, skip_bg, gamma, alpha = cfg
    return _lib.PwaSegLoss(B, K, nvox, act, squared, focal, skip_bg, gamma, alpha)


def segloss_workspace_size(B: int, K: int, nvox: int) -> int:
    """Bytes of device workspace the forward kernel needs (one fp32 slot [4][B][K] per CTA column); needs no GPU."""
    return int(_lib.lib.pwa_segloss_workspace_size(_shape(B, K, nvox, _cfg(0, False, 0, False, 0.0, None))))


class _SegLossSums(torch.autograd.Function):
    """logits [B, K, nvox] (contiguous), labels [B, nvox] (uint8 / int32 / int64) -> sums fp32 [4, B, K] (I, P, G, F)."""

    @staticmethod
    def forward(ctx, logits, labels, cfg):
        B, K, nvox = logits.shape
        shape = _shape(B, K, nvox, cfg)
        nbytes = int(_lib.lib.pwa_segloss_workspace_size(shape))
        _lib.check(min(nbytes, 0), "pwa_segloss_workspace_size")
        work = torch.empty(nbytes, dtype=torch.uint8, device=logits.device)
        sums = torch.empty((4, B, K), dtype=torch.float32, device=logits.device)
        with torch.cuda.device(logits.device):
            _lib.check(_lib.lib.pwa_segloss_fwd(_ptr(logits), _dtype_code(logits), _ptr(labels), _LABEL_DT[labels.dtype], shape,
                                                _ptr(sums), _ptr(work), nbytes, _stream(logits)), "pwa_segloss_fwd")
        ctx.save_for_backward(logits, labels)
        ctx.cfg = cfg
        return sums

    @staticmethod
    def backward(ctx, dsums):
        logits, labels = ctx.saved_tensors
        B, K, nvox = logits.shape
        dsums = dsums.float().contiguous()
        dlogits = torch.empty_like(logits)
        with torch.cuda.device(logits.device):
            _lib.check(_lib.lib.pwa_segloss_bwd(_ptr(logits), _dtype_code(logits), _ptr(labels), _LABEL_DT[labels.dtype],
                                                _shape(B, K, nvox, ctx.cfg), _ptr(dsums), _ptr(dlogits), _stream(logits)),
                       "pwa_segloss_bwd")
        return dlogits, None, None


def _prepare(input: torch.Tensor, target: torch.Tensor, who: str):
    """Checks shapes, then flattens to logits [B, K, nvox] and labels [B, nvox]; returns (logits, labels, number of spatial dims)."""
    if not isinstance(input, torch.Tensor) or input.dim() < 3:
        raise ValueError(f"{who}: input must be a tensor [B, K, *spatial], got "
                         f"{tuple(input.shape) if isinstance(input, torch.Tensor) else type(input).__name__}")
    B, K, spatial = input.shape[0], input.shape[1], tuple(input.shape[2:])
    if K < 2:
        raise ValueError(f"{who}: needs K >= 2 channels (one-hot of integer labels), got K={K}")
    if K > _lib.PWA_SEGLOSS_MAX_K:
        raise NotImplementedError(f"{who}: at most {_lib.PWA_SEGLOSS_MAX_K} classes are supported, got K={K}")
    if tuple(target.shape) not in ((B, 1) + spatial, (B,) + spatial):
        raise ValueError(f"{who}: target must be [B, 1, *spatial] or [B, *spatial] = {(B, 1) + spatial}, got {tuple(target.shape)}")
    if not (input.is_cuda and target.is_cuda):
        raise RuntimeError("pwa_b200 has no CPU path: tensors must live on a CUDA device (sm_100a)")
    _dtype_code(input)
    nvox = math.prod(spatial)
    if nvox < 1 or B < 1:
        raise ValueError(f"{who}: empty input {tuple(input.shape)}")
    labels = target.reshape(B, nvox)
    if labels.dtype not in _LABEL_DT:
        if labels.is_complex():
            raise TypeError(f"{who}: target must hold integer labels, got {labels.dtype}")
        labels = labels.long()
    return input.contiguous().view(B, K, nvox), labels.contiguous(), len(spatial)


def _check_common(who, to_onehot_y, other_act, weight, reduction):
    if not to_onehot_y:
        raise NotImplementedError(f"{who}: only integer label maps are supported (to_onehot_y=True); one-hot or soft targets are not")
    if other_act is not None:
        raise NotImplementedError(f"{who}: other_act is not supported (use sigmoid=True or softmax=True)")
    if weight is not None:
        raise NotImplementedError(f"{who}: class weights are not supported")
    if reduction not in _REDUCTIONS:
        raise ValueError(f"{who}: reduction must be one of {_REDUCTIONS}, got {reduction!r}")


def _check_focal(who, gamma, alpha, use_softmax, include_background, reduction, focal_weight=None):
    if focal_weight is not None:
        raise NotImplementedError(f"{who}: focal_weight (class weights) is not supported")
    if reduction == "none":
        raise NotImplementedError(f"{who}: the focal term with reduction='none' (a per-voxel loss map) is not supported")
    if not (gamma >= 0 and math.isfinite(gamma)):
        raise ValueError(f"{who}: gamma must be finite and >= 0, got {gamma}")
    if alpha is not None and use_softmax and not include_background:
        raise NotImplementedError(f"{who}: alpha with the softmax focal form and include_background=False is not defined "
                                  "(MONAI ignores alpha there)")


def _reduce(f: torch.Tensor, reduction: str, nspatial: int) -> torch.Tensor:
    if reduction == "mean":
        return f.mean()
    if reduction == "sum":
        return f.sum()
    return f.reshape(tuple(f.shape) + (1,) * nspatial)


def _dice(sums, include_background, jaccard, batch, smooth_nr, smooth_dr, reduction, nspatial):
    inter, pred, gt = sums[0], sums[1], sums[2]
    if not include_background:
        inter, pred, gt = inter[:, 1:], pred[:, 1:], gt[:, 1:]
    if batch:
        inter, pred, gt = inter.sum(0), pred.sum(0), gt.sum(0)
    den = gt + pred
    if jaccard:
        den = 2.0 * (den - inter)
    f = 1.0 - (2.0 * inter + smooth_nr) / (den + smooth_dr)
    return _reduce(f, reduction, nspatial)


def _focal(sums, include_background, reduction, nvox):
    f = sums[3] if include_background else sums[3][:, 1:]
    if reduction == "mean":
        return f.sum() / (f.numel() * nvox)
    return (f / nvox).sum()


def _act(who, sigmoid, softmax):
    if sigmoid and softmax:
        raise ValueError(f"{who}: sigmoid=True and softmax=True are mutually exclusive")
    return _lib.PWA_ACT_SIGMOID if sigmoid else _lib.PWA_ACT_SOFTMAX if softmax else _lib.PWA_ACT_NONE


class DiceLoss(nn.Module):
    """MONAI's DiceLoss for integer label maps (formulas in the module docstring)."""

    def __init__(self, include_background: bool = True, to_onehot_y: bool = False, sigmoid: bool = False, softmax: bool = False,
                 other_act=None, squared_pred: bool = False, jaccard: bool = False, reduction: str = "mean",
                 smooth_nr: float = 1e-5, smooth_dr: float = 1e-5, batch: bool = False, weight=None):
        super().__init__()
        _check_common("DiceLoss", to_onehot_y, other_act, weight, reduction)
        self.include_background, self.jaccard, self.batch = include_background, jaccard, batch
        self.reduction, self.smooth_nr, self.smooth_dr = reduction, float(smooth_nr), float(smooth_dr)
        self.cfg = _cfg(_act("DiceLoss", sigmoid, softmax), squared_pred, _lib.PWA_FOCAL_OFF, False, 0.0, None)

    def forward(self, input: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
        x, y, nsp = _prepare(input, target, "DiceLoss")
        sums = _SegLossSums.apply(x, y, self.cfg)
        return _dice(sums, self.include_background, self.jaccard, self.batch, self.smooth_nr, self.smooth_dr, self.reduction, nsp)


class FocalLoss(nn.Module):
    """MONAI's FocalLoss for integer label maps on logits: the sigmoid form per channel, or with use_softmax=True the softmax
    form (formulas in the module docstring)."""

    def __init__(self, include_background: bool = True, to_onehot_y: bool = False, gamma: float = 2.0,
                 alpha: Optional[float] = None, weight=None, reduction: str = "mean", use_softmax: bool = False):
        super().__init__()
        _check_common("FocalLoss", to_onehot_y, None, weight, reduction)
        _check_focal("FocalLoss", gamma, alpha, use_softmax, include_background, reduction)
        self.include_background, self.reduction = include_background, reduction
        focal = _lib.PWA_FOCAL_SOFTMAX if use_softmax else _lib.PWA_FOCAL_SIGMOID
        self.cfg = _cfg(_lib.PWA_ACT_NONE, False, focal, use_softmax and not include_background, gamma, alpha)

    def forward(self, input: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
        x, y, _ = _prepare(input, target, "FocalLoss")
        sums = _SegLossSums.apply(x, y, self.cfg)
        return _focal(sums, self.include_background, self.reduction, x.shape[2])


class DiceFocalLoss(nn.Module):
    """MONAI's DiceFocalLoss for integer label maps: lambda_dice * Dice + lambda_focal * Focal from ONE kernel pass (formulas
    in the module docstring)."""

    def __init__(self, include_background: bool = True, to_onehot_y: bool = False, sigmoid: bool = False, softmax: bool = False,
                 other_act=None, squared_pred: bool = False, jaccard: bool = False, reduction: str = "mean",
                 smooth_nr: float = 1e-5, smooth_dr: float = 1e-5, batch: bool = False, gamma: float = 2.0,
                 focal_weight=None, weight=None, lambda_dice: float = 1.0, lambda_focal: float = 1.0,
                 alpha: Optional[float] = None, use_softmax: bool = False):
        super().__init__()
        _check_common("DiceFocalLoss", to_onehot_y, other_act, weight, reduction)
        _check_focal("DiceFocalLoss", gamma, alpha, use_softmax, include_background, reduction, focal_weight)
        if lambda_dice < 0.0 or lambda_focal < 0.0:
            raise ValueError("DiceFocalLoss: lambda_dice and lambda_focal should be no less than 0.0")
        self.include_background, self.jaccard, self.batch = include_background, jaccard, batch
        self.reduction, self.smooth_nr, self.smooth_dr = reduction, float(smooth_nr), float(smooth_dr)
        self.lambda_dice, self.lambda_focal = float(lambda_dice), float(lambda_focal)
        focal = _lib.PWA_FOCAL_SOFTMAX if use_softmax else _lib.PWA_FOCAL_SIGMOID
        self.cfg = _cfg(_act("DiceFocalLoss", sigmoid, softmax), squared_pred, focal, use_softmax and not include_background,
                        gamma, alpha)

    def forward(self, input: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
        x, y, nsp = _prepare(input, target, "DiceFocalLoss")
        sums = _SegLossSums.apply(x, y, self.cfg)
        dice = _dice(sums, self.include_background, self.jaccard, self.batch, self.smooth_nr, self.smooth_dr, self.reduction, nsp)
        return self.lambda_dice * dice + self.lambda_focal * _focal(sums, self.include_background, self.reduction, x.shape[2])
