"""float64 torch restatement of MONAI's DiceLoss / FocalLoss / DiceFocalLoss (1.3-series formulas) for integer label maps,
written the way MONAI computes them: an explicit one-hot target [B, K, *S], the activation, channel 0 dropped from input and
target when include_background=False, then the reductions.  Differentiated by autograd, its gradients are the reference of
the GPU tests.  Independent of the product: it imports torch only.

`seg_sums` restates the per-(sample, class) sums [4, B, K] (I, P, G, F) that the fused kernel returns, with the sums of the
absolute values of their terms (the scale of each sum's rounding error).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F


def one_hot(labels: torch.Tensor, K: int, spatial_dims: int) -> torch.Tensor:
    """[B, 1, *S] or [B, *S] labels (any dtype: .long() truncation, as MONAI's one_hot) -> float64 [B, K, *S]; a label outside
    [0, K) gives an all-zero row."""
    lab = labels.long()
    if lab.dim() == spatial_dims + 2:
        lab = lab[:, 0]
    cls = torch.arange(K, device=lab.device).view((1, K) + (1,) * spatial_dims)
    return (lab.unsqueeze(1) == cls).double()


def _activate(x, sigmoid, softmax):
    if sigmoid:
        return torch.sigmoid(x)
    if softmax:
        return torch.softmax(x, 1)
    return x


def _sigmoid_focal(x, y, gamma, alpha):
    loss = x - x * y - F.logsigmoid(x)
    loss = torch.exp(gamma * F.logsigmoid(-x * (y * 2 - 1))) * loss
    if alpha is not None:
        loss = (y * alpha + (1 - y) * (1 - alpha)) * loss
    return loss


def _softmax_focal(x, y, gamma, alpha):
    ls = x.log_softmax(1)
    loss = -(1 - ls.exp()).pow(gamma) * ls * y
    if alpha is not None:
        fac = torch.tensor([1 - alpha] + [alpha] * (y.shape[1] - 1), dtype=x.dtype, device=x.device)
        loss = fac.view((1, -1) + (1,) * (x.dim() - 2)) * loss
    return loss


def focal_map(x, y, gamma=2.0, alpha=None, use_softmax=False, include_background=True):
    """Per-voxel focal terms [B, K', *S] (MONAI drops channel 0 before the focal computation)."""
    if not include_background:
        x, y = x[:, 1:], y[:, 1:]
    return _softmax_focal(x, y, gamma, alpha) if use_softmax else _sigmoid_focal(x, y, gamma, alpha)


def dice_loss(x, labels, include_background=True, sigmoid=False, softmax=False, squared_pred=False, jaccard=False,
              reduction="mean", smooth_nr=1e-5, smooth_dr=1e-5, batch=False):
    nsp = x.dim() - 2
    y = one_hot(labels, x.shape[1], nsp).to(x.device)
    p = _activate(x, sigmoid, softmax)
    if not include_background:
        p, y = p[:, 1:], y[:, 1:]
    axes = list(range(2, x.dim()))
    if batch:
        axes = [0] + axes
    inter = torch.sum(y * p, dim=axes)
    gt = torch.sum(y, dim=axes)
    pred = torch.sum(p * p if squared_pred else p, dim=axes)
    den = gt + pred
    if jaccard:
        den = 2.0 * (den - inter)
    f = 1.0 - (2.0 * inter + smooth_nr) / (den + smooth_dr)
    if reduction == "mean":
        return f.mean()
    if reduction == "sum":
        return f.sum()
    return f.reshape(tuple(f.shape) + (1,) * nsp)


def focal_loss(x, labels, include_background=True, gamma=2.0, alpha=None, reduction="mean", use_softmax=False):
    y = one_hot(labels, x.shape[1], x.dim() - 2).to(x.device)
    loss = focal_map(x, y, gamma, alpha, use_softmax, include_background)
    if reduction == "sum":
        return loss.mean(dim=list(range(2, x.dim()))).sum()
    return loss.mean()


def dice_focal_loss(x, labels, include_background=True, sigmoid=False, softmax=False, squared_pred=False, jaccard=False,
                    reduction="mean", smooth_nr=1e-5, smooth_dr=1e-5, batch=False, gamma=2.0, lambda_dice=1.0,
                    lambda_focal=1.0, alpha=None, use_softmax=False):
    d = dice_loss(x, labels, include_background, sigmoid, softmax, squared_pred, jaccard, reduction, smooth_nr, smooth_dr, batch)
    f = focal_loss(x, labels, include_background, gamma, alpha, reduction, use_softmax)
    return lambda_dice * d + lambda_focal * f


def seg_sums(x, labels, sigmoid=False, softmax=False, squared_pred=False, focal=None, gamma=2.0, alpha=None,
             include_background=True):
    """The kernel's sums, float64 [4, B, K] (I, P, G, F over all K channels; focal = None, "sigmoid" or "softmax"), and the
    sums of the absolute values of their terms.  The softmax focal form with include_background=False has F = 0 at channel 0
    and its softmax over channels 1 .. K-1."""
    B, K = x.shape[:2]
    y = one_hot(labels, K, x.dim() - 2).to(x.device)
    p = _activate(x, sigmoid, softmax)
    terms = [p * y, p * p if squared_pred else p, y]
    if focal == "sigmoid":
        terms.append(_sigmoid_focal(x, y, gamma, alpha))
    elif focal == "softmax":
        fm = focal_map(x, y, gamma, alpha, True, include_background)
        terms.append(fm if include_background else torch.cat([torch.zeros_like(fm[:, :1]), fm], 1))
    else:
        terms.append(torch.zeros_like(x))
    sums = torch.stack([t.reshape(B, K, -1).sum(-1) for t in terms])
    abs_sums = torch.stack([t.abs().reshape(B, K, -1).sum(-1) for t in terms])
    return sums, abs_sums
