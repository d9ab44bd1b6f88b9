"""Trainer-side glue around the hot path (SURVEY.md §8f-4): student / teacher pair with a multi-tensor EMA update, the
phase-1 / phase-2 SSL losses, the segmentation losses of the downstream and supervised heads (Dice, focal and Dice-focal on the
fused kernels of csrc/segloss.cu, a drop-in for monai.losses), synthetic loaders for the three training modes, and a
data-parallel training step."""
from .momentum import MomentumModel
from .losses import ClusteredPrototypeLoss, ContrastivePairLoss
from .seg_losses import DiceLoss, FocalLoss, DiceFocalLoss
from .synthetic import synthetic_loader_multi_view, synthetic_loader_students_teacher, synthetic_loader_downstream

__all__ = ['MomentumModel', 'ClusteredPrototypeLoss', 'ContrastivePairLoss', 'DiceLoss', 'FocalLoss', 'DiceFocalLoss',
           'synthetic_loader_multi_view',
           'synthetic_loader_students_teacher', 'synthetic_loader_downstream']
