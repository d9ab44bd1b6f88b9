"""Whole-volume sliding-window inference on the sm_100a tiling kernels (include/pwa.h, "whole-volume sliding-window inference").

The downstream model is scored by Dice and IoU per class on whole CT volumes (the reference's SegmentationTrainer.test,
SURVEY.md §3(4)): the volume is cut into roi-sized patches, the model runs on sub-batches of them and the predictions are
added back with overlap weights.  Here the cutting (`pwa_tile_gather`), the weighted adding (`pwa_tile_stitch`) and the final
normalise / argmax pass (`pwa_tile_finalize`) are CUDA kernels, the patch table lives on the device, and with `graph=True` one
sub-batch (gather -> predictor -> stitch -> cursor advance) is captured once as a CUDA graph and replayed over the volume.
Only one sub-batch of patches exists at a time: the volume is never unfolded.

Tiling rule (MONAI's `sliding_window_inference`), per axis a with volume size d, roi r and overlap in [0, 1):
    stride = max(1, int(r * (1 - overlap)))
    d <= r : one origin, 0 (the patch reaches past the volume; those voxels read `cval` and are not stitched back)
    d >  r : n = ceil((d - r) / stride) + 1 origins min(i * stride, d - r), i < n
Patches are ordered by sample, then in raster order over (x, y, z) origins; every voxel's weighted sum is formed in that order.
Importance map w (fp32 [r0][r1][r2]): all ones for mode="constant"; for mode="gaussian"
    prod_a exp(-(i_a - (r_a - 1) / 2)^2 / (2 sigma_a^2)),  sigma_a = sigma_scale * r_a,
normalised to a maximum of 1 and clamped below at its smallest positive value.
The result is sum_p w * pred_p / sum_p w over the patches p covering each voxel.  This follows the published MONAI rule; it is
not claimed to match the reference's own test routine bit for bit.
"""
from __future__ import annotations

import ctypes as C
import math
import weakref
from typing import Callable, Optional, Sequence, Tuple, Union

import torch

from . import _lib
from .functional import _DT, _dtype_code, _ptr, _stream
from .graphs import GraphedStep

_LABEL_DT = {torch.uint8: _lib.PWA_LABEL_U8, torch.int32: _lib.PWA_LABEL_I32, torch.int64: _lib.PWA_LABEL_I64}


def tile_starts(d: int, r: int, overlap: float) -> list:
    """Patch origins along one axis of size d for a roi of r voxels (the rule in the module docstring)."""
    if d <= r:
        return [0]
    stride = max(1, int(r * (1 - overlap)))
    n = math.ceil((d - r) / stride) + 1
    return [min(i * stride, d - r) for i in range(n)]


def tile_origins(batch: int, dims: Sequence[int], roi_size: Sequence[int], overlap: float) -> torch.Tensor:
    """int32 [n][4] table of (b, x0, y0, z0) in patch order: sample, then raster order over (x, y, z)."""
    axes = [torch.tensor(tile_starts(d, r, overlap), dtype=torch.int32) for d, r in zip(dims, roi_size)]
    grid = torch.cartesian_prod(torch.arange(batch, dtype=torch.int32), *axes)
    return grid.reshape(-1, 4).contiguous()


def importance_map(roi_size: Sequence[int], mode: str = "constant", sigma_scale: float = 0.125) -> torch.Tensor:
    """fp32 [r0][r1][r2] weight of each patch position (CPU tensor)."""
    if mode == "constant":
        return torch.ones(tuple(roi_size), dtype=torch.float32)
    if mode != "gaussian":
        raise ValueError(f"mode must be 'constant' or 'gaussian', got {mode!r}")
    g = []
    for r in roi_size:
        sigma = sigma_scale * r
        i = torch.arange(r, dtype=torch.float32)
        g.append(torch.exp(-((i - (r - 1) / 2) ** 2) / (2 * sigma * sigma)))
    w = g[0][:, None, None] * g[1][None, :, None] * g[2][None, None, :]
    w = w / w.max()
    return w.clamp_min(w[w > 0].min()).contiguous()


def _i3(v):
    return (C.c_int32 * 3)(*v)


class _Plan:
    """The device state of one (image shape, roi, sub-batch, dtypes) tiling: patch table, importance map, patch buffer,
    cursor and, once the predictor's class count is known, the accumulators."""

    def __init__(self, image, roi, sw, overlap, mode, sigma_scale, cval, in_dtype):
        dev = image.device
        self.B, self.Cin = image.shape[:2]
        self.dims, self.roi, self.sw, self.cval = tuple(image.shape[2:]), roi, sw, float(cval)
        self.origins = tile_origins(self.B, self.dims, roi, overlap).to(dev)
        self.n = self.origins.shape[0]
        self.steps = -(-self.n // sw)
        self.weight = importance_map(roi, mode, sigma_scale).to(dev)
        self.patches = torch.empty((sw, self.Cin) + roi, dtype=in_dtype, device=dev)
        self.cursor_init = torch.tensor([0, min(sw, self.n)], dtype=torch.int32).to(dev)
        self.cursor = self.cursor_init.clone()
        self.acc = self.wsum = None
        self.K = None

    def gather(self, image, cursor):
        _lib.check(_lib.lib.pwa_tile_gather(_ptr(image), _dtype_code(image), self.B, self.Cin, _i3(self.dims), _ptr(self.origins),
                                            self.n, _ptr(cursor), _i3(self.roi), self.sw, self.cval, _ptr(self.patches),
                                            _dtype_code(self.patches), _stream(image)), "pwa_tile_gather")

    def check_pred(self, pred):
        if not isinstance(pred, torch.Tensor) or pred.dim() != 5 or pred.shape[0] != self.sw or tuple(pred.shape[2:]) != self.roi:
            shape = tuple(pred.shape) if isinstance(pred, torch.Tensor) else type(pred).__name__
            raise ValueError(f"sliding_window_inference: the predictor must map [sw, Cin, *roi] = {tuple(self.patches.shape)} "
                             f"to [sw, K, *roi], got {shape}")
        if pred.dtype not in _DT or not pred.is_cuda:
            raise TypeError(f"sliding_window_inference: predictions must be float32, bfloat16 or float16 CUDA tensors, got {pred.dtype}")
        if self.K is None:
            self.K = pred.shape[1]
            self.acc = torch.zeros((self.B, self.K) + self.dims, dtype=torch.float32, device=pred.device)
            self.wsum = torch.zeros((self.B,) + self.dims, dtype=torch.float32, device=pred.device)
        elif pred.shape[1] != self.K:
            raise ValueError(f"sliding_window_inference: the predictor returned {pred.shape[1]} classes, earlier {self.K}")
        return pred.contiguous()

    def stitch(self, pred, cursor):
        _lib.check(_lib.lib.pwa_tile_stitch(_ptr(pred), _dtype_code(pred), _ptr(self.weight), self.B, self.K, _i3(self.dims),
                                            _ptr(self.origins), self.n, _ptr(cursor), _i3(self.roi), self.sw, _ptr(self.acc),
                                            _ptr(self.wsum), _stream(pred)), "pwa_tile_stitch")
        _lib.check(_lib.lib.pwa_tile_advance(_ptr(cursor), self.sw, self.n, _stream(pred)), "pwa_tile_advance")

    def reset(self):
        self.acc.zero_()
        self.wsum.zero_()

    def finalize(self, want_logits, want_labels):
        dev = self.acc.device
        out = torch.empty_like(self.acc) if want_logits else None
        labels = None
        if want_labels:
            labels = torch.empty((self.B,) + self.dims, dtype=torch.uint8 if self.K <= 256 else torch.int32, device=dev)
        _lib.check(_lib.lib.pwa_tile_finalize(_ptr(self.acc), _ptr(self.wsum), self.B, self.K, _i3(self.dims), _ptr(out),
                                              _lib.PWA_F32, _ptr(labels), None, 0, None, None, None, _stream(self.acc)),
                   "pwa_tile_finalize")
        return out, labels


# predictor -> (key, plan, GraphedStep): one captured sub-batch per live predictor, replaced when the shapes change
_GRAPHS: "weakref.WeakKeyDictionary" = weakref.WeakKeyDictionary()


def _capture(predictor, plan, image):
    try:
        pref = weakref.ref(predictor)        # a cached entry must not keep its own key alive
    except TypeError:                        # not weak-referenceable: never cached, a strong reference is fine
        pref = lambda: predictor             # noqa: E731

    def step_fn(img, cursor):
        plan.gather(img, cursor)
        pred = plan.check_pred(pref()(plan.patches))
        plan.stitch(pred, cursor)
        return pred

    # Autocast caches the low-precision copy of each fp32 weight it casts and frees the cache when the outermost autocast
    # context exits.  A graph captured on cache hits would keep reading those copies after they are freed (and never see
    # in-place weight updates), so the capture runs with the cache off: the casts are recorded and read the parameters.
    with torch.autocast("cuda", dtype=torch.get_autocast_dtype("cuda"), enabled=torch.is_autocast_enabled("cuda"),
                        cache_enabled=False):
        # the first sub-batch runs once eagerly to learn the class count (the accumulators' shape) before anything is captured
        plan.gather(image, plan.cursor)
        plan.check_pred(predictor(plan.patches))
        step = GraphedStep(step_fn, [image, plan.cursor_init], [], warmup=2)
    plan.cursor = step.static_inputs[1]
    return step


def sliding_window_inference(predictor: Callable[[torch.Tensor], torch.Tensor], image: torch.Tensor,
                             roi_size: Union[int, Sequence[int]], sw_batch_size: int = 4, overlap: float = 0.5,
                             mode: str = "constant", sigma_scale: float = 0.125, cval: float = 0.0,
                             input_dtype: Optional[torch.dtype] = None, output: str = "logits", graph: bool = True):
    """Run `predictor` over a whole volume in roi-sized patches and stitch the predictions back.

    predictor: callable from patches [sw_batch_size, Cin, *roi] (dtype `input_dtype`, default the image's) to predictions
        [sw_batch_size, K, *roi] (fp32, bf16 or fp16), e.g. `lambda x: model(x)["downstream"]` for a downstream SwinUnetR in
        eval mode.  A partial last sub-batch is filled with `cval` patches; their predictions are ignored.
    image: CUDA tensor [B, Cin, X, Y, Z] (fp32, bf16 or fp16).
    Returns logits fp32 [B, K, X, Y, Z] (the weighted mean of the covering predictions, see the module docstring for the
    tiling and weighting rule), labels [B, X, Y, Z] (argmax over K of the fp32 logits, uint8 for K <= 256, else int32) or
    both as (logits, labels), for output = "logits", "labels" or "both".

    Runs under torch.no_grad() rather than torch.inference_mode(): the model hosts cache device tensors across calls, and
    inference tensors among them would break a later training step.  The stitched sums are formed in patch order without
    float atomics: bitwise the same for every sw_batch_size and from run to run, given the same predictions.  graph=True captures one sub-batch (gather -> predictor -> stitch -> cursor advance) as a
    CUDA graph and replays it ceil(n_patches / sw_batch_size) times with no host synchronisation; graph=False runs the same
    kernels eagerly and gives bitwise the same result when the predictor does.  The captured graph, a static copy of the image
    and the accumulators are kept while `predictor` lives and reused by the next call with the same shapes, dtypes and
    autocast state: keep the predictor in a variable to evaluate many volumes with one capture.  The graph reads the model's
    parameters by address (autocast's weight casts are recorded in it, not taken from autocast's cache), so it sees in-place
    updates (optimizer steps, load_state_dict) but not parameters that were replaced (e.g. module.half()): pass a new
    predictor after such a change.
    Memory: the accumulators (fp32, K + 1 values per voxel), the outputs and a few sub-batches of patches and predictions;
    with graph=True also the static image copy and the predictor's activations for one sub-batch in the graph's pool.
    """
    if not isinstance(image, torch.Tensor) or image.dim() != 5:
        raise ValueError("sliding_window_inference: image must be a tensor [B, Cin, X, Y, Z]")
    if not image.is_cuda:
        raise RuntimeError("pwa_b200 has no CPU path: tensors must live on a CUDA device (sm_100a)")
    roi = (int(roi_size),) * 3 if isinstance(roi_size, int) else tuple(int(r) for r in roi_size)
    if len(roi) != 3 or min(roi) < 1:
        raise ValueError(f"sliding_window_inference: roi_size must be 3 positive ints, got {roi_size}")
    if not 1 <= sw_batch_size <= _lib.PWA_TILE_MAX_SW:
        raise ValueError(f"sliding_window_inference: sw_batch_size must be in [1, {_lib.PWA_TILE_MAX_SW}], got {sw_batch_size}")
    if not 0.0 <= overlap < 1.0:
        raise ValueError(f"sliding_window_inference: overlap must be in [0, 1), got {overlap}")
    if output not in ("logits", "labels", "both"):
        raise ValueError(f"sliding_window_inference: output must be 'logits', 'labels' or 'both', got {output!r}")
    if mode not in ("constant", "gaussian"):
        raise ValueError(f"mode must be 'constant' or 'gaussian', got {mode!r}")
    in_dtype = image.dtype if input_dtype is None else input_dtype
    _dtype_code(image), _dtype_code(torch.empty(0, dtype=in_dtype))
    # torch.no_grad, not torch.inference_mode: the model hosts cache device tensors (index maps, tables) across calls, and
    # inference tensors in those caches would break a later training step
    with torch.no_grad(), torch.cuda.device(image.device):
        image = image.contiguous()
        key = (tuple(image.shape), image.dtype, image.device, roi, sw_batch_size, float(overlap), mode, float(sigma_scale),
               float(cval), in_dtype, torch.is_autocast_enabled("cuda"), torch.get_autocast_dtype("cuda"))
        if graph:
            entry = None
            try:
                entry = _GRAPHS.get(predictor)
            except TypeError:                    # not weak-referenceable (or unhashable): captured for this call only
                pass
            if entry is None or entry[0] != key:
                plan = _Plan(image, roi, sw_batch_size, overlap, mode, sigma_scale, cval, in_dtype)
                entry = (key, plan, _capture(predictor, plan, image))
                try:
                    _GRAPHS[predictor] = entry
                except TypeError:
                    pass
            _, plan, step = entry
            plan.reset()
            step(image, plan.cursor_init)        # copies the image and the cursor start into the graph's inputs
            for _ in range(plan.steps - 1):
                step(*step.static_inputs)
        else:
            plan = _Plan(image, roi, sw_batch_size, overlap, mode, sigma_scale, cval, in_dtype)
            for _ in range(plan.steps):
                plan.gather(image, plan.cursor)
                plan.stitch(plan.check_pred(predictor(plan.patches)), plan.cursor)
        logits, labels = plan.finalize(output != "labels", output != "logits")
    if output == "logits":
        return logits
    if output == "labels":
        return labels
    return logits, labels


def segmentation_counts(labels: torch.Tensor, target: torch.Tensor, num_classes: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Per (sample, class) true positives, false positives and false negatives, int64 [B, K] each, of a label map against a
    target ([B, ...] CUDA tensors of the same shape, uint8, int32 or int64).  Voxels whose label or target is outside
    [0, num_classes) are not counted.  Exact integer counts; num_classes <= 1024."""
    if not (labels.is_cuda and target.is_cuda):
        raise RuntimeError("pwa_b200 has no CPU path: tensors must live on a CUDA device (sm_100a)")
    if labels.shape != target.shape or labels.dim() < 1:
        raise ValueError(f"segmentation_counts: labels {tuple(labels.shape)} and target {tuple(target.shape)} must match")
    for name, t in (("labels", labels), ("target", target)):
        if t.dtype not in _LABEL_DT:
            raise TypeError(f"segmentation_counts: {name} must be uint8, int32 or int64, got {t.dtype}")
    labels, target = labels.contiguous(), target.contiguous()
    B = labels.shape[0]
    tp, fp, fn = (torch.empty((B, num_classes), dtype=torch.int64, device=labels.device) for _ in range(3))
    with torch.cuda.device(labels.device):
        _lib.check(_lib.lib.pwa_seg_counts(_ptr(labels), _LABEL_DT[labels.dtype], _ptr(target), _LABEL_DT[target.dtype], B,
                                           labels[0].numel(), num_classes, _ptr(tp), _ptr(fp), _ptr(fn), _stream(labels)),
                   "pwa_seg_counts")
    return tp, fp, fn


def dice_iou(tp: torch.Tensor, fp: torch.Tensor, fn: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Dice 2TP / (2TP + FP + FN) and IoU TP / (TP + FP + FN), float64, NaN where the denominator is 0 (a class absent from
    both the prediction and the target)."""
    tp, fp, fn = tp.double(), fp.double(), fn.double()
    nan = torch.full_like(tp, float("nan"))
    d_den, i_den = 2 * tp + fp + fn, tp + fp + fn
    dice = torch.where(d_den > 0, 2 * tp / d_den.clamp_min(1), nan)
    iou = torch.where(i_den > 0, tp / i_den.clamp_min(1), nan)
    return dice, iou
