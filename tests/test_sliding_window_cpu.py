"""CPU-only checks of whole-volume sliding-window inference: the tiling rule against a plain restatement, the Gaussian
importance map formula, and PWA_ERR_ARG from malformed calls of the tiling entry points (returned before any CUDA call)."""
import ctypes
import itertools
import math

import pytest
import torch

import pwa_b200
from pwa_b200 import _lib
from pwa_b200.inference import importance_map, tile_origins, tile_starts

L = _lib.lib
F32, BF16 = _lib.PWA_F32, _lib.PWA_BF16


def _starts_ref(d, r, overlap):
    stride = max(1, int(r * (1 - overlap)))
    if d <= r:
        return [0]
    n = math.ceil((d - r) / stride) + 1
    return [min(i * stride, d - r) for i in range(n)]


@pytest.mark.parametrize("overlap", [0.0, 0.25, 0.5, 0.75])
def test_tile_origins_follow_the_rule(overlap):
    rois = [(32, 32, 32), (64, 48, 16), (5, 7, 3)]
    for roi in rois:
        for dims in itertools.product(*[(r - 3, r, r + 1, 2 * r + 5, 3 * r) for r in roi]):
            dims = tuple(max(1, d) for d in dims)
            got = tile_origins(2, dims, roi, overlap)
            axes = [_starts_ref(d, r, overlap) for d, r in zip(dims, roi)]
            ref = [(b, x, y, z) for b in range(2) for x in axes[0] for y in axes[1] for z in axes[2]]
            assert got.dtype == torch.int32 and got.tolist() == [list(t) for t in ref], (dims, roi, overlap)
            for d, r, a in zip(dims, roi, axes):
                # every voxel is covered, the last patch ends at the volume's end when the volume is longer than the roi
                assert a[0] == 0 and (a[-1] + r == d if d > r else a == [0])
                assert all(q > p for p, q in zip(a, a[1:]))


def test_tile_starts_reference_stride():
    # overlap 0.5 with a cubic roi gives the reference's roi/2 stride
    assert tile_starts(512, 96, 0.5) == [0, 48, 96, 144, 192, 240, 288, 336, 384, 416]
    assert tile_starts(256, 96, 0.5) == [0, 48, 96, 144, 160]
    assert tile_starts(96, 96, 0.5) == [0] and tile_starts(40, 96, 0.5) == [0]
    assert tile_starts(10, 3, 0.9) == list(range(8))            # stride clamps at 1


@pytest.mark.parametrize("roi,sigma", [((16, 16, 16), 0.125), ((9, 12, 5), 0.125), ((96, 96, 96), 0.125), ((8, 8, 8), 0.02)])
def test_gaussian_importance_map(roi, sigma):
    w = importance_map(roi, "gaussian", sigma)
    assert w.dtype == torch.float32 and tuple(w.shape) == roi
    ref = torch.ones(roi, dtype=torch.float64)
    for a, r in enumerate(roi):
        i = torch.arange(r, dtype=torch.float64)
        g = torch.exp(-((i - (r - 1) / 2) ** 2) / (2 * (sigma * r) ** 2))
        shape = [1, 1, 1]
        shape[a] = r
        ref = ref * g.view(shape)
    ref = ref / ref.max()
    ref = ref.clamp_min(ref[ref > 0].min())
    assert w.max().item() == 1.0 and w.min().item() > 0
    # products below fp32's range underflow to 0 and take the clamp value, the smallest positive weight
    normal = ref > 1e-30
    assert torch.allclose(w.double()[normal], ref[normal], rtol=1e-5, atol=0)
    assert torch.all(w[~normal] == w.min())
    assert torch.equal(importance_map(roi, "constant"), torch.ones(roi))
    with pytest.raises(ValueError):
        importance_map(roi, "triangle")


def _i3(*v):
    return (ctypes.c_int32 * 3)(*v)


def _err(rc, needle):
    assert rc == -1, rc
    assert needle in L.pwa_last_error().decode()


def test_tile_entry_points_reject_malformed_calls():
    d, r = _i3(8, 8, 8), _i3(4, 4, 4)
    buf, org = 64, 16                                             # non-null, aligned fake pointers: never dereferenced
    g = L.pwa_tile_gather
    _err(g(buf, F32, 1, 1, d, None, 1, buf, r, 1, 0.0, buf, F32, None), "null origins")
    _err(g(buf, F32, 1, 1, d, org, 1, buf, r, 0, 0.0, buf, F32, None), "sw=0")
    _err(g(buf, F32, 1, 1, d, org, 1, buf, r, 1025, 0.0, buf, F32, None), "sw=1025")
    _err(g(buf, F32, 0, 1, d, org, 1, buf, r, 1, 0.0, buf, F32, None), "B=0")
    _err(g(buf, F32, 1, 1, _i3(8, 0, 8), org, 1, buf, r, 1, 0.0, buf, F32, None), "positive")
    _err(g(buf, F32, 1, 1, d, org, 1, buf, _i3(4, -1, 4), 1, 0.0, buf, F32, None), "positive")
    _err(g(buf, F32, 1, 1, d, org + 4, 1, buf, r, 1, 0.0, buf, F32, None), "aligned")
    _err(g(buf, 3, 1, 1, d, org, 1, buf, r, 1, 0.0, buf, F32, None), "dtype")
    _err(g(buf, F32, 1, 1, d, org, 1, buf, r, 1, 0.0, buf, 7, None), "dtype")
    _err(g(None, F32, 1, 1, d, org, 1, buf, r, 1, 0.0, buf, F32, None), "null image")
    _err(g(buf, F32, 1, 1, d, org, -1, buf, r, 1, 0.0, buf, F32, None), "n_total")
    _err(g(buf, F32, 1, 1, None, org, 1, buf, r, 1, 0.0, buf, F32, None), "null dims")
    s = L.pwa_tile_stitch
    _err(s(buf, BF16, buf, 1, 2, d, org, 4, buf, r, 4, buf, None, None), "null pred")
    _err(s(buf, 5, buf, 1, 2, d, org, 4, buf, r, 4, buf, buf, None), "dtype")
    _err(s(buf, BF16, buf, 1, 0, d, org, 4, buf, r, 4, buf, buf, None), "C=0")
    _err(s(buf, BF16, buf, 1, 2, d, org, 4, None, r, 4, buf, buf, None), "null origins")
    _err(s(buf, BF16, buf, 1, 2, d, org, 4, buf, r, 0, buf, buf, None), "sw=0")
    a = L.pwa_tile_advance
    _err(a(None, 4, 10, None), "null cursor")
    _err(a(buf, 0, 10, None), "sw=0")
    f = L.pwa_tile_finalize
    _err(f(None, buf, 1, 2, d, None, F32, None, None, 0, None, None, None, None), "null acc")
    _err(f(buf, buf, 1, 0, d, None, F32, None, None, 0, None, None, None, None), "K=0")
    _err(f(buf, buf, 1, 2, d, buf, 9, None, None, 0, None, None, None, None), "output dtype")
    _err(f(buf, buf, 1, 2, d, None, F32, None, buf, 3, buf, buf, buf, None), "target dtype")
    _err(f(buf, buf, 1, 2, d, None, F32, None, buf, 0, buf, None, buf, None), "tp, fp and fn")
    _err(f(buf, buf, 1, 1025, d, None, F32, None, buf, 0, buf, buf, buf, None), "at most 1024")
    c = L.pwa_seg_counts
    _err(c(None, 0, buf, 0, 1, 64, 2, buf, buf, buf, None), "null labels")
    _err(c(buf, 4, buf, 0, 1, 64, 2, buf, buf, buf, None), "label dtype")
    _err(c(buf, 0, buf, 0, 1, 64, 0, buf, buf, buf, None), "K=0")
    _err(c(buf, 0, buf, 0, 1, 64, 2, None, buf, buf, None), "tp, fp and fn")


def test_python_api_rejects_cpu_tensors_and_bad_arguments():
    x = torch.zeros(1, 1, 8, 8, 8)
    with pytest.raises(RuntimeError, match="no CPU path"):
        pwa_b200.sliding_window_inference(lambda t: t, x, 4)
    with pytest.raises(RuntimeError, match="no CPU path"):
        pwa_b200.segmentation_counts(torch.zeros(1, 4, dtype=torch.uint8), torch.zeros(1, 4, dtype=torch.uint8), 2)
    with pytest.raises(ValueError):
        pwa_b200.sliding_window_inference(lambda t: t, torch.zeros(8, 8, 8), 4)


def test_dice_iou_hand_made():
    tp = torch.tensor([[5, 0, 0, 3]])
    fp = torch.tensor([[1, 0, 2, 0]])
    fn = torch.tensor([[2, 0, 0, 1]])
    dice, iou = pwa_b200.dice_iou(tp, fp, fn)
    assert dice.dtype == torch.float64
    assert dice[0, 0].item() == 10 / 13 and iou[0, 0].item() == 5 / 8
    assert math.isnan(dice[0, 1].item()) and math.isnan(iou[0, 1].item())     # class absent from prediction and target
    assert dice[0, 2].item() == 0.0 and iou[0, 2].item() == 0.0
    assert dice[0, 3].item() == 6 / 7 and iou[0, 3].item() == 3 / 4
