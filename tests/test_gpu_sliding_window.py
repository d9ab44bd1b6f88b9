"""Whole-volume sliding-window inference on the GPU (pwa_b200.inference, csrc/tiles.cu):
  1. pwa_tile_gather is bit-exact against torch slicing + F.pad + .to();
  2. stitching is within 1e-6 of a float64 torch loop, bitwise the same for every sub-batch size, across runs and between
     graph=True and graph=False, and returns the predictions themselves for overlap 0;
  3. the final pass: labels are torch.argmax of the stitched output, counts match a torch.bincount restatement;
  4. end to end with a small downstream SwinUnetR: graph replay == eager, float64 stitching of the same per-batch outputs,
     no host synchronisation in the replay loop, and peak memory bounded by the accumulators plus a few sub-batches."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

import pwa_b200
from pwa_b200 import _lib
from pwa_b200.inference import _Plan, importance_map, tile_origins

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
L = _lib.lib


def _gather_ref(img, origins, roi, sw, first, count, cval, out_dtype):
    B, Cin = img.shape[:2]
    out = []
    for s in range(sw):
        if s < count:
            b, x0, y0, z0 = origins[first + s]
            p = img[b, :, x0:x0 + roi[0], y0:y0 + roi[1], z0:z0 + roi[2]]
            pad = (0, roi[2] - p.shape[3], 0, roi[1] - p.shape[2], 0, roi[0] - p.shape[1])
            p = F.pad(p, pad, value=cval)
        else:
            p = torch.full((Cin,) + tuple(roi), cval, dtype=img.dtype, device=img.device)
        out.append(p.to(out_dtype))
    return torch.stack(out)


GATHER_CASES = [  # B, Cin, dims, roi, sw, overlap, cval
    (2, 2, (37, 21, 19), (16, 16, 16), 3, 0.5, -1.5),      # borders, odd Z (rows not 16-byte aligned), partial last batch
    (1, 1, (10, 40, 9), (16, 16, 16), 4, 0.5, 0.1),        # two axes shorter than the roi
    (2, 1, (33, 30, 64), (16, 12, 8), 5, 0.25, 0.0),       # anisotropic roi, aligned rows: vector path
    (1, 3, (20, 18, 17), (8, 6, 7), 4, 0.75, 2.0),         # roi[2] odd: element kernel
]


@pytest.mark.parametrize("case", GATHER_CASES)
@pytest.mark.parametrize("in_dtype,out_dtype", [(torch.float32, torch.float32), (torch.float32, torch.bfloat16),
                                                (torch.float32, torch.float16), (torch.bfloat16, torch.float32),
                                                (torch.float16, torch.bfloat16)])
def test_gather_bit_exact(case, in_dtype, out_dtype):
    B, Cin, dims, roi, sw, overlap, cval = case
    g = torch.Generator().manual_seed(1)
    img = (torch.randn((B, Cin) + dims, generator=g) * 3).to(DEV, in_dtype)
    plan = _Plan(img, roi, sw, overlap, "constant", 0.125, cval, out_dtype)
    origins = plan.origins.cpu().tolist()
    first = 0
    for _ in range(plan.steps):
        count = min(sw, plan.n - first)
        plan.patches.fill_(float("nan"))
        plan.gather(img, plan.cursor)
        ref = _gather_ref(img, origins, roi, sw, first, count, cval, out_dtype)
        assert torch.equal(plan.patches.view(torch.int8 if out_dtype != torch.float32 else torch.int32),
                           ref.view(torch.int8 if out_dtype != torch.float32 else torch.int32)), (first, count)
        _lib.check(L.pwa_tile_advance(ctypes.c_void_p(plan.cursor.data_ptr()), sw, plan.n,
                                      ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "advance")
        first += count
        assert plan.cursor.tolist() == [first, min(sw, plan.n - first)]


def _elementwise_predictor(K):
    """A deterministic predictor whose outputs depend on the patch values (elementwise, so that the same voxel gives the same
    prediction in every patch that covers it)."""
    def pred(x):
        x = x.float()
        return torch.cat([torch.sin((k + 1) * x[:, :1]) + 0.1 * k for k in range(K)], 1)
    return pred


def _stitch_ref64(img, preds, origins, roi, w):
    """float64 torch restatement: sum_p w * pred_p / sum_p w over the covering patches (patches past the volume cropped)."""
    B = img.shape[0]
    K = preds[0].shape[0]
    X, Y, Z = img.shape[2:]
    acc = torch.zeros((B, K, X, Y, Z), dtype=torch.float64, device=img.device)
    wsum = torch.zeros((B, X, Y, Z), dtype=torch.float64, device=img.device)
    w = w.double().to(img.device)
    for (b, x0, y0, z0), p in zip(origins, preds):
        ex, ey, ez = min(roi[0], X - x0), min(roi[1], Y - y0), min(roi[2], Z - z0)
        ww = w[:ex, :ey, :ez]
        acc[b, :, x0:x0 + ex, y0:y0 + ey, z0:z0 + ez] += ww * p[:, :ex, :ey, :ez].double()
        wsum[b, x0:x0 + ex, y0:y0 + ey, z0:z0 + ez] += ww
    return acc / wsum[:, None]


def _record(predictor):
    calls = []

    def f(x):
        y = predictor(x)
        calls.append(y.detach().clone())
        return y
    return f, calls


def _per_patch(calls, n):
    return [c for call in calls for c in call][:n]


def _rel(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max()).item()


@pytest.mark.parametrize("mode", ["constant", "gaussian"])
def test_stitch_matches_float64_and_is_bitwise_stable(mode):
    K, roi, overlap = 3, (16, 12, 16), 0.5
    g = torch.Generator().manual_seed(2)
    img = torch.rand((2, 1, 41, 29, 35), generator=g).to(DEV)
    pred = _elementwise_predictor(K)
    outs = []
    for sw in (1, 3, 8):
        for graph in (True, False):
            rec, calls = _record(pred)
            out = pwa_b200.sliding_window_inference(rec, img, roi, sw, overlap, mode=mode, graph=graph)
            outs.append(out)
            if sw == 3 and not graph:
                origins = tile_origins(2, img.shape[2:], roi, overlap).tolist()
                ref = _stitch_ref64(img, _per_patch(calls, len(origins)), origins, roi, importance_map(roi, mode))
                assert out.dtype == torch.float32 and out.shape == (2, K) + tuple(img.shape[2:])
                assert _rel(out, ref) < 1e-6
    again = pwa_b200.sliding_window_inference(pred, img, roi, 3, overlap, mode=mode)
    for o in outs[1:] + [again]:
        assert torch.equal(o, outs[0])


def test_overlap_zero_returns_the_predictions():
    img = torch.randn((1, 1, 32, 24, 48), generator=torch.Generator().manual_seed(3)).to(DEV)
    pred = _elementwise_predictor(2)
    out = pwa_b200.sliding_window_inference(pred, img, (16, 12, 16), 4, 0.0, mode="constant")
    assert torch.equal(out, pred(img))


@pytest.mark.parametrize("K", [3, 300])
def test_finalize_labels_and_counts(K):
    g = torch.Generator().manual_seed(4)
    B, dims, roi = 2, (30, 21, 26), (16, 16, 16)
    img = torch.rand((B, 1) + dims, generator=g).to(DEV)
    w = torch.randn(K, generator=g).to(DEV)

    def pred(x):                             # near-ties between classes, so that argmax order matters
        return torch.sin(x * w.view(1, K, 1, 1, 1) * 7).round(decimals=1)
    logits, labels = pwa_b200.sliding_window_inference(pred, img, roi, 4, 0.5, mode="gaussian", output="both")
    assert labels.dtype == (torch.uint8 if K <= 256 else torch.int32)
    assert torch.equal(labels.long(), torch.argmax(logits, 1))
    assert torch.equal(pwa_b200.sliding_window_inference(pred, img, roi, 4, 0.5, mode="gaussian", output="labels"), labels)

    target = torch.randint(0, K + 2, (B,) + dims, generator=g).to(DEV)       # values >= K are ignored
    ref = []
    for b in range(B):
        p, t = labels[b].long().flatten(), target[b].flatten()
        valid = t < K
        hit, miss = valid & (p == t), valid & (p != t)
        ref.append([torch.bincount(p[hit], minlength=K), torch.bincount(p[miss], minlength=K), torch.bincount(t[miss], minlength=K)])
    ref_tp, ref_fp, ref_fn = (torch.stack([r[i] for r in ref]) for i in range(3))
    for tgt in (target, target.to(torch.int32)) + ((target.to(torch.uint8),) if K <= 256 else ()):
        tp, fp, fn = pwa_b200.segmentation_counts(labels, tgt, K)
        assert torch.equal(tp, ref_tp) and torch.equal(fp, ref_fp) and torch.equal(fn, ref_fn)

    # the same counts fused into the final pass (pwa_tile_finalize with a target)
    plan = _Plan(img, roi, 4, 0.5, "gaussian", 0.125, 0.0, img.dtype)
    for _ in range(plan.steps):
        plan.gather(img, plan.cursor)
        plan.stitch(plan.check_pred(pred(plan.patches)), plan.cursor)
    cnt = [torch.full((B, K), -7, dtype=torch.int64, device=DEV) for _ in range(3)]
    lab2 = torch.empty_like(labels)
    i3 = (ctypes.c_int32 * 3)(*dims)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    _lib.check(L.pwa_tile_finalize(p(plan.acc), p(plan.wsum), B, K, i3, None, 0, p(lab2), p(target), _lib.PWA_LABEL_I64,
                                   *[p(c) for c in cnt], ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "finalize")
    assert torch.equal(lab2, labels)
    assert torch.equal(cnt[0], ref_tp) and torch.equal(cnt[1], ref_fp) and torch.equal(cnt[2], ref_fn)


def test_dice_iou_from_counts():
    labels = torch.tensor([[0, 1, 1, 2, 2, 2]], dtype=torch.uint8, device=DEV)
    target = torch.tensor([[0, 1, 2, 2, 2, 9]], dtype=torch.int64, device=DEV)
    tp, fp, fn = pwa_b200.segmentation_counts(labels, target, 4)
    assert tp.tolist() == [[1, 1, 2, 0]] and fp.tolist() == [[0, 1, 0, 0]] and fn.tolist() == [[0, 0, 1, 0]]
    dice, iou = pwa_b200.dice_iou(tp, fp, fn)
    assert dice[0, :3].tolist() == [1.0, 2 / 3, 4 / 5] and iou[0, :3].tolist() == [1.0, 1 / 2, 2 / 3]
    assert torch.isnan(dice[0, 3]) and torch.isnan(iou[0, 3])


def test_predictor_output_shape_is_checked():
    img = torch.rand((1, 1, 20, 20, 20), device=DEV)
    with pytest.raises(ValueError, match="predictor"):
        pwa_b200.sliding_window_inference(lambda x: x[:, :, :8], img, 16, 2, graph=False)
    with pytest.raises(ValueError, match="predictor"):
        pwa_b200.sliding_window_inference(lambda x: x[:, :, :8], img, 16, 2, graph=True)


def _small_downstream_model():
    torch.manual_seed(0)
    conf = pwa_b200.SwinUnetRConfig(training_mode="downstream", hidden_channels=[12, 24, 48, 96], use_encoder_prompting=True,
                                    use_decoder_prompting=True, use_checkpoint=False, attn_drop=0.0, proj_drop=0.0,
                                    contrastive_coding_dim=32)
    return pwa_b200.SwinUnetR(conf).to(DEV).eval()


def test_swin_unetr_end_to_end():
    old = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        model = _small_downstream_model()
        img = torch.rand((1, 1, 150, 130, 110), generator=torch.Generator().manual_seed(5)).to(DEV)
        roi, sw, overlap = (64, 64, 64), 2, 0.5

        def predictor(x):
            return model(x)["downstream"]
        rec, calls = _record(predictor)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            eager = pwa_b200.sliding_window_inference(rec, img, roi, sw, overlap, mode="gaussian", graph=False)
            graphed = pwa_b200.sliding_window_inference(predictor, img, roi, sw, overlap, mode="gaussian", graph=True)
            torch.cuda.synchronize()
            # the second call replays the cached graph: no host synchronisation anywhere in it
            torch.cuda.set_sync_debug_mode("error")
            try:
                replayed = pwa_b200.sliding_window_inference(predictor, img, roi, sw, overlap, mode="gaussian", graph=True)
            finally:
                torch.cuda.set_sync_debug_mode(0)
        assert eager.shape == (1, 2, 150, 130, 110)
        assert torch.equal(graphed, eager) and torch.equal(replayed, eager)
        origins = tile_origins(1, img.shape[2:], roi, overlap).tolist()
        ref = _stitch_ref64(img, _per_patch(calls, len(origins)), origins, roi, importance_map(roi, "gaussian"))
        assert _rel(eager, ref) < 1e-5
        # tensors the model cached during inference do not get in the way of a training step afterwards
        model.train()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            y = model(img[:, :, :64, :64, :64])["downstream"]
        y.float().square().mean().backward()
        assert all(torch.isfinite(p.grad).all() for p in model.parameters() if p.grad is not None)
    finally:
        torch.backends.cudnn.deterministic = old


def test_cached_graph_outlives_the_autocast_context():
    """A graph captured in one autocast context and replayed in another reads the parameters, not autocast's freed cache of
    their bf16 copies, and sees in-place weight updates made between the two."""
    old = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        model = _small_downstream_model()
        for p in model.parameters():
            p.requires_grad_(True)                       # autocast caches the casts of leaf weights that require grad
        img = torch.rand((1, 1, 80, 72, 70), generator=torch.Generator().manual_seed(6)).to(DEV)
        roi, sw = (64, 64, 64), 2

        def predictor(x):
            return model(x)["downstream"]
        with torch.autocast("cuda", dtype=torch.bfloat16):
            first = pwa_b200.sliding_window_inference(predictor, img, roi, sw, 0.5, graph=True)
        # the context has exited: whatever autocast cached is freed; refill that memory and change the weights in place
        junk = [torch.full((1 << 20,), float("nan"), device=DEV) for _ in range(256)]
        with torch.no_grad():
            for m in model.modules():
                if isinstance(m, (torch.nn.Conv3d, torch.nn.ConvTranspose3d, torch.nn.Linear)):
                    m.weight.mul_(0.75)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            replayed = pwa_b200.sliding_window_inference(predictor, img, roi, sw, 0.5, graph=True)
            eager = pwa_b200.sliding_window_inference(predictor, img, roi, sw, 0.5, graph=False)
        del junk
        assert torch.isfinite(replayed).all()
        assert torch.equal(replayed, eager)
        assert not torch.equal(replayed, first)
    finally:
        torch.backends.cudnn.deterministic = old


def test_peak_memory_is_accumulators_plus_sub_batches():
    img = torch.rand((1, 1, 160, 160, 160), device=DEV)
    roi, sw, K = (32, 32, 32), 4, 2

    def predictor(x):
        return torch.cat([x, -x], 1) * 0.5
    n = tile_origins(1, img.shape[2:], roi, 0.5).shape[0]
    vox = img.numel()
    sub_batch = sw * 32 ** 3 * 4 * (1 + K)                 # patches + predictions of one sub-batch, fp32
    fixed = vox * 4 * (K + 1) + vox * 4 * K + vox * 4      # acc + wsum, logits, static image copy
    bound = fixed + 8 * sub_batch + (1 << 20)
    assert bound < n * 32 ** 3 * 4 * K                     # far below the unfolded predictions alone
    for graph in (False, True):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = pwa_b200.sliding_window_inference(predictor, img, roi, sw, 0.5, graph=graph)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        assert peak <= bound, (graph, peak, bound)
        del out
