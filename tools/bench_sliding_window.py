"""Whole-volume sliding-window inference of the downstream SwinUnetR: volumes/s and the tiling kernels' time.

    python tools/bench_sliding_window.py [--rounds 3] [--sw 4 8] [--out profiles/sliding_window.json]

Workload: SwinUnetR(feature_size=48) in downstream mode with encoder and decoder prompting (the bench.py --workload model
--mode downstream network), eval, bf16 autocast, on a synthetic 1 x 1 x 512 x 512 x 256 volume (a CT of 512 x 512 pixels and 256
slices), roi 96^3, overlap 0.5, Gaussian weighting: 10 x 10 x 5 = 500 patches per volume.  For each sub-batch size:
  - graph:  pwa_b200.sliding_window_inference(graph=True) (captured once, then replayed per volume)
  - eager:  the same with graph=False
  - torch:  a loop shaped like the reference's test routine: slice each patch, eager forward per sub-batch, weighted
            accumulation with torch indexing
run alternately in one process, `rounds` volumes each, timed with CUDA events (the host waits at the end of each volume).
Then CUDA events around 50 eager calls of each tiling kernel at this shape, with the bytes each call must move.
Prints one JSON object (GPU name and power limit included) and writes it to --out."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import pwa_b200  # noqa: E402
from pwa_b200.inference import _Plan, importance_map, tile_origins  # noqa: E402

DEV = "cuda:0"
DIMS, ROI, OVERLAP, MODE = (512, 512, 256), (96, 96, 96), 0.5, "gaussian"


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True).stdout.strip().split("\n")[0]
        name, pl, clk = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": pl, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def torch_loop(predictor, img, sw):
    """The reference's routine restated in torch (every axis here is longer than the roi): slice, eager forward per sub-batch, accumulate by indexing."""
    B, _, X, Y, Z = img.shape
    w = importance_map(ROI, MODE).to(img.device)
    origins = tile_origins(B, (X, Y, Z), ROI, OVERLAP).tolist()
    acc = wsum = None
    for i in range(0, len(origins), sw):
        chunk = origins[i:i + sw]
        x = torch.stack([img[b, :, x0:x0 + ROI[0], y0:y0 + ROI[1], z0:z0 + ROI[2]] for b, x0, y0, z0 in chunk])
        pred = predictor(x).float()
        if acc is None:
            acc = torch.zeros((B, pred.shape[1], X, Y, Z), device=img.device)
            wsum = torch.zeros((B, 1, X, Y, Z), device=img.device)
        for (b, x0, y0, z0), p in zip(chunk, pred):
            sl = (b, slice(None), slice(x0, x0 + ROI[0]), slice(y0, y0 + ROI[1]), slice(z0, z0 + ROI[2]))
            acc[sl] += p * w
            wsum[sl] += w
    return acc / wsum


def time_volume(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / 1e3, out


def kernel_times(img, sw, K, reps=50):
    """Event-timed eager calls of the three kernels at the first sub-batch of the volume, with their algorithmic bytes."""
    plan = _Plan(img, ROI, sw, OVERLAP, MODE, 0.125, 0.0, img.dtype)
    pred = torch.randn((sw, K) + ROI, device=DEV).to(torch.bfloat16)
    plan.K = K
    plan.acc = torch.zeros((1, K) + DIMS, device=DEV)
    plan.wsum = torch.zeros((1,) + DIMS, device=DEV)
    # voxels the first sub-batch covers (each read and written once by the stitch)
    cover = torch.zeros(DIMS, dtype=torch.bool, device=DEV)
    for b, x0, y0, z0 in plan.origins[:sw].tolist():
        cover[x0:x0 + ROI[0], y0:y0 + ROI[1], z0:z0 + ROI[2]] = True
    covered = int(cover.sum().item())
    patch = sw * ROI[0] * ROI[1] * ROI[2]
    nvox = img.numel()
    out = {}
    for name, fn, nbytes in (
            ("pwa_tile_gather", lambda: plan.gather(img, plan.cursor), patch * 4 * 2),
            ("pwa_tile_stitch", lambda: plan.stitch(pred, plan.cursor), patch * K * 2 + covered * (K + 1) * 4 * 2),
            ("pwa_tile_finalize", lambda: plan.finalize(True, True), nvox * (K + 1) * 4 + nvox * (K * 4 + 1))):
        for _ in range(3):
            fn()
            plan.cursor.copy_(plan.cursor_init)
        es = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for e0, e1 in es:
            e0.record()
            fn()
            e1.record()
            plan.cursor.copy_(plan.cursor_init)
        torch.cuda.synchronize()
        us = sorted(e0.elapsed_time(e1) * 1e3 for e0, e1 in es)[reps // 2]
        out[name] = {"median_us": round(us, 2), "bytes": nbytes, "GB_per_s": round(nbytes / us / 1e3, 1)}
    out["pwa_tile_stitch"]["note"] = ("stitch timing includes the 1-thread cursor advance; bytes = bf16 predictions read once + "
                                      f"{covered} covered voxels' K + 1 fp32 accumulators read and written once")
    out["pwa_tile_gather"]["note"] = "fp32 image -> fp32 patches, every patch voxel inside the volume"
    out["pwa_tile_finalize"]["note"] = "acc + wsum read, fp32 logits + uint8 labels written"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--sw", type=int, nargs="+", default=[4, 8])
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sliding_window.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sliding_window.py needs a GPU")
    torch.manual_seed(0)
    conf = pwa_b200.SwinUnetRConfig(training_mode="downstream", use_encoder_prompting=True, use_decoder_prompting=True,
                                    use_checkpoint=False)
    model = pwa_b200.SwinUnetR(conf).to(DEV).eval()
    img = torch.rand((1, 1) + DIMS, generator=torch.Generator().manual_seed(1)).to(DEV)
    n = tile_origins(1, DIMS, ROI, OVERLAP).shape[0]

    def predictor(x):
        return model(x)["downstream"]

    res = {"workload": f"SwinUnetR(feature_size=48) downstream, eval, bf16 autocast; volume 1x1x{DIMS[0]}x{DIMS[1]}x{DIMS[2]}, "
                       f"roi {ROI[0]}^3, overlap {OVERLAP}, {MODE} weighting, {n} patches per volume",
           **gpu_info(), "torch": torch.__version__, "rounds": args.rounds, "sw": {}}
    for sw in args.sw:
        runs = {"graph": lambda: pwa_b200.sliding_window_inference(predictor, img, ROI, sw, OVERLAP, mode=MODE, graph=True),
                "eager": lambda: pwa_b200.sliding_window_inference(predictor, img, ROI, sw, OVERLAP, mode=MODE, graph=False),
                "torch": lambda: torch_loop(predictor, img, sw)}
        times = {k: [] for k in runs}
        outs = {}
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            for k, fn in runs.items():                    # warm-up (and the graph capture)
                outs[k] = fn()
            for _ in range(args.rounds):
                for k, fn in runs.items():
                    t, _ = time_volume(fn)
                    times[k].append(t)
        d_ge = (outs["graph"] - outs["eager"]).abs().max().item()
        d_gt = ((outs["graph"] - outs["torch"]).abs().max() / outs["torch"].abs().max()).item()
        res["sw"][sw] = {k: {"volumes_per_s": round(1 / min(v), 4), "seconds_per_volume": [round(x, 4) for x in v],
                             "patches_per_s": round(n / min(v), 1)} for k, v in times.items()}
        res["sw"][sw]["graph_vs_eager_max_abs_diff"] = d_ge
        res["sw"][sw]["graph_vs_torch_rel_linf"] = d_gt
        res["sw"][sw]["kernels"] = kernel_times(img, sw, outs["graph"].shape[1])
        del outs
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
