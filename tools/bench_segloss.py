"""Segmentation losses: the fused Dice / focal kernels against the same loss written as fp32 torch ops, and the config-4 step.

    python tools/bench_segloss.py [--iters 50] [--rounds 3] [--steps 10] [--out profiles/segloss.json]

1. Kernel time of pwa_segloss_fwd (incl. its slot sum) and pwa_segloss_bwd at the two production shapes, bf16 logits and int64
   labels: [8, 2, 96^3] (the config-4 downstream head) and [4, 5, 96^3] (the phase-2 seg_pred head).  CUDA events around
   `iters` back-to-back launches, rotating over input sets that together exceed the 126 MB L2; GB/s against the bytes each call
   must move (forward B nvox (K e + 8), backward B nvox (2 K e + 8), e = 2 bytes).
2. The loss (DiceFocalLoss(to_onehot_y=True, softmax=True), the focal part in its sigmoid form) forward + backward: the fused
   module, and MONAI's formulas written as fp32 torch ops (float one-hot by scatter, softmax, sums; standing in for MONAI,
   which is not installed), each eager and captured as a CUDA graph.
3. The config-4 training step: downstream SwinUnetR(feature_size=48), encoder and decoder prompting, frozen backbone, batch 8,
   96^3, bf16 autocast, dropout 0, one GraphedStep replay per step, with three losses on the `downstream` head: the fused
   DiceFocalLoss, the torch-ops loss, and bench.py's `_MeanSquare` stand-in.  Patches/s from CUDA events over `steps` replays.
All arms run alternately in one process, `rounds` times; the median is reported.  Prints one JSON object (GPU name and power
limit included) and writes it to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import pwa_b200  # noqa: E402
from pwa_b200 import _lib  # noqa: E402
from pwa_b200.functional import _ptr, _stream  # noqa: E402
from pwa_b200.graphs import GraphedStep  # noqa: E402
from pwa_b200.trainer import DiceFocalLoss  # noqa: E402
from pwa_b200.trainer import seg_losses as S  # noqa: E402

DEV = "cuda:0"
SHAPES = [(8, 2), (4, 5)]
SPATIAL = (96, 96, 96)
L2_BYTES = 126e6


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True).stdout.strip().split("\n")[0]
        name, pl, clk = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": pl, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def torch_dice_focal(x, lab, gamma=2.0, smooth=1e-5):
    """DiceFocalLoss(to_onehot_y=True, softmax=True) as MONAI computes it, in fp32 torch ops."""
    xf = x.float()
    y = torch.zeros_like(xf).scatter_(1, lab, 1.0)                 # monai.networks.utils.one_hot
    p = torch.softmax(xf, 1)
    axes = list(range(2, x.dim()))
    inter = torch.sum(y * p, dim=axes)
    den = torch.sum(y, dim=axes) + torch.sum(p, dim=axes)
    dice = (1.0 - (2.0 * inter + smooth) / (den + smooth)).mean()
    loss = xf - xf * y - F.logsigmoid(xf)
    focal = (torch.exp(gamma * F.logsigmoid(-xf * (y * 2 - 1))) * loss).mean()
    return dice + focal


def time_events(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / n          # us per call


def capture(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def kernel_arms(B, K):
    nvox = SPATIAL[0] * SPATIAL[1] * SPATIAL[2]
    fwd_bytes = B * nvox * (K * 2 + 8)
    bwd_bytes = B * nvox * (2 * K * 2 + 8)
    R = max(2, int(3 * L2_BYTES // fwd_bytes) + 1)            # rotating sets: > 3 x L2 together
    gen = torch.Generator().manual_seed(B * 10 + K)
    xs = [torch.randn((B, K, nvox), generator=gen).to(DEV, torch.bfloat16) for _ in range(R)]
    labs = [torch.randint(0, K, (B, nvox), generator=gen).to(DEV) for _ in range(R)]
    mod = DiceFocalLoss(to_onehot_y=True, softmax=True)
    shape = S._shape(B, K, nvox, mod.cfg)
    nbytes = S.segloss_workspace_size(B, K, nvox)
    work = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    sums = torch.empty((4, B, K), device=DEV)
    dsums = torch.randn((4, B, K), device=DEV)
    dls = [torch.empty_like(x) for x in xs]
    st = _stream(xs[0])

    def fwd(i):
        x, lab = xs[i % R], labs[i % R]
        _lib.check(_lib.lib.pwa_segloss_fwd(_ptr(x), _lib.PWA_BF16, _ptr(lab), _lib.PWA_LABEL_I64, shape, _ptr(sums), _ptr(work),
                                            nbytes, st), "fwd")

    def bwd(i):
        x, lab = xs[i % R], labs[i % R]
        _lib.check(_lib.lib.pwa_segloss_bwd(_ptr(x), _lib.PWA_BF16, _ptr(lab), _lib.PWA_LABEL_I64, shape, _ptr(dsums),
                                            _ptr(dls[i % R]), st), "bwd")

    # whole loss forward + backward, [B, K, 96, 96, 96] views of the same sets
    x5 = [x.view((B, K) + SPATIAL).requires_grad_(True) for x in xs]
    l5 = [lab.view((B, 1) + SPATIAL) for lab in labs]
    def loss_fused(i):
        j = i % R
        x5[j].grad = None
        mod(x5[j], l5[j]).backward()

    def loss_torch(i):
        j = i % R
        x5[j].grad = None
        torch_dice_focal(x5[j], l5[j]).backward()

    # captured: one graph per input set, replayed in rotation
    def graphs_of(step):
        gs = []
        for j in range(R):
            gs.append(capture(lambda j=j: step(j)))
        return gs
    g_fused, g_torch = graphs_of(loss_fused), graphs_of(loss_torch)
    arms = {"fused_fwd": (fwd, fwd_bytes), "fused_bwd": (bwd, bwd_bytes), "loss_fused_eager": (loss_fused, None),
            "loss_fused_graph": (lambda i: g_fused[i % R].replay(), None), "loss_torch_eager": (loss_torch, None),
            "loss_torch_graph": (lambda i: g_torch[i % R].replay(), None)}
    return arms, {"B": B, "K": K, "nvox": nvox, "rotating_sets": R, "fwd_bytes": fwd_bytes, "bwd_bytes": bwd_bytes}


def step_arms(steps):
    torch.manual_seed(0)
    conf = pwa_b200.SwinUnetRConfig(training_mode="downstream", use_encoder_prompting=True, use_decoder_prompting=True,
                                    use_checkpoint=False, attn_drop=0.0, proj_drop=0.0)
    model = pwa_b200.SwinUnetR(conf).to(DEV).train()
    params = [p for p in model.parameters() if p.requires_grad]
    B, K = 8, conf.output_channels_downstream
    gen = torch.Generator().manual_seed(1)
    img = torch.rand((B, 1) + SPATIAL, generator=gen).to(DEV)
    mask = torch.randint(0, K, (B, 1) + SPATIAL, generator=gen).to(DEV)
    import bench
    fused = DiceFocalLoss(to_onehot_y=True, softmax=True)
    losses = {"DiceFocalLoss_fused": lambda o, m: fused(o, m), "torch_ops": torch_dice_focal,
              "MeanSquare_standin": lambda o, m: bench._MeanSquare.apply(o)}
    def make(fn):
        def step(x, m):
            with torch.autocast("cuda", dtype=torch.bfloat16):
                out = model(x)["downstream"]
            loss = fn(out, m)
            loss.backward()
            return loss.detach()
        return lambda: GraphedStep(step, [img, mask], params, warmup=2)
    return {name: make(fn) for name, fn in losses.items()}, B


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "segloss.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_segloss.py needs a GPU"
    res = {"device": gpu_info(), "torch": torch.__version__, "iters": args.iters, "rounds": args.rounds, "kernels": []}
    for B, K in SHAPES:
        arms, meta = kernel_arms(B, K)
        for fn, _ in arms.values():
            fn(0)
        torch.cuda.synchronize()
        times = {n: [] for n in arms}
        for _ in range(args.rounds):
            for n, (fn, _) in arms.items():
                times[n].append(time_events(fn, args.iters))
        row = dict(meta)
        for n, (fn, nbytes) in arms.items():
            us = statistics.median(times[n])
            row[n + "_us"] = round(us, 2)
            if nbytes:
                row[n + "_GBps"] = round(nbytes / us / 1e3, 1)
        res["kernels"].append(row)
        del arms
        torch.cuda.empty_cache()
    makers, B = step_arms(args.steps)
    times = {n: [] for n in makers}
    for _ in range(args.rounds):
        for n, make in makers.items():          # one captured step alive at a time (each holds a step's activations)
            gs = make()
            gs(*gs.static_inputs)
            torch.cuda.synchronize()
            times[n].append(time_events(lambda i, gs=gs: gs(*gs.static_inputs), args.steps))
            del gs
            torch.cuda.empty_cache()
    res["config4_step"] = {"batch": B, "patch": list(SPATIAL), "steps": args.steps}
    for n, t in times.items():
        ms = statistics.median(t) / 1e3
        res["config4_step"][n] = {"ms_per_step": round(ms, 3), "patches_per_s": round(B / ms * 1e3, 1),
                                  "all_ms": [round(v / 1e3, 3) for v in t]}
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
