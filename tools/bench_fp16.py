"""fp16 against bf16 on the B200, in one process, alternating: the bench.py headline workload (EncoderWorkload: 3 encoder
stages of SwinUNETR(feature_size=48), 96^3 patches, B = 4, dropout 0.1, GraphedStep replays) with bf16 and with fp16
inputs, and the whole SwinUnetR cfg2 model (ssl_encoder, raw image in) under torch.autocast(bfloat16) and
torch.autocast(float16).  Also counts, on the encoder's real activations, how many (window, head) units of each stage take
the exact-row-maximum sweep of the tcgen05 forward under the bf16 rule (norm bound > 80 binades loose) and the fp16 rule
(> 24).  Prints one JSON object (GPU name and power limit included) and writes it to --out.

    python tools/bench_fp16.py --out profiles/bench_fp16.json
"""
import argparse
import json
import os
import subprocess
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import pwa_b200  # noqa: E402
from pwa_b200 import functional as PF  # noqa: E402
from pwa_b200.graphs import GraphedStep  # noqa: E402
from oracle import restatement as R  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=20).stdout.strip().split("\n")[0]
        name, pl, clk = [v.strip() for v in q.split(",")]
        return {"gpu": name, "power_limit": pl, "sm_max_clock": clk}
    except Exception as e:                      # (the name from torch still identifies the card)
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def time_replays(fn, x, n):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(n):
        fn(x)
    end.record()
    torch.cuda.synchronize()
    return start.elapsed_time(end) / n


def sweep_census(wl, x):
    """One eager step with the attention call wrapped: per stage, the share of (sample, window, head) units whose norm bound
    is looser than the bf16 / fp16 thresholds of the tcgen05 forward (restated from attn_tc_ws.cu in torch)."""
    out, real = {}, PF.prompted_window_attention_packed

    def spy(qkv, kvp, th, tw, td, tok, ids, heads, ws, scale, impl, p_drop=0.0, seed=None):
        with torch.no_grad():
            B, P, N, C3 = qkv.shape
            C, dh = C3 // 3, C3 // 3 // heads
            q = qkv[..., :C].float().view(B, P, N, heads, dh)
            k = qkv[..., C:2 * C].float().view(B, P, N, heads, dh)
            kp = kvp[..., :C].float().view(B, 1, -1, heads, dh).expand(B, P, -1, heads, dh)
            kmax = torch.cat([k, kp], 2).norm(dim=-1).amax(2)                              # [B, P, h]
            qn = q.norm(dim=-1)                                                            # [B, P, N, h]
            bias = R.dense_bias(th.double(), tw.double(), td.double(), tok.double()).float()   # [h, N, N + I]
            rb = (bias.amax(-1) / scale).t()                                               # [N, h]
            c2 = scale * 1.4426950408889634
            qk = qn * kmax[:, :, None, :]
            mbt = c2 * 1.01 * (qk + rb.clamp(min=0))
            gap_b = mbt - c2 * (rb - qk)
            gap_h = mbt - c2 * ((rb - qk).clamp(max=0) if ids is not None else rb - qk)
            key = f"C{C}_{'shift' if ids is not None else 'noshift'}"
            out[key] = {"bf16_sweep": float((gap_b > 80).any(2).float().mean()),
                        "fp16_sweep": float((gap_h > 24).any(2).float().mean()),
                        "median_gap_binades": float(gap_h.median())}
        return real(qkv, kvp, th, tw, td, tok, ids, heads, ws, scale, impl, p_drop=p_drop, seed=seed)

    PF.prompted_window_attention_packed = spy
    try:
        wl.step(x.clone().requires_grad_(True))
    finally:
        PF.prompted_window_attention_packed = real
    for p in wl.params:
        p.grad = None
    return out


class _ModelStep:
    def __init__(self, wl, dtype):
        self.wl, self.dtype = wl, dtype

    def __call__(self, x):
        with torch.autocast("cuda", dtype=self.dtype):
            out = self.wl.model(x.float())
        loss = 0.0
        for _, t in out.items():
            for u in (t if isinstance(t, list) else [t]):
                if u.requires_grad:
                    loss = loss + bench._MeanSquare.apply(u)
        loss.backward()
        return loss.detach()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed replays per round and dtype")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--model-batch", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    res = {"what": "EncoderWorkload 96^3 B=%d dropout 0.1 GraphedStep, bf16 vs fp16 inputs; SwinUnetR cfg2 autocast bf16 vs "
                   "fp16" % args.batch, **gpu_info(), "torch": torch.__version__}

    # ---- encoder headline workload ----
    wargs = types.SimpleNamespace(patch=96, batch=args.batch, dropout=0.1, frozen=False)
    gen = torch.Generator().manual_seed(1234)
    runs = {}
    for name, dt in (("bf16", torch.bfloat16), ("fp16", torch.float16)):
        wl = bench.EncoderWorkload(dev, wargs, use_checkpoint=False)
        x = wl.host_batch(gen, dt).to(dev)
        if name == "fp16":
            res["sweep_census"] = sweep_census(wl, x)
        g = GraphedStep(wl.step, [x.clone().requires_grad_(True)], wl.params)
        time_replays(g, x, 3)
        runs[name] = (g, x, [])
    for _ in range(args.rounds):
        for name in ("bf16", "fp16"):
            g, x, ts = runs[name]
            ts.append(time_replays(g, x, args.steps))
    enc = {}
    for name, (_, _, ts) in runs.items():
        ms = sorted(ts)[len(ts) // 2]
        enc[name] = {"step_ms_median": round(ms, 3), "step_ms_all": [round(t, 3) for t in ts],
                     "patches_per_s": round(args.batch / ms * 1e3, 1)}
    enc["fp16_over_bf16"] = round(enc["fp16"]["patches_per_s"] / enc["bf16"]["patches_per_s"], 4)
    res["encoder"] = enc
    del runs
    torch.cuda.empty_cache()

    # ---- whole model cfg2 under autocast ----
    margs = types.SimpleNamespace(mode="ssl_encoder", dropout=0.1, dtype="bf16", batch=args.model_batch, patch=96)
    mruns = {}
    for name, dt in (("autocast_bf16", torch.bfloat16), ("autocast_fp16", torch.float16)):
        wl = bench.ModelWorkload(dev, margs, use_checkpoint=False)
        x = wl.host_batch(gen, torch.float32).to(dev)
        g = GraphedStep(_ModelStep(wl, dt), [x], wl.params)
        time_replays(g, x, 3)
        mruns[name] = (g, x, [])
    for _ in range(args.rounds):
        for name in mruns:
            g, x, ts = mruns[name]
            ts.append(time_replays(g, x, max(1, args.steps // 2)))
    mod = {}
    for name, (_, _, ts) in mruns.items():
        ms = sorted(ts)[len(ts) // 2]
        mod[name] = {"step_ms_median": round(ms, 3), "step_ms_all": [round(t, 3) for t in ts],
                     "patches_per_s": round(args.model_batch / ms * 1e3, 1)}
    mod["fp16_over_bf16"] = round(mod["autocast_fp16"]["patches_per_s"] / mod["autocast_bf16"]["patches_per_s"], 4)
    res["model_cfg2"] = mod
    s = json.dumps(res)
    print(s)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
