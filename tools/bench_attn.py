"""Kernel-level timing of the fused attention forward / backward and partition / reverse at the BASELINE stage
shapes (CUDA events on the launching stream, inputs larger than L2 or rotated).  Run on the GPU box:
    python tools/bench_attn.py [--what attn,part] [--iters 20]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import pwa_b200  # noqa: E402
from pwa_b200 import functional as PF  # noqa: E402

WS = (8, 8, 4)
STAGES = {  # name: (C, heads, dims)
    "enc0": (48, 4, (48, 48, 48)), "enc1": (96, 8, (24, 24, 24)), "enc2": (192, 16, (12, 12, 24)),
    "dec0": (192, 4, (12, 12, 24)), "dec1": (96, 4, (24, 24, 24)),
}


def timeit(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3  # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--what", default="attn,part")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--stages", default="enc0,enc1,enc2,dec0")
    ap.add_argument("--dropout", type=float, default=0.0)
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp16"], help="element type of the attention kernels")
    args = ap.parse_args()
    adt = torch.bfloat16 if args.dtype == "bf16" else torch.float16
    dev = torch.device("cuda")
    B, I = args.batch, 64
    torch.manual_seed(0)
    for name in args.stages.split(","):
        C, heads, dims = STAGES[name]
        for shifted in (False, True):
            g = pwa_b200.get_geometry(dims, WS, (4, 4, 2) if shifted else (0, 0, 0))
            P, N = g.P, g.N
            if "attn" in args.what:
                qkv = torch.randn(B, P, N, 3 * C, device=dev).to(adt).requires_grad_(True)
                kvp = torch.randn(B, I, 2 * C, device=dev).to(adt).requires_grad_(True)
                th, tw, td = (0.3 * torch.randn(heads, w, w, device=dev) for w in WS)
                tok = 0.3 * torch.randn(heads, I, device=dev)
                ids = g.region_ids(dev) if g.masked else None
                scale = (C // heads) ** -0.5
                seed = torch.tensor([1234, 5678], dtype=torch.int32, device=dev) if args.dropout > 0 else None
                out = PF.prompted_window_attention_packed(qkv, kvp, th, tw, td, tok, ids, heads, WS, scale, PF.IMPL_TC,
                                                          p_drop=args.dropout, seed=seed)
                go = torch.randn_like(out)
                fwd = lambda: PF.prompted_window_attention_packed(qkv, kvp, th, tw, td, tok, ids, heads, WS, scale, PF.IMPL_TC,
                                                                  p_drop=args.dropout, seed=seed)
                t_f = timeit(lambda: fwd(), args.iters)
                t_fb = timeit(lambda: fwd().backward(go), args.iters)
                fl = 4.0 * B * P * N * (N + I) * C
                print(json.dumps({"kernel": "attn", "dtype": args.dtype, "stage": name, "shifted": shifted, "B": B, "P": P, "drop": args.dropout, "fwd_us": round(t_f, 1),
                                  "bwd_us": round(t_fb - t_f, 1), "fwd_tflops": round(fl / t_f / 1e6, 1),
                                  "bwd_tflops": round(2 * fl / max(t_fb - t_f, 1e-3) / 1e6, 1),
                                  "fwd_Gexp_s": round(B * P * heads * N * (N + I) / t_f / 1e3, 1)}))
            if "part" in args.what:
                for dt in (torch.bfloat16, torch.float32):
                    xs = [torch.randn(B, C, *dims, device=dev).to(dt) for _ in range(4)]
                    k = [0]

                    def part():
                        k[0] += 1
                        return PF._partition_raw(xs[k[0] % 4], g, 0)
                    toks = [part() for _ in range(4)]

                    def rev():
                        k[0] += 1
                        return PF._reverse_raw(toks[k[0] % 4], g, 1)
                    nbytes = 2.0 * toks[0].numel() * toks[0].element_size()
                    tp, tr = timeit(part, args.iters), timeit(rev, args.iters)
                    print(json.dumps({"kernel": "partition/reverse", "stage": name, "shifted": shifted, "dtype": str(dt), "B": B,
                                      "MB": round(nbytes / 1e6, 1), "part_us": round(tp, 1), "rev_us": round(tr, 1),
                                      "part_GBs": round(nbytes / tp / 1e3, 1), "rev_GBs": round(nbytes / tr / 1e3, 1)}))


if __name__ == "__main__":
    main()
