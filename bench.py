#!/usr/bin/env python
"""bench.py -- throughput of the prompted 3D shifted-window attention hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload encoder|model] [--mode ssl_encoder|ssl_all|downstream] [--patch 96|128] [--batch B]
                    [--dtype bf16|fp32] [--dropout 0.1] [--checkpoint] [--frozen] [--dump-outputs DIR]

One "step" = forward + backward of the hot path over one batch of synthetic input.
  --workload encoder (default, BASELINE config[1]): the Swin encoder of SwinUNETR(feature_size=48) on 96^3 patches with
      encoder prompting -- three ConsecutiveSwinBlocks stages = 6 prompted window-attention blocks (+ the 3 PatchMerging
      layers that chain them) on the patch-embedded feature map [B, 48, 48, 48, 48], in the reference's training
      configuration attn_drop = proj_drop = 0.1 (configurations/example_configs.yml:18-19).  `use_checkpoint` (a memory
      saving, :17) is measured both ways; the headline runs without it, the other value is in `variants`.
  --workload model: the MONAI-free SwinUnetR host around the blocks, from the raw image [B, 1, R, R, R]:
      --mode ssl_encoder (config[1] with patch embedding and SSL heads), ssl_all (config[2]: encoder + decoder prompting,
      12 prompted blocks), downstream (config[3]: frozen backbone, prompt-token-only gradients); --patch 128 = config[4].
Metric: 3D patches / s, whole job.  Prints ONE JSON line (rank 0).  Under torchrun (N > 1) every rank processes its own
batch shard (weak scaling: fixed per-GPU batch); gradients are all-reduced over NCCL once per step.
--dump-outputs DIR: after the HBM-resident timed steps, rank 0 writes what the last of them returned to its caller (loss,
every trainable parameter's gradient, the input's gradient where the input takes one) as DIR/<name>.npy, 64 MB at most.
Weights, inputs and dropout seeds are seeded, so two builds run with the same arguments can be compared array by array.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WS = (8, 8, 4)
E = 64
I_PROMPT = 64
FEATURE = 48
HEADS_ENC = 4
METRIC = "3D patches/sec fwd+bwd (96^3 SwinUNETR+prompts) at 1/2/4/8 B200; attn TFLOP/s"
UNIT = "patches/s"


def stage_specs(patch=96, feature=FEATURE):
    """(C, heads, dims) of the three encoder stages after the 2x2x2 patch embedding (swin_unetr.py:146-178)."""
    d = patch // 2
    return [(feature, HEADS_ENC, (d, d, d)), (2 * feature, 2 * HEADS_ENC, (d // 2, d // 2, d // 2)),
            (4 * feature, 4 * HEADS_ENC, (d // 4, d // 4, d // 2))]


def decoder_specs(patch=96, feature=FEATURE):
    """(C, heads, dims) of the three decoder stages (unet_blocks.py:57-69, num_heads_decoder = 4)."""
    d = patch // 2
    return [(4 * feature, 4, (d // 4, d // 4, d // 2)), (2 * feature, 4, (d // 2, d // 2, d // 2)), (feature, 4, (d, d, d))]


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sus=1400.0, src="fallback")


# --------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [v.strip() for v in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# our arm: workloads
# --------------------------------------------------------------------------------------------------
class _MeanSquare(torch.autograd.Function):
    """mean(x.float() ** 2), the stand-in loss on every output, as ONE reduction kernel forward and ONE scaling kernel
    backward (the plain torch expression costs nine elementwise passes over every stage output)."""

    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        n = torch.linalg.vector_norm(x, 2, dtype=torch.float32)
        return n * n / x.numel()

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        coef = (g * (2.0 / x.numel())).to(x.dtype)
        return torch._foreach_mul((x,), coef)[0]


class EncoderWorkload:
    """BASELINE config[1] hot path: 3 stages x (2 prompted blocks + PatchMerging) on the patch-embedded map."""

    def __init__(self, dev, args, use_checkpoint):
        import pwa_b200
        torch.manual_seed(0)
        stages, prompts = [], []
        self.specs = stage_specs(args.patch)
        for i, (c, h, _) in enumerate(self.specs):
            stages.append(pwa_b200.ConsecutiveSwinBlocks(hidden_channels=c, num_heads=h, pos_bias_embed_dim=E, max_prompts=1,
                                                         tokens_per_prompt=I_PROMPT, window_size=WS, use_token_params=True,
                                                         down=True, merge_last_dim=(i < 1), use_checkpoint=use_checkpoint,
                                                         attn_drop=args.dropout, proj_drop=args.dropout))
            for _ in range(2):   # prompt_tokens['enc'][2j], [2j+1]  (swin_unetr.py:400-409), xavier-uniform
                prompts.append(torch.nn.Parameter(torch.nn.init.xavier_uniform_(torch.empty(I_PROMPT, c))))
        self.model = torch.nn.ModuleList(stages).to(dev).train()
        self.prompts = torch.nn.ParameterList(prompts).to(dev)
        if args.frozen:          # config[3] on the encoder: only prompt tokens + their bias parameters train
            keep = {id(p) for st in self.model for _, p in st.named_parameters_bias_prompt_tokens()}
            for p in self.model.parameters():
                p.requires_grad_(id(p) in keep)
        named = list(self.model.named_parameters()) + [("prompts." + n, p) for n, p in self.prompts.named_parameters()]
        self.named_params = [(n, p) for n, p in named if p.requires_grad]
        self.params = [p for _, p in self.named_params]
        c0, _, d0 = self.specs[0]
        self.in_shape = (args.batch, c0, *d0)
        self.n_blocks = 6
        self.desc = (f"SwinUNETR(feature_size=48) encoder hot path, {args.patch}^3 patches: 3 ConsecutiveSwinBlocks stages = 6 "
                     f"prompted window-attention blocks (ws 8x8x4, 64 prompt tokens/block) + 3 PatchMerging, fwd+bwd")

    def host_batch(self, gen, dtype):
        return torch.randn(self.in_shape, generator=gen).to(dtype)

    def step(self, x):
        b = x.shape[0]
        loss = 0.0
        ps = [self.prompts[k].to(x.dtype).unsqueeze(0).expand(b, -1, -1) for k in range(2 * len(self.model))]
        for j, stage in enumerate(self.model):      # (what SwinUnetR.forward does at its top: feature-map-independent inputs
            stage.prefetch_side_inputs((ps[2 * j], ps[2 * j + 1]), x)     # of every stage start on the side stream now)
        for j, stage in enumerate(self.model):
            x = stage(x, (ps[2 * j], ps[2 * j + 1]))
            loss = loss + _MeanSquare.apply(x)          # every stage output feeds the decoder / heads in the real model
        loss.backward()
        return loss.detach()


class ModelWorkload:
    """The MONAI-free SwinUnetR host (modules/swin_unetr) from the raw image; bf16 = torch.autocast, as a user runs it."""
    MODES = {"ssl_encoder": ("self_supervised_learning_encoder", True, False, 6),
             "ssl_all": ("self_supervised_learning_all", True, True, 12),
             "downstream": ("downstream", True, True, 12)}

    def __init__(self, dev, args, use_checkpoint):
        import pwa_b200
        mode, enc_p, dec_p, self.n_blocks = self.MODES[args.mode]
        torch.manual_seed(0)
        conf = pwa_b200.SwinUnetRConfig(training_mode=mode, use_encoder_prompting=enc_p, use_decoder_prompting=dec_p,
                                        use_checkpoint=use_checkpoint, attn_drop=args.dropout, proj_drop=args.dropout)
        self.model = pwa_b200.SwinUnetR(conf).to(dev).train()
        self.named_params = [(n, p) for n, p in self.model.named_parameters() if p.requires_grad]
        self.params = [p for _, p in self.named_params]
        self.in_shape = (args.batch, 1, args.patch, args.patch, args.patch)
        self.autocast = args.dtype == "bf16"
        self.desc = (f"SwinUnetR(feature_size=48) {mode}, {args.patch}^3 single-channel patches, encoder"
                     f"{' + decoder' if dec_p else ''} prompting ({self.n_blocks} prompted window-attention blocks), fwd+bwd; "
                     "conv / BatchNorm / upsampling layers of the host are library calls (cuDNN / ATen)")

    def host_batch(self, gen, dtype):
        return torch.rand(self.in_shape, generator=gen)            # CT values scaled to [0, 1) (transforms.py:142-147)

    def step(self, x):
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=self.autocast):
            out = self.model(x.float())
        loss = 0.0
        for k, t in out.items():
            for u in (t if isinstance(t, list) else [t]):
                if u.requires_grad:
                    loss = loss + _MeanSquare.apply(u)
        loss.backward()
        return loss.detach()


def algorithmic_attn_flops(args, batch):
    """Per step: attention FLOPs 12*B*P*N*N'*C fwd+bwd over every prompted block (SURVEY §8d)."""
    import pwa_b200
    n = WS[0] * WS[1] * WS[2]
    specs = list(stage_specs(args.patch))
    if args.workload == "model" and args.mode != "ssl_encoder":
        specs += decoder_specs(args.patch)
    flops = 0.0
    for c, h, dims in specs:
        g = pwa_b200.get_geometry(dims, WS, (0, 0, 0))
        flops += 2 * 12.0 * batch * g.P * n * (n + I_PROMPT) * c
    return flops


# --------------------------------------------------------------------------------------------------
# per-kernel device times: each kernel class captured as a CUDA graph of back-to-back launches (rotating inputs)
# --------------------------------------------------------------------------------------------------
def _graph_time(fn, reps, rounds=3):
    """us per call of fn(i), `reps` calls captured into one CUDA graph, best of `rounds` replays."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for i in range(3):
            fn(i)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(reps):
            fn(i)
    g.replay()
    torch.cuda.synchronize()
    best = 1e30
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) * 1e3 / reps)
    return best


def kernel_microbench(args, dev, dtype):
    """Device time of every hot-path kernel class at the step's own shapes (launch-gap free: graph replays), and the
    step's attention launches one by one.  Returns ({class: {...}}, [(name, flops, us)] per attention launch of a step)."""
    import pwa_b200
    from pwa_b200 import functional as PF
    B, I = args.batch, I_PROMPT
    specs = list(stage_specs(args.patch))
    if args.workload == "model" and args.mode != "ssl_encoder":
        specs += decoder_specs(args.patch)
    out, attn_launches = {}, []
    n = WS[0] * WS[1] * WS[2]
    R = 3                                                   # rotating input sets (beyond L2 together)
    for si, (C, heads, dims) in enumerate(specs):
        for shifted in (False, True):
            g = pwa_b200.get_geometry(dims, WS, (4, 4, 2) if shifted else (0, 0, 0))
            P = g.P
            qkv = [torch.randn(B, P, n, 3 * C, device=dev).to(dtype).requires_grad_(True) for _ in range(R)]
            kvp = torch.randn(B, I, 2 * C, device=dev).to(dtype).requires_grad_(True)
            th, tw, td = (0.3 * torch.randn(heads, w, w, device=dev) for w in WS)
            tok = 0.3 * torch.randn(heads, I, device=dev)
            ids = g.region_ids(dev) if g.masked else None
            scale = (C // heads) ** -0.5
            seed = PF.new_dropout_seed(dev) if args.dropout > 0 else None
            go = torch.randn(B, P, n, C, device=dev).to(dtype)
            fwd = lambda i: PF.prompted_window_attention_packed(qkv[i % R], kvp, th, tw, td, tok, ids, heads, WS, scale,
                                                                PF.IMPL_AUTO, p_drop=args.dropout, seed=seed)

            def fwdbwd(i):
                fwd(i).backward(go)
            t_f = _graph_time(fwd, 6)
            t_fb = _graph_time(fwdbwd, 6)
            fl = 4.0 * B * P * n * (n + I) * C
            tag = f"stage{si}{'s' if shifted else 'u'}"
            attn_launches.append(("attn_fwd", tag, fl, t_f))
            attn_launches.append(("attn_bwd", tag, 2 * fl, max(t_fb - t_f, 1e-3)))
            del qkv, go
    # memory-bound classes at the first stage's shape (the step's largest)
    C, heads, dims = specs[0]
    g0 = pwa_b200.get_geometry(dims, WS, (0, 0, 0))
    g1 = pwa_b200.get_geometry(dims, WS, (4, 4, 2))
    from pwa_b200.geometry import rowmap_regroup
    xs = [torch.randn(B, C, *dims, device=dev).to(dtype) for _ in range(R)]
    toks = [PF._partition_raw(x, g1, 0) for x in xs]
    es = xs[0].element_size()
    nb = 2.0 * toks[0].numel() * es
    res = {}
    res["partition"] = (nb, _graph_time(lambda i: PF._partition_raw(xs[i % R], g1, 0), 10))
    res["reverse"] = (nb, _graph_time(lambda i: PF._reverse_raw(toks[i % R], g1, 1), 10))
    rm = rowmap_regroup(g0, g1)
    fwd_map, _ = rm.on(dev)
    flat = [t.view(B, -1, C) for t in toks]
    res["gather_rows"] = (nb, _graph_time(lambda i: PF._gather_rows_raw(flat[i % R], None, fwd_map, rm.rows_src, rm.rows_dst), 10))
    gamma, beta = torch.ones(C, device=dev), torch.zeros(C, device=dev)
    with torch.no_grad():
        res["ln_fwd"] = (nb, _graph_time(lambda i: PF.layer_norm(toks[i % R], gamma, beta, 1e-6), 10))
    for name, (bytes_, us) in res.items():
        out[name] = {"shape": f"stage0 B={B}", "us": round(us, 2), "GB/s": round(bytes_ / us / 1e3, 1)}
    return out, attn_launches


DUMP_BYTES = 60 << 20                       # array data; the .npy headers fit in the rest of the 64 MB


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """Writes {name: tensor} as out_dir/<name>.npy in float32 (float64 stays float64).  Taken smallest first, an array is
    written whole when it fits an even share of the budget still left; a larger one becomes a 1-D sample of that many
    elements at sorted random flat indices from a fixed seed, so every run with the same shapes stores the same elements."""
    os.makedirs(out_dir, exist_ok=True)
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel())
    left = budget
    for i, (name, t) in enumerate(items):
        t = t.detach().cpu()
        t = t.double() if t.dtype == torch.float64 else t.float()
        share = left // (len(items) - i) // t.element_size()
        if t.numel() > share:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:share].sort().values
            t = t.reshape(-1)[idx]
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())
        left -= t.numel() * t.element_size()


def run_ours(args):
    import torch.distributed as dist
    import pwa_b200
    from pwa_b200.functional import KernelStats
    from pwa_b200.graphs import GraphedStep, InputPrefetcher

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:
        emit(json.dumps({"error": "launch with torchrun for --gpus > 1"}))
        return 2
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    B = args.batch
    Workload = EncoderWorkload if args.workload == "encoder" else ModelWorkload

    def build(use_checkpoint, policy=None):
        wl = Workload(dev, args, use_checkpoint)
        if policy is not None:             # 'selective' (default) | 'full': see SwinTransformerBlock._tokens_forward_ckpt
            for m in wl.model.modules():
                if hasattr(m, "checkpoint_policy"):
                    m.checkpoint_policy = policy
        in_dtype = dtype if args.workload == "encoder" else torch.float32
        x0 = torch.zeros(wl.in_shape, dtype=in_dtype, device=dev)
        graphed = None
        if not args.no_graph:
            graphed = GraphedStep(wl.step, [x0.clone().requires_grad_(args.workload == "encoder")], wl.params, flat_grads=world > 1)
        return wl, graphed, in_dtype

    wl, graphed, in_dtype = build(args.checkpoint)
    gen = torch.Generator().manual_seed(1234 + rank)
    # several distinct pinned host batches; every step's working set (inputs + saved activations, > 1 GB) is far larger
    # than the 126 MB L2, so no explicit flush is needed between timed iterations
    host = [wl.host_batch(gen, in_dtype).pin_memory() for _ in range(2)]
    xdev = [h.to(dev) for h in host]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}                                         # what the latest step handed back: its loss and input gradient

    def run_step(w, gr, x_src):
        if gr is not None:
            loss = gr(x_src)                          # copy into the static input (H2D or D2D) + one graph launch
            if world > 1:
                gr.allreduce_flat()                   # ONE in-place NCCL all-reduce of the flat gradient buffer
            last.update(loss=loss, input_grad=gr.input_grads[0])
        else:
            for p in w.params:
                p.grad = None
            x = x_src.to(dev, non_blocking=True).clone().requires_grad_(args.workload == "encoder")
            loss = w.step(x)
            if world > 1:
                grads = [p.grad for p in w.params if p.grad is not None]
                flat = torch.cat([g.reshape(-1) for g in grads])
                dist.all_reduce(flat)
                flat.div_(world)
            last.update(loss=loss, input_grad=x.grad)
        return loss

    def timed(w, gr, steps, warmup, count=False):
        for i in range(warmup):
            run_step(w, gr, xdev[i % len(xdev)])
        barrier()
        if count:                                   # gpu_launches: kernels of the K timed steps only, not of the warm-up
            KernelStats.reset(enabled=True, timing=False)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(steps):
            run_step(w, gr, xdev[i % len(xdev)])
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    # ---- timed region 1: inputs resident in HBM ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    KernelStats.reset(enabled=True, timing=False)
    if args.cuda_profiler_range:
        for i in range(args.warmup):
            run_step(wl, graphed, xdev[i % len(xdev)])
        barrier()
        torch.cuda.profiler.start()
        ms = timed(wl, graphed, args.steps, 0, count=True)
        torch.cuda.profiler.stop()
    else:
        ms = timed(wl, graphed, args.steps, args.warmup, count=True)
    launches = KernelStats.launches
    KernelStats.reset(enabled=False)
    if args.dump_outputs and rank == 0:
        outs = {"loss": last["loss"]}
        if last["input_grad"] is not None:
            outs["input_grad"] = last["input_grad"]
        for n, p in wl.named_params:                 # (a parameter the step never reaches has no gradient: zeros)
            outs["grad." + n] = p.grad if p.grad is not None else torch.zeros_like(p)
        dump_outputs(args.dump_outputs, outs)

    # ---- timed region 2: end to end through the public module API with host buffers ----
    feeder = InputPrefetcher(xdev[0], dev)
    loss_host = torch.empty(2, dtype=torch.float32).pin_memory()
    loss_events = [torch.cuda.Event(), torch.cuda.Event()]

    def run_e2e(n):
        """n steps from pinned host batches: the H2D copy of step i+1 runs on a side stream while step i computes.  The
        loss of EVERY step is read on the host, one step late (as a training loop logs it); the last one is read before
        the function returns (inside the timed region)."""
        feeder.prefetch(host[0])
        total = 0.0
        for i in range(n):
            x = feeder.get()
            if i + 1 < n:
                feeder.prefetch(host[(i + 1) % len(host)])
            loss = run_step(wl, graphed, x)
            loss_host[i % 2:i % 2 + 1].copy_(loss.reshape(1), non_blocking=True)
            loss_events[i % 2].record()
            if i > 0:
                loss_events[(i - 1) % 2].synchronize()
                total += float(loss_host[(i - 1) % 2])
        loss_events[(n - 1) % 2].synchronize()
        total += float(loss_host[(n - 1) % 2])
        return total

    run_e2e(min(2, args.warmup))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    run_e2e(args.steps)
    e1.record()
    barrier()
    ms_e2e = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    clocks = sampler.stop() if rank == 0 else None

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()

    # ---- the other use_checkpoint setting (reference example config: use_checkpoint true), same run, fewer steps ----
    variants = {}
    if not args.no_variants and not args.no_graph:
        del graphed, wl
        torch.cuda.empty_cache()
        wl2, gr2, _ = build(not args.checkpoint)
        ms2 = timed(wl2, gr2, args.steps, args.warmup)
        t2 = torch.tensor([ms2], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        ms2 = t2.item()
        variants[f"use_checkpoint_{str(not args.checkpoint).lower()}"] = {
            "value": round(B * world * args.steps / (ms2 / 1e3), 3), "ms_per_step": round(ms2 / args.steps, 3)}
        if not args.checkpoint:
            variants["use_checkpoint_true"]["policy"] = ("selective: token segments recomputed, attention results kept "
                                                         "(the default of use_checkpoint=True here)")
        del gr2, wl2
        torch.cuda.empty_cache()
        if not args.checkpoint and world == 1:
            # whole-block recomputation, attention included: what torch.utils.checkpoint around forward_attn_mlp does in
            # the reference (swin_block.py:257-260)
            wl3, gr3, _ = build(True, "full")
            ms3 = timed(wl3, gr3, args.steps, args.warmup)
            variants["use_checkpoint_true_full_recompute"] = {
                "value": round(B * args.steps / (ms3 / 1e3), 3), "ms_per_step": round(ms3 / args.steps, 3)}
            del gr3, wl3
            torch.cuda.empty_cache()

    kern, attn_launches = {}, []
    if rank == 0 and not args.no_kernels and args.dtype == "bf16":
        kern, attn_launches = kernel_microbench(args, dev, dtype)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_sample(args)

    if rank == 0:
        pk = peaks()
        value = B * world * args.steps / (ms / 1e3)
        e2e_v = B * world * args.steps / (ms_e2e / 1e3)
        roof = None
        if attn_launches:
            # dominant kernel = the attention backward: algorithmic FLOPs of its launches in one step / their device time
            by = {}
            for name, tag, fl, us in attn_launches:
                a = by.setdefault(name, [0.0, 0.0, 0])
                a[0] += fl
                a[1] += us
                a[2] += 1
            for name, (fl, us, cnt) in by.items():
                kern[name] = {"launches_per_step": cnt, "us_per_step": round(us, 1), "TFLOP/s": round(fl / us / 1e6, 2),
                              "frac_of_peak": round(fl / us / 1e6 / pk["tf_sus"], 4),
                              "per_launch_us": {tag: round(u, 1) for n2, tag, _, u in attn_launches if n2 == name}}
            dom = max(by.items(), key=lambda kv: kv[1][1])
            name, (fl, us, cnt) = dom
            try:
                traffic_tab = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
            except Exception:
                traffic_tab = {}
            ach = fl / us / 1e6
            roof = {"kernel": name, "bound": "tensor", "achieved": round(ach, 3), "peak": pk["tf_sus"], "unit": "TFLOP/s",
                    "frac": round(ach / pk["tf_sus"], 5), "traffic": traffic_tab.get(name, {}).get("bytes"),
                    "traffic_of": traffic_tab.get(name, {}).get("launch"),
                    "peak_source": pk["src"] + " (sustained bf16 cuBLAS)", "avg_launch_ms": round(us / cnt / 1e3, 4),
                    "share_of_step": round(us / 1e3 / (ms / args.steps), 4),
                    "timed": "CUDA events around graph replays of back-to-back launches at the step's shapes (rotating inputs)",
                    "note": "at head_dim 12 the softmax exponentials (MUFU, 16/clk/SM), not the tensor pipe, bound this path: "
                            "see DESIGN.md"}
        line = {
            "metric": METRIC, "value": round(value, 4), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": f"{wl_desc(args)}; batch {B}/GPU, {args.dtype}; random-init weights",
                       "per_gpu_batch": B, "global_batch": B * world, "patch": args.patch, "parallelism": f"dp{world}",
                       "l2": "per-step working set (>1 GB of activations) exceeds the 126 MB L2; inputs rotate",
                       "launch": "eager" if args.no_graph else "whole step (fwd+loss+bwd) replayed as one CUDA graph",
                       "attn_drop": args.dropout, "proj_drop": args.dropout, "use_checkpoint": bool(args.checkpoint),
                       "frozen_backbone": bool(args.frozen or (args.workload == "model" and args.mode == "downstream"))},
            "e2e": {"value": round(e2e_v, 4), "unit": UNIT,
                    "h2d_bytes_per_step": host[0].numel() * host[0].element_size(), "d2h_bytes_per_step": 4},
            "gpu_launches": launches, "variants": variants,
            "attn_tflops": round(algorithmic_attn_flops(args, B * world) * args.steps / (ms / 1e3) / 1e12, 3),
            "roofline": roof, "kernels": kern, "clocks": clocks, "cpu_baseline": cpu,
        }
        emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def wl_desc(args):
    if args.workload == "encoder":
        return (f"SwinUNETR(feature_size=48) encoder hot path, {args.patch}^3 patches: 3 ConsecutiveSwinBlocks stages = 6 prompted "
                f"window-attention blocks (ws 8x8x4, 64 prompt tokens/block) + 3 PatchMerging, fwd+bwd"
                + (", frozen backbone (prompt-token-only gradients)" if args.frozen else ""))
    mode, _, dec_p, nb = ModelWorkload.MODES[args.mode]
    return (f"SwinUnetR(feature_size=48) {mode} from the raw {args.patch}^3 single-channel image, {nb} prompted "
            f"window-attention blocks, fwd+bwd (conv / norm / upsampling layers of the host = cuDNN / ATen)")


# --------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the reference's algorithm for this path on the host cores.  Nothing of the product is
# imported here: parameters come from oracle/model_init.py (plain torch initialisers), compute is oracle/restatement.py.
# --------------------------------------------------------------------------------------------------
def _oracle_encoder(args, threads):
    from oracle import restatement as R
    from oracle import model_init
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    specs = stage_specs(args.patch)
    sds, prompts = [], []
    for i, (c, h, _) in enumerate(specs):
        sd = model_init.pair_state_dict(c, h, E, I_PROMPT, WS, down=True, merge_last_dim=(i < 1))
        sds.append({k: v.requires_grad_(v.is_floating_point()) for k, v in sd.items()})
        prompts += [torch.nn.init.xavier_uniform_(torch.empty(I_PROMPT, c)).requires_grad_(True) for _ in range(2)]

    def step(x):
        loss = 0.0
        for j, (c, h, _) in enumerate(specs):
            pw = prompts[2 * j].unsqueeze(0).repeat(x.shape[0], 1, 1)
            ps = prompts[2 * j + 1].unsqueeze(0).repeat(x.shape[0], 1, 1)
            x = R.pair_forward(sds[j], x, (pw, ps), WS, h, True, j < 1, attn_drop=args.dropout, proj_drop=args.dropout)
            loss = loss + x.square().mean()
        loss.backward()
        return float(loss.detach())
    return step


def cpu_baseline_sample(args, steps=8, warmup=1, batch=1):
    threads = os.cpu_count() or 1
    step = _oracle_encoder(args, threads)
    c0, _, d0 = stage_specs(args.patch)[0]
    gen = torch.Generator().manual_seed(1234)
    x = torch.randn(batch, c0, *d0, generator=gen)
    for _ in range(warmup):
        step(x.clone().requires_grad_(True))
    t0 = time.perf_counter()
    for _ in range(steps):
        step(x.clone().requires_grad_(True))
    dt = time.perf_counter() - t0
    return {"value": round(batch * steps / dt, 5), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{steps} step(s) of the same 6-block encoder workload ({args.patch}^3, attn_drop = proj_drop = {args.dropout}) at "
                      f"batch {batch}, fp32, oracle restatement (torch CPU, {threads} threads), {dt:.1f} s"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps, warmup = args.steps, max(1, min(args.warmup, 1))
    cpu = cpu_baseline_sample(args, steps=steps, warmup=warmup, batch=1)
    line = {
        "impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": round(1e3 / cpu["value"], 1), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": f"same 6-block SwinUNETR encoder hot path, {args.patch}^3, fwd+bwd, attn_drop = proj_drop = "
                               f"{args.dropout}; reference algorithm on the host CPU (oracle port, batch 1 per step)",
                   "per_gpu_batch": 1, "patch": args.patch, "attn_drop": args.dropout, "proj_drop": args.dropout},
        "cpu_baseline": cpu,
        "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(json.dumps(line))
    return 0


_JSON_FD = None


def _claim_stdout():
    """stdout carries exactly ONE JSON line.  Libraries print there too (NCCL's version banner, through C stdio, whatever
    NCCL_DEBUG_FILE says), so file descriptor 1 is pointed at stderr for the whole run and the result line is written
    to a private duplicate of the original stdout."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: str):
    if _JSON_FD is None:
        print(line, flush=True)
    else:
        os.write(_JSON_FD, (line + "\n").encode())


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 20; 5 for --impl reference, whose steps take seconds)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="encoder", choices=["encoder", "model"])
    ap.add_argument("--mode", default="ssl_encoder", choices=list(ModelWorkload.MODES))
    ap.add_argument("--patch", type=int, default=96, choices=[64, 96, 128])
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=4, help="per-GPU batch (BASELINE config[1]: 4)")
    ap.add_argument("--dropout", type=float, default=0.1,
                    help="attn_drop = proj_drop of the blocks; default = the reference's training config (example_configs.yml:18-19)")
    ap.add_argument("--checkpoint", action="store_true",
                    help="use_checkpoint=True for the headline value (the other setting is measured into `variants` either way)")
    ap.add_argument("--frozen", action="store_true", help="encoder workload with a frozen backbone (config[3])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--no-kernels", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying a CUDA graph")
    ap.add_argument("--cuda-profiler-range", action="store_true",
                    help="bracket the HBM-resident timed region with cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and gradients of the last HBM-resident timed step as DIR/<name>.npy (64 MB at most)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 5 if args.impl == "reference" else 20
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what --impl ours computes")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
