"""Cost of deterministic mode (torch.use_deterministic_algorithms(True)) on the headline encoder step, and per sibling.

    python tools/bench_deterministic.py [--rounds 5] [--replays 20] [--out profiles/deterministic_cost.json]

1. Step: the bench.py encoder workload (96^3, B = 4, bf16, dropout 0.1) as a GraphedStep captured with the flag off and one
   captured with it on (the flag is read when the backward is recorded), replayed alternately: `rounds` x `replays` each.
2. Siblings at the enc0 shapes (442 368 tokens of C = 48, attention B = 4, P = 432, 4 heads, I = 64, shifted, dropout 0.1):
   each entry point against its `_det` sibling, CUDA events around 50 eager calls after a warm-up.
Prints one JSON object (GPU name and power limit included) and writes it to --out."""
import argparse
import json
import os
import subprocess
import sys
import types

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
import pwa_b200  # noqa: E402
from pwa_b200 import functional as PF  # noqa: E402
from pwa_b200.graphs import GraphedStep  # noqa: E402

DEV = "cuda:0"


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True).stdout.strip().split("\n")[0]
        name, pl, clk = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": pl, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def events_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def step_cost(rounds, replays):
    args = types.SimpleNamespace(patch=96, dropout=0.1, frozen=False, batch=4)
    graphs = {}
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        wl = bench.EncoderWorkload(torch.device(DEV), args, use_checkpoint=False)
        x0 = torch.randn(wl.in_shape, generator=torch.Generator().manual_seed(1)).to(DEV, torch.bfloat16)
        graphs[det] = (GraphedStep(wl.step, [x0.clone().requires_grad_(True)], wl.params), x0)
    torch.use_deterministic_algorithms(False)
    times = {False: [], True: []}
    for g, x in graphs.values():
        for _ in range(3):
            g(x)
    torch.cuda.synchronize()
    for _ in range(rounds):
        for det in (False, True):
            g, x = graphs[det]
            times[det].append(events_ms(lambda: g(x), replays))
    B = args.batch
    out = {}
    for det, name in ((False, "default"), (True, "deterministic")):
        ms = sorted(times[det])
        out[name] = {"ms_per_step_median": ms[len(ms) // 2], "ms_per_step_all": ms, "patches_per_s": B * 1e3 / ms[len(ms) // 2]}
    out["slowdown"] = out["deterministic"]["ms_per_step_median"] / out["default"]["ms_per_step_median"] - 1.0
    return out


def sibling_costs(reps=50):
    res = {}
    rows, C = 442368, 48
    gen = torch.Generator(device=DEV).manual_seed(0)
    x, dy, dres = (torch.randn(rows, C, generator=gen, device=DEV).bfloat16() for _ in range(3))
    gamma = torch.ones(C, device=DEV)
    mean, rstd = torch.zeros(rows, device=DEV), torch.ones(rows, device=DEV)
    dx = torch.empty_like(x)
    f = [torch.empty(C, device=DEV) for _ in range(4)]
    seed = torch.tensor([1, 2], dtype=torch.int32, device=DEV)
    L, p, st, code = PF._lib.lib, PF._ptr, PF._stream(x), PF._dtype_code(x)

    def ws(n):
        return torch.empty(max(int(n), 1), dtype=torch.uint8, device=DEV)

    w_ln, w_dr, w_cs = (ws(L.pwa_ln_bwd2_det_workspace_size(rows, C, code)), ws(L.pwa_dropout_colsum_det_workspace_size(rows, C, code)),
                        ws(L.pwa_colsum_rows_det_workspace_size(rows, C, code)))
    ln_args = [p(dy), p(x), p(gamma), p(mean), p(rstd), p(dres), p(dx), *[p(t) for t in f], rows, C, code]
    calls = {
        "ln_bwd2": (lambda: L.pwa_ln_bwd2(*ln_args, st), lambda: L.pwa_ln_bwd2_det(*ln_args, p(w_ln), w_ln.numel(), st)),
        "dropout_colsum": (lambda: L.pwa_dropout_colsum(p(dy), p(dx), rows, C, 0.1, p(seed), p(f[0]), code, st),
                           lambda: L.pwa_dropout_colsum_det(p(dy), p(dx), rows, C, 0.1, p(seed), p(f[0]), code, p(w_dr), w_dr.numel(), st)),
        "colsum_rows": (lambda: L.pwa_colsum_rows(p(x), p(f[0]), rows, C, code, st),
                        lambda: L.pwa_colsum_rows_det(p(x), p(f[0]), rows, C, code, p(w_cs), w_cs.numel(), st)),
    }
    for name, (a, d) in calls.items():
        for fn in (a, d):
            for _ in range(3):
                assert fn() == 0, PF._lib.lib.pwa_last_error()
        torch.cuda.synchronize()
        res[name] = {"atomic_us": 1e3 * events_ms(a, reps), "det_us": 1e3 * events_ms(d, reps)}

    from tests.test_gpu_multiwindow import _inputs
    ten, ids, go, heads, _ = _inputs("enc0", True, seed=11, dtype=torch.bfloat16)
    dev = [None if t is None else t.to(DEV).requires_grad_(True) for t in ten]
    out = PF.prompted_window_attention(*dev, torch.from_numpy(ids).to(DEV), heads, bench.WS, 12 ** -0.5, p_drop=0.1,
                                       seed=seed)
    g = go.to(DEV)
    for det in (False, True):
        torch.use_deterministic_algorithms(det)
        for _ in range(3):
            out.backward(g, retain_graph=True)
        torch.cuda.synchronize()
        res.setdefault("attn_bwd", {})["det_us" if det else "atomic_us"] = 1e3 * events_ms(
            lambda: out.backward(g, retain_graph=True), reps)
    torch.use_deterministic_algorithms(False)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "deterministic_cost.json"))
    a = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"what": "encoder step (96^3, B=4, bf16, dropout 0.1, GraphedStep) with torch.use_deterministic_algorithms off / on, "
                   "and each deterministic sibling against its atomic entry point at the enc0 shapes",
           **gpu_info(), "step": step_cost(a.rounds, a.replays), "siblings": sibling_costs()}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
