"""The benchmarked training step (bench.EncoderWorkload.step replayed through GraphedStep) against the float64 oracle.

What only the composed, captured step does, and what this file holds to oracle/restatement.py:
  - side inputs (bias tables, packed weights, prompt K|V, the four dropout seed words of each block) prefetched on a side
    stream under capture and claimed by the forward;
  - both projection-dropout paths in one step: the fused dropout + residual + LayerNorm GEMM at C = 48 and project_out ->
    seeded_dropout at C = 96 / 192, and the attention dropout of every block;
  - activation checkpointing under both policies, flat gradient buffers, a frozen backbone, fp32, 128^3 patches;
  - replays after optimizer updates of the parameters.

The seed words are caught where they are drawn: pwa_b200.functional.new_dropout_seed is wrapped while the step is
captured, and the tensors it returned are static outputs of the graph, so after each replay they hold that replay's words.
The oracle (R.pair_forward per stage, float64 torch ops on the GPU, none of the kernels) gets float64 copies of the fp32
master parameters and prompts, the exact input and the masks restated from those words (R.block_keep_factors).

Two comparisons:
  literal -- the replay of bench's own step: loss, input gradient, every parameter and prompt gradient against the
             oracle of the whole chain, loss = sum of mean(y_j^2) over the stage outputs;
  staged  -- the same step with each stage's input and output kept, and tensor hooks on an identity view of each stage
             input and on each stage output (module hooks would switch the stages off their token pipeline).  Each stage
             is checked on its own from the kernels' stage input and upstream gradient: output, input gradient, parameter
             and prompt gradients.  Errors then do not compound over six blocks, and a failure names the stage.
Metric: normalised L-inf (tests/util.rel_linf).  Bounds per (dtype, comparison, stage, tensor group): 1.5x the worst error
measured over input seeds 1, 2 and 3 on a B200 (1000 W power limit), rounded up to two digits (BOUNDS).  Every bound is shown able to fail: the
same comparison against the oracle given the previous replay's seed words (dropout cases), or the parameters before the
last optimizer update (training case), misses its bounds by at least NEG_MARGIN."""
import time
import types
from typing import NamedTuple, Optional

import pytest
import torch

import bench
from pwa_b200 import functional as PF
from pwa_b200.graphs import GraphedStep
from oracle import restatement as R
from tests.util import rel_linf

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
F64 = torch.float64
NEG_MARGIN = 5.0
# Adam: the first updates move every element by about lr, so every parameter tensor by about lr / max|p| (LayerNorm gains
# are ~1: 1.5 %).  Larger rates blow the loss up (0.05: x500 in two updates) and with it the bf16 errors
TRAIN_LR = 0.02
GRAPH_WARMUP = 3           # GraphedStep's default, as bench.py builds it


class Case(NamedTuple):
    name: str
    mode: str                       # 'literal' | 'staged' | 'train' (literal comparison after two optimizer updates)
    batch: int = 2
    patch: int = 96
    dropout: float = 0.1
    ckpt: Optional[str] = None      # None: use_checkpoint=False; else the checkpoint_policy of every module
    frozen: bool = False
    flat: bool = False
    dtype: str = "bf16"
    seed: int = 1                   # input batch


CASES = [
    Case("headline", "literal"),
    Case("headline_staged", "staged"),
    Case("headline_b4", "literal", batch=4),
    Case("ckpt_selective", "staged", ckpt="selective"),
    Case("ckpt_full", "staged", ckpt="full"),
    Case("no_dropout", "staged", dropout=0.0),
    Case("frozen", "literal", frozen=True),
    Case("flat_grads", "literal", flat=True),
    Case("fp32", "staged", dtype="fp32"),
    Case("patch128_b1", "literal", batch=1, patch=128),
    Case("train", "train"),
]

# (dtype, comparison) -> tensor group -> bound.  Groups: loss, dx (input gradient), s<j>.out / s<j>.dx (stage j output /
# input gradient), s<j>.param / s<j>.prompt (the worst parameter / prompt-token gradient of stage j).
BOUNDS = {
    ("bf16", "literal"): {"loss": 2.4e-5, "dx": 2.4e-2, "s0.param": 2.2e-2, "s1.param": 2.2e-2, "s2.param": 2.1e-2,
                          "s0.prompt": 1.7e-2, "s1.prompt": 1.6e-2, "s2.prompt": 1.7e-2},
    ("bf16", "staged"): {"s0.out": 8.8e-3, "s0.dx": 1.4e-2, "s0.param": 1.6e-2, "s0.prompt": 1.3e-2,
                         "s1.out": 8.7e-3, "s1.dx": 1.5e-2, "s1.param": 1.6e-2, "s1.prompt": 1.3e-2,
                         "s2.out": 9.1e-3, "s2.dx": 1.3e-2, "s2.param": 1.8e-2, "s2.prompt": 1.4e-2},
    ("fp32", "staged"): {"s0.out": 1.5e-6, "s0.dx": 6.0e-7, "s0.param": 2.2e-6, "s0.prompt": 6.2e-7,
                         "s1.out": 1.4e-6, "s1.dx": 7.3e-7, "s1.param": 2.0e-6, "s1.prompt": 7.0e-7,
                         "s2.out": 1.9e-6, "s2.dx": 1.1e-6, "s2.param": 2.2e-6, "s2.prompt": 8.2e-7},
    # after two updates (literal comparison): larger activations, larger bf16 errors
    ("bf16", "train"): {"loss": 7.6e-4, "dx": 1.9e-2, "s0.param": 1.6e-2, "s1.param": 2.6e-2, "s2.param": 2.6e-2,
                        "s0.prompt": 1.6e-2, "s1.prompt": 3.1e-2, "s2.prompt": 3.2e-2},
}


def _group(name):
    head, _, tail = name.partition(".")
    if name in ("loss", "dx"):
        return name
    if head == "prompts":
        return f"s{int(tail) // 2}.prompt"
    return f"s{head}.{tail}" if tail in ("out", "dx") else f"s{head}.param"


def _bounds(case):
    return BOUNDS[(case.dtype, case.mode)]


# ---- the step ------------------------------------------------------------------------------------------------------------
class _Record:
    """What the staged step keeps of the captured replay: stage inputs / outputs and the gradients reaching them."""

    def __init__(self, n):
        self.ins, self.outs, self.din, self.dout = [None] * n, [None] * n, [None] * n, [None] * n


def _staged_step(wl, rec):
    """bench.EncoderWorkload.step plus: an identity view at each stage input with a hook recording its gradient (the
    stage's input gradient), and a hook on each stage output (the total upstream gradient the stage's backward consumed:
    next stage + this stage's loss term)."""
    def put(lst, j):
        def hook(g):
            lst[j] = g.detach().clone()
        return hook

    def step(x):
        b = x.shape[0]
        loss = 0.0
        ps = [wl.prompts[k].to(x.dtype).unsqueeze(0).expand(b, -1, -1) for k in range(2 * len(wl.model))]
        for j, stage in enumerate(wl.model):
            stage.prefetch_side_inputs((ps[2 * j], ps[2 * j + 1]), x)
        for j, stage in enumerate(wl.model):
            x = x.view_as(x)
            x.register_hook(put(rec.din, j))
            rec.ins[j] = x.detach()
            x = stage(x, (ps[2 * j], ps[2 * j + 1]))
            rec.outs[j] = x.detach()
            x.register_hook(put(rec.dout, j))
            loss = loss + bench._MeanSquare.apply(x)
        loss.backward()
        return loss.detach()
    return step


def _build(case, step_kind):
    """Workload, graphed step, captured seed tensors (one per block, in stage/block order), eager draw count, record."""
    args = types.SimpleNamespace(patch=case.patch, batch=case.batch, dropout=case.dropout, frozen=case.frozen)
    draws = []
    real = PF.new_dropout_seed

    def recording(device, words=2):
        t = real(device, words)
        draws.append((t, torch.cuda.is_current_stream_capturing()))
        return t

    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(PF, "new_dropout_seed", recording)
        wl = bench.EncoderWorkload(DEV, args, case.ckpt is not None)
        if case.ckpt is not None:
            for m in wl.model.modules():
                if hasattr(m, "checkpoint_policy"):
                    m.checkpoint_policy = case.ckpt
        dtype = torch.bfloat16 if case.dtype == "bf16" else torch.float32
        x0 = torch.zeros(wl.in_shape, dtype=dtype, device=DEV)
        rec = _Record(len(wl.model))
        fn = _staged_step(wl, rec) if step_kind == "staged" else wl.step
        g = GraphedStep(fn, [x0.clone().requires_grad_(True)], wl.params, flat_grads=case.flat)
    captured = [t for t, cap in draws if cap]
    return wl, g, captured, len(draws) - len(captured), rec, dtype


# ---- the oracle ------------------------------------------------------------------------------------------------------------
def _leaves(wl, values=None):
    """float64 leaves: one state dict per stage, and the prompts.  values: {name in wl.named_params: tensor} overrides."""
    sds = [{k: v.detach().to(DEV, F64) for k, v in st.state_dict().items() if v.is_floating_point()} for st in wl.model]
    prompts = [p.detach().to(DEV, F64) for p in wl.prompts]
    for n, v in (values or {}).items():
        head, _, tail = n.partition(".")
        if head == "prompts":
            prompts[int(tail)] = v.detach().to(DEV, F64)
        else:
            sds[int(head)][tail] = v.detach().to(DEV, F64)
    for t in [v for sd in sds for v in sd.values()] + prompts:
        t.requires_grad_(True)
    return sds, prompts


def _grads(wl, sds, prompts):
    out = {}
    for n, _ in wl.named_params:
        head, _, tail = n.partition(".")
        t = prompts[int(tail)] if head == "prompts" else sds[int(head)][tail]
        out[n] = t.grad if t.grad is not None else torch.zeros_like(t)
    return out


def _stage_oracle(wl, j, x64, sds, prompts, words, p_drop):
    _, heads, _ = wl.specs[j]
    keep = None
    if p_drop > 0:
        keep = [R.block_keep_factors(words[2 * j + i], x64.shape, bench.WS, heads, bench.I_PROMPT, p_drop, p_drop, DEV)
                for i in range(2)]
    b = x64.shape[0]
    pp = [prompts[2 * j + i].unsqueeze(0).expand(b, -1, -1) for i in range(2)]
    return R.pair_forward(sds[j], x64, pp, bench.WS, heads, True, j < 1, keep=keep)


def _grad_of(p):
    return p.grad if p.grad is not None else torch.zeros_like(p)


def _errors_literal(wl, g, x, words, p_drop, values=None):
    sds, prompts = _leaves(wl, values)
    x64 = x.to(DEV, F64).requires_grad_(True)
    y, loss = x64, 0.0
    for j in range(len(wl.model)):
        y = _stage_oracle(wl, j, y, sds, prompts, words, p_drop)
        loss = loss + y.square().mean()
    loss.backward()
    ref = _grads(wl, sds, prompts)
    errs = {"loss": abs(g.loss.item() - loss.item()) / abs(loss.item()), "dx": rel_linf(g.input_grads[0], x64.grad)}
    for n, p in wl.named_params:
        errs[n] = rel_linf(_grad_of(p), ref[n])
    return errs


def _errors_staged(wl, rec, words, p_drop):
    sds, prompts = _leaves(wl)
    errs = {}
    for j in range(len(wl.model)):
        x64 = rec.ins[j].to(F64).requires_grad_(True)
        y = _stage_oracle(wl, j, x64, sds, prompts, words, p_drop)
        y.backward(rec.dout[j].to(F64))
        errs[f"{j}.out"] = rel_linf(rec.outs[j], y)
        errs[f"{j}.dx"] = rel_linf(rec.din[j], x64.grad)
        del y, x64
    ref = _grads(wl, sds, prompts)
    for n, p in wl.named_params:
        errs[n] = rel_linf(_grad_of(p), ref[n])
    return errs


# ---- one case --------------------------------------------------------------------------------------------------------------
def run_case(case, seed=None, negative=True):
    """Builds and replays the case's step, checks the seed plumbing, and returns
    {errs: {tensor: error}, neg: [{tensor: error}, ...] (negative controls), moved: min relative update or None, ...}."""
    t0 = time.perf_counter()
    step_kind = "staged" if case.mode == "staged" else "literal"
    wl, g, seeds, n_eager, rec, dtype = _build(case, step_kind)
    per_step = 2 * len(wl.model) if case.dropout > 0 else 0
    # one draw per block per step: the prefetched side inputs are the ones the forward claimed (an unclaimed prefetch draws
    # again), and checkpoint recomputation draws nothing
    assert len(seeds) == per_step, f"{len(seeds)} seed draws captured, {per_step} expected"
    assert n_eager == GRAPH_WARMUP * per_step, (n_eager, GRAPH_WARMUP * per_step)
    assert all(t.numel() == 4 and t.dtype == torch.int32 for t in seeds)
    x = wl.host_batch(torch.Generator().manual_seed(case.seed if seed is None else seed), dtype).to(DEV)
    words_of = lambda: [[int(v) for v in t.tolist()] for t in seeds]

    moved, before, losses = None, None, []
    if case.mode == "train":
        opt = torch.optim.Adam(wl.params, lr=TRAIN_LR)
        losses.append(g(x).item())
        g.bind_grads()
        opt.step()
        losses.append(g(x).item())
        prev = words_of()
        before = {n: p.detach().clone() for n, p in wl.named_params}
        g.bind_grads()
        opt.step()
        moved = min(rel_linf(p, before[n]) for n, p in wl.named_params)
    else:
        g(x)
        prev = words_of()
    losses.append(g(x).item())
    words = words_of()
    if case.dropout > 0:
        for a, b in zip(prev, words):
            assert a != b, "seed words repeat from one replay to the next"

    torch.cuda.reset_peak_memory_stats()
    mem0 = torch.cuda.memory_allocated()
    if step_kind == "staged":
        errs = _errors_staged(wl, rec, words, case.dropout)
    else:
        errs = _errors_literal(wl, g, x, words, case.dropout)
    peak = torch.cuda.max_memory_allocated() - mem0
    neg = []
    if negative and case.dropout > 0:
        neg.append(("previous replay's seed words", _errors_staged(wl, rec, prev, case.dropout) if step_kind == "staged"
                    else _errors_literal(wl, g, x, prev, case.dropout)))
    if negative and case.mode == "train":
        neg.append(("parameters before the last update", _errors_literal(wl, g, x, words, case.dropout, values=before)))
    return {"errs": errs, "neg": neg, "moved": moved, "oracle_peak_gb": peak / 2 ** 30,
            "losses": losses, "seconds": time.perf_counter() - t0}


def _worst_by_group(errs):
    out = {}
    for n, e in errs.items():
        k = _group(n)
        if e > out.get(k, (-1.0, None))[0]:
            out[k] = (e, n)
    return out


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_bench_step_vs_float64_oracle(case):
    res = run_case(case)
    bounds = _bounds(case)
    print(f"\n{case.name}: {res['seconds']:.1f} s, oracle peak {res['oracle_peak_gb']:.1f} GB above the step's own memory")
    for n, e in res["errs"].items():
        print(f"  {n:48s} {e:.2e}  bound {bounds[_group(n)]:.1e}")
    bad = {n: (e, bounds[_group(n)]) for n, e in res["errs"].items() if not e < bounds[_group(n)]}
    assert not bad, (case.name, bad)
    if case.mode == "train":
        print(f"  loss over the three replays {['%.3g' % v for v in res['losses']]}, smallest relative parameter update "
              f"{res['moved']:.3f}")
        assert res["moved"] >= 0.01
    expected = (case.dropout > 0) + (case.mode == "train")
    assert len(res["neg"]) == expected
    for what, errs in res["neg"]:
        miss = max(e / bounds[_group(n)] for n, e in errs.items())
        print(f"  negative control ({what}): misses by {miss:.0f}x")
        assert miss >= NEG_MARGIN, (case.name, what, miss)
