"""Whole-step CUDA-graph capture for training steps built on the pwa kernels.

One forward+backward of the prompted Swin encoder is ~280 kernel launches (ours + cuBLAS + a few torch
elementwise ops), most of them 3-50 us long: launched eagerly from Python the step is bound by the host, not
by the GPU.  Every pwa C-ABI entry point launches on the caller's stream, allocates nothing and never
synchronises (include/pwa.h), so a whole step -- forward, loss, backward -- can be captured ONCE into a CUDA
graph and replayed with a single launch.  This is the "streams and graphs" replacement for a tracing compiler:
the Python module code still defines the step; the graph only removes the per-launch host cost.

    step = GraphedStep(lambda x: encoder_step(model, prompts, x), [x_example], params)
    loss = step(x_batch)          # copies x_batch into the static input, replays, returns the static loss tensor
    # parameter gradients are in p.grad (static tensors, overwritten by every replay)
"""
from __future__ import annotations

from typing import Callable, Iterable, List, Sequence

import torch

from .functional import KernelStats


class GraphedStep:
    def __init__(self, step_fn: Callable[..., torch.Tensor], example_inputs: Sequence[torch.Tensor],
                 params: Iterable[torch.nn.Parameter], warmup: int = 3, flat_grads: bool = False):
        """step_fn(*inputs) must run forward AND backward and return a (scalar) loss tensor; it is called `warmup`
        times eagerly on a side stream (lazy initialisation: cuBLAS handles, kernel attributes, cached index maps),
        then once more under capture.  Inputs that require grad get a static .grad too (`input_grads`).
        The graph replays the kernels the capture recorded: under torch.use_deterministic_algorithms(True) at capture time
        every replay runs the deterministic backward kernels (see INTEGRATION.md), whatever the flag says at replay time.
        flat_grads=True makes every parameter's .grad a view into ONE flat fp32 buffer (`flat_grad`), so that the
        data-parallel exchange is a single in-place all-reduce of that buffer (`allreduce_flat`).  Inside the graph the
        backward produces its gradients as usual (autograd hands the freshly computed tensors over without a kernel) and
        ONE multi-tensor copy at the end of the step moves them into the flat buffer.  (Pointing .grad at the views during
        the backward instead made autograd ACCUMULATE into them: one tiny add kernel per parameter, ~150 launches and
        0.1-0.2 ms per step -- most of what the 2/4/8-GPU lines lost against one GPU.)"""
        if not example_inputs or not all(t.is_cuda for t in example_inputs):
            raise RuntimeError("GraphedStep: CUDA tensors only (pwa_b200 has no CPU path)")
        self.params: List[torch.nn.Parameter] = [p for p in params]
        self.static_inputs = [t.detach().clone().requires_grad_(t.requires_grad) for t in example_inputs]
        self._step_fn = step_fn
        self.flat_grad = None
        if flat_grads:
            if any(p.dtype != torch.float32 for p in self.params):
                raise RuntimeError("GraphedStep(flat_grads=True) needs fp32 master parameters")
            self.flat_grad = torch.zeros(sum(p.numel() for p in self.params), dtype=torch.float32,
                                         device=self.static_inputs[0].device)
            o = 0
            self._grad_views = []
            for p in self.params:
                self._grad_views.append(self.flat_grad[o:o + p.numel()].view_as(p))
                o += p.numel()
            inner = step_fn

            def step_fn(*inputs):
                loss = inner(*inputs)
                pairs = [(v, p.grad) for p, v in zip(self.params, self._grad_views) if p.grad is not None]
                with torch.no_grad():               # (parameters the step never reaches keep their zeros)
                    torch._foreach_copy_([v for v, _ in pairs], [g for _, g in pairs])
                return loss
        # CUDA events cannot be recorded inside a capture; launches are counted during the capture pass
        saved = (KernelStats.enabled, KernelStats.timing, KernelStats.launches)
        KernelStats.enabled, KernelStats.timing = True, False
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(max(1, warmup)):
                    self._zero()
                    step_fn(*self.static_inputs)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self._zero()
            self.graph = torch.cuda.CUDAGraph()
            launches0 = KernelStats.launches
            with torch.cuda.graph(self.graph):
                self.loss = step_fn(*self.static_inputs)
            self.launches_per_replay = KernelStats.launches - launches0   # pwa kernels inside one replay
            # the tensors every replay writes the parameter gradients into (None for parameters the step never reaches)
            self.static_grads = [p.grad for p in self.params] if self.flat_grad is None else list(self._grad_views)
            if self.flat_grad is not None:
                self.bind_grads()
        finally:
            KernelStats.enabled, KernelStats.timing, KernelStats.launches = saved

    def _zero(self):
        for p in self.params:
            p.grad = None
        for t in self.static_inputs:
            t.grad = None

    def bind_grads(self):
        """Point every p.grad back at the tensor the graph writes (after code that reset or replaced p.grad, e.g.
        optimizer.zero_grad(set_to_none=True) or an eager step in between): a replay does not touch p.grad itself."""
        for p, g in zip(self.params, self.static_grads):
            p.grad = g

    def allreduce_flat(self, group=None):
        """Average the flat gradient buffer over the data-parallel group: ONE NCCL all-reduce with the 1/world scale folded
        into the reduction (ReduceOp.AVG; gloo has no AVG: sum + scale there).
        (Capturing bucketed all-reduces INSIDE the step's graph, on a branch parallel to the backward, was tried in round 2:
        the 2-GPU run hung under capture and was dropped -- the exchange stays one launch after the replay.)"""
        import torch.distributed as dist
        world = dist.get_world_size(group)
        if world > 1:
            if dist.get_backend(group) == "nccl":
                dist.all_reduce(self.flat_grad, op=dist.ReduceOp.AVG, group=group)
            else:
                dist.all_reduce(self.flat_grad, group=group)
                self.flat_grad.div_(world)

    @property
    def input_grads(self):
        return [t.grad for t in self.static_inputs]

    def __call__(self, *inputs: torch.Tensor) -> torch.Tensor:
        with torch.no_grad():
            for s, t in zip(self.static_inputs, inputs):
                if t is not s:
                    s.copy_(t, non_blocking=True)
        self.graph.replay()
        if KernelStats.enabled:
            KernelStats.launches += self.launches_per_replay
        return self.loss


class InputPrefetcher:
    """Double-buffered host -> device input feed on a side stream: the pinned-host batch of step i+1 is copied while
    step i computes.  `prefetch(t)` enqueues the copy, `get()` makes the current stream wait for the oldest pending
    copy and returns the device buffer (valid until two more prefetches have been issued)."""

    def __init__(self, example: torch.Tensor, device):
        self.stream = torch.cuda.Stream(device=device)
        self.bufs = [torch.empty(example.shape, dtype=example.dtype, device=device) for _ in range(2)]
        self.events = [torch.cuda.Event(), torch.cuda.Event()]
        self.head = self.tail = 0

    def prefetch(self, host_batch: torch.Tensor):
        k = self.head % 2
        self.stream.wait_stream(torch.cuda.current_stream())    # the buffer's previous consumer has been enqueued
        with torch.cuda.stream(self.stream):
            self.bufs[k].copy_(host_batch, non_blocking=True)
            self.events[k].record(self.stream)
        self.head += 1

    def get(self) -> torch.Tensor:
        if self.tail >= self.head:
            raise RuntimeError("InputPrefetcher.get() without a pending prefetch")
        k = self.tail % 2
        torch.cuda.current_stream().wait_event(self.events[k])
        self.tail += 1
        return self.bufs[k]
