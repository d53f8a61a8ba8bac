"""Whole-step CUDA graph: forward + loss + backward (+ gradient all-reduce) + optimizer step captured once and
replayed, so the ~100 kernel launches of a training step cost one graph launch.

The C ABI is enqueue-only on the current stream, allocates nothing and never synchronises (include/nbody_b200.h), so
it is capture-safe; PyTorch supplies the graph-private memory pool and the capturable optimizer.

    step = GraphedStep(fn, static_inputs, optimizer)      # fn(**static_inputs) -> scalar loss
    loss = step(**new_inputs)                              # copies into the static buffers, replays, returns the loss
"""
from __future__ import annotations

from typing import Callable, Dict, Optional

import torch


class GraphedStep:
    def __init__(self, fn: Callable[..., torch.Tensor], static_inputs: Dict[str, torch.Tensor],
                 optimizer: Optional[torch.optim.Optimizer] = None, warmup: int = 3):
        if not torch.cuda.is_available():
            raise RuntimeError("GraphedStep needs a CUDA device")
        self.fn, self.opt = fn, optimizer
        self.static = {k: v.clone() for k, v in static_inputs.items()}
        dev = next(iter(self.static.values())).device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):          # warm-up off the capture stream (allocator, lazy optimizer state)
            for _ in range(warmup):
                self._eager()
        torch.cuda.current_stream(dev).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        if self.opt is not None:
            self.opt.zero_grad(set_to_none=True)
        from ._lib import load_library

        lib = load_library()
        n0 = lib.nb_launch_count()
        with torch.cuda.graph(self.graph):
            self.loss = self._eager(zero=False)
        self.launches_per_replay = int(lib.nb_launch_count() - n0)   # kernels of this library inside the graph
        # the gradient buffers every replay writes, in the optimizer's parameter order (None: no gradient); p.grad itself
        # points elsewhere once another step over the same parameters is captured
        self.grads = [p.grad for g in self.opt.param_groups for p in g["params"]] if self.opt is not None else []

    def _eager(self, zero: bool = True) -> torch.Tensor:
        if self.opt is not None and zero:
            self.opt.zero_grad(set_to_none=True)
        loss = self.fn(**self.static)
        if self.opt is not None:
            loss.backward()
            self.opt.step()
            # keep no reference to the autograd graph: its AccumulateGrad nodes are bound to the capture stream and would
            # otherwise outlive the capture (PyTorch warns about, and may synchronise on, the stream mismatch later)
            loss = loss.detach()
        return loss

    def __call__(self, **inputs: torch.Tensor) -> torch.Tensor:
        for k, v in inputs.items():
            self.static[k].copy_(v, non_blocking=True)
        self.graph.replay()
        return self.loss.detach()
