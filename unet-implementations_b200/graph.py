"""CUDA-graph replay of the training step (SURVEY.md section 8d: "CUDA events around a CUDA-graph-replayed step").

One step of the fused UNet is ~230 kernel launches enqueued from Python (ctypes calls + torch allocations).  The GPU
is the bottleneck at batch 32, but the deep levels are runs of 5-20 us kernels where the host can fall behind;
capturing forward + loss + backward once and replaying the graph removes the host from the step entirely.

    gs = GraphedStep(lambda: step_fn(static_batch))   # step_fn: zero_grad(set_to_none) -> model -> loss -> backward
    loss = gs.replay()                                # same static inputs; refresh them with .copy_() between replays

Do not keep the loss tensor (or anything else that holds the autograd graph) of an EAGER step alive across the capture:
its AccumulateGrad nodes belong to the stream that step ran on, and torch would synchronise the capture with it.

What is captured: every kernel of libb200unet.so on the capture stream, the side stream of the weight gradients
(forked and joined inside the capture), the dropout draws (torch's graph-safe Philox offsets: every replay draws new
masks) and the allocations of the step (a private pool: replays reuse the same addresses, which is also why the TMA
descriptors baked into the kernel parameters stay valid).  The reference has no counterpart (its loop is eager,
Our_UNet/src/train.py:630-670).  The optimizer step can be part of the graph: `FusedSGD(..., model=model,
capturable=True)` and `FusedAdam(..., model=model, capturable=True)` read their learning rate from a device scalar,
which replay() refreshes from `param_groups` -- what LambdaLR / CosineAnnealingLR change every epoch (train.py:454-477)
-- so the schedule works without re-capturing.
"""
from __future__ import annotations

from typing import Callable

import torch


class GraphedStep:
    """step_fn: zero_grad(set_to_none=True) -> forward -> loss -> backward [-> optimizer.step()], returning the loss.
    optimizer: a `FusedSGD(..., model=model, capturable=True)` or `FusedAdam(..., model=model, capturable=True)` whose
    step() is INSIDE step_fn -- the whole training step
    then replays as one graph; its learning rate lives in a device scalar that replay() refreshes from param_groups
    (what LambdaLR updates), so the schedule keeps working without re-capturing."""

    def __init__(self, step_fn: Callable[[], torch.Tensor], warmup: int = 2, optimizer=None):
        if not torch.cuda.is_available():
            raise RuntimeError("b200unet: GraphedStep needs a CUDA device; there is no CPU path")
        self.optimizer = optimizer
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):  # warm-up on a side stream, as torch's capture rules ask
            for _ in range(max(1, warmup)):
                step_fn()
        cur.wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = step_fn()
        torch.cuda.synchronize()
        self.num_nodes = None
        try:  # diagnostic only
            from cuda.bindings import runtime as cudart  # noqa: F401
            g = self.graph.raw_cuda_graph() if hasattr(self.graph, "raw_cuda_graph") else None
            if g is not None:
                err, _, n = cudart.cudaGraphGetNodes(g, 0)
                self.num_nodes = int(n)
        except Exception:  # noqa: BLE001
            pass

    def replay(self) -> torch.Tensor:
        if self.optimizer is not None and hasattr(self.optimizer, "sync_lr"):
            self.optimizer.sync_lr()
        self.graph.replay()
        return self.loss
