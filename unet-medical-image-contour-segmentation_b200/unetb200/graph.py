"""Whole-step CUDA graph for the UNet training step.

One training step of the path is ~350 kernel launches issued from Python through ctypes; on a B200 the step
is 25 ms, so launch gaps are a few per cent of it.  ``GraphedStep`` captures the caller's step function
(forward + loss + backward [+ gradient all-reduce] + clip + optimizer step) once into a ``torch.cuda.CUDAGraph``
and replays it: every kernel of the library enqueues on the stream it is given (the capture stream), buffers come
from PyTorch's graph-private pool so the addresses baked into the TMA descriptors stay valid, and nothing on the
path synchronises with the host (the reference's boundary_loss has six syncs; ours none).

The step function must be capture-safe: no ``.item()``, optimizer constructed with ``capturable=True``.
"""
from __future__ import annotations

import torch

from .functional import graph_replayed


class GraphedStep:
    def __init__(self, step_fn, example_inputs, warmup=3):
        """step_fn(*inputs) -> loss tensor.  ``example_inputs`` give shapes/dtypes/layouts of the static inputs."""
        self.step_fn = step_fn
        self.static_inputs = [torch.empty_like(a).copy_(a) for a in example_inputs]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                      # warm-up on a side stream, as CUDA-graph capture requires
            for _ in range(warmup):
                step_fn(*self.static_inputs)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graph = torch.cuda.CUDAGraph()
        # thread_local: other threads of the process (NCCL's watchdog polls CUDA events) must not invalidate the
        # capture -- with 8 ranks per box the default "global" mode failed with cudaErrorStreamCaptureInvalidated
        with torch.cuda.graph(self.graph, capture_error_mode="thread_local"):
            self.static_loss = step_fn(*self.static_inputs)
        torch.cuda.synchronize()

    def load(self, *inputs):
        """Device-to-device copy of a new batch into the graph's static input buffers (current stream)."""
        for s, a in zip(self.static_inputs, inputs):
            s.copy_(a, non_blocking=True)

    def replay(self):
        self.graph.replay()
        graph_replayed()                # the weights and running statistics moved: drop the cached operands
        return self.static_loss

    def __call__(self, *inputs):
        self.load(*inputs)
        return self.replay()
