"""Whole-step CUDA-graph capture.

At pose-0 size a training step is ~70 small kernels whose roofline time is a few
hundred microseconds in total, so launch latency dominates an eager step.  Every
entry point of the C ABI is capture-safe (no allocation, no sync, stream passed in),
so forward + loss + backward can be recorded once and replayed.

Per-step inputs (e.g. the negatives resampled every epoch, ``GripNet-pose.py:131``)
live in static buffers that the caller overwrites with ``copy_`` before ``replay()``;
the index structures derived from them (endpoint CSR of the negative edges) are
rebuilt by the captured K1 kernels on every replay.
"""
import torch

from . import _lib, streams


class CapturedStep:
    """Capture ``outputs = fn(); outputs[0].backward()`` into one CUDA graph.

    ``fn`` must read its per-step inputs from the tensors listed in ``dynamic_inputs``.
    After construction: overwrite those tensors in place, call ``replay()``, read
    ``outputs`` and the parameters' ``.grad``.
    """

    def __init__(self, fn, parameters, dynamic_inputs=(), warmup=3, post_backward=None):
        self.params = [p for p in parameters]
        post = post_backward if post_backward is not None else (lambda: None)
        cur = torch.cuda.current_stream()
        # warm-up and capture run on ONE high-priority stream: the chain's kernels keep that priority in the graph,
        # the background branches (streams.Branch(background=True)) stay below it
        side = torch.cuda.Stream(priority=streams.CHAIN_PRIORITY)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(max(int(warmup), 1)):      # builds and caches every static graph structure
                self._drop_grads()
                out = fn()
                out[0].backward()
                post()
            # static seed of the backward pass: `backward()` alone fills a fresh ones_like(loss) every replay —
            # one more kernel at the head of the backward's dependency chain
            self._seed = torch.ones_like(out[0])
        cur.wait_stream(side)
        torch.cuda.synchronize()
        for t in dynamic_inputs:
            t.add_(0)                                  # new tensor version: structures of per-step inputs
        self._drop_grads()                             # are (re)built INSIDE the graph, not served from cache
        self.graph = torch.cuda.CUDAGraph()
        before = _lib.launch_count()
        with torch.cuda.graph(self.graph, stream=side):
            self.outputs = fn()
            self.outputs[0].backward(self._seed)
            post()                                     # e.g. the bucketed gradient all-reduce of a partitioned run
        self.launches_per_replay = _lib.launch_count() - before
        torch.cuda.synchronize()

    def _drop_grads(self):
        for p in self.params:
            p.grad = None

    def replay(self):
        self.graph.replay()
        return self.outputs
