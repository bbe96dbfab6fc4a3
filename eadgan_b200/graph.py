"""Whole-step CUDA graph: the training step (all phases, backward passes, Adam updates) is captured once
and replayed, so the ~600 kernel launches per step cost no host time (SURVEY.md section 8f rank 3; the
reference issues ~10^4 ATen dispatches per step, section 3.2).

    step = CelebAStep(...)
    gstep = GraphedStep(step, example_inputs)      # eager warm-up steps, then capture
    losses = gstep(imgs, z, code, labels)          # copies into the static inputs, replays

What makes the step capturable: no host synchronisation anywhere in it (the affine glue has a closed-form
inverse, eadgan_b200/affine.py); every kernel is launched on the caller's current stream; tensor maps are
kernel *arguments* (baked into the graph, valid because the graph's private memory pool keeps every
address); Adam's step count lives on the device while capturing (eadgan_adam_step_dev).
"""
from __future__ import annotations

import torch

from . import _lib, tc


class GraphedStep:
    def __init__(self, step, example_inputs, warmup=3):
        self.step = step
        self.static_in = [t.clone() for t in example_inputs]
        self.opts = list(step.optimizers())
        cur = torch.cuda.current_stream()
        side = torch.cuda.Stream()
        side.wait_stream(cur)
        with torch.cuda.stream(side):        # warm-up on a side stream, as torch's capture protocol asks
            for _ in range(max(1, warmup)):
                step(*self.static_in)
        cur.wait_stream(side)
        torch.cuda.synchronize()
        for o in self.opts:
            o.prepare_capture()
            # Drop every gradient tensor left by the warm-up.  A phase's backward also accumulates into the
            # gradients of parameters its optimiser does NOT own (phase G reaches D's parameters); with warm-up
            # leftovers in place that accumulation would be captured as an in-place add into REGULAR-pool memory
            # which the next zero_grad() frees -- the graph would then write through a dangling address on every
            # replay (silent corruption, or an illegal access once the allocator releases the block).
            for grp in o.param_groups:
                for p in grp["params"]:
                    p.grad = None
        self.graph = torch.cuda.CUDAGraph()
        k0 = _lib.lib().eadgan_kernel_launches()
        # packed-weight cache: a hit during capture would leave the pack kernel OUT of the graph (stale weights on
        # replay), and an entry filled during capture holds nothing until the first replay -> clear on both sides
        tc.invalidate_caches()
        # Capture on the SAME side stream the warm-up ran on.  AccumulateGrad nodes created during warm-up outlive it
        # and keep running on the stream they were created on; with torch's default (separate) capture stream their
        # kernels were pulled into the capture through an event while their allocations came from the REGULAR pool
        # (only the capture stream allocates from the graph's private pool) -- memory the allocator was free to
        # release (torch.cuda.empty_cache(), or the empty_cache() a later capture begins with) under the graph.
        tc.capture_births = []
        try:
            with torch.cuda.graph(self.graph, stream=side):
                self.static_out = step(*self.static_in)
        finally:
            births, tc.capture_births = tc.capture_births, None
        for b in births:
            b.zero_()        # see tc.alloc_padded: make the recorded zero fills real before anyone else reuses them
        # The graph has baked in the addresses of every pooled halo buffer and per-stream workspace the step used --
        # regular-pool memory that only module-level caches keep alive.  Hold strong references for the life of the
        # graph: tc.clear_pool(), or a larger workspace replacing a cache entry, can then no longer free memory under
        # the graph.  (The warm-up steps filled the pool, so capture creates almost no buffer: a buffer first created
        # INSIDE a capture has its zero fill recorded and re-executed by every replay.)
        self._keepalive = [b for free in tc._pool.values() for b in free] + births + list(tc._ws_cache.values())
        tc.invalidate_caches()
        self.kernels_per_replay = int(_lib.lib().eadgan_kernel_launches() - k0)
        self._first = True
        # input pipeline: the NEXT step's host batch is copied into a staging set on a copy stream while the
        # current replay runs; the replay then only does a device-to-device copy into its static inputs
        self._copy_stream = torch.cuda.Stream()
        self._staging = None
        self._staged_key = None
        self._staged_ready = torch.cuda.Event()
        self._staging_free = torch.cuda.Event()
        self._staging_free.record()

    @staticmethod
    def _key(inputs):
        return tuple((t.data_ptr(), t._version) for t in inputs)

    def prefetch(self, inputs):
        """start copying ``inputs`` (pinned host or device tensors) for a later ``__call__(*inputs)``"""
        if self._staging is None:
            self._staging = [torch.empty_like(t) for t in self.static_in]
        self._copy_stream.wait_event(self._staging_free)     # the previous consumer has read the staging set
        with torch.cuda.stream(self._copy_stream):
            for dst, src in zip(self._staging, inputs):
                dst.copy_(src, non_blocking=True)
            self._staged_ready.record(self._copy_stream)
        self._staged_key = self._key(inputs)

    def __call__(self, *inputs, prefetch=None):
        """copies ``inputs`` into the static inputs and replays; ``prefetch``: the inputs of the NEXT call, whose
        host-to-device copy then overlaps this replay"""
        if self._staged_key is not None and self._staged_key == self._key(inputs):
            cur = torch.cuda.current_stream()
            cur.wait_event(self._staged_ready)
            for dst, src in zip(self.static_in, self._staging):
                dst.copy_(src, non_blocking=True)
            self._staging_free.record(cur)
            self._staged_key = None
            inputs = ()
        for dst, src in zip(self.static_in, inputs):
            if dst.data_ptr() != src.data_ptr():
                dst.copy_(src, non_blocking=True)
        if self._first:
            self._first = False          # the capture pass already advanced the python step mirrors once
        else:
            for o in self.opts:
                o.on_replay()
        self.graph.replay()
        _lib.bump_weights_epoch()        # the replay ran Adam steps: eager code must re-pack afterwards
        if prefetch is not None:
            self.prefetch(prefetch)
        return self.static_out
