"""Data parallelism for the training step: one process per GPU (torchrun), NCCL over
NVLink 5 / NVSwitch.  The reference has no multi-GPU support at all (it only prints the
device count, celebA/EAD-GAN_celebA.py:178-179), so this layer is new; its contract is
"N-GPU step on global batch B == 1-device step on batch B" (SURVEY.md section 8e).

What is exchanged (one exchange per optimisation phase, nothing else):
  * gradients of exactly the parameter set the phase's optimiser owns -- phase G reduces
    only G's gradients, phase D only D's, the info phase both (SURVEY.md section 7.3-8).
    ``Adam.zero_grad()`` arms the optimiser that the coming backward is for; as autograd
    accumulates each of its parameters' gradients a hook copies it into a flat bucket and,
    when a bucket is full, launches its all-reduce on a side stream, so communication
    overlaps the rest of the backward pass; ``Adam.step()`` waits for the buckets and feeds
    the reduced flat views straight to the fused Adam kernel (scaled by 1/world_size there).
  * BatchNorm statistics: the [2C] fp64 partial sums of every train-mode BN forward and
    backward are summed across ranks between the reduce and apply kernels (SyncBN).
  * nothing for spectral norm: u, v are deterministic functions of the replicated weights.
The global batch is drawn once from the seeded host RNG and split contiguously
(``shard``): rank r takes rows [r*B/N, (r+1)*B/N).
"""
from __future__ import annotations

import os

import torch
import torch.distributed as dist

from . import functional as Fn

_state = None


class DataParallel:
    def __init__(self, rank, world_size, device, bucket_bytes=None, overlap=True):
        if bucket_bytes is None:
            bucket_bytes = int(os.environ.get("EADGAN_DP_BUCKET_MB", "32")) << 20
        self.rank, self.world_size, self.device = rank, world_size, device
        self.bucket_elems = max(1, bucket_bytes // 4)
        self.overlap = overlap  # on CPU (gloo, tests) the buckets are reduced asynchronously too, without a side stream
        self.comm_stream = torch.cuda.Stream(device=device) if device.type == "cuda" else None
        self._plans = {}      # id(optimizer) -> plan
        self._armed = None
        self._hooks_installed = set()

    # ---- SyncBN -----------------------------------------------------------------------
    def allreduce_sum_(self, t):
        dist.all_reduce(t, op=dist.ReduceOp.SUM)

    # ---- gradient buckets ---------------------------------------------------------------
    def _plan(self, opt):
        plan = self._plans.get(id(opt))
        if plan is not None:
            return plan
        params = [p for g in opt.param_groups for p in g["params"] if p.requires_grad]
        # reverse registration order ~ the order gradients become ready in backward
        order = list(reversed(params))
        buckets, cur, cur_n = [], [], 0
        for p in order:
            cur.append(p)
            cur_n += p.numel()
            if cur_n >= self.bucket_elems:
                buckets.append(cur)
                cur, cur_n = [], 0
        if cur:
            buckets.append(cur)
        plan = {"buckets": [], "where": {}}
        for bi, ps in enumerate(buckets):
            n = sum(p.numel() for p in ps)
            flat = torch.zeros(n, device=ps[0].device, dtype=torch.float32)
            off = 0
            views = []
            for p in ps:
                v = flat[off:off + p.numel()].view_as(p)
                views.append(v)
                plan["where"][p] = (bi, len(views) - 1)
                off += p.numel()
            plan["buckets"].append({"params": ps, "flat": flat, "views": views, "pending": 0, "work": None,
                                    "filled": set(), "dirty": False})
        self._plans[id(opt)] = plan
        for p in params:
            if p not in self._hooks_installed:
                p.register_post_accumulate_grad_hook(self._on_grad)
                self._hooks_installed.add(p)
        return plan

    def arm(self, opt):
        """called from Adam.zero_grad(): the next backward's gradients belong to ``opt``."""
        plan = self._plan(opt)
        for b in plan["buckets"]:
            b["filled"].clear()
            b["work"] = None
            b["dirty"] = False
        self._armed = plan

    def _on_grad(self, p):
        plan = self._armed
        if plan is None or not self.overlap:
            return
        loc = plan["where"].get(p)
        if loc is None:
            return  # gradient of a parameter this phase's optimiser does not own: never communicated
        b = plan["buckets"][loc[0]]
        if p in b["filled"]:
            # second accumulation into the same .grad in one phase: fall back to reduce-at-step (the in-flight
            # all-reduce, if any, is waited for there before ``flat`` is rewritten)
            b["dirty"] = True
            return
        b["views"][loc[1]].copy_(p.grad)
        b["filled"].add(p)
        if len(b["filled"]) == len(b["params"]) and b["work"] is None:
            self._launch(b)

    def _launch(self, b):
        if self.comm_stream is not None:
            self.comm_stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self.comm_stream):
                b["work"] = dist.all_reduce(b["flat"], op=dist.ReduceOp.SUM, async_op=True)
        else:
            b["work"] = dist.all_reduce(b["flat"], op=dist.ReduceOp.SUM, async_op=True)

    def reduce(self, opt):
        """called from Adam.step(): returns {param: summed-over-ranks gradient view}."""
        plan = self._plan(opt)
        out = {}
        for b in plan["buckets"]:
            if b["work"] is None or b["dirty"]:
                if b["work"] is not None:
                    # an all-reduce launched before the second accumulation is still writing ``flat``
                    b["work"].wait()
                    if self.comm_stream is not None:
                        torch.cuda.current_stream().wait_stream(self.comm_stream)
                for p, v in zip(b["params"], b["views"]):
                    if p.grad is not None:
                        v.copy_(p.grad)
                    else:
                        v.zero_()
                b["work"] = None
                b["dirty"] = False
                self._launch(b)
        for b in plan["buckets"]:
            b["work"].wait()
            if self.comm_stream is not None:
                torch.cuda.current_stream().wait_stream(self.comm_stream)
            for p, v in zip(b["params"], b["views"]):
                out[p] = v
            b["work"] = None
            b["filled"].clear()
        self._armed = None
        return out


def get():
    return _state


def attach(*optimizers):
    """Make the given eadgan_b200.optim.Adam instances data-parallel (no-op when world_size == 1)."""
    if _state is None:
        return
    for o in optimizers:
        o._dp = _state


def detach(*optimizers):
    """the given optimisers step on local gradients only (single-device reference runs inside a DP process)"""
    for o in optimizers:
        o._dp = None


def init(rank, world_size, device, backend=None, **kw):
    """Create the process group (if needed) and the DP state; wires SyncBN."""
    global _state
    if world_size <= 1:
        _state = None
        Fn.set_allreduce(None, 1)
        return None
    if not dist.is_initialized():
        backend = backend or ("nccl" if device.type == "cuda" else "gloo")
        dist.init_process_group(backend=backend, rank=rank, world_size=world_size)
    _state = DataParallel(rank, world_size, device, **kw)
    Fn.set_allreduce(_state.allreduce_sum_, world_size)
    return _state


def init_from_env():
    """torchrun entry: RANK / LOCAL_RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT."""
    ws = int(os.environ.get("WORLD_SIZE", "1"))
    if ws <= 1:
        return None
    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if torch.cuda.is_available():
        torch.cuda.set_device(local)
        dev = torch.device("cuda", local)
    else:
        dev = torch.device("cpu")
    return init(rank, ws, dev)


def shard(t, rank=None, world_size=None):
    """contiguous batch shard of a globally drawn tensor (rows [r*B/N, (r+1)*B/N))."""
    if rank is None:
        if _state is None:
            return t
        rank, world_size = _state.rank, _state.world_size
    B = t.shape[0]
    if B % world_size != 0:
        raise ValueError(f"global batch {B} is not divisible by world size {world_size}")
    per = B // world_size
    return t[rank * per:(rank + 1) * per]
