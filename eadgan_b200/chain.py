"""bf16 tensor-core execution of a whole ``nn.Sequential`` conv stack as ONE autograd node.

When ``EADGAN_PRECISION=bf16`` (default), a Sequential made only of
  Conv2d | ConvTranspose2d  [+ BatchNorm2d]  [+ LeakyReLU | ReLU | Tanh | Sigmoid]
groups (every G / D / Encoder trunk of the reference: celebA/EAD-GAN_celebA.py:75-92,
109-122; dSprites/rp.py:65-76,94-105,128-142,164-175) is run by ``_ChainFn``:

  * module-boundary tensors stay ordinary fp32 NCHW; everything in between lives in PRIVATE
    halo-padded NHWC bf16 buffers [n, h+2, w+2, c] (SURVEY.md section 8b);
  * k4 s2 p1 layers with tensor-core-friendly channel counts run on the tcgen05/TMEM/TMA
    kernels (csrc/tc_conv.cu): Conv forward = fprop, ConvTranspose forward = dgrad, and the
    opposite direction for input gradients, wgrad for both;
  * bias + activation are fused into the producing kernel's epilogue; BatchNorm statistics
    are accumulated in the ConvTranspose epilogue (fp64 atomics) and the normalise + ReLU pass
    is one streaming kernel; the LeakyReLU/ReLU backward of layer L is fused into the epilogue
    of layer L+1's input-gradient kernel (mask = saved output of layer L);
  * a BatchNorm in eval mode (``.eval()``, torch semantics) normalises with its running statistics:
    no fused statistics, no cross-rank all-reduce, no running-statistics update; its backward is
    one pass (dx in place, plus the fp64 sums that give dgamma, dbeta and the conv-bias gradient).
    The conv output before BatchNorm is kept exactly as in training mode, and the kernel families
    are the training-mode ones; the stage's BatchNorm mode is recorded in its plan by the forward;
  * layers the tensor-core path does not cover run on the generic SIMT kernels directly on the
    same buffers (strided bf16 views) -- there is no torch / cuDNN fallback anywhere.
    ``_plan_kernels`` picks the kernel family of every stage and direction, in one place.

Forward pre-hooks of the wrapped modules (legacy spectral_norm) are honoured: they run before
the chain and the chain consumes ``module.weight`` (= weight_orig / sigma, an autograd tensor).
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _lib as L
from . import functional as Fn
from . import tc
from ._lib import ACT_NONE, call, ptr, stream, t4


def precision():
    return os.environ.get("EADGAN_PRECISION", "bf16")


# tests only (tests/gates.py): when this is a list, every chain forward appends (sequential, [gate masks]) to it,
# one bool NCHW mask per ReLU / LeakyReLU stage: mask = saved output > 0, which is exactly the gate the fused
# backward kernels read.  A parity test replays these gates in the oracle so that both runs differentiate the
# same piecewise-linear function (SURVEY.md section 7.3-1: a single flipped gate moves every upstream gradient).
gate_log = None


def _pow2(v):
    return v > 0 and (v & (v - 1)) == 0


class _Stage:
    __slots__ = ("kind", "conv", "bn", "act", "stride", "pad", "r")

    def __init__(self, kind, conv):
        self.kind, self.conv, self.bn, self.act = kind, conv, None, (ACT_NONE, 0.0)
        self.stride = conv.stride[0]
        self.pad = conv.padding[0]
        self.r = conv.kernel_size[0]


def _compile(seq):
    from . import nn as enn
    mods = list(seq._modules.values())
    stages, i = [], 0
    while i < len(mods):
        m = mods[i]
        if isinstance(m, enn.Conv2d):
            kind = "conv"
        elif isinstance(m, enn.ConvTranspose2d):
            kind = "convT"
        else:
            return None
        if (m.groups != 1 or m.dilation != (1, 1) or m.kernel_size[0] != m.kernel_size[1]
                or m.stride[0] != m.stride[1] or m.padding[0] != m.padding[1] or m._forward_hooks
                or m._backward_hooks or getattr(m, "padding_mode", "zeros") != "zeros"
                or (kind == "convT" and m.output_padding != (0, 0))):
            return None
        st = _Stage(kind, m)
        i += 1
        if i < len(mods) and isinstance(mods[i], enn.BatchNorm2d) and enn._plain(mods[i]):
            bn = mods[i]
            if not (bn.affine and bn.track_running_stats) or bn.momentum is None:
                return None
            st.bn = bn
            i += 1
        if i < len(mods) and isinstance(mods[i], enn._Act) and enn._plain(mods[i]):
            st.act = mods[i].act()
            i += 1
        stages.append(st)
    if not stages or stages[-1].bn is not None:
        return None
    return stages


def _plan(seq):
    key = tuple(id(m) for m in seq._modules.values())
    cached = seq.__dict__.get("_eadgan_plan")
    if cached is None or cached[0] != key:
        cached = (key, _compile(seq))
        seq.__dict__["_eadgan_plan"] = cached
    return cached[1]


_sn_streams = {}
prefetch_enabled = True     # False: prefetch_spectral_norm is a no-op and every forward runs its own power iteration
                            # (state snapshots taken BETWEEN phases then hold u / v exactly as far as the forwards got)


def _side_stream(dev):
    """the per-device side stream of the prefetches, ordered after everything queued on the current stream so far
    (the last optimiser step, every earlier u / v update and every earlier consumer of the old packs)"""
    side = _sn_streams.get(dev)
    if side is None:
        side = _sn_streams[dev] = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    return side


def prefetch_spectral_norm(seq, count=1):
    """Run the spectral-norm power iterations of the NEXT ``count`` forwards of ``seq`` now, on a side stream.

    The legacy spectral_norm hook depends only on weight_orig and the u / v buffers -- not on the activations --
    so a step driver that knows how many forwards of a network follow before its weights change can issue their
    power iterations early; they then overlap whatever the main stream is doing (the other network's forward, a
    backward pass) instead of sitting, 4 small launches per layer, on the critical path in front of every conv
    stack.  Results are queued per module in forward order; ``try_run`` consumes them (and waits on the side
    stream's event) instead of calling the hooks.  Same arithmetic, same order of u / v updates."""
    if precision() != "bf16" or not prefetch_enabled:
        return
    stages = _plan(seq)
    if stages is None:
        return
    convs = [st.conv for st in stages if st.conv._forward_pre_hooks]
    if not convs:
        return
    w0 = getattr(convs[0], "weight_orig", None)
    if w0 is None or not w0.is_cuda:
        return
    side = _side_stream(w0.device)
    with torch.cuda.stream(side):
        for _ in range(count):
            done = []
            Fn.sn_skip_scale = True
            try:
                for conv in convs:
                    conv.__dict__.pop("_eadgan_sn_src", None)
                    for hook in conv._forward_pre_hooks.values():
                        hook(conv, (None,))
                    done.append((conv.weight, conv.__dict__.get("_eadgan_sn_src")))
            finally:
                Fn.sn_skip_scale = False
            ev = torch.cuda.Event()
            ev.record(side)
            for conv, entry in zip(convs, done):
                tag = getattr(getattr(conv, "weight_orig", None), "_eadgan_stepped", 0)
                conv.__dict__.setdefault("_eadgan_sn_queue", []).append((entry, ev, tag))


def prefetch_packs(module):
    """Re-pack the bf16 GEMM operands of every conv stack inside ``module`` now, on the side stream.

    The packs depend only on the raw weights (sigma of a spectral-normalised layer is applied in the kernel
    epilogue), so a step driver calls this right after the optimiser step that changed them; the ~30 small
    permutation kernels per step then overlap the main stream's work instead of preceding the first GEMM that needs
    them.  The layouts are the ones each parameter was consumed in so far (tc._note_use), i.e. nothing happens on the
    first step.  Every pack built here carries an event which its consumer's stream waits on (tc._adopt)."""
    if precision() != "bf16" or not prefetch_enabled:
        return
    todo = []
    for seq in module.modules():
        if not isinstance(seq, torch.nn.Sequential):
            continue
        stages = _plan(seq)
        if stages is None:
            continue
        for st in stages:
            p = getattr(st.conv, "weight_orig", None)
            if p is None:
                p = st.conv.weight
            if isinstance(p, torch.nn.Parameter) and p.is_cuda and getattr(p, "_eadgan_pack_uses", None):
                todo.append(p)
    if not todo:
        return
    with torch.cuda.stream(_side_stream(todo[0].device)):
        for p in todo:
            tc.prefetch_packs(p)


def set_trainable(module, flag):
    """Step drivers freeze the networks the current phase's optimiser does not own (celebA/EAD-GAN_celebA.py:334-345:
    phase G back-propagates THROUGH D, and the reference also computes D's weight gradients there, which
    ``optimizer_D.zero_grad()`` (:353) discards unread).  With the parameters frozen autograd asks the chain for
    input gradients only, so those dead weight-gradient GEMMs are never launched (SURVEY.md section 7.3-8)."""
    for p in module.parameters():
        p.requires_grad_(flag)


def clear_prefetch(seq):
    for m in seq._modules.values():
        m.__dict__.pop("_eadgan_sn_queue", None)


def try_run(seq, x):
    """Returns the Sequential's output, or None when the chain path does not apply."""
    if precision() != "bf16" or not torch.is_tensor(x) or not x.is_cuda or x.dim() != 4 or x.dtype != torch.float32:
        return None
    stages = _plan(seq)
    if stages is None:
        return None
    params, srcs = [], []
    for st in stages:
        queue = st.conv.__dict__.get("_eadgan_sn_queue")
        if queue:
            # this forward's power iteration was issued ahead of time (prefetch_spectral_norm): adopt its results
            (w_pre, sn_pre), ev, tag = queue.pop(0)
            if tag != getattr(getattr(st.conv, "weight_orig", None), "_eadgan_stepped", 0):
                raise RuntimeError("eadgan_b200.chain: a prefetched spectral-norm result is older than the layer's "
                                   "weights (an optimiser stepped them after prefetch_spectral_norm); the step driver "
                                   "must prefetch only forwards that run before the owning optimiser steps")
            cur = torch.cuda.current_stream()
            cur.wait_event(ev)
            for t in (w_pre,) + (tuple(sn_pre[1:3]) if sn_pre is not None else ()):
                if torch.is_tensor(t):
                    t.record_stream(cur)
            setattr(st.conv, "weight", w_pre)
            if sn_pre is not None:
                st.conv.__dict__["_eadgan_sn_src"] = sn_pre
            else:
                st.conv.__dict__.pop("_eadgan_sn_src", None)
        else:
            st.conv.__dict__.pop("_eadgan_sn_src", None)
            Fn.sn_skip_scale = True      # W / sigma is materialised only if a SIMT / dense consumer asks for it
            try:
                for hook in st.conv._forward_pre_hooks.values():  # legacy spectral_norm lives here
                    hook(st.conv, (x,))
            finally:
                Fn.sn_skip_scale = False
        w = st.conv.weight
        # what the tensor-core path packs: the parameter itself (cached until it changes), with sigma applied
        # in the kernel epilogue for spectral-normalised layers; any other weight tensor is packed as is
        sn = st.conv.__dict__.get("_eadgan_sn_src")
        if sn is not None and sn[2] is w and isinstance(sn[0], torch.nn.Parameter):
            srcs.append((sn[0], sn[1], sn[3]))
        elif sn is not None and sn[3]:
            Fn.spectral_norm_materialize(sn[0], sn[1], sn[2])   # not packable from weight_orig: needs the values now
            srcs.append(None)
        elif isinstance(w, torch.nn.Parameter):
            srcs.append((w, None))
        else:
            srcs.append(None)
        params += [w, st.conv.bias]
        if st.bn is not None:
            if st.bn.training:
                st.bn.num_batches_tracked.add_(1)
            params += [st.bn.weight, st.bn.bias]
    if gate_log is not None:
        gate_log.append((seq, []))
    return _ChainFn.apply(x, stages, srcs, *params)


# ------------------------------------------------------------------------------------------
class _Buf:
    """an activation in one of the two formats: 'ext' fp32 NCHW tensor, 'pad' padded NHWC bf16."""
    __slots__ = ("t", "fmt")

    def __init__(self, t, fmt):
        self.t, self.fmt = t, fmt

    @property
    def nchw(self):  # logical (n, c, h, w)
        if self.fmt == "ext":
            return tuple(self.t.shape)
        n, hp, wp, c = self.t.shape
        return (n, c, hp - 2, wp - 2)

    def view(self):  # logical NCHW view usable with t4()
        return self.t if self.fmt == "ext" else tc.interior(self.t)

    def padded(self):
        return self.t if self.fmt == "pad" else tc.to_padded(self.t)


def _geom(st, in_shape):
    """conv-view descriptor (always stated as the forward conv x[n,c,h,w] -> y[n,k,p,q])."""
    w = st.conv.weight
    r, s_, pad = st.r, st.stride, st.pad
    if st.kind == "conv":
        n, c, h, ww = in_shape
        k = w.shape[0]
        p = (h + 2 * pad - r) // s_ + 1
        q = (ww + 2 * pad - r) // s_ + 1
    else:
        n, k, p, q = in_shape
        c = w.shape[1]
        h = (p - 1) * s_ - 2 * pad + r
        ww = (q - 1) * s_ - 2 * pad + r
    return L.ConvDesc(n, c, h, ww, k, r, r, p, q, s_, pad)


def _calloc(d):
    """big-map channel count the tensor-core kernels run with: d.c, or 32 when the layer has fewer than
    32 real channels (the 1- / 3-channel image layers are zero-padded to 32), or None if unsupported."""
    if d.c % 32 == 0:
        return d.c
    return 32 if d.c < 32 else None


def _tc_ok(d, direction):
    if not (d.r == 4 and d.stride == 2 and d.pad == 1 and d.h == 2 * d.p and d.w == 2 * d.q):
        return False
    if not (_pow2(d.p) and _pow2(d.q)) or _calloc(d) is None:
        return False
    if direction == "fprop":
        return d.k % 32 == 0 and d.q <= 128
    if direction == "dgrad":
        return (d.k % 64 == 0 or d.k == 32) and d.q <= 128
    return d.k % 32 == 0 and d.q <= 64  # wgrad


def _thin_ok(d, direction):
    """the "thin" kernels: k4 s2 p1 with a 1..4-channel big map (the image)"""
    if not (d.r == 4 and d.stride == 2 and d.pad == 1 and d.h == 2 * d.p and d.w == 2 * d.q and d.c <= 4):
        return False
    if not (_pow2(d.p) and _pow2(d.q)):
        return False
    if direction == "fprop":
        return d.k % 32 == 0 and d.q <= 128
    if direction == "dgrad":      # GEMM + col2im epilogue: 32-wide small map of 2-row tiles, <= 3 image channels
        return (d.k % 64 == 0 or d.k == 32) and d.q == 32 and d.p >= 2 and d.c <= 3
    return d.k % 32 == 0 and d.q <= 64  # wgrad


# the tensor-core epilogues stage a fused bias and accumulate fused BatchNorm statistics for at most this many output
# channels (STAT_MAX_CH in csrc/tc_conv.cu)
FUSE_MAX_CH = 1024


def _impl(st, d, last):
    """which kernel family runs the forward of this stage (called by _plan_kernels)."""
    out_ch = d.k if st.kind == "conv" else d.c
    if out_ch > FUSE_MAX_CH and (st.conv.bias is not None or st.bn is not None):
        return "simt"      # bias / statistics too wide for the fused epilogues: the SIMT kernels have no such limit
    unit = d.r == 4 and d.stride == 1 and d.pad == 0 and d.h == 4 and d.w == 4 and d.p == 1 and d.q == 1
    plain = st.bn is None and st.act[0] == ACT_NONE
    if unit and plain and d.c % 128 == 0:
        if st.kind == "convT" and d.k <= 256 and not last:
            return "dense_T"
        if st.kind == "conv" and d.k <= 32 and last:
            return "dense_C"
    direction = "fprop" if st.kind == "conv" else "dgrad"
    if _thin_ok(d, direction) and (st.kind == "conv" or (last and st.bn is None)):
        return "thin"      # big map = the 1..4-channel image: row-expanded buffer, K = 64 (csrc/tc_conv.cu, "thin")
    if _tc_ok(d, direction):
        if _calloc(d) != d.c and st.kind == "convT" and not (last and st.bn is None):
            return "simt"  # zero-padded OUTPUT channels are only supported for an fp32 NCHW result
        return "tc"
    return "simt"


class _StagePlan:
    """How one stage runs: its geometry ``d``, the kernel family of its forward (``fwd``), weight gradient
    (``wgrad``) and input gradient (``dx``), the mode of its BatchNorm (``bn``: None, "train" or "eval"), and the
    layout of the buffers around it.

    Families: "tc" (tcgen05 implicit GEMM, csrc/tc_conv.cu), "thin" (the same kernels with the 1..4-channel image as
    big map, row-expanded to K = 64), "dense_T" / "dense_C" / "dense" (the 1x1 <-> 4x4 layers as batch GEMMs) and
    "simt" (the any-geometry SIMT kernels, csrc/simt_conv.cu).

    The BatchNorm mode is read from ``bn.training`` when the forward builds the plan; the backward follows the plan,
    so switching the module between ``.train()`` and ``.eval()`` after a forward does not change its backward."""
    __slots__ = ("d", "ca", "fwd", "wgrad", "dx", "bn", "fuse", "in_fmt", "out_fmt", "in_shape", "out_shape")


def _plan_kernels(stages, in_shape):
    """-> one _StagePlan per stage of a compiled chain (``_plan(seq)``) run on an NCHW input of ``in_shape``.

    This is the only place that picks kernels.  The executor asks autograd only WHETHER a planned kernel runs (a
    frozen weight, an input that needs no gradient), never which one."""
    plans = []
    for si, st in enumerate(stages):
        last, conv = si == len(stages) - 1, st.kind == "conv"
        prev = stages[si - 1] if si > 0 else None
        p = _StagePlan()
        d = p.d = _geom(st, in_shape)
        p.in_shape = tuple(in_shape)
        p.out_shape = (d.n, d.k, d.p, d.q) if conv else (d.n, d.c, d.h, d.w)
        p.bn = None if st.bn is None else ("train" if st.bn.training else "eval")
        p.fwd = _impl(st, d, last)
        p.ca = _calloc(d) if p.fwd == "tc" else d.c
        if p.fwd in ("dense_T", "dense_C"):
            p.wgrad = "dense"
            p.dx = "dense" if p.fwd == "dense_C" and si > 0 else "simt"
        elif p.fwd == "thin":
            if conv and last:
                raise RuntimeError("eadgan_b200.chain: a thin conv cannot be the last stage")
            p.wgrad = "thin" if _thin_ok(d, "wgrad") else "simt"
            if conv:    # the image gradient of the chain's input: GEMM + col2im epilogue
                p.dx = "thin" if si == 0 and _thin_ok(d, "dgrad") else "simt"
            else:       # a small-map gradient from the row-expanded image gradient
                p.dx = "thin" if si > 0 else "simt"
        elif p.fwd == "tc":
            p.wgrad = "tc" if _tc_ok(d, "wgrad") else "simt"
            # zero-padded result channels need the fp32 NCHW epilogue: a conv's input gradient onto fewer than 32
            # channels runs on the tensor cores only for the chain's input
            tc_dx = _tc_ok(d, "dgrad" if conv else "fprop") and not (conv and si > 0 and p.ca != d.c)
            p.dx = "tc" if tc_dx else "simt"
        else:
            p.wgrad = p.dx = "simt"
        # the first stage reads the caller's fp32 NCHW tensor where its kernel can, every other buffer is padded
        # NHWC bf16; only the chain's result is fp32 NCHW again
        p.in_fmt = "ext" if si == 0 and (p.fwd in ("dense_T", "simt") or (p.fwd == "thin" and conv)) else "pad"
        p.out_fmt = "ext" if last else "pad"
        # the previous stage's LeakyReLU / ReLU backward runs in the epilogue of this stage's input-gradient kernel
        # (mask = this stage's saved input, a padded buffer)
        p.fuse = prev is not None and prev.bn is None and prev.act[0] != ACT_NONE
        plans.append(p)
        in_shape = p.out_shape
    return plans


def _chan_sums(buf, c):
    """per-channel sum of a buffer in either format -> fp32 [c]"""
    n, cc, h, w = buf.nchw
    if buf.fmt == "ext" and h * w == 1 and cc == c and buf.t.dtype == torch.float32:
        return Fn.channel_sum(buf.t)          # [n, c, 1, 1] head outputs: one block per channel, a few microseconds
    sums = torch.zeros(2 * c, device=buf.t.device, dtype=torch.float64)
    d = t4(buf.view())
    call("eadgan_bn_stats", C.byref(d), n, c, h, w, ptr(sums), stream())
    return sums[:c].float()


def _r64(v):
    return (v + 63) // 64 * 64


class _Arena:
    """one zero-filled fp64 buffer handed out in slices (16-byte aligned)"""

    def __init__(self, n, dev):
        self.buf = torch.zeros(n + 2, device=dev, dtype=torch.float64) if n > 0 else None
        self.off = 0

    def take(self, n):
        n2 = (n + 1) // 2 * 2
        if self.buf is None or self.off + n2 > self.buf.numel():
            return torch.zeros(n, device=self.buf.device if self.buf is not None else "cuda", dtype=torch.float64)
        out = self.buf[self.off:self.off + n]
        self.off += n2
        return out


class _Saved:
    """what the forward of one stage leaves for its backward, and the stage's weight in every form a kernel reads"""
    # a BatchNorm stage keeps its conv output ``pre`` and the normalisation it applied: ``mean`` / ``invstd`` of the
    # batch in training mode; in eval mode ``mean`` / ``invstd`` are running_mean / running_var, with ``eps``
    __slots__ = ("w", "src", "lazy", "pi", "has_b", "inp", "y", "R", "a", "pre", "mean", "invstd", "eps", "gamma",
                 "beta", "count", "sum_x")

    def __init__(self, w, src, pi, has_b):
        self.w, self.src, self.pi, self.has_b = w, src, pi, has_b
        self.lazy = src is not None and len(src) > 2 and bool(src[2])
        self.R = self.a = self.pre = None

    def values(self):
        """the weight VALUES (W / sigma for spectral-normalised layers), materialised on first use"""
        if self.lazy:
            Fn.spectral_norm_materialize(self.src[0], self.src[1], self.w)
            self.lazy = False
        return self.w.contiguous()

    def packed(self, direction, ca):
        """(bf16 GEMM operand of the weight for `direction`, sigma or None)"""
        if self.src is not None:
            return tc.pack_w_cached(self.src[0], direction, ca), self.src[1]
        return tc.pack_w(self.values(), None, direction, ca), None

    def packed_thin(self, direction):
        if self.src is not None:
            return tc.thin_pack_w_cached(self.src[0], direction), self.src[1]
        return tc.thin_pack_w(self.values(), direction), None


class _ChainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, stages, srcs, *params):
        st_ = stream()
        dev = x.device
        plans = _plan_kernels(stages, tuple(x.shape))
        cur = _Buf(x.contiguous(), "ext")
        saved = []
        pi = 0
        # ONE zero fill for all per-channel fp64 statistics vectors of this forward (a fill kernel per BatchNorm layer
        # was ~40 launches of a few microseconds per step)
        arena = _Arena(sum(2 * p.out_shape[1] for p in plans if p.bn == "train"), dev)
        for si, (st, p) in enumerate(zip(stages, plans)):
            sv = _Saved(params[pi], srcs[si], pi, params[pi + 1] is not None)
            b = params[pi + 1]
            pi += 4 if st.bn is not None else 2
            d, conv, last = p.d, st.kind == "conv", si == len(stages) - 1
            out_shape = p.out_shape
            cout = out_shape[1]
            epi_act = st.act if st.bn is None else (ACT_NONE, 0.0)
            stats = arena.take(2 * cout) if p.bn == "train" else None   # eval: running statistics, nothing to fuse
            # a conv reads its big map zero-padded to p.ca channels: a padded buffer of fewer channels (the output of a
            # SIMT stage onto 5..31 channels) is copied into a channel-padded one
            in_c = p.ca if conv else p.in_shape[1]
            if cur.fmt == p.in_fmt and (cur.fmt == "ext" or cur.t.shape[3] == in_c):
                inp = cur
            else:
                inp = _Buf(tc.to_padded(cur.view(), in_c), "pad")
            if p.fwd == "thin" and conv:
                sv.R = tc.thin_expand(inp.view())
                wpk, sg = sv.packed_thin("fprop")
                out_t = tc.thin_fprop(sv.R, wpk, b, d.c, cout, *epi_act, stats=stats, sigma=sg)
            elif p.fwd == "thin":      # ConvTranspose onto the image: GEMM over input pixels + col2im epilogue
                wpk, sg = sv.packed_thin("dgrad")
                out_t = tc.thin_dgrad(inp.t, wpk, b, d.c, *epi_act, sigma=sg)
            elif p.fwd == "dense_T":
                sv.a = tc.pad_rows(inp.t.reshape(d.n, d.k), _r64(d.k))
                out_t = tc.dense_scatter(sv.a, tc.dense_pack(sv.values(), _r64(d.k), False), b, d.c)
            elif p.fwd == "dense_C":
                out_t = tc.dense_gather(inp.t, tc.dense_pack(sv.values(), 32, True), b, d.k).view(out_shape)
            elif p.fwd == "tc" and conv:
                wpk, sg = sv.packed("fprop", p.ca)
                out_t = tc.fprop(inp.t, wpk, b, cout, *epi_act, out_f32_nchw=last, stats=stats, sigma=sg)
            elif p.fwd == "tc":
                wpk, sg = sv.packed("dgrad", p.ca)
                out_t = tc.dgrad(inp.t, wpk, b, p.ca, *epi_act, out_f32_nchw=last, stats=stats,
                                 c_real=d.c if p.ca != d.c else 0, sigma=sg)
            else:
                out_t = (torch.empty(out_shape, device=dev, dtype=torch.float32) if last
                         else tc.alloc_padded(out_shape[0], out_shape[2], out_shape[3], cout, dev))
                ind, outd = t4(inp.view()), t4(out_t if last else tc.interior(out_t))
                call("eadgan_conv_fprop" if conv else "eadgan_conv_dgrad", C.byref(d), C.byref(ind),
                     ptr(sv.values()), ptr(b), epi_act[0], float(epi_act[1]), C.byref(outd), None, ACT_NONE, 0.0, st_)
                if stats is not None:
                    call("eadgan_bn_stats", C.byref(outd), out_shape[0], cout, out_shape[2], out_shape[3],
                         ptr(stats), st_)
            out = _Buf(out_t, p.out_fmt)
            sv.inp = inp
            if p.bn is not None:
                bn = st.bn
                gamma, beta = params[pi - 2], params[pi - 1]
                y = _Buf(tc.alloc_padded(out_shape[0], out_shape[2], out_shape[3], cout, dev), "pad")
                if p.bn == "eval":
                    # running statistics: no statistics pass, no finalize, no cross-rank communication, no update
                    xd, yd = t4(out.view()), t4(y.view())
                    call("eadgan_bn_eval", C.byref(xd), out_shape[0], cout, out_shape[2], out_shape[3],
                         ptr(bn.running_mean), ptr(bn.running_var), float(bn.eps), ptr(gamma), ptr(beta), st.act[0],
                         float(st.act[1]), C.byref(yd), st_)
                    sv.mean, sv.invstd, sv.eps = bn.running_mean, bn.running_var, float(bn.eps)
                else:
                    sv.mean, sv.invstd, sv.count, sv.sum_x = Fn.bn_train_forward(
                        out.view(), stats, gamma, beta, bn.running_mean, bn.running_var, bn.momentum, bn.eps, *st.act,
                        y.view(), keep_sum_x=True)
                sv.pre, sv.gamma, sv.beta = out, gamma, beta
                out = y
            sv.y = out
            if gate_log is not None and st.act[0] in (L.ACT_RELU, L.ACT_LRELU):
                gate_log[-1][1].append(out.view() > 0)
            saved.append(sv)
            cur = out
        # the returned tensor is saved through autograd (no ctx <-> output reference cycle)
        saved[-1].y = None
        ctx.save_for_backward(cur.t)
        ctx.stages, ctx.plans, ctx.saved = stages, plans, saved
        return cur.t

    @staticmethod
    def backward(ctx, gout):
        stages, plans, saved = ctx.stages, ctx.plans, ctx.saved
        saved[-1].y = _Buf(ctx.saved_tensors[0], "ext")
        st_ = stream()
        dev = gout.device
        g = _Buf(gout.contiguous(), "ext")
        g_masked = False
        db_sums = None   # fp64 per-channel sums of g, accumulated by the epilogue of the kernel that produced g
        grads = []
        arena = _Arena(sum(3 * max(p.d.k, p.d.c) for p in plans), dev)   # every fp64 sum vector of this backward
        for si in range(len(stages) - 1, -1, -1):
            st, p, sv = stages[si], plans[si], saved[si]
            d, conv = p.d, st.kind == "conv"
            cout = p.out_shape[1]
            dgamma = dbeta = None
            # which parameter gradients autograd actually wants (inputs: x, stages, srcs, then w, b[, gamma, beta] per
            # stage).  A step driver freezes the networks a phase's optimiser does not own (phase G: D), so their
            # weight-gradient GEMMs, bias sums and spectral-norm backward are never launched (SURVEY.md section 7.3-8)
            need_dw = ctx.needs_input_grad[3 + sv.pi]
            need_db = sv.has_b and ctx.needs_input_grad[3 + sv.pi + 1]
            need_dx = si > 0 or ctx.needs_input_grad[0]
            # ---- 1. gradient w.r.t. the conv output (pre-BN / pre-activation) ----------------
            if p.bn is not None:
                # in place: dz overwrites g.  dgamma, dbeta and the conv-bias gradient come from the pass's fp64 sums
                sums, gv = arena.take(2 * cout), g.view()
                if p.bn == "eval":
                    dgamma, dbeta, db_bn = Fn.bn_eval_backward(gv, sv.pre.view(), sv.y.view(), sv.mean, sv.invstd,
                                                               sv.eps, sv.gamma, sv.beta, *st.act, sums, gv,
                                                               want_dbias=sv.has_b)
                else:
                    dgamma, dbeta, db_bn = Fn.bn_train_backward(gv, sv.pre.view(), sv.y.view(), sv.mean, sv.invstd,
                                                                sv.gamma, sv.beta, *st.act, sv.count, sums, gv,
                                                                sum_x=sv.sum_x if sv.has_b else None)
                dz = g
            elif st.act[0] != ACT_NONE and not g_masked:
                if g.fmt != "ext" or sv.y.fmt != "ext":
                    raise RuntimeError("eadgan_b200.chain: unfused activation backward on a private buffer")
                dz = _Buf(Fn.act_bwd(g.t, sv.y.t, st.act[0], st.act[1]), "ext")
            else:
                dz = g
            if not need_db:
                db = None
            elif st.bn is not None:
                db = db_bn
            elif db_sums is not None and dz is g:
                db = torch.empty(cout, device=dev, dtype=torch.float32)
                call("eadgan_f64_to_f32", ptr(db_sums), ptr(db), cout, st_)
            else:
                db = _chan_sums(dz, cout)
            db_sums = None
            # the dx computed here IS the previous stage's pre-activation gradient when that stage has no BN (its
            # activation backward, if any, is fused): let the producing epilogue also sum it per channel (= that
            # stage's bias gradient), instead of a separate pass over dx
            want_sums = (si > 0 and stages[si - 1].bn is None and saved[si - 1].has_b
                         and ctx.needs_input_grad[3 + saved[si - 1].pi + 1] and p.in_shape[1] <= 1024)
            sums_buf = arena.take(p.in_shape[1]) if want_sums else None
            # ---- 2. weight gradient ------------------------------------------------------------------
            x_big, dy_small = (sv.inp, dz) if conv else (dz, sv.inp)
            r, a = sv.R, sv.a       # row-expanded image (thin) / small map as GEMM rows (dense) of the forward
            if p.fwd == "thin" and not conv and (need_dw or (need_dx and p.dx == "thin")):
                r = tc.thin_expand(dz.view())          # the image gradient is this stage's big map
            if p.fwd == "dense_C":
                a = tc.pad_rows(dz.t.reshape(d.n, d.k), 64)
            dw = None
            if not need_dw:
                pass
            elif p.wgrad == "thin":
                dw = tc.thin_wgrad(r, dy_small.padded(), d.c)
            elif p.wgrad == "dense":
                dw = tc.dense_wgrad(a, x_big.padded(), d.k)
            elif p.wgrad == "tc":
                xb = x_big.t if x_big.fmt == "pad" else tc.to_padded(x_big.t, p.ca)
                if not conv and p.ca != d.c:
                    dz = _Buf(xb, "pad")  # reuse the channel-padded copy for the input gradient below
                dw = tc.wgrad(xb, dy_small.padded(), c_real=d.c if p.ca != d.c else 0)
            else:
                dw = torch.empty_like(sv.w, memory_format=torch.contiguous_format)
                Fn.conv_wgrad(d, t4(x_big.view()), t4(dy_small.view()), dw)
            # ---- 3. input gradient -------------------------------------------------------------------
            if need_dx:
                mask = sv.inp.t if p.fuse else None
                mask_act, mask_slope = stages[si - 1].act if p.fuse else (ACT_NONE, 0.0)
                if p.dx == "thin" and conv:
                    wpk, sg = sv.packed_thin("dgrad")
                    dx_t = tc.thin_dgrad(dz.padded(), wpk, None, d.c, sigma=sg)
                elif p.dx == "thin":
                    wpk, sg = sv.packed_thin("fprop")
                    dx_t = tc.thin_fprop(r, wpk, None, d.c, d.k, mask=mask, mask_mode=mask_act, slope=mask_slope,
                                         stats=sums_buf, stats_mode=2, sigma=sg)
                elif p.dx == "dense":
                    dx_t = tc.dense_scatter(a, tc.dense_pack(sv.values(), 64, False), None, d.c, mask=mask,
                                            mask_act=mask_act, slope=mask_slope, chan_sums=sums_buf)
                elif p.dx == "tc" and conv:
                    wpk, sg = sv.packed("dgrad", p.ca)
                    dx_t = tc.dgrad(dz.padded(), wpk, None, p.ca, mask=mask, mask_mode=mask_act, slope=mask_slope,
                                    out_f32_nchw=si == 0, c_real=d.c if p.ca != d.c else 0, stats=sums_buf,
                                    stats_mode=2, sigma=sg)
                elif p.dx == "tc":
                    wpk, sg = sv.packed("fprop", p.ca)
                    dzp = dz.t if dz.fmt == "pad" else tc.to_padded(dz.t, p.ca)
                    dx_t = tc.fprop(dzp, wpk, None, d.k, mask=mask, mask_mode=mask_act, slope=mask_slope,
                                    out_f32_nchw=si == 0, stats=sums_buf, stats_mode=2, sigma=sg)
                else:
                    ic, ih, iw = p.in_shape[1:]
                    dx_t = (tc.alloc_padded(d.n, ih, iw, ic, dev) if si > 0
                            else torch.empty(p.in_shape, device=dev, dtype=torch.float32))
                    dzd, dxd = t4(dz.view()), t4(dx_t if si == 0 else tc.interior(dx_t))
                    md = t4(sv.inp.view()) if p.fuse else None
                    call("eadgan_conv_dgrad" if conv else "eadgan_conv_fprop", C.byref(d), C.byref(dzd),
                         ptr(sv.values()), None, ACT_NONE, 0.0, C.byref(dxd), C.byref(md) if p.fuse else None,
                         mask_act, float(mask_slope), st_)
                g, g_masked = _Buf(dx_t, "ext" if si == 0 else "pad"), p.fuse
                db_sums = sums_buf if p.dx != "simt" else None
            stage_grads = [dw, db]
            if st.bn is not None:
                stage_grads += [dgamma, dbeta]
            grads = stage_grads + grads
        dx0 = g.t if ctx.needs_input_grad[0] else None
        ctx.saved = ctx.plans = None
        return (dx0, None, None, *grads)
