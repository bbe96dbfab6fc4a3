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
  * layers the tensor-core path does not cover (Cin = 3 first layer, Cout = 3 / 19 last layers,
    the 1x1-input ConvTranspose) run on the generic SIMT kernels directly on the same buffers
    (strided bf16 views) -- there is no torch / cuDNN fallback anywhere.

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
    cur = torch.cuda.current_stream()
    side = _sn_streams.get(w0.device)
    if side is None:
        side = _sn_streams[w0.device] = torch.cuda.Stream(device=w0.device)
    side.wait_stream(cur)          # the weights (last optimiser step) and every earlier u / v update are visible
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
    dev = todo[0].device
    cur = torch.cuda.current_stream()
    side = _sn_streams.get(dev)
    if side is None:
        side = _sn_streams[dev] = torch.cuda.Stream(device=dev)
    side.wait_stream(cur)          # the optimiser step (and every earlier consumer of the old packs) comes first
    with torch.cuda.stream(side):
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
    if any(st.bn is not None and not st.bn.training for st in stages):
        return None  # eval-mode BN: per-op path
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
    if direction == "dgrad":      # GEMM + col2im epilogue: 32-wide small map, <= 3 image channels
        return (d.k % 64 == 0 or d.k == 32) and d.q == 32 and d.c <= 3
    return d.k % 32 == 0 and d.q <= 64  # wgrad


def _impl(st, d, last):
    """which kernel family runs the forward of this stage."""
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


class _ChainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, stages, srcs, *params):
        st_ = stream()
        dev = x.device
        cur = _Buf(x.contiguous(), "ext")
        saved = []
        pi = 0
        # ONE zero fill for all per-channel fp64 statistics vectors of this forward (a fill kernel per BatchNorm layer
        # was ~40 launches of a few microseconds per step)
        arena = _Arena(sum(2 * (s_.conv.weight.shape[0] if s_.kind == "conv" else s_.conv.weight.shape[1])
                           for s_ in stages if s_.bn is not None), dev)
        for si, st in enumerate(stages):
            w, b = params[pi], params[pi + 1]
            pi += 2
            gamma = beta = None
            if st.bn is not None:
                gamma, beta = params[pi], params[pi + 1]
                pi += 2
            last = si == len(stages) - 1
            d = _geom(st, cur.nchw)
            direction = "fprop" if st.kind == "conv" else "dgrad"
            out_shape = (d.n, d.k, d.p, d.q) if st.kind == "conv" else (d.n, d.c, d.h, d.w)
            cout = out_shape[1]
            epi_act = st.act if st.bn is None else (ACT_NONE, 0.0)
            stats = arena.take(2 * cout) if st.bn is not None else None
            wc = w.contiguous()
            impl = _impl(st, d, last)
            rec = {"d": d, "w": wc, "has_b": b is not None, "impl": impl, "pi": pi - (4 if st.bn is not None else 2)}
            src = srcs[si]
            lazy = [src is not None and len(src) > 2 and bool(src[2])]

            def wvals(_src=src, _wc=wc, _w=w, _lazy=lazy):
                """the weight VALUES (W / sigma for spectral-normalised layers), materialised on first use"""
                if _lazy[0]:
                    Fn.spectral_norm_materialize(_src[0], _src[1], _w)
                    _lazy[0] = False
                return _wc if _wc.data_ptr() == _w.data_ptr() else _w.contiguous()
            rec["wvals"] = wvals

            def packed(direction, ca, _src=src):
                """(bf16 GEMM operand, sigma) of this stage's weight for `direction`"""
                if _src is not None and tuple(_src[0].shape[2:]) == (4, 4):
                    return tc.pack_w_cached(_src[0], direction, ca), _src[1]
                return tc.pack_w(wvals(), None, direction, ca), None
            rec["packed"] = packed

            def packed_thin(direction, _src=src):
                if _src is not None:
                    return tc.thin_pack_w_cached(_src[0], direction), _src[1]
                return tc.thin_pack_w(wvals(), direction), None
            rec["packed_thin"] = packed_thin
            if impl == "thin" and st.kind == "conv":
                inp = cur
                r = tc.thin_expand(cur.view())
                rec["R"] = r
                wpk, sg = packed_thin("fprop")
                if last:
                    raise RuntimeError("eadgan_b200.chain: a thin conv cannot be the last stage")
                out = _Buf(tc.thin_fprop(r, wpk, b, d.c, cout, epi_act[0], epi_act[1], stats=stats, sigma=sg), "pad")
            elif impl == "thin":       # ConvTranspose onto the image: GEMM over input pixels + col2im epilogue
                inp = _Buf(cur.padded(), "pad")
                wpk, sg = packed_thin("dgrad")
                out = _Buf(tc.thin_dgrad(inp.t, wpk, b, d.c, epi_act[0], epi_act[1], sigma=sg), "ext")
            elif impl == "dense_T":      # 1x1 -> 4x4 ConvTranspose: batch GEMM, scatter epilogue
                a = tc.pad_rows(cur.t.reshape(d.n, d.k), _r64(d.k))
                out = _Buf(tc.dense_scatter(a, tc.dense_pack(wvals(), _r64(d.k), False), b, d.c), "pad")
                inp = cur
                rec["a"] = a
            elif impl == "dense_C":    # 4x4 -> 1x1 Conv head: batch GEMM, gather prologue
                inp = _Buf(cur.padded(), "pad")
                o = tc.dense_gather(inp.t, tc.dense_pack(wvals(), 32, True), b, d.k)
                out = _Buf(o.view(d.n, d.k, 1, 1), "ext")
            elif impl == "tc":
                ca = _calloc(d)
                if st.kind == "conv":
                    inp = _Buf(cur.t if cur.fmt == "pad" else tc.to_padded(cur.t, ca), "pad")
                    wpk, sg = packed("fprop", ca)
                    out_t = tc.fprop(inp.t, wpk, b, cout, epi_act[0], epi_act[1], out_f32_nchw=last, stats=stats,
                                     sigma=sg)
                else:
                    inp = _Buf(cur.padded(), "pad")
                    wpk, sg = packed("dgrad", ca)
                    out_t = tc.dgrad(inp.t, wpk, b, ca, epi_act[0], epi_act[1], out_f32_nchw=last, stats=stats,
                                     c_real=d.c if ca != d.c else 0, sigma=sg)
                out = _Buf(out_t, "ext" if last else "pad")
            else:
                inp = cur
                if last:
                    out = _Buf(torch.empty(out_shape, device=dev, dtype=torch.float32), "ext")
                else:
                    out = _Buf(tc.alloc_padded(out_shape[0], out_shape[2], out_shape[3], cout, dev), "pad")
                ind, outd = t4(inp.view()), t4(out.view())
                call("eadgan_conv_fprop" if st.kind == "conv" else "eadgan_conv_dgrad", C.byref(d), C.byref(ind),
                     ptr(wvals()), ptr(b), epi_act[0], float(epi_act[1]), C.byref(outd), None, ACT_NONE, 0.0, st_)
                if stats is not None:
                    call("eadgan_bn_stats", C.byref(outd), out_shape[0], cout, out_shape[2], out_shape[3],
                         ptr(stats), st_)
            rec["inp"] = inp
            if st.bn is not None:
                bn = st.bn
                n_local = float(out_shape[0] * out_shape[2] * out_shape[3])
                count = n_local
                sum_x = stats                      # this rank's S(x) (first C entries), kept for backward
                if Fn._allreduce_sum is not None:
                    sum_x = stats[:cout].clone()
                    Fn._allreduce_sum(stats)
                    count *= Fn._world_size
                mean = torch.empty(cout, device=dev, dtype=torch.float32)
                invstd = torch.empty(cout, device=dev, dtype=torch.float32)
                call("eadgan_bn_finalize", ptr(stats), count, cout, float(bn.eps), float(bn.momentum), ptr(mean),
                     ptr(invstd), ptr(bn.running_mean), ptr(bn.running_var), st_)
                y = _Buf(tc.alloc_padded(out_shape[0], out_shape[2], out_shape[3], cout, dev), "pad")
                xd, yd = t4(out.view()), t4(y.view())
                call("eadgan_bn_apply", C.byref(xd), out_shape[0], cout, out_shape[2], out_shape[3], ptr(mean),
                     ptr(invstd), ptr(gamma), ptr(beta), st.act[0], float(st.act[1]), C.byref(yd), st_)
                rec.update(pre=out, mean=mean, invstd=invstd, gamma=gamma, beta=beta, count=count, n_local=n_local,
                           sum_x=sum_x)
                out = y
            rec["y"] = out
            if gate_log is not None and st.act[0] in (L.ACT_RELU, L.ACT_LRELU):
                gate_log[-1][1].append(out.view() > 0)
            saved.append(rec)
            cur = out
        # the returned tensor is saved through autograd (no ctx <-> output reference cycle)
        saved[-1]["y"] = None
        ctx.save_for_backward(cur.t)
        ctx.stages, ctx.saved = stages, saved
        return cur.t

    @staticmethod
    def backward(ctx, gout):
        stages, saved = ctx.stages, ctx.saved
        saved[-1]["y"] = _Buf(ctx.saved_tensors[0], "ext")
        st_ = stream()
        dev = gout.device
        g = _Buf(gout.contiguous(), "ext")
        g_masked = False
        db_sums = None   # fp64 per-channel sums of g, accumulated by the epilogue of the kernel that produced g
        grads = []
        arena = _Arena(sum(3 * max(sv_["d"].k, sv_["d"].c) for sv_ in saved), dev)   # every fp64 sum vector of this backward
        for si in range(len(stages) - 1, -1, -1):
            st, sv = stages[si], saved[si]
            d, impl = sv["d"], sv["impl"]
            cout = d.k if st.kind == "conv" else d.c
            n, _, oh, ow = sv["y"].nchw
            dgamma = dbeta = None
            # which parameter gradients autograd actually wants (inputs: x, stages, srcs, then w, b[, gamma, beta] per
            # stage).  A step driver freezes the networks a phase's optimiser does not own (phase G: D), so their
            # weight-gradient GEMMs, bias sums and spectral-norm backward are never launched (SURVEY.md section 7.3-8)
            need_dw = ctx.needs_input_grad[3 + sv["pi"]]
            need_db = sv["has_b"] and ctx.needs_input_grad[3 + sv["pi"] + 1]
            # ---- 1. gradient w.r.t. the conv output (pre-BN / pre-activation) ----------------
            if st.bn is not None:
                sums = arena.take(2 * cout)
                gd, xd, yd = t4(g.view()), t4(sv["pre"].view()), t4(sv["y"].view())
                call("eadgan_bn_bwd_reduce", C.byref(gd), C.byref(xd), C.byref(yd), n, cout, oh, ow, ptr(sv["mean"]),
                     ptr(sv["invstd"]), ptr(sv["gamma"]), ptr(sv["beta"]), st.act[0], float(st.act[1]), ptr(sums), st_)
                local = sums
                if Fn._allreduce_sum is not None:
                    local = sums.clone()
                    Fn._allreduce_sum(sums)
                call("eadgan_bn_bwd_apply", C.byref(gd), C.byref(xd), C.byref(yd), n, cout, oh, ow, ptr(sv["mean"]),
                     ptr(sv["invstd"]), ptr(sv["gamma"]), ptr(sv["beta"]), st.act[0], float(st.act[1]), ptr(sums),
                     float(sv["count"]), C.byref(gd), st_)  # in place: dz overwrites g
                # dgamma / dbeta, and the conv-bias gradient (= sum of dx, zero up to rounding) in closed
                # form from the fp64 sums: no extra pass over dz
                small = torch.empty(3 * cout, device=dev, dtype=torch.float32)
                dgamma, dbeta, db_bn = small[:cout], small[cout:2 * cout], small[2 * cout:]
                call("eadgan_bn_bwd_finalize", ptr(local), ptr(sums), ptr(sv["sum_x"]), float(sv["n_local"]),
                     float(sv["count"]), ptr(sv["mean"]), ptr(sv["invstd"]), ptr(sv["gamma"]), cout, ptr(dgamma),
                     ptr(dbeta), ptr(db_bn) if sv["has_b"] else None, st_)
                dz = g
            elif st.act[0] != ACT_NONE and not g_masked:
                if g.fmt != "ext" or sv["y"].fmt != "ext":
                    raise RuntimeError("eadgan_b200.chain: unfused activation backward on a private buffer")
                dz = _Buf(Fn.act_bwd(g.t, sv["y"].t, st.act[0], st.act[1]), "ext")
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
            prev = stages[si - 1] if si > 0 else None
            need_dx = si > 0 or ctx.needs_input_grad[0]
            fuse = need_dx and prev is not None and prev.bn is None and prev.act[0] != ACT_NONE
            mask_act, mask_slope = (prev.act if fuse else (ACT_NONE, 0.0))
            in_shape = (d.n, d.c, d.h, d.w) if st.kind == "conv" else (d.n, d.k, d.p, d.q)
            dx = None
            # the dx computed here IS the previous stage's pre-activation gradient when that stage has no BN and
            # its activation backward is fused (or absent): let the producing epilogue also sum it per channel
            # (= that stage's bias gradient), instead of a separate pass over dx
            want_sums = (need_dx and prev is not None and prev.bn is None and saved[si - 1]["has_b"]
                         and ctx.needs_input_grad[3 + saved[si - 1]["pi"] + 1]
                         and (fuse or prev.act[0] == ACT_NONE) and in_shape[1] <= 1024)
            sums_buf = arena.take(in_shape[1]) if want_sums else None
            sums_used = False
            # ---- 2./3. weight gradient and input gradient -----------------------------------------
            if impl == "thin":
                dw = None
                if st.kind == "conv":      # big map = stage input (image), small map = dz
                    r = sv["R"]
                    if not need_dw:
                        pass
                    elif _thin_ok(d, "wgrad"):
                        dw = tc.thin_wgrad(r, dz.padded(), d.c)
                    else:
                        dw = torch.empty_like(sv["w"])
                        Fn.conv_wgrad(d, t4(sv["inp"].view()), t4(dz.view()), dw)
                    if need_dx and si == 0 and _thin_ok(d, "dgrad"):
                        wpk, sg = sv["packed_thin"]("dgrad")
                        dx = _Buf(tc.thin_dgrad(dz.padded(), wpk, None, d.c, sigma=sg), "ext")
                else:                      # big map = dz (image gradient), small map = stage input
                    r = tc.thin_expand(dz.view()) if (need_dw or (need_dx and si > 0)) else None
                    if not need_dw:
                        pass
                    elif _thin_ok(d, "wgrad"):
                        dw = tc.thin_wgrad(r, sv["inp"].t, d.c)
                    else:
                        dw = torch.empty_like(sv["w"])
                        Fn.conv_wgrad(d, t4(dz.view()), t4(sv["inp"].view()), dw)
                    if need_dx and si > 0:
                        wpk, sg = sv["packed_thin"]("fprop")
                        dx = _Buf(tc.thin_fprop(r, wpk, None, d.c, in_shape[1], mask=sv["inp"].t if fuse else None,
                                                mask_mode=mask_act, slope=mask_slope, stats=sums_buf, stats_mode=2,
                                                sigma=sg), "pad")
                        sums_used = want_sums
            elif impl == "dense_T":
                dw = tc.dense_wgrad(sv["a"], dz.padded(), d.k) if need_dw else None
            elif impl == "dense_C":
                a = tc.pad_rows(dz.t.reshape(d.n, d.k), 64)
                dw = tc.dense_wgrad(a, sv["inp"].t, d.k) if need_dw else None
                if need_dx and (si > 0) and (not fuse or sv["inp"].fmt == "pad"):
                    dx = _Buf(tc.dense_scatter(a, tc.dense_pack(sv["wvals"](), 64, False), None, d.c,
                                               mask=sv["inp"].t if fuse else None, mask_act=mask_act,
                                               slope=mask_slope, chan_sums=sums_buf), "pad")
                    sums_used = want_sums
            else:
                ca = _calloc(d) if impl == "tc" else d.c
                x_big, dy_small = (sv["inp"], dz) if st.kind == "conv" else (dz, sv["inp"])
                if not need_dw:
                    dw = None
                elif impl == "tc" and _tc_ok(d, "wgrad"):
                    xb = x_big.t if x_big.fmt == "pad" else tc.to_padded(x_big.t, ca)
                    if st.kind == "convT" and ca != d.c:
                        dz = _Buf(xb, "pad")  # reuse the channel-padded copy for the input gradient below
                        x_big = dz
                    dw = tc.wgrad(xb, dy_small.padded(), c_real=d.c if ca != d.c else 0)
                else:
                    dw = torch.empty_like(sv["w"])
                    Fn.conv_wgrad(d, t4(x_big.view()), t4(dy_small.view()), dw)
                if need_dx:
                    direction = "dgrad" if st.kind == "conv" else "fprop"
                    tc_dx = impl == "tc" and _tc_ok(d, direction) and (not fuse or sv["inp"].fmt == "pad")
                    if tc_dx and ca != d.c and st.kind == "conv" and si > 0:
                        tc_dx = False  # zero-padded result channels need the fp32 NCHW epilogue (si == 0)
                    if tc_dx:
                        wpk, sg = sv["packed"](direction, ca)
                        if st.kind == "conv":
                            dx_t = tc.dgrad(dz.padded(), wpk, None, ca, mask=sv["inp"].t if fuse else None,
                                            mask_mode=mask_act, slope=mask_slope, out_f32_nchw=(si == 0),
                                            c_real=d.c if ca != d.c else 0, stats=sums_buf, stats_mode=2, sigma=sg)
                        else:
                            dzp = dz.t if dz.fmt == "pad" else tc.to_padded(dz.t, ca)
                            dx_t = tc.fprop(dzp, wpk, None, in_shape[1], mask=sv["inp"].t if fuse else None,
                                            mask_mode=mask_act, slope=mask_slope, out_f32_nchw=(si == 0),
                                            stats=sums_buf, stats_mode=2, sigma=sg)
                        dx = _Buf(dx_t, "ext" if si == 0 else "pad")
                        sums_used = want_sums
            if need_dx and dx is None:   # generic SIMT input gradient on the same buffers
                if si > 0:
                    dx = _Buf(tc.alloc_padded(in_shape[0], in_shape[2], in_shape[3], in_shape[1], dev), "pad")
                else:
                    dx = _Buf(torch.empty(in_shape, device=dev, dtype=torch.float32), "ext")
                dzv = dz.view()
                if dzv.shape[1] != cout:
                    dzv = dzv[:, :cout]
                dzd, dxd = t4(dzv), t4(dx.view())
                md = t4(sv["inp"].view()) if fuse else None
                call("eadgan_conv_dgrad" if st.kind == "conv" else "eadgan_conv_fprop", C.byref(d), C.byref(dzd),
                     ptr(sv["wvals"]()), None, ACT_NONE, 0.0, C.byref(dxd), C.byref(md) if fuse else None, mask_act,
                     float(mask_slope), st_)
            if need_dx:
                g, g_masked = dx, fuse
                db_sums = sums_buf if sums_used else None
            stage_grads = [dw, db]
            if st.bn is not None:
                stage_grads += [dgamma, dbeta]
            grads = stage_grads + grads
        dx0 = g.t if ctx.needs_input_grad[0] else None
        ctx.saved = None
        return (dx0, None, None, *grads)
