"""Test helper: a stock-torch evaluation of a conv stack that rounds to bf16 at exactly the
points where eadgan_b200.chain stores bf16 (activations between layers, and the operands of the
tensor-core layers).  With the rounding points matched, ReLU / LeakyReLU gates agree between the
two runs, so what is left is accumulation order -- this is the "plain PyTorch fp32 reference of the
same op" for the bf16 mode.  (Against the un-rounded fp32 oracle a bf16 run of ANY implementation
flips ~0.1 % of the LeakyReLU(0.1)/ReLU gates, which alone moves max-normalised gradient errors to
5-20 % at small batch: see DESIGN.md "parity protocol".)

By default rounding is straight-through in backward (gradients are not rounded; ours rounds them to
bf16 when it stores them, a smooth <=0.4 % perturbation).  The options of ``emulate`` turn it into an
fp64 referee that also matches the backward: forced gates, gradients rounded where the chain stores them,
and spectral-normalised tensor-core layers evaluated the way their kernels evaluate them.

BatchNorm follows the mode the chain planned for it (``_StagePlan.bn``): the batch's statistics in training mode, the
running statistics in eval mode, with the same bf16 rounding points in both.
"""
import torch
import torch.nn.functional as TF
from torch.nn.utils.spectral_norm import SpectralNorm

from eadgan_b200 import chain
from eadgan_b200._lib import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_TANH


def _bf(x):
    return x.bfloat16().to(x.dtype)


class _RoundSTE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return _bf(x)

    @staticmethod
    def backward(ctx, g):
        return g


class _RoundGrad(torch.autograd.Function):
    """identity in forward; rounds the gradient to bf16 in backward (a gradient the chain stores in a bf16 buffer)"""
    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return _bf(g)


def rb(x):
    return _RoundSTE.apply(x)


class _SmoothAct(torch.autograd.Function):
    """tanh / sigmoid whose derivative is taken from the output as the chain saves it: rounded to bf16 when the
    output is a private buffer (every stage but the last), fp32 / fp64 for the chain's result"""
    @staticmethod
    def forward(ctx, h, kind, stored_bf16):
        y = torch.tanh(h) if kind == ACT_TANH else torch.sigmoid(h)
        ctx.kind = kind
        ctx.save_for_backward(_bf(y) if stored_bf16 else y)
        return y

    @staticmethod
    def backward(ctx, g):
        y, = ctx.saved_tensors
        return g * (1 - y * y if ctx.kind == ACT_TANH else y * (1 - y)), None, None


class _Conv(torch.autograd.Function):
    """y = fn(x, w) whose backward reads what the chain's backward kernels read: the incoming gradient rounded to
    bf16 for a direction whose kernel takes it as a bf16 operand (``round_w`` / ``round_x``), and the weight
    ``w_dx`` for the input gradient (the SIMT kernels read fp32 weights where the forward read a bf16 pack)"""
    @staticmethod
    def forward(ctx, x, w, w_dx, fn, round_w, round_x):
        ctx.save_for_backward(x, w, w_dx)
        ctx.fn, ctx.round_w, ctx.round_x = fn, round_w, round_x
        return fn(x, w)

    @staticmethod
    def backward(ctx, g):
        x, w, w_dx = ctx.saved_tensors
        gx = gw = None
        with torch.enable_grad():
            if ctx.needs_input_grad[0]:
                xx = x.detach().requires_grad_()
                gx = torch.autograd.grad(ctx.fn(xx, w_dx.detach()), xx, _bf(g) if ctx.round_x else g)[0]
            if ctx.needs_input_grad[1]:
                ww = w.detach().requires_grad_()
                gw = torch.autograd.grad(ctx.fn(x.detach(), ww), ww, _bf(g) if ctx.round_w else g)[0]
        return gx, gw, None, None, None, None


def _act(h, a):
    kind, slope = a
    if kind == ACT_RELU:
        return torch.relu(h)
    if kind == ACT_LRELU:
        return TF.leaky_relu(h, slope)
    if kind == ACT_TANH:
        return torch.tanh(h)
    if kind == ACT_SIGMOID:
        return torch.sigmoid(h)
    return h


def _sn_sigma(conv):
    """(weight_orig, sigma) of a torch spectral-normalised conv after its pre-forward hook ran, else None"""
    for hook in conv._forward_pre_hooks.values():
        if isinstance(hook, SpectralNorm):
            w = getattr(conv, hook.name + "_orig")
            u, v = getattr(conv, hook.name + "_u"), getattr(conv, hook.name + "_v")
            return w, torch.dot(u, torch.mv(hook.reshape_weight_to_matrix(w), v))
    return None


def emulate(ours_seq, ref_seq, x, update_running=False, gates=None, round_grads=False, sn_epilogue=False):
    """ours_seq: eadgan_b200.nn.Sequential (only its structure / geometry decisions are used);
    ref_seq: torch.nn.Sequential with the same layout holding the parameters to differentiate.

    The computation runs in the dtype of ``x`` and ``ref_seq`` (float64 for a referee); rounding is to bf16 either way.
    A BatchNorm that is in eval mode in ``ours_seq`` (the chain's plan says so) normalises with the running statistics
    of its ref_seq twin and updates nothing.
      update_running: training-mode BatchNorm layers of ref_seq update running_mean / running_var as torch's do;
      gates:        the gate masks of this forward from ``chain.gate_log`` (one per ReLU / LeakyReLU stage, in order),
                    applied as where(mask, h, slope * h), so that both runs differentiate the same branch;
      round_grads:  gradients are rounded to bf16 where the chain stores them (every inter-stage buffer, the
                    BatchNorm dz) and where a tensor-core kernel reads the chain's fp32 result gradient; input gradients
                    on SIMT kernels use the fp32 weights; tanh / sigmoid derivatives come from the stored output;
      sn_epilogue:  a spectral-normalised tensor-core / thin layer is conv(x, rb(weight_orig)) / sigma, as its kernel
                    computes it (bf16 pack of weight_orig, 1 / sigma in the epilogue), not conv(x, rb(weight_orig / sigma)).
    """
    stages = chain._compile(ours_seq)
    assert stages is not None, "not a chain-able Sequential"
    plans = chain._plan_kernels(stages, tuple(x.shape))
    idx = {id(m): i for i, m in enumerate(ours_seq._modules.values())}
    ref_mods = list(ref_seq._modules.values())
    gates = list(gates) if gates is not None else None
    h = x
    for si, (st, p) in enumerate(zip(stages, plans)):
        last = si == len(stages) - 1
        conv = ref_mods[idx[id(st.conv)]]
        for hook in conv._forward_pre_hooks.values():  # spectral norm on the torch side
            hook(conv, (h,))
        tensor_core = p.fwd != "simt"
        w, sigma = conv.weight, None
        hin = rb(h) if (tensor_core or si > 0) else h   # private buffers / tensor-core operands are bf16
        sn = _sn_sigma(conv) if sn_epilogue and p.fwd in ("tc", "thin") else None
        if sn is not None:
            w_orig, sigma = sn
            w = rb(w_orig)
            w_dx = w if p.dx != "simt" else w_orig
        elif tensor_core:
            w = rb(w)
            w_dx = w if p.dx != "simt" else conv.weight
        else:
            w_dx = w
        if st.kind == "conv":
            def fn(a, b, _st=st):
                return TF.conv2d(a, b, None, stride=_st.stride, padding=_st.pad)
        else:
            def fn(a, b, _st=st):
                return TF.conv_transpose2d(a, b, None, stride=_st.stride, padding=_st.pad)
        if round_grads or sigma is not None:
            # the chain's result gradient is fp32: a tensor-core kernel of the last stage reads it rounded to bf16
            h = _Conv.apply(hin, w, w_dx, fn, round_grads and last and p.wgrad != "simt",
                            round_grads and last and p.dx != "simt") if round_grads else fn(hin, w)
            if sigma is not None:
                h = h / sigma
            # the gradient below this stage's output is stored bf16 (the BatchNorm dz, or the next stage's input
            # gradient with this stage's activation backward applied).  The bias gradient sums it BEFORE that rounding
            # where the sums are fused into the producing epilogue or taken in closed form from BatchNorm's fp64 sums,
            # and sums the stored bf16 buffer where the next stage's input gradient runs on SIMT
            round_here = round_grads and not last
            sums_rounded = st.bn is None and not last and (plans[si + 1].dx == "simt"
                                                           or p.out_shape[1] > chain.FUSE_MAX_CH)
            if round_here and not sums_rounded:
                h = _RoundGrad.apply(h)
            if conv.bias is not None:
                h = h + conv.bias[None, :, None, None]
            if round_here and sums_rounded:
                h = _RoundGrad.apply(h)
        elif st.kind == "conv":
            h = TF.conv2d(hin, w, conv.bias, stride=st.stride, padding=st.pad)
        else:
            h = TF.conv_transpose2d(hin, w, conv.bias, stride=st.stride, padding=st.pad)
        if p.bn is not None:
            # both modes round the conv output to bf16 before normalising it (the chain stores it so), and the
            # BatchNorm dz the chain stores in bf16 is the _RoundGrad above
            bn = ref_mods[idx[id(st.bn)]]
            if p.bn == "eval":
                mean, var = bn.running_mean.to(h.dtype), bn.running_var.to(h.dtype)
            else:
                mean = h.mean((0, 2, 3))
                var = h.var((0, 2, 3), unbiased=False)
                if update_running:
                    with torch.no_grad():
                        cnt = h.numel() // h.shape[1]
                        bn.running_mean.mul_(1 - bn.momentum).add_(bn.momentum * mean.detach())
                        bn.running_var.mul_(1 - bn.momentum).add_(bn.momentum * var.detach() * cnt / (cnt - 1))
                        bn.num_batches_tracked.add_(1)
            hb = rb(h)
            h = (hb - mean[None, :, None, None]) * torch.rsqrt(var + bn.eps)[None, :, None, None]
            h = h * bn.weight[None, :, None, None] + bn.bias[None, :, None, None]
        if gates is not None and st.act[0] in (ACT_RELU, ACT_LRELU):
            mask = gates.pop(0)
            h = torch.where(mask, h, h * (0.0 if st.act[0] == ACT_RELU else st.act[1]))
        elif round_grads and st.act[0] in (ACT_TANH, ACT_SIGMOID):
            h = _SmoothAct.apply(h, st.act[0], not last)
        else:
            h = _act(h, st.act)
        if not last:
            if round_grads and st.bn is not None:
                h = _RoundGrad.apply(h)     # the next stage's input gradient, stored bf16 (no activation fused)
            h = rb(h)
    assert not gates, "more gate masks than ReLU / LeakyReLU stages"
    return h
