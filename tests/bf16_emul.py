"""Test helper: a stock-torch fp32 evaluation of a conv stack that rounds to bf16 at exactly the
points where eadgan_b200.chain stores bf16 (activations between layers, and the operands of the
tensor-core layers).  With the rounding points matched, ReLU / LeakyReLU gates agree between the
two runs, so what is left is accumulation order -- this is the "plain PyTorch fp32 reference of the
same op" for the bf16 mode.  (Against the un-rounded fp32 oracle a bf16 run of ANY implementation
flips ~0.1 % of the LeakyReLU(0.1)/ReLU gates, which alone moves max-normalised gradient errors to
5-20 % at small batch: see DESIGN.md "parity protocol".)

Rounding is straight-through in backward (gradients are not rounded; ours rounds them to bf16 when
it stores them, a smooth <=0.4 % perturbation).
"""
import torch
import torch.nn.functional as TF

from eadgan_b200 import chain
from eadgan_b200._lib import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_TANH


class _RoundSTE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.bfloat16().float()

    @staticmethod
    def backward(ctx, g):
        return g


def rb(x):
    return _RoundSTE.apply(x)


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


def emulate(ours_seq, ref_seq, x, update_running=False):
    """ours_seq: eadgan_b200.nn.Sequential (only its structure / geometry decisions are used);
    ref_seq: torch.nn.Sequential with the same layout holding the parameters to differentiate."""
    stages = chain._compile(ours_seq)
    assert stages is not None, "not a chain-able Sequential"
    plans = chain._plan_kernels(stages, tuple(x.shape))
    idx = {id(m): i for i, m in enumerate(ours_seq._modules.values())}
    ref_mods = list(ref_seq._modules.values())
    h = x
    for si, st in enumerate(stages):
        last = si == len(stages) - 1
        conv = ref_mods[idx[id(st.conv)]]
        for hook in conv._forward_pre_hooks.values():  # spectral norm on the torch side
            hook(conv, (h,))
        tensor_core = plans[si].fwd != "simt"
        w = conv.weight
        hin = rb(h) if (tensor_core or si > 0) else h   # private buffers / tensor-core operands are bf16
        if tensor_core:
            w = rb(w)
        if st.kind == "conv":
            h = TF.conv2d(hin, w, conv.bias, stride=st.stride, padding=st.pad)
        else:
            h = TF.conv_transpose2d(hin, w, conv.bias, stride=st.stride, padding=st.pad)
        if st.bn is not None:
            bn = ref_mods[idx[id(st.bn)]]
            mean = h.mean((0, 2, 3))
            var = h.var((0, 2, 3), unbiased=False)
            hb = rb(h)
            h = (hb - mean[None, :, None, None]) * torch.rsqrt(var + bn.eps)[None, :, None, None]
            h = h * bn.weight[None, :, None, None] + bn.bias[None, :, None, None]
        h = _act(h, st.act)
        if not last:
            h = rb(h)
    return h
