"""freeze(): an inference-only snapshot of a trained network, with every eval-mode BatchNorm2d that directly follows a
Conv2d / ConvTranspose2d / Linear and every legacy spectral norm folded into that layer's weight and bias.

A ``.eval()`` network stays differentiable (inverting the generator needs it): each forward stores the pre-BatchNorm
output and normalises it in a separate pass, and recomputes sigma = u^T W v of every spectral-normalised layer.  A
frozen copy does neither.  Its stacks hold only Conv / ConvTranspose (+ bias) (+ activation) stages, which the bf16
chain (eadgan_b200.chain) and the per-operator path run with bias and activation in the GEMM epilogue.

``plan`` decides what folds; ``freeze`` builds the copy.  The argument of ``freeze`` is only read: its parameters,
buffers and the project's per-object caches (packed weights, chain plans, prefetched spectral-norm results) stay as
they are, and the copy shares none of them.
"""
from __future__ import annotations

import copy
import importlib
import itertools
import types
from typing import NamedTuple, Optional

import torch

from . import chain
from . import functional as Fn

_tsn = importlib.import_module("torch.nn.utils.spectral_norm")

# per-object state of the chain executor and of the spectral-norm hooks (modules), and of the pack cache and the fused
# Adam (parameters): a frozen copy starts without any of it
_MODULE_CACHES = ("_eadgan_plan", "_eadgan_sn_queue", "_eadgan_sn_src", "_eadgan_sigma")
_PARAM_CACHES = ("_eadgan_pack_uses", "_eadgan_stepped")
_LAYERS = (torch.nn.Conv2d, torch.nn.ConvTranspose2d, torch.nn.Linear)


class Fold(NamedTuple):
    """One layer of a frozen copy whose weight and bias differ from the original's."""
    layer: str              # qualified name of the Conv2d / ConvTranspose2d / Linear
    bn: Optional[str]       # qualified name of the BatchNorm2d folded into it (dropped from the copy), or None
    sigma: bool             # its legacy spectral norm is folded: weight = weight_orig / sigma, no hook


def _sn_hook(m):
    """the legacy spectral-norm hook of ``m`` that a fold can replace (on ``weight``, over dim 0), else None"""
    hooks = list(m._forward_pre_hooks.values())
    if len(hooks) == 1 and isinstance(hooks[0], _tsn.SpectralNorm) and hooks[0].name == "weight" and hooks[0].dim == 0:
        return hooks[0]
    return None


def _foldable_layer(m):
    """no hooks but (at most) one foldable spectral norm: nothing observes the weight or the output being folded"""
    if m._forward_hooks or m._backward_hooks or m._backward_pre_hooks:
        return False
    return not m._forward_pre_hooks or _sn_hook(m) is not None


def _out_channels(m):
    return m.out_features if isinstance(m, torch.nn.Linear) else m.out_channels


def _foldable_bn(bn, layer):
    """a BatchNorm2d that normalises ``layer``'s output with its running statistics and an affine transform"""
    return (isinstance(bn, torch.nn.BatchNorm2d) and bn.affine and bn.track_running_stats
            and bn.running_mean is not None and bn.num_features == _out_channels(layer)
            and not (bn._forward_hooks or bn._forward_pre_hooks or bn._backward_hooks or bn._backward_pre_hooks))


def plan(module):
    """-> (folds, kept): the ``Fold`` of every layer whose weight ``freeze(module)`` rewrites, in module order, and the
    qualified names of the BatchNorm2d layers it keeps.  A pure function of the module tree; these are the only rules.

    * A Conv2d / ConvTranspose2d / Linear directly followed, inside a Sequential, by a BatchNorm2d with running
      statistics folds it: W' = W * s along the output channels (dim 1 of a ConvTranspose2d weight, dim 0 otherwise),
      b' = (b - running_mean) * s + beta with s = gamma / sqrt(running_var + eps) and b = 0 without a bias.  An
      activation after the BatchNorm stays, and runs fused into the layer's epilogue.
    * A legacy spectral norm folds sigma = u^T W v (torch's eval mode: no power iteration): W' = weight_orig / sigma,
      combined with the BatchNorm's s where both apply.
    * Any other BatchNorm2d stays, and runs as in eval mode: one in front of a conv, or after an activation, would
      fold into the next layer's input side, which is inexact at the zero padding."""
    after = {}
    for seq in module.modules():
        if isinstance(seq, torch.nn.Sequential):
            mods = list(seq._modules.values())
            after.update((id(a), b) for a, b in zip(mods, mods[1:]))
    names = {id(m): n for n, m in module.named_modules()}
    folds, folded = [], set()
    for name, m in module.named_modules():
        if not isinstance(m, _LAYERS) or not _foldable_layer(m):
            continue
        bn = after.get(id(m))
        bn = bn if _foldable_bn(bn, m) else None
        sigma = _sn_hook(m) is not None
        if bn is not None or sigma:
            folds.append(Fold(name, None if bn is None else names[id(bn)], sigma))
            if bn is not None:
                folded.add(id(bn))
    kept = [n for n, m in module.named_modules() if isinstance(m, torch.nn.BatchNorm2d) and id(m) not in folded]
    return folds, kept


def _refuse_train(self, mode=True):
    if mode:
        raise RuntimeError("eadgan_b200.freeze: a frozen copy is inference-only and cannot be put in training mode; "
                           "train the original and call freeze() again")
    return torch.nn.Module.train(self, False)


def _refuse_load(self, *args, **kwargs):
    raise RuntimeError("eadgan_b200.freeze: a frozen copy cannot load a state_dict (its BatchNorm layers and spectral "
                       "norms are folded into the weights); load it into the original and call freeze() again")


def _refuse_grad(module, args, kwargs):
    if any(torch.is_tensor(t) and t.requires_grad for t in itertools.chain(args, kwargs.values())):
        raise RuntimeError("eadgan_b200.freeze: a frozen copy is inference-only and does not differentiate its "
                           "input; use the original in .eval() mode for that")


def _remove_spectral_norm(m, hook):
    """torch.nn.utils.remove_spectral_norm without its final compute_weight (the caller sets the folded weight)"""
    for hooks in (m._forward_pre_hooks, m._state_dict_hooks, m._load_state_dict_pre_hooks):
        for k, h in list(hooks.items()):
            if h is hook or getattr(getattr(h, "hook", h), "fn", None) is hook:
                del hooks[k]
    del m._parameters["weight_orig"], m._buffers["weight_u"], m._buffers["weight_v"]
    m.__dict__.pop("weight", None)


def freeze(module):
    """Return an inference-only copy of ``module`` (a CUDA module built from eadgan_b200.nn, or under patch()) with its
    eval-mode BatchNorm layers and spectral norms folded into the conv / linear weights (the rules are ``plan``'s).

    The copy is a snapshot: it is in eval mode, none of its tensors requires grad, and later changes to ``module``
    (optimiser steps, load_state_dict) do not reach it -- call freeze() again for new weights.  Its forward refuses an
    input that requires grad, and ``.train()`` and ``load_state_dict`` raise.  ``module`` itself is not modified."""
    for t in itertools.chain(module.parameters(), module.buffers()):
        if not t.is_cuda:
            raise RuntimeError(f"eadgan_b200.freeze: expected a CUDA module, found a {t.device} tensor (the fold runs "
                               "on the sm_100a kernels; there is no CPU fallback)")
    folds, _ = plan(module)
    # power iterations prefetched on the chain's side streams write u / v in place: read them after those writes
    cur = torch.cuda.current_stream()
    for side in chain._sn_streams.values():
        cur.wait_stream(side)

    # the copy: deepcopy with the private caches (and the spectral-norm hooks' last W / sigma, an autograd result that
    # deepcopy refuses) mapped to None, then removed
    memo = {}
    for m in module.modules():
        for k in _MODULE_CACHES:
            if k in m.__dict__:
                memo[id(m.__dict__[k])] = None
        for h in m._forward_pre_hooks.values():
            if isinstance(h, _tsn.SpectralNorm) and torch.is_tensor(m.__dict__.get(h.name)):
                memo[id(m.__dict__[h.name])] = None
    frozen = copy.deepcopy(module, memo)
    for m in frozen.modules():
        for k in _MODULE_CACHES:
            m.__dict__.pop(k, None)

    with torch.no_grad():
        for f in folds:
            layer = frozen.get_submodule(f.layer)
            hook = _sn_hook(layer) if f.sigma else None
            bn = frozen.get_submodule(f.bn) if f.bn is not None else None
            w = layer.weight_orig if hook is not None else layer.weight
            sigma = Fn.spectral_norm_sigma(w, layer.weight_u, layer.weight_v, hook.eps) if hook is not None else None
            w_new, b_new = Fn.fold_bn_sn(w, 1 if isinstance(layer, torch.nn.ConvTranspose2d) else 0, sigma, bn,
                                         layer.bias)
            if hook is not None:
                _remove_spectral_norm(layer, hook)
            layer.weight = torch.nn.Parameter(w_new, requires_grad=False)
            if b_new is not None:
                layer.bias = torch.nn.Parameter(b_new, requires_grad=False)
        for f in folds:
            if f.bn is not None:
                parent, _, key = f.bn.rpartition(".")
                delattr(frozen.get_submodule(parent), key)

    torch.nn.Module.train(frozen, False)
    for t in itertools.chain(frozen.parameters(), frozen.buffers()):
        t.requires_grad_(False)
        for k in _PARAM_CACHES:
            t.__dict__.pop(k, None)
    for m in frozen.modules():
        m.train = types.MethodType(_refuse_train, m)
        m._load_from_state_dict = types.MethodType(_refuse_load, m)
        if m is frozen or m._modules:
            # containers only: a hook on a leaf would keep the chain from fusing it
            m.register_forward_pre_hook(_refuse_grad, with_kwargs=True)
    return frozen
