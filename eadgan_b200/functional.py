"""torch.autograd.Function wrappers over the C ABI (one per operator the reference's
modules use).  Tensors in and out are ordinary fp32 torch tensors; all device work is
done by libeadgan.so on the caller's current CUDA stream.  No torch compute op is used
on the data path (allocation via torch.empty / zeros only).

Reference operators replaced (SURVEY.md section 8a): F.conv2d / F.conv_transpose2d /
F.linear (a5), F.batch_norm (a6), LeakyReLU / ReLU / Tanh / sigmoid / softmax /
Upsample (a7), spectral_norm's compute_weight (a8), BCE / MSE / CE-on-softmax /
mutual_info_loss (a9).
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L
from . import tc
from ._lib import ACT_NONE, ACT_LRELU, ACT_RELU, ACT_SIGMOID, ACT_TANH, call, ptr, stream, t4

# ----------------------------------------------------------------------------------
# data-parallel hook: set by eadgan_b200.parallel when WORLD_SIZE > 1
# ----------------------------------------------------------------------------------
_allreduce_sum = None  # callable(tensor) -> None (in place, sum over ranks)
_world_size = 1


def set_allreduce(fn, world_size):
    global _allreduce_sum, _world_size
    _allreduce_sum, _world_size = fn, int(world_size)


def _f32(t, who):
    L.require_cuda(t, who)
    if t.dtype != torch.float32:
        raise RuntimeError(f"{who}: expected float32, got {t.dtype}")
    return t


def _conv_desc(n, c, h, w, k, r, s, stride, pad):
    p = (h + 2 * pad - r) // stride + 1
    q = (w + 2 * pad - s) // stride + 1
    return L.ConvDesc(n, c, h, w, k, r, s, p, q, stride, pad), p, q


def act_fwd_(x, kind, slope=0.0, out=None):
    out = x if out is None else out
    call("eadgan_act_fwd", ptr(x), ptr(out), x.numel(), kind, float(slope), stream())
    return out


def act_bwd(dy, y, kind, slope=0.0):
    dy = dy.contiguous()
    dx = torch.empty_like(dy)
    call("eadgan_act_bwd", ptr(dy), ptr(y), ptr(dx), dy.numel(), kind, float(slope), stream())
    return dx


def channel_sum(t):
    """[N,C,H,W] or [N,C] -> [C] (bias gradients)."""
    if t.dim() == 2:
        n, c, h, w = t.shape[0], t.shape[1], 1, 1
    else:
        n, c, h, w = t.shape
    out = torch.empty(c, device=t.device, dtype=torch.float32)
    d = t4(t)
    call("eadgan_channel_sum", C.byref(d), n, c, h, w, ptr(out), stream())
    return out


# ----------------------------------------------------------------------------------
# convolution family (fp32 SIMT path)
# ----------------------------------------------------------------------------------
def conv_wgrad(d, x_t4, dy_t4, dw):
    """dw (overwritten) = SIMT weight gradient; split partials go through the per-(device, stream) workspace of
    eadgan_b200.tc (the library allocates nothing) and are summed in a fixed order: deterministic."""
    need = L.lib().eadgan_conv_wgrad_workspace(C.byref(d))
    ws = tc._workspace(need, dw.device) if need else None
    call("eadgan_conv_wgrad", C.byref(d), C.byref(x_t4), C.byref(dy_t4), ptr(dw), ptr(ws),
         C.c_size_t(need), stream())


class _ConvFn(torch.autograd.Function):
    """y = act(conv2d(x, w, b)); nn.Linear is the 1x1 case on [N,C] tensors."""

    @staticmethod
    def forward(ctx, x, w, b, stride, pad, act, slope):
        _f32(x, "conv2d")
        _f32(w, "conv2d")
        x = x if x.is_contiguous() else x.contiguous()
        w = w.contiguous()
        two_d = x.dim() == 2
        if two_d:
            n, c, h, ww = x.shape[0], x.shape[1], 1, 1
            k, r, s = w.shape[0], 1, 1
        else:
            n, c, h, ww = x.shape
            k, _, r, s = w.shape
        if w.shape[1] != c:
            raise RuntimeError(f"conv2d: weight {tuple(w.shape)} does not match input channels {c}")
        d, p, q = _conv_desc(n, c, h, ww, k, r, s, stride, pad)
        y = torch.empty((n, k) if two_d else (n, k, p, q), device=x.device, dtype=torch.float32)
        xd, yd = t4(x), t4(y)
        call("eadgan_conv_fprop", C.byref(d), C.byref(xd), ptr(w), ptr(b), act, float(slope),
             C.byref(yd), None, ACT_NONE, 0.0, stream())
        ctx.save_for_backward(x, w, y if act != ACT_NONE else None)
        ctx.cfg = (d, act, slope, b is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, y = ctx.saved_tensors
        d, act, slope, has_b = ctx.cfg
        dy = dy.contiguous()
        dz = act_bwd(dy, y, act, slope) if act != ACT_NONE else dy
        dx = dw = db = None
        dzd = t4(dz)
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            dxd = t4(dx)
            call("eadgan_conv_dgrad", C.byref(d), C.byref(dzd), ptr(w), None, ACT_NONE, 0.0,
                 C.byref(dxd), None, ACT_NONE, 0.0, stream())
        if ctx.needs_input_grad[1]:
            dw = torch.empty_like(w)
            conv_wgrad(d, t4(x), dzd, dw)
        if has_b and ctx.needs_input_grad[2]:
            db = channel_sum(dz)
        return dx, dw, db, None, None, None, None


class _ConvTFn(torch.autograd.Function):
    """y = act(conv_transpose2d(x, w, b)); w is [Cin, Cout, r, s] (torch ConvTranspose2d layout)."""

    @staticmethod
    def forward(ctx, x, w, b, stride, pad, act, slope):
        _f32(x, "conv_transpose2d")
        _f32(w, "conv_transpose2d")
        x = x if x.is_contiguous() else x.contiguous()
        w = w.contiguous()
        n, k, p, q = x.shape
        kk, c, r, s = w.shape
        if kk != k:
            raise RuntimeError(f"conv_transpose2d: weight {tuple(w.shape)} does not match input channels {k}")
        h = (p - 1) * stride - 2 * pad + r
        ww = (q - 1) * stride - 2 * pad + s
        d = L.ConvDesc(n, c, h, ww, k, r, s, p, q, stride, pad)
        y = torch.empty((n, c, h, ww), device=x.device, dtype=torch.float32)
        xd, yd = t4(x), t4(y)
        call("eadgan_conv_dgrad", C.byref(d), C.byref(xd), ptr(w), ptr(b), act, float(slope),
             C.byref(yd), None, ACT_NONE, 0.0, stream())
        ctx.save_for_backward(x, w, y if act != ACT_NONE else None)
        ctx.cfg = (d, act, slope, b is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w, y = ctx.saved_tensors
        d, act, slope, has_b = ctx.cfg
        dy = dy.contiguous()
        dz = act_bwd(dy, y, act, slope) if act != ACT_NONE else dy
        dx = dw = db = None
        dzd = t4(dz)
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            dxd = t4(dx)
            call("eadgan_conv_fprop", C.byref(d), C.byref(dzd), ptr(w), None, ACT_NONE, 0.0,
                 C.byref(dxd), None, ACT_NONE, 0.0, stream())
        if ctx.needs_input_grad[1]:
            dw = torch.empty_like(w)
            xd = t4(x)
            # conv view: "x" is the big map (dz), "dy" is the small map (module input)
            conv_wgrad(d, dzd, xd, dw)
        if has_b and ctx.needs_input_grad[2]:
            db = channel_sum(dz)
        return dx, dw, db, None, None, None, None


def conv2d(x, w, b=None, stride=1, padding=0, act=ACT_NONE, slope=0.0):
    return _ConvFn.apply(x, w, b, int(stride), int(padding), act, slope)


def conv_transpose2d(x, w, b=None, stride=1, padding=0, act=ACT_NONE, slope=0.0):
    return _ConvTFn.apply(x, w, b, int(stride), int(padding), act, slope)


def linear(x, w, b=None, act=ACT_NONE, slope=0.0):
    if x.dim() != 2:
        raise RuntimeError("linear: expected a [N, in_features] input")
    return _ConvFn.apply(x, w, b, 1, 0, act, slope)


# ----------------------------------------------------------------------------------
# batch norm (+ fused activation), SyncBN across ranks when data-parallel
# ----------------------------------------------------------------------------------
# The host sequence of both callers, _BatchNormFn and the bf16 chain (eadgan_b200.chain).  Tensors are [N, C, H, W]
# views in any layout bn.cu takes (fp32 NCHW, or the chain's padded bf16 NHWC interiors); the fp64 [2C] sum buffers
# belong to the caller, zero-filled.
def _ref(t):
    return None if t is None else C.byref(t4(t))


def bn_train_forward(x, sums, gamma, beta, rmean, rvar, momentum, eps, act, slope, y, keep_sum_x=False):
    """y = act(BatchNorm(x)) with the batch's statistics, from sums = [S x | S x^2] of this rank's x.  When data-parallel
    the sums are all-reduced in place first.  Updates rmean / rvar.  Returns (mean, invstd, count, sum_x): count is the
    element count per channel over all ranks; with keep_sum_x, sum_x is this rank's S x, which bn_train_backward needs
    for the gradient of a conv bias in front of the BatchNorm."""
    n, c, h, w = x.shape
    count = float(n * h * w)
    sum_x = sums[:c] if keep_sum_x else None
    if _allreduce_sum is not None:
        if keep_sum_x:
            sum_x = sum_x.clone()
        _allreduce_sum(sums)
        count *= _world_size
    mean = torch.empty(c, device=x.device, dtype=torch.float32)
    invstd = torch.empty(c, device=x.device, dtype=torch.float32)
    st = stream()
    call("eadgan_bn_finalize", ptr(sums), count, c, float(eps), float(momentum), ptr(mean), ptr(invstd), ptr(rmean),
         ptr(rvar), st)
    call("eadgan_bn_apply", _ref(x), n, c, h, w, ptr(mean), ptr(invstd), ptr(gamma), ptr(beta), act, float(slope),
         _ref(y), st)
    return mean, invstd, count, sum_x


def bn_train_backward(dy, x, y, mean, invstd, gamma, beta, act, slope, count, sums, dx, sum_x=None):
    """Backward of bn_train_forward: writes dx (which may be dy) and returns (dgamma, dbeta, dbias).  y is the forward's
    output (None without an activation); sums is scratch.  The fp64 sums [S dz | S dz*xhat] are all-reduced between the
    two passes; dgamma and dbeta are this rank's, as every other parameter gradient.  dbias, the gradient of a conv bias
    in front of the BatchNorm, is computed when sum_x (bn_train_forward's) is given, else None."""
    n, c, h, w = x.shape
    st = stream()
    call("eadgan_bn_bwd_reduce", _ref(dy), _ref(x), _ref(y), n, c, h, w, ptr(mean), ptr(invstd), ptr(gamma), ptr(beta),
         act, float(slope), ptr(sums), st)
    local = sums
    if _allreduce_sum is not None:
        local = sums.clone()
        _allreduce_sum(sums)
    call("eadgan_bn_bwd_apply", _ref(dy), _ref(x), _ref(y), n, c, h, w, ptr(mean), ptr(invstd), ptr(gamma), ptr(beta),
         act, float(slope), ptr(sums), float(count), _ref(dx), st)
    small = torch.empty((2 if sum_x is None else 3) * c, device=x.device, dtype=torch.float32)
    dgamma, dbeta, dbias = small[:c], small[c:2 * c], small[2 * c:] if sum_x is not None else None
    # in closed form from the fp64 sums: no extra pass over dx
    call("eadgan_bn_bwd_finalize", ptr(local), ptr(sums), ptr(sum_x), float(n * h * w), float(count), ptr(mean),
         ptr(invstd), ptr(gamma), c, ptr(dgamma), ptr(dbeta), ptr(dbias), st)
    return dgamma, dbeta, dbias


def bn_eval_backward(dy, x, y, rmean, rvar, eps, gamma, beta, act, slope, sums, dx, want_dbias=False):
    """Backward of y = act(BatchNorm(x)) with the running statistics, one pass: writes dx (which may be dy) and returns
    (dgamma, dbeta, dbias), dbias (the gradient of a conv bias in front of the BatchNorm) only with want_dbias.  No
    all-reduce: the normalisation does not depend on other ranks' data."""
    n, c, h, w = x.shape
    small = torch.empty((3 if want_dbias else 2) * c, device=x.device, dtype=torch.float32)
    dgamma, dbeta, dbias = small[:c], small[c:2 * c], small[2 * c:] if want_dbias else None
    call("eadgan_bn_eval_bwd", _ref(dy), _ref(x), _ref(y), n, c, h, w, ptr(rmean), ptr(rvar), float(eps), ptr(gamma),
         ptr(beta), act, float(slope), ptr(sums), _ref(dx), ptr(dgamma), ptr(dbeta), ptr(dbias), stream())
    return dgamma, dbeta, dbias


class _BatchNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, rmean, rvar, training, momentum, eps, act, slope):
        _f32(x, "batch_norm")
        x = x if x.is_contiguous() else x.contiguous()
        n, c, h, w = x.shape
        y = torch.empty_like(x)
        ctx.training = training
        if not training:
            call("eadgan_bn_eval", _ref(x), n, c, h, w, ptr(rmean), ptr(rvar), float(eps), ptr(gamma), ptr(beta), act,
                 float(slope), _ref(y), stream())
            ctx.save_for_backward(x, gamma, beta, rmean, rvar, y if act != ACT_NONE else None)
            ctx.cfg = (eps, act, slope)
            return y
        sums = torch.zeros(2 * c, device=x.device, dtype=torch.float64)
        call("eadgan_bn_stats", _ref(x), n, c, h, w, ptr(sums), stream())
        mean, invstd, count, _ = bn_train_forward(x, sums, gamma, beta, rmean, rvar, momentum, eps, act, slope, y)
        ctx.save_for_backward(x, gamma, beta, mean, invstd, y if act != ACT_NONE else None)
        ctx.cfg = (count, act, slope)
        return y

    @staticmethod
    def backward(ctx, dy):
        dy = dy.contiguous()
        x, gamma, beta, a, b, y = ctx.saved_tensors     # a, b: mean, invstd (training) / running_mean, running_var
        c = x.shape[1]
        sums = torch.zeros(2 * c, device=x.device, dtype=torch.float64)
        dx = torch.empty_like(x)
        if ctx.training:
            count, act, slope = ctx.cfg
            dgamma, dbeta, _ = bn_train_backward(dy, x, y, a, b, gamma, beta, act, slope, count, sums, dx)
        else:
            eps, act, slope = ctx.cfg
            dgamma, dbeta, _ = bn_eval_backward(dy, x, y, a, b, eps, gamma, beta, act, slope, sums, dx)
        return dx, dgamma, dbeta, None, None, None, None, None, None, None


def batch_norm(x, gamma, beta, rmean, rvar, training, momentum, eps, act=ACT_NONE, slope=0.0):
    return _BatchNormFn.apply(x, gamma, beta, rmean, rvar, bool(training), momentum, eps, act, slope)


# ----------------------------------------------------------------------------------
# pointwise
# ----------------------------------------------------------------------------------
class _ActFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, kind, slope, inplace):
        _f32(x, "activation")
        if inplace and x.is_contiguous():
            ctx.mark_dirty(x)
            y = act_fwd_(x, kind, slope)
        else:
            xc = x.contiguous()
            y = torch.empty_like(xc)
            act_fwd_(xc, kind, slope, out=y)
        ctx.save_for_backward(y)
        ctx.cfg = (kind, slope)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        kind, slope = ctx.cfg
        return act_bwd(dy, y, kind, slope), None, None, None


def activation(x, kind, slope=0.0, inplace=False):
    return _ActFn.apply(x, kind, float(slope), bool(inplace))


class _SoftmaxFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        _f32(x, "softmax")
        if x.dim() != 2:
            raise RuntimeError("softmax: only [rows, cols] inputs (implicit dim=1) are on the hot path")
        x = x.contiguous()
        y = torch.empty_like(x)
        call("eadgan_softmax_fwd", ptr(x), ptr(y), x.shape[0], x.shape[1], stream())
        ctx.save_for_backward(y)
        return y

    @staticmethod
    def backward(ctx, dy):
        (y,) = ctx.saved_tensors
        dy = dy.contiguous()
        dx = torch.empty_like(y)
        call("eadgan_softmax_bwd", ptr(dy), ptr(y), ptr(dx), y.shape[0], y.shape[1], stream())
        return dx


def softmax(x):
    return _SoftmaxFn.apply(x)


class _Upsample2xFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        _f32(x, "upsample")
        x = x.contiguous()
        n, c, h, w = x.shape
        y = torch.empty((n, c, 2 * h, 2 * w), device=x.device, dtype=torch.float32)
        call("eadgan_upsample2x_fwd", ptr(x), ptr(y), n * c, h, w, stream())
        ctx.shape = (n, c, h, w)
        return y

    @staticmethod
    def backward(ctx, dy):
        n, c, h, w = ctx.shape
        dy = dy.contiguous()
        dx = torch.empty((n, c, h, w), device=dy.device, dtype=torch.float32)
        call("eadgan_upsample2x_bwd", ptr(dy), ptr(dx), n * c, h, w, stream())
        return dx


def upsample2x(x):
    return _Upsample2xFn.apply(x)


# ----------------------------------------------------------------------------------
# legacy spectral norm
# ----------------------------------------------------------------------------------
class _SpectralNormFn(torch.autograd.Function):
    """weight = weight_orig / sigma with one in-place power iteration on u, v
    (torch/nn/utils/spectral_norm.py::SpectralNorm.compute_weight, dim=0)."""

    @staticmethod
    def forward(ctx, w_orig, u, v, do_power_iter, eps):
        _f32(w_orig, "spectral_norm")
        w = w_orig.contiguous()
        rows = w.shape[0]
        cols = w.numel() // rows
        sigma = torch.empty(1, device=w.device, dtype=torch.float32)
        w_sn = torch.empty_like(w)
        scratch = torch.empty(L.lib().eadgan_spectral_norm_scratch_floats(rows, cols, 0), device=w.device,
                              dtype=torch.float32)
        # sn_skip_scale (set by the bf16 chain executor around the pre-forward hooks): W / sigma is NOT written --
        # the chain packs weight_orig and applies 1/sigma in the conv epilogue; spectral_norm_materialize() fills
        # w_sn later if some consumer needs its values
        call("eadgan_spectral_norm_fwd", ptr(w), rows, cols, ptr(u), ptr(v), 1 if do_power_iter else 0,
             float(eps), ptr(sigma), None if sn_skip_scale else ptr(w_sn), ptr(scratch), stream())
        ctx.mark_non_differentiable(sigma)
        # u, v are cloned exactly like the reference does, so later in-place power
        # iterations (6 per CelebA step) do not corrupt this graph's backward
        ctx.save_for_backward(w, u.clone(), v.clone(), sigma)
        return w_sn, sigma

    @staticmethod
    def backward(ctx, dw_sn, _dsigma):
        w, u, v, sigma = ctx.saved_tensors
        dw_sn = dw_sn.contiguous()
        rows = w.shape[0]
        cols = w.numel() // rows
        dw = torch.empty_like(w)
        scratch = torch.empty(L.lib().eadgan_spectral_norm_scratch_floats(rows, cols, 1), device=w.device,
                              dtype=torch.float32)
        call("eadgan_spectral_norm_bwd", ptr(dw_sn), ptr(w), ptr(u), ptr(v), ptr(sigma), rows, cols, ptr(dw),
             ptr(scratch), stream())
        return dw, None, None, None, None


sn_skip_scale = False


def spectral_norm_materialize(w_orig, sigma, w_sn):
    """w_sn <- w_orig / sigma (for a forward that ran with sn_skip_scale)."""
    call("eadgan_spectral_norm_scale", ptr(w_orig.detach().contiguous()), ptr(sigma), ptr(w_sn), w_sn.numel(), stream())


def spectral_norm_sigma(w_orig, u, v, eps):
    """sigma = u^T W v from the stored u, v: the eval-mode spectral norm (no power iteration; u, v are only read)
    -> fp32 [1] device tensor."""
    w = _f32(w_orig, "spectral_norm").detach().contiguous()
    rows = w.shape[0]
    cols = w.numel() // rows
    sigma = torch.empty(1, device=w.device, dtype=torch.float32)
    scratch = torch.empty(L.lib().eadgan_spectral_norm_scratch_floats(rows, cols, 0), device=w.device,
                          dtype=torch.float32)
    call("eadgan_spectral_norm_fwd", ptr(w), rows, cols, ptr(u), ptr(v), 0, float(eps), ptr(sigma), None,
         ptr(scratch), stream())
    return sigma


def fold_bn_sn(w, channel_dim, sigma=None, bn=None, bias=None):
    """(W', b') of a layer with its legacy spectral norm (sigma: the fp32 [1] device scalar) and / or the eval-mode
    BatchNorm2d after it folded in, along the output-channel axis ``channel_dim`` of W (0: Conv2d / Linear, 1:
    ConvTranspose2d).  b' is None without a BatchNorm (the bias is unchanged then)."""
    w = _f32(w, "fold_bn_sn").detach().contiguous()
    c = w.shape[channel_dim]
    outer = w.shape[0] if channel_dim == 1 else 1
    w_out = torch.empty_like(w)
    b_out = torch.empty(c, device=w.device, dtype=torch.float32) if bn is not None else None
    g = (bn.weight, bn.bias, bn.running_mean, bn.running_var) if bn is not None else (None,) * 4
    call("eadgan_fold_bn_sn", ptr(w), outer, c, w.numel() // (outer * c), ptr(sigma), *(ptr(t) for t in g),
         float(bn.eps) if bn is not None else 0.0, ptr(bias), ptr(w_out), ptr(b_out), stream())
    return w_out, b_out


def spectral_norm_weight(w_orig, u, v, do_power_iter, eps):
    return _SpectralNormFn.apply(w_orig, u, v, bool(do_power_iter), float(eps))


# ----------------------------------------------------------------------------------
# losses (scalar, mean reduction)
# ----------------------------------------------------------------------------------
def _same_shape(a, b, who):
    if a.shape != b.shape:
        raise ValueError(f"{who}: input {tuple(a.shape)} and target {tuple(b.shape)} must have the same shape")


class _BCEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p, target):
        _f32(p, "BCELoss")
        _same_shape(p, target, "BCELoss")
        p, target = p.contiguous(), target.contiguous().float()
        loss = torch.empty((), device=p.device, dtype=torch.float32)
        call("eadgan_bce_fwd", ptr(p), ptr(target), p.numel(), ptr(loss), stream())
        ctx.save_for_backward(p, target)
        return loss

    @staticmethod
    def backward(ctx, g):
        p, target = ctx.saved_tensors
        dp = torch.empty_like(p)
        g = g.contiguous().float()
        call("eadgan_bce_bwd", ptr(p), ptr(target), ptr(g), p.numel(), ptr(dp), stream())
        return dp, None


class _MSEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b):
        _f32(a, "MSELoss")
        _same_shape(a, b, "MSELoss")
        a, b = a.contiguous(), b.contiguous().float()
        loss = torch.empty((), device=a.device, dtype=torch.float32)
        call("eadgan_mse_fwd", ptr(a), ptr(b), a.numel(), ptr(loss), stream())
        ctx.save_for_backward(a, b)
        return loss

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        g = g.contiguous().float()
        da = torch.empty_like(a) if ctx.needs_input_grad[0] else None
        db = torch.empty_like(b) if ctx.needs_input_grad[1] else None
        if da is None and db is None:
            return None, None
        call("eadgan_mse_bwd", ptr(a), ptr(b), ptr(g), a.numel(), ptr(da), ptr(db), stream())
        return da, db


class _CEFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, labels):
        _f32(x, "CrossEntropyLoss")
        if x.dim() != 2 or labels.dim() != 1 or labels.dtype != torch.int64:
            raise RuntimeError("CrossEntropyLoss: expected [N,C] float input and [N] int64 class labels")
        x, labels = x.contiguous(), labels.contiguous()
        loss = torch.empty((), device=x.device, dtype=torch.float32)
        call("eadgan_ce_fwd", ptr(x), ptr(labels), x.shape[0], x.shape[1], ptr(loss), stream())
        ctx.save_for_backward(x, labels)
        return loss

    @staticmethod
    def backward(ctx, g):
        x, labels = ctx.saved_tensors
        g = g.contiguous().float()
        dx = torch.empty_like(x)
        call("eadgan_ce_bwd", ptr(x), ptr(labels), ptr(g), x.shape[0], x.shape[1], ptr(dx), stream())
        return dx, None


class _MIFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, c):
        _f32(q, "mutual_info_loss")
        _same_shape(q, c, "mutual_info_loss")
        q, c = q.contiguous(), c.contiguous().float()
        loss = torch.empty((), device=q.device, dtype=torch.float32)
        call("eadgan_mi_fwd", ptr(q), ptr(c), q.shape[0], q.shape[1], ptr(loss), stream())
        ctx.save_for_backward(q, c)
        return loss

    @staticmethod
    def backward(ctx, g):
        q, c = ctx.saved_tensors
        g = g.contiguous().float()
        dq = torch.empty_like(q)
        call("eadgan_mi_bwd", ptr(q), ptr(c), ptr(g), q.shape[0], q.shape[1], ptr(dq), stream())
        return dq, None


def bce_loss(p, target):
    return _BCEFn.apply(p, target)


def mse_loss(a, b):
    return _MSEFn.apply(a, b)


def cross_entropy(x, labels):
    return _CEFn.apply(x, labels)


def mutual_info_loss(q, c):
    """dSprites/rp.py:225-232; the target c carries no gradient (one-hot or detached)."""
    return _MIFn.apply(q, c.detach())


# ---- fused affine glue (csrc/glue.cu) ----------------------------------------------------------------------
REL_CELEBA, REL_DSPRITES, REL_MNIST = 0, 1, 2
_REL_DIMS = {REL_CELEBA: (5, 5), REL_DSPRITES: (4, 4), REL_MNIST: (7, 6)}


def _rows(t, k, who):
    """[B, >=k] fp32 CUDA tensor with unit column stride -> (tensor kept alive, row stride)"""
    if not (t.is_cuda and t.dtype == torch.float32 and t.dim() == 2 and t.shape[1] >= k):
        raise RuntimeError(f"{who}: expected a CUDA fp32 [B, >= {k}] tensor")
    if t.stride(1) != 1:
        t = t.contiguous()
    return t, t.stride(0)


class _RelCodeFn(torch.autograd.Function):
    """relative affine code of two code vectors (mode-specific closed form) with a stored Jacobian"""

    @staticmethod
    def forward(ctx, real, trans, mode):
        k, ko = _REL_DIMS[mode]
        real_k, rs = _rows(real.detach(), k, "relative_code")
        trans_k, ts = _rows(trans.detach(), k, "relative_code")
        n = real.shape[0]
        out = torch.empty((n, ko), device=real.device, dtype=torch.float32)
        jac = torch.empty((n, ko, 2 * k), device=real.device, dtype=torch.float32)
        call("eadgan_relcode_fwd", mode, ptr(real_k), rs, ptr(trans_k), ts, n, ptr(out), ptr(jac), stream())
        ctx.save_for_backward(jac)
        ctx.cfg = (mode, k, real.shape[1], trans.shape[1])
        return out

    @staticmethod
    def backward(ctx, g):
        (jac,) = ctx.saved_tensors
        mode, k, real_w, trans_w = ctx.cfg
        n = jac.shape[0]
        g = g.contiguous()
        # gradients w.r.t. the first k columns; any further columns of the inputs get zero
        d_real = torch.zeros((n, real_w), device=g.device, dtype=torch.float32) if real_w != k else None
        d_trans = torch.zeros((n, trans_w), device=g.device, dtype=torch.float32) if trans_w != k else None
        dr = torch.empty((n, k), device=g.device, dtype=torch.float32)
        dt = torch.empty((n, k), device=g.device, dtype=torch.float32)
        call("eadgan_relcode_bwd", mode, ptr(g), ptr(jac), n, ptr(dr), ptr(dt), stream())
        if d_real is not None:
            d_real[:, :k] = dr
            dr = d_real
        if d_trans is not None:
            d_trans[:, :k] = dt
            dt = d_trans
        return dr, dt, None


def relative_code(real, trans, mode):
    return _RelCodeFn.apply(real, trans, mode)


def stn_fwd(img, theta23, border=True):
    """F.grid_sample(img, F.affine_grid(theta, img.size()), padding_mode) with align_corners=False; forward only."""
    if not (img.is_cuda and img.dtype == torch.float32 and img.dim() == 4):
        raise RuntimeError("stn_fwd: expected a CUDA fp32 [N, C, H, W] image")
    img = img.contiguous()
    theta = theta23.detach().to(torch.float32).contiguous()
    n, c, h, w = img.shape
    if tuple(theta.shape) != (n, 2, 3):
        raise RuntimeError("stn_fwd: theta must be [N, 2, 3]")
    out = torch.empty_like(img)
    call("eadgan_stn_fwd", ptr(img), ptr(theta), n, c, h, w, 1 if border else 0, ptr(out), stream())
    return out


# ---- F.affine_grid / F.grid_sample as differentiable operators (csrc/glue.cu) --------------------------------------------
class _AffineGridFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, theta, n, h, w):
        grid = torch.empty((n, h, w, 2), device=theta.device, dtype=torch.float32)
        call("eadgan_affine_grid_fwd", ptr(theta), n, h, w, ptr(grid), stream())
        ctx.dims = (n, h, w)
        return grid

    @staticmethod
    def backward(ctx, dgrid):
        n, h, w = ctx.dims
        dtheta = torch.empty((n, 2, 3), device=dgrid.device, dtype=torch.float32)
        call("eadgan_affine_grid_bwd", ptr(dgrid.contiguous()), n, h, w, ptr(dtheta), stream())
        return dtheta, None, None, None


def affine_grid(theta, size, align_corners=None):
    """F.affine_grid(theta [N,2,3], size (N,C,H,W), align_corners=False) -> [N,H,W,2]
    (celebA/EAD-GAN_celebA.py:150, dSprites/rp.py:205)."""
    if align_corners:
        raise RuntimeError("eadgan_b200 affine_grid: align_corners=True is not used by the reference and unsupported")
    if not (theta.is_cuda and theta.dtype == torch.float32 and theta.dim() == 3 and tuple(theta.shape[1:]) == (2, 3)):
        raise RuntimeError("eadgan_b200 affine_grid: theta must be a CUDA fp32 [N, 2, 3] tensor (no CPU fallback)")
    size = tuple(int(v) for v in size)
    if len(size) != 4 or size[0] != theta.shape[0]:
        raise RuntimeError("eadgan_b200 affine_grid: size must be (N, C, H, W) with N = theta.shape[0]")
    return _AffineGridFn.apply(theta.contiguous(), size[0], size[2], size[3])


class _GridSampleFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img, grid, border):
        n, c, h, w = img.shape
        oh, ow = grid.shape[1], grid.shape[2]
        out = torch.empty((n, c, oh, ow), device=img.device, dtype=torch.float32)
        call("eadgan_grid_sample_fwd", ptr(img), ptr(grid), n, c, h, w, oh, ow, int(border), ptr(out), stream())
        ctx.save_for_backward(img, grid)
        ctx.border = int(border)
        return out

    @staticmethod
    def backward(ctx, gout):
        img, grid = ctx.saved_tensors
        n, c, h, w = img.shape
        oh, ow = grid.shape[1], grid.shape[2]
        dimg = torch.zeros_like(img) if ctx.needs_input_grad[0] else None
        dgrid = torch.empty_like(grid) if ctx.needs_input_grad[1] else None
        if dimg is not None or dgrid is not None:
            call("eadgan_grid_sample_bwd", ptr(gout.contiguous()), ptr(img), ptr(grid), n, c, h, w, oh, ow, ctx.border,
                 ptr(dimg), ptr(dgrid), stream())
        return dimg, dgrid, None


def grid_sample(input, grid, mode="bilinear", padding_mode="zeros", align_corners=None):
    """F.grid_sample(input [N,C,H,W], grid [N,Ho,Wo,2], 'bilinear', 'border' | 'zeros', align_corners=False)
    (celebA/EAD-GAN_celebA.py:151, colored_dSprites/pxy_color.py:90) with both gradients."""
    if mode != "bilinear" or padding_mode not in ("border", "zeros") or align_corners:
        raise RuntimeError("eadgan_b200 grid_sample: only bilinear, padding_mode 'border' | 'zeros', align_corners=False")
    if not (input.is_cuda and grid.is_cuda and input.dtype == torch.float32 and grid.dtype == torch.float32
            and input.dim() == 4 and grid.dim() == 4 and grid.shape[0] == input.shape[0] and grid.shape[3] == 2):
        raise RuntimeError("eadgan_b200 grid_sample: CUDA fp32 input [N,C,H,W] and grid [N,Ho,Wo,2] required "
                           "(no CPU fallback)")
    return _GridSampleFn.apply(input.contiguous(), grid.contiguous(), padding_mode == "border")
