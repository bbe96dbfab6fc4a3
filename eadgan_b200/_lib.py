"""ctypes binding of libeadgan.so (the C ABI declared in include/eadgan.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``eadgan_b200.build``
(``nvcc -gencode arch=compute_100a,code=sm_100a``).  There is NO fallback: if the
shared object is missing, or an entry point returns a non-zero status, a
RuntimeError is raised (SURVEY.md section 8b "Errors").
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libeadgan.so")

ACT_NONE, ACT_RELU, ACT_LRELU, ACT_TANH, ACT_SIGMOID = 0, 1, 2, 3, 4
F32, BF16 = 0, 1
ADAM_MAX_TENSORS = 48


class Tensor4(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("sn", C.c_int64), ("sc", C.c_int64), ("sh", C.c_int64),
                ("sw", C.c_int64), ("dtype", C.c_int32), ("_pad", C.c_int32)]


class ConvDesc(C.Structure):
    _fields_ = [("n", C.c_int32), ("c", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
                ("k", C.c_int32), ("r", C.c_int32), ("s", C.c_int32), ("p", C.c_int32),
                ("q", C.c_int32), ("stride", C.c_int32), ("pad", C.c_int32)]


class TcDesc(C.Structure):
    _fields_ = [("n", C.c_int32), ("c", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
                ("k", C.c_int32), ("act", C.c_int32), ("slope", C.c_float),
                ("out_f32_nchw", C.c_int32), ("want_stats", C.c_int32), ("c_real", C.c_int32),
                ("mask_mode", C.c_int32)]


class AdamTensors(C.Structure):
    _fields_ = [("p", C.c_void_p * ADAM_MAX_TENSORS), ("g", C.c_void_p * ADAM_MAX_TENSORS),
                ("m", C.c_void_p * ADAM_MAX_TENSORS), ("v", C.c_void_p * ADAM_MAX_TENSORS),
                ("numel", C.c_int64 * ADAM_MAX_TENSORS), ("count", C.c_int32), ("_pad", C.c_int32)]


_P = C.c_void_p
_T4 = C.POINTER(Tensor4)
_I, _F, _D, _L = C.c_int, C.c_float, C.c_double, C.c_int64

# name -> argtypes (every function returns int status unless listed in _SPECIAL)
_PROTOS = {
    "eadgan_conv_fprop": [C.POINTER(ConvDesc), _T4, _P, _P, _I, _F, _T4, _T4, _I, _F, _P],
    "eadgan_conv_dgrad": [C.POINTER(ConvDesc), _T4, _P, _P, _I, _F, _T4, _T4, _I, _F, _P],
    "eadgan_conv_wgrad": [C.POINTER(ConvDesc), _T4, _T4, _P, _P, C.c_size_t, _P],
    "eadgan_channel_sum": [_T4, _I, _I, _I, _I, _P, _P],
    "eadgan_tc_pack_w_fprop": [_P, _P, _I, _I, _I, _P, _P],
    "eadgan_tc_pack_w_dgrad": [_P, _P, _I, _I, _I, _P, _P],
    "eadgan_tc_dense_pack": [_P, _I, _I, _I, _I, _P, _P],
    "eadgan_tc_dense_gather": [_P, _P, _P, _P, _I, _I, _I, _P, C.c_size_t, _P],
    "eadgan_tc_dense_scatter": [_P, _P, _P, _P, _P, _I, _F, _I, _I, _I, _P, _P],
    "eadgan_tc_dense_wgrad": [_P, _P, _P, _P, C.c_size_t, _I, _I, _I, _I, _P],
    "eadgan_tc_fprop": [C.POINTER(TcDesc), _P, _P, _P, _P, _P, _P, _P, _P],
    "eadgan_tc_dgrad": [C.POINTER(TcDesc), _P, _P, _P, _P, _P, _P, _P, _P],
    "eadgan_tc_wgrad": [C.POINTER(TcDesc), _P, _P, _P, _P, C.c_size_t, _P],
    "eadgan_tc_gemm": [_P, _P, _P, _I, _I, _I, _P],
    "eadgan_tc_thin_expand": [_T4, _T4, _I, _F, _I, _I, _I, _I, _P, _P],
    "eadgan_tc_thin_pack_w": [_P, _I, _I, _I, _P, _P],
    "eadgan_tc_thin_fprop": [C.POINTER(TcDesc), _P, _P, _P, _P, _P, _P, _P, _P],
    "eadgan_tc_thin_wgrad": [C.POINTER(TcDesc), _P, _P, _P, _P, C.c_size_t, _P],
    "eadgan_tc_thin_dgrad": [C.POINTER(TcDesc), _P, _P, _P, _P, _P, _P],
    "eadgan_copy4": [_T4, _T4, _I, _I, _I, _I, _P],
    "eadgan_bn_stats": [_T4, _I, _I, _I, _I, _P, _P],
    "eadgan_bn_finalize": [_P, _D, _I, _F, _F, _P, _P, _P, _P, _P],
    "eadgan_bn_apply": [_T4, _I, _I, _I, _I, _P, _P, _P, _P, _I, _F, _T4, _P],
    "eadgan_bn_bwd_reduce": [_T4, _T4, _T4, _I, _I, _I, _I, _P, _P, _P, _P, _I, _F, _P, _P],
    "eadgan_bn_bwd_apply": [_T4, _T4, _T4, _I, _I, _I, _I, _P, _P, _P, _P, _I, _F, _P, _D, _T4, _P],
    "eadgan_bn_bwd_finalize": [_P, _P, _P, _D, _D, _P, _P, _P, _I, _P, _P, _P, _P],
    "eadgan_bn_eval": [_T4, _I, _I, _I, _I, _P, _P, _F, _P, _P, _I, _F, _T4, _P],
    "eadgan_bn_eval_bwd": [_T4, _T4, _T4, _I, _I, _I, _I, _P, _P, _F, _P, _P, _I, _F, _P, _T4, _P, _P, _P, _P],
    "eadgan_act_fwd": [_P, _P, _L, _I, _F, _P],
    "eadgan_act_bwd": [_P, _P, _P, _L, _I, _F, _P],
    "eadgan_softmax_fwd": [_P, _P, _I, _I, _P],
    "eadgan_softmax_bwd": [_P, _P, _P, _I, _I, _P],
    "eadgan_upsample2x_fwd": [_P, _P, _I, _I, _I, _P],
    "eadgan_upsample2x_bwd": [_P, _P, _I, _I, _I, _P],
    "eadgan_spectral_norm_fwd": [_P, _I, _I, _P, _P, _I, _F, _P, _P, _P, _P],
    "eadgan_spectral_norm_scale": [_P, _P, _P, C.c_longlong, _P],
    "eadgan_spectral_norm_bwd": [_P, _P, _P, _P, _P, _I, _I, _P, _P, _P],
    "eadgan_fold_bn_sn": [_P, C.c_longlong, _I, C.c_longlong, _P, _P, _P, _P, _P, _D, _P, _P, _P, _P],
    "eadgan_bce_fwd": [_P, _P, _L, _P, _P],
    "eadgan_bce_bwd": [_P, _P, _P, _L, _P, _P],
    "eadgan_mse_fwd": [_P, _P, _L, _P, _P],
    "eadgan_mse_bwd": [_P, _P, _P, _L, _P, _P, _P],
    "eadgan_ce_fwd": [_P, _P, _I, _I, _P, _P],
    "eadgan_ce_bwd": [_P, _P, _P, _I, _I, _P, _P],
    "eadgan_mi_fwd": [_P, _P, _I, _I, _P, _P],
    "eadgan_mi_bwd": [_P, _P, _P, _I, _I, _P, _P],
    "eadgan_adam_step": [C.POINTER(AdamTensors), _D, _D, _D, _D, _D, _F, _P],
    "eadgan_adam_step_dev": [C.POINTER(AdamTensors), _D, _D, _D, _D, _P, _F, _P],
    "eadgan_adam_advance": [_P, _P],
    "eadgan_fill_f32": [_P, _L, _F, _P],
    "eadgan_f64_to_f32": [_P, _P, _L, _P],
    "eadgan_zero_halo": [_P, _I, _I, _I, _I, _P],
    "eadgan_stn_fwd": [_P, _P, _I, _I, _I, _I, _I, _P, _P],
    "eadgan_affine_grid_fwd": [_P, _I, _I, _I, _P, _P],
    "eadgan_affine_grid_bwd": [_P, _I, _I, _I, _P, _P],
    "eadgan_grid_sample_fwd": [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P],
    "eadgan_grid_sample_bwd": [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P],
    "eadgan_relcode_dims": [_I, _P, _P],
    "eadgan_relcode_fwd": [_I, _P, C.c_longlong, _P, C.c_longlong, _I, _P, _P, _P],
    "eadgan_relcode_bwd": [_I, _P, _P, _I, _P, _P, _P],
    "eadgan_philox": [_I, C.c_ulonglong, _P, C.c_longlong, _I, C.c_longlong, C.c_longlong, C.c_longlong, _F, _F, _I, _P, _P],
}
_SPECIAL = {
    "eadgan_last_error": ([], C.c_char_p),
    "eadgan_version": ([], C.c_int),
    "eadgan_sm_count": ([], C.c_int),
    "eadgan_kernel_launches": ([], C.c_int64),
    "eadgan_tc_workspace_bytes": ([C.POINTER(TcDesc), _I], C.c_size_t),
    "eadgan_conv_wgrad_workspace": ([C.POINTER(ConvDesc)], C.c_size_t),
    "eadgan_tc_thin_buffer_elems": ([_I, _I, _I], C.c_size_t),
    "eadgan_tc_dense_gather_workspace": ([_I], C.c_size_t),
    "eadgan_tc_thin_wgrad_workspace": ([C.POINTER(TcDesc)], C.c_size_t),
    "eadgan_tc_dense_wgrad_workspace": ([_I, _I], C.c_size_t),
    "eadgan_spectral_norm_scratch_floats": ([_I, _I, _I], C.c_size_t),
}
EXPORTED = sorted(list(_PROTOS) + list(_SPECIAL))

weights_epoch = 0  # bumped whenever parameters may have changed behind torch's version counters (Adam.step,
                   # load_state_dict): invalidates the packed-weight cache of eadgan_b200.tc


def bump_weights_epoch():
    global weights_epoch
    weights_epoch += 1


step_serial = 0    # one number per Adam.step() call; the parameters it updates carry it as ``_eadgan_stepped`` so that
                   # only THEIR cached packs / prefetched spectral-norm results go stale (phase G's step leaves D's alone)


def next_step_serial():
    global step_serial
    step_serial += 1
    return step_serial


_lib = None
launches = 0  # number of C-ABI compute calls issued (bench.py reports kernel launches from it)


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m eadgan_b200.build` "
                "(nvcc, sm_100a). eadgan_b200 has no CPU or cuDNN fallback.")
        l = C.CDLL(LIB_PATH)
        for name, args in _PROTOS.items():
            fn = getattr(l, name)
            fn.argtypes = args
            fn.restype = C.c_int
        for name, (args, res) in _SPECIAL.items():
            fn = getattr(l, name)
            fn.argtypes = args
            fn.restype = res
        _lib = l
    return _lib


_prof = None  # list of (name, flops, start_event, end_event) while profiling


def _flops(name, args):
    """algorithmic FLOPs (2*MAC) of one convolution-family call, from its descriptor."""
    try:
        d = args[0]._obj
    except AttributeError:
        return 0
    if isinstance(d, ConvDesc):
        return 2 * d.n * d.p * d.q * d.k * d.c * d.r * d.s
    if isinstance(d, TcDesc):
        return 2 * d.n * (d.h // 2) * (d.w // 2) * d.k * d.c * 16
    return 0


def _shape_tag(args):
    try:
        d = args[0]._obj
    except (AttributeError, IndexError):
        return ""
    if isinstance(d, ConvDesc):
        return f"[n{d.n} c{d.c} h{d.h} k{d.k} r{d.r} s{d.stride}]"
    if isinstance(d, TcDesc):
        return f"[n{d.n} c{d.c} h{d.h} k{d.k}]"
    return ""


def profile_start():
    """time every C-ABI call with CUDA events on the launching stream (bench.py roofline leg)."""
    global _prof
    _prof = []


def profile_stop():
    """-> {entry point: {"calls", "ms", "flops"}}"""
    global _prof
    rec, _prof = _prof, None
    torch.cuda.synchronize()
    out = {}
    for name, fl, e0, e1 in rec or []:
        r = out.setdefault(name, {"calls": 0, "ms": 0.0, "flops": 0})
        r["calls"] += 1
        r["ms"] += e0.elapsed_time(e1)
        r["flops"] += fl
    return out


def call(name, *args):
    """Invoke a status-returning entry point; raise RuntimeError on failure."""
    global launches
    if _prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = getattr(lib(), name)(*args)
        e1.record()
        _prof.append((name + _shape_tag(args), _flops(name, args), e0, e1))
    else:
        rc = getattr(lib(), name)(*args)
    launches += 1
    if rc != 0:
        msg = lib().eadgan_last_error()
        raise RuntimeError(f"{name} failed ({rc}): {msg.decode() if msg else '?'}")


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _dt(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise RuntimeError(f"eadgan_b200: unsupported dtype {t.dtype}")


def t4(t: torch.Tensor) -> Tensor4:
    """Describe a [N,C,H,W] (or [N,C]) tensor, whatever its strides."""
    if t.dim() == 2:
        return Tensor4(t.data_ptr(), t.stride(0), t.stride(1), 0, 0, _dt(t), 0)
    assert t.dim() == 4, t.shape
    return Tensor4(t.data_ptr(), t.stride(0), t.stride(1), t.stride(2), t.stride(3), _dt(t), 0)


def require_cuda(t: torch.Tensor, who: str):
    if not t.is_cuda:
        raise RuntimeError(
            f"{who}: eadgan_b200 operators run only on CUDA tensors (sm_100a kernels, no CPU "
            f"fallback); got a {t.device} tensor")
