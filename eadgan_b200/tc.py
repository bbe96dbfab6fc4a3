"""Host-side helpers for the tcgen05 path: private halo-padded NHWC bf16 buffers, weight
repacking and thin wrappers over the eadgan_tc_* entry points (include/eadgan.h)."""
from __future__ import annotations

import ctypes as C
import weakref

import torch

from . import _lib as L
from ._lib import ACT_NONE, call, ptr, stream, t4


# Pool of halo-padded buffers.  A buffer's halo (and, for channel-padded image buffers, its padding channels)
# is zeroed ONCE, when the buffer is first created; after that only interiors are ever written, so a recycled
# buffer needs no clearing at all.  Buffers are recycled per (shape, real-channel count, device) when the
# tensor object handed out dies (the chain executor always holds the padded tensor itself, views are
# temporaries); reuse is stream-ordered exactly like the caching allocator's.
_pool = {}
_pool_enabled = True
capture_births = None   # list while a CUDA-graph capture is running (eadgan_b200.graph): buffers first created inside it


_pool_gen = 0           # bumped by clear_pool(): buffers handed out before it are NOT recycled into the new pool


def _recycle(key, base, gen):
    if gen == _pool_gen:
        _pool.setdefault(key, []).append(base)


def alloc_padded(n, h, w, c, device, zero_interior=False, c_real=None):
    """[n, h+2, w+2, c] bf16 with a zero halo.  The interior is NOT initialised (every producing kernel
    overwrites it completely) unless ``zero_interior``.  ``c_real`` < c: channels >= c_real are guaranteed zero
    (the producing copy writes only the first c_real)."""
    shape = (n, h + 2, w + 2, c)
    if zero_interior or not _pool_enabled:
        return torch.zeros(shape, device=device, dtype=torch.bfloat16)
    key = (shape, c_real or c, str(device))
    free = _pool.get(key)
    if free:
        base = free.pop()
    else:
        base = torch.zeros(shape, device=device, dtype=torch.bfloat16)
        if capture_births is not None:
            # created during capture: the zero fill is only RECORDED, the memory holds garbage until the graph's first
            # replay.  GraphedStep zeroes these for real right after the capture, because the buffer now circulates
            # in the pool and eager code (or another capture) may pick it up before this graph ever runs.
            capture_births.append(base)
    t = base.view(shape)
    weakref.finalize(t, _recycle, key, base, _pool_gen)
    return t


def clear_pool():
    """drop every pooled buffer and workspace (frees the memory back to torch's allocator); buffers still in use are
    dropped when they die instead of being recycled.  eadgan_b200.graph.GraphedStep calls this on both sides of a
    capture, so that everything a captured step touches is allocated from -- and stays inside -- the graph's
    private memory pool: nothing a later eager call (or another capture) can free or reuse under a live graph."""
    global _pool_gen
    _pool_gen += 1
    _pool.clear()
    _ws_cache.clear()


def interior(xp):
    """logical [n, c, h, w] view of the interior of a padded NHWC buffer."""
    n, hp, wp, c = xp.shape
    return xp.permute(0, 3, 1, 2)[:, :, 1:hp - 1, 1:wp - 1]


def to_padded(x, c_alloc=None):
    """fp32/bf16 NCHW tensor -> padded NHWC bf16 (copy4 kernel); channels zero-padded to c_alloc."""
    n, c, h, w = x.shape
    xp = alloc_padded(n, h, w, c_alloc or c, x.device, c_real=c)
    src, dst = t4(x), t4(interior(xp)[:, :c])
    call("eadgan_copy4", C.byref(src), C.byref(dst), n, c, h, w, stream())
    return xp


def pad_rows(x2d, m_pad):
    """fp32 [n, m] -> bf16 [n, m_pad] (zero padded columns)."""
    n, m = x2d.shape
    out = torch.zeros((n, m_pad), device=x2d.device, dtype=torch.bfloat16)
    src, dst = t4(x2d), t4(out[:, :m])
    call("eadgan_copy4", C.byref(src), C.byref(dst), n, m, 1, 1, stream())
    return out


def from_padded(xp, dtype=torch.float32):
    n, hp, wp, c = xp.shape
    out = torch.empty((n, c, hp - 2, wp - 2), device=xp.device, dtype=dtype)
    src, dst = t4(interior(xp)), t4(out)
    call("eadgan_copy4", C.byref(src), C.byref(dst), n, c, hp - 2, wp - 2, stream())
    return out


def pack_w(w, sigma=None, direction="fprop", c_alloc=None):
    """fp32 [k, c, 4, 4] -> bf16 GEMM operand ([k,16c] for fprop, [4c,4k] for dgrad), / sigma;
    the c axis is zero-padded to c_alloc."""
    k, c = w.shape[0], w.shape[1]
    ca = c_alloc or c
    assert tuple(w.shape[2:]) == (4, 4)
    out = torch.empty(k * 16 * ca, device=w.device, dtype=torch.bfloat16)
    call("eadgan_tc_pack_w_fprop" if direction == "fprop" else "eadgan_tc_pack_w_dgrad",
         ptr(w.contiguous()), ptr(sigma), k, c, ca, ptr(out), stream())
    return out


_pack_cache = {}


def pack_w_cached(param, direction="fprop", c_alloc=None):
    """pack_w of a PARAMETER object (a G weight, or the weight_orig of a spectral-normalised layer), cached until
    the parameter changes (``_cached_pack``)."""
    return _cached_pack(param, "wide", direction, c_alloc)


def _cached_pack(param, kind, direction, c_alloc):
    """pack_w ("wide") or thin_pack_w ("thin") of a parameter, cached until the parameter changes: torch's version
    counter catches in-place torch ops (load_state_dict, stock optimisers), the ``_eadgan_stepped`` serial our fused
    Adam leaves on every parameter it updates (through raw pointers) catches that one, _lib.weights_epoch everything
    wholesale (load_state_dict, graph replays).  Entries are tied to the parameter OBJECT (weak reference), never to
    an address that a later tensor could reuse.  Code that rewrites a parameter through ``.data`` must call
    eadgan_b200.invalidate_caches()."""
    key = (id(param), direction if kind == "wide" else "thin_" + direction, c_alloc)
    token = (param._version, param.data_ptr(), L.weights_epoch, getattr(param, "_eadgan_stepped", 0))
    _note_use(param, kind, direction, c_alloc)
    hit = _pack_cache.get(key)
    if hit is not None and hit[0]() is param and hit[1] == token:
        return _adopt(hit)
    w = param.detach()
    out = thin_pack_w(w, direction) if kind == "thin" else pack_w(w, None, direction, c_alloc)
    if hit is None or hit[0]() is not param:
        weakref.finalize(param, _pack_cache.pop, key, None)
    _pack_cache[key] = (weakref.ref(param), token, out) + _built_on()
    return out


_ahead = False      # True while prefetch_packs builds on a side stream: those entries carry an event


def _built_on():
    """(stream the pack was built on, event recorded behind the build or None)"""
    cur = torch.cuda.current_stream()
    ev = None
    if _ahead:
        ev = torch.cuda.Event()
        ev.record(cur)
    return (cur.cuda_stream, ev)


def _adopt(hit):
    """a cached pack that was built ahead of time on ANOTHER stream: the consumer's stream waits for that build"""
    if hit[4] is not None:
        cur = torch.cuda.current_stream()
        if cur.cuda_stream != hit[3]:
            cur.wait_event(hit[4])
            hit[2].record_stream(cur)     # allocated on the builder's stream, read on this one
    return hit[2]


def _note_use(param, kind, direction, c_alloc):
    """remember which operand layouts a parameter is consumed in, so that they can be rebuilt ahead of time"""
    uses = getattr(param, "_eadgan_pack_uses", None)
    if uses is None:
        uses = set()
        param._eadgan_pack_uses = uses
    uses.add((kind, direction, c_alloc))


def prefetch_packs(param):
    """Rebuild, on the CURRENT stream, every operand layout ``param`` was consumed in so far (no-op for layouts whose
    cached pack is still current).  chain.prefetch_packs calls this on a side stream right after an optimiser step;
    every entry built here carries an event, and whichever stream later takes it from the cache waits on that event
    (``_adopt``), so no consumer -- chain executor, per-op module path, autograd worker -- can read a pack early."""
    global _ahead
    _ahead = True
    try:
        for kind, direction, c_alloc in tuple(getattr(param, "_eadgan_pack_uses", ())):
            _cached_pack(param, kind, direction, c_alloc)
    finally:
        _ahead = False


def invalidate_caches():
    _pack_cache.clear()
    L.bump_weights_epoch()


def _desc(n, c, h, w, k, act=ACT_NONE, slope=0.0, out_f32_nchw=False, want_stats=False, mask_mode=0, c_real=0):
    return L.TcDesc(n, c, h, w, k, act, float(slope), int(out_f32_nchw), int(want_stats), int(c_real), int(mask_mode))


def fprop(xp, wpk, bias, k, act=ACT_NONE, slope=0.0, out_f32_nchw=False, mask=None, mask_mode=0, stats=None,
          out=None, stats_mode=1, sigma=None):
    """big map xp [n,h+2,w+2,c] -> small map [n,p+2,q+2,k] (or fp32 NCHW [n,k,p,q])."""
    n, hp, wp, c = xp.shape
    h, w = hp - 2, wp - 2
    d = _desc(n, c, h, w, k, act, slope, out_f32_nchw, stats_mode if stats is not None else 0, mask_mode)
    if out is None:
        out = (torch.empty((n, k, h // 2, w // 2), device=xp.device, dtype=torch.float32) if out_f32_nchw
               else alloc_padded(n, h // 2, w // 2, k, xp.device))
    call("eadgan_tc_fprop", C.byref(d), ptr(xp), ptr(wpk), ptr(bias), ptr(out), ptr(mask), ptr(stats), ptr(sigma),
         stream())
    return out


def dgrad(yp, wpk, bias, c, act=ACT_NONE, slope=0.0, out_f32_nchw=False, mask=None, mask_mode=0, stats=None,
          out=None, c_real=0, stats_mode=1, sigma=None):
    """small map yp [n,p+2,q+2,k] -> big map [n,2p+2,2q+2,c] (or fp32 NCHW [n,c_real or c,2p,2q])."""
    n, pp, qp, k = yp.shape
    h, w = 2 * (pp - 2), 2 * (qp - 2)
    d = _desc(n, c, h, w, k, act, slope, out_f32_nchw, stats_mode if stats is not None else 0, mask_mode, c_real)
    if out is None:
        out = (torch.empty((n, c_real or c, h, w), device=yp.device, dtype=torch.float32) if out_f32_nchw
               else alloc_padded(n, h, w, c, yp.device))
    call("eadgan_tc_dgrad", C.byref(d), ptr(yp), ptr(wpk), ptr(bias), ptr(out), ptr(mask), ptr(stats), ptr(sigma),
         stream())
    return out


_ws_cache = {}


def _workspace(need, device):
    """scratch of at least ``need`` bytes for the kernels that split a reduction over CTAs (every wgrad, the dense
    gather): one per (device, stream), reused by every such launch on that stream, grown when a launch needs more"""
    key = (device, torch.cuda.current_stream().cuda_stream)
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < need:
        ws = torch.empty(need, device=device, dtype=torch.uint8)
        _ws_cache[key] = ws
    return ws


def dense_pack(w, m_pad, rows_major):
    """w viewed as [m][C][16] -> bf16 [m_pad][16C] (rows_major) or [16C][m_pad]."""
    m, Cc = w.shape[0], w.shape[1]
    out = torch.empty(m_pad * 16 * Cc, device=w.device, dtype=torch.bfloat16)
    call("eadgan_tc_dense_pack", ptr(w.contiguous()), m, m_pad, Cc, 1 if rows_major else 0, ptr(out), stream())
    return out


def dense_gather(yp, w_rows, bias, m_real):
    n, _, _, Cc = yp.shape
    out = torch.empty((n, m_real), device=yp.device, dtype=torch.float32)
    ws = _workspace(L.lib().eadgan_tc_dense_gather_workspace(n), yp.device)
    call("eadgan_tc_dense_gather", ptr(yp), ptr(w_rows), ptr(bias), ptr(out), n, Cc, m_real, ptr(ws),
         C.c_size_t(ws.numel()), stream())
    return out


def dense_scatter(a, w_cols, bias, Cc, mask=None, mask_act=0, slope=0.0, chan_sums=None):
    n, m_pad = a.shape
    out = alloc_padded(n, 4, 4, Cc, a.device)
    call("eadgan_tc_dense_scatter", ptr(a), ptr(w_cols), ptr(bias), ptr(out), ptr(mask), int(mask_act), float(slope),
         n, Cc, m_pad, ptr(chan_sums), stream())
    return out


def dense_wgrad(a, yp, m_real):
    n, m_pad = a.shape
    Cc = yp.shape[3]
    need = L.lib().eadgan_tc_dense_wgrad_workspace(Cc, m_pad)
    ws = _workspace(need, a.device)
    dw = torch.empty((m_real, Cc, 4, 4), device=a.device, dtype=torch.float32)
    call("eadgan_tc_dense_wgrad", ptr(a), ptr(yp), ptr(dw), ptr(ws), C.c_size_t(ws.numel()), n, Cc, m_real, m_pad,
         stream())
    return dw


def wgrad(xp, yp, c_real=0):
    """dw[k,c_real or c,4,4] fp32 from the big map xp and the small map yp (both padded NHWC bf16)."""
    n, hp, wp, c = xp.shape
    k = yp.shape[3]
    d = _desc(n, c, hp - 2, wp - 2, k, c_real=c_real)
    need = L.lib().eadgan_tc_workspace_bytes(C.byref(d), 2)
    if need == 0:
        raise RuntimeError(f"tc wgrad: unsupported geometry n={n} c={c} h={hp - 2} k={k}")
    ws = _workspace(need, xp.device)
    dw = torch.empty((k, c_real or c, 4, 4), device=xp.device, dtype=torch.float32)
    call("eadgan_tc_wgrad", C.byref(d), ptr(xp), ptr(yp), ptr(dw), ptr(ws), C.c_size_t(ws.numel()), stream())
    return dw


# ---- "thin" image layers (1..4-channel big map): row-expanded image buffer R[n][h/2][w+2][4][4] bf16 ----------
def thin_expand(x, mask_y=None, act=ACT_NONE, slope=0.0):
    """fp32 image [n,c<=4,h,w] (any strides) [* act'(mask_y)] -> row-expanded bf16 buffer (every element written)."""
    n, c, h, w = x.shape
    r = torch.empty((n, h // 2, w + 2, 4, 4), device=x.device, dtype=torch.bfloat16)
    src = t4(x)
    mk = t4(mask_y) if mask_y is not None else None
    call("eadgan_tc_thin_expand", C.byref(src), C.byref(mk) if mk is not None else None, int(act), float(slope), n, c, h, w,
         ptr(r), stream())
    return r


def thin_pack_w(w, direction):
    """fp32 [k, c<=4, 4, 4] -> bf16 [k][64] ("fprop") or [64][k] ("dgrad")."""
    k, c = w.shape[0], w.shape[1]
    assert tuple(w.shape[2:]) == (4, 4) and c <= 4
    out = torch.empty(k * 64, device=w.device, dtype=torch.bfloat16)
    call("eadgan_tc_thin_pack_w", ptr(w.contiguous()), k, c, 0 if direction == "fprop" else 1, ptr(out), stream())
    return out


def thin_pack_w_cached(param, direction):
    """thin_pack_w of a parameter, cached until it changes (``_cached_pack``)."""
    return _cached_pack(param, "thin", direction, None)


def thin_fprop(r, wpk, bias, c, k, act=ACT_NONE, slope=0.0, mask=None, mask_mode=0, stats=None, stats_mode=1, sigma=None,
               out=None):
    """row-expanded image r -> small map [n,p+2,q+2,k] padded NHWC bf16."""
    n, p, wp = r.shape[0], r.shape[1], r.shape[2]
    h, w = 2 * p, wp - 2
    d = _desc(n, c, h, w, k, act, slope, False, stats_mode if stats is not None else 0, mask_mode)
    if out is None:
        out = alloc_padded(n, h // 2, w // 2, k, r.device)
    call("eadgan_tc_thin_fprop", C.byref(d), ptr(r), ptr(wpk), ptr(bias), ptr(out), ptr(mask), ptr(stats), ptr(sigma),
         stream())
    return out


def thin_wgrad(r, yp, c):
    """dw[k,c,4,4] fp32 from the row-expanded image r and the small map yp (padded NHWC bf16)."""
    n, p, wp = r.shape[0], r.shape[1], r.shape[2]
    k = yp.shape[3]
    d = _desc(n, c, 2 * p, wp - 2, k)
    need = L.lib().eadgan_tc_thin_wgrad_workspace(C.byref(d))
    if need == 0:
        raise RuntimeError(f"tc thin wgrad: unsupported geometry n={n} c={c} h={2 * p} k={k}")
    ws = _workspace(need, r.device)
    dw = torch.empty((k, c, 4, 4), device=r.device, dtype=torch.float32)
    call("eadgan_tc_thin_wgrad", C.byref(d), ptr(r), ptr(yp), ptr(dw), ptr(ws), C.c_size_t(ws.numel()), stream())
    return dw


def thin_dgrad(yp, wpk, bias, c, act=ACT_NONE, slope=0.0, sigma=None, out=None):
    """small map yp [n,p+2,34,k] -> fp32 NCHW image [n,c,2p,64] = act(conv_transpose(yp, W/sigma) + bias)."""
    n, pp, qp, k = yp.shape
    h, w = 2 * (pp - 2), 2 * (qp - 2)
    d = _desc(n, c, h, w, k, act, slope, True)
    if out is None:
        out = torch.empty((n, c, h, w), device=yp.device, dtype=torch.float32)
    call("eadgan_tc_thin_dgrad", C.byref(d), ptr(yp), ptr(wpk), ptr(bias), ptr(out), ptr(sigma), stream())
    return out


def gemm(a, b):
    """C[m,n] fp32 = A[m,k] bf16 @ B[n,k]^T bf16 through the tcgen05 mainloop."""
    m, kk = a.shape
    n = b.shape[0]
    c = torch.empty((m, n), device=a.device, dtype=torch.float32)
    call("eadgan_tc_gemm", ptr(a.contiguous()), ptr(b.contiguous()), ptr(c), m, n, kk, stream())
    return c
