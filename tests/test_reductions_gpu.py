"""The fp32 streaming kernels (losses, spectral norm, Adam, BatchNorm, SIMT split-K and split wgrad, softmax, upsample,
channel_sum) against an fp64 referee, at the shapes where their work is split: block partitions, partial sums, vector
tails and alignment fallbacks.

BRANCHES names, for each parametrised shape, the launch branch it is there to reach.  The *_branch helpers restate only
the size arithmetic the C code selects that branch with (loss_blocks, sn_small, ADAM_CHUNK, CHUNK / cb, pick_ksplit,
wgrad_split), with the SM count as an argument.  test_branch_table (no GPU) checks the table at the B200's 148 SMs, and
every GPU test asserts that its shape still takes its branch on the device it runs on, so a threshold change cannot
move a shape off its branch silently.

Referee (test_ops_gpu._ok): the kernel's error against fp64 is at most max(tol, 2 x the error of stock torch fp32)."""
import ctypes as C
import itertools
import math

import pytest
import torch
import torch.nn.functional as TF

from conftest import rel_err
from test_ops_gpu import TOL, _ok

B200_SMS = 148


def _cdiv(a, b):
    return -(-a // b)


# ---- branch selection, restated from the C sources --------------------------------------------------------------
def loss_branch(shape, sms):
    """loss_adam.cu loss_blocks: one block per LCHUNK = 8192 elements (rows for cross-entropy), at most 256."""
    kind, rows, cols = shape
    n = rows if kind == "ce" else rows * cols
    blocks = _cdiv(n, 8192)
    if blocks <= 1:
        return "one block"
    return "capped grid" if blocks > 256 else "multi-block"


def sn_branch(shape, sms):
    """spectral_norm.cu: sn_small (one block), else W^T u split over row ranges of >= 16 rows (sn_wtu / sn_vsum),
    float4 bodies of sn_wv / sn_bwd when cols % 4 == 0 and of sn_dot when rows * cols % 4 == 0, and a v slice of
    ceil(cols / rows) per sn_wv block."""
    rows, cols = shape
    if rows * cols <= 16 * 1024 and cols <= 4096 and rows <= 1024:
        return "small"
    splits = max(1, min(_cdiv(4 * sms, _cdiv(cols, 128)), _cdiv(rows, 16)))
    splits = _cdiv(rows, _cdiv(rows, splits))
    tags = ["multi", "split" if splits > 1 else "splits=1", "vec4" if cols % 4 == 0 else "scalar"]
    if rows * cols % 4:
        tags.append("dot-scalar")
    if _cdiv(cols, rows) == 1:
        tags.append("v-slice=1")
    return " ".join(tags)


def adam_branch(numel, sms):
    """loss_adam.cu adam_kernel on 16-byte aligned tensors: ADAM_CHUNK = 16384 elements per block, float4 body and a
    scalar tail inside each chunk."""
    blocks = _cdiv(numel, 16384)
    last = numel - (blocks - 1) * 16384
    return f"blocks={blocks} last={last} f4={last // 4 * 4} tail={last % 4}"


def adam_align_branch(offset, sms):
    """adam_kernel takes the float4 body only when p, g, m and v are all 16-byte aligned; `offset` is the parameter's
    element offset into a flat fp32 buffer."""
    return "float4" if offset * 4 % 16 == 0 else "scalar"


def adam_launch_branch(steps, sms):
    """optim.Adam.step: one launch per run of parameters with equal step counts, split at 48 tensors
    (EADGAN_ADAM_MAX_TENSORS)."""
    runs = [len(list(g)) for _, g in itertools.groupby(steps)]
    return f"launches={sum(_cdiv(r, 48) for r in runs)}"


def bn_branch(shape, sms):
    """bn.cu, fp32: kind 0 (NCHW) warp jobs of CHUNK = 2048 plane elements; kind 1 (channels last) cb = min(c, 256)
    channels per pass and 256 // cb pixel lanes per block."""
    n, c, h, w, layout = shape
    if layout == "nchw":
        return f"kind0 jobs/plane={_cdiv(h * w, 2048)}" + (" ragged" if h * w % 2048 else "")
    cb = min(c, 256)
    lanes = 256 // cb
    return f"kind1 cb={cb} lanes={lanes} idle={256 - cb * lanes} passes={_cdiv(c, cb)}" + (" partial" if c % cb else "")


def _gemm_extents(shape):
    dirn, n, c, h, k, r, stride, pad = shape
    p = (h + 2 * pad - r) // stride + 1
    return (n * p * p, k, c * r * r) if dirn == "fprop" else (n * h * h, c, k * r * r)


def ksplit_branch(shape, sms):
    """simt_conv.cu pick_ksplit: clusters of ksplit CTAs along K for <= 37 output tiles and >= 16 k tiles (BK = 16),
    ksplit in {8, 4, 2} with >= 4 k tiles per CTA and <= 296 CTAs; CTA z reduces tiles [z * per, (z + 1) * per)."""
    M, N, K = _gemm_extents(shape)
    ctas, k_tiles = _cdiv(M, 64) * _cdiv(N, 64), _cdiv(K, 16)
    ks = 1
    if ctas <= 37 and k_tiles >= 16:
        ks = 8
        while ks > 1 and (k_tiles // ks < 4 or ctas * ks > 296):
            ks //= 2
    tags = [f"ksplit={ks}"]
    if ks > 1 and (ks - 1) * _cdiv(k_tiles, ks) >= k_tiles:
        tags.append("empty-rank")
    if K % 16:
        tags.append("K-tail")
    return " ".join(tags)


def wgrad_branch(shape, sms):
    """simt_conv.cu wgrad_split: the n*p*q reduction split to fill 4 x SMs CTAs, >= 4 BK-chunks per split, split
    length rounded up to BK = 16 rows."""
    n, c, h, k, r, stride, pad = shape
    p = (h + 2 * pad - r) // stride + 1
    K = n * p * p
    tiles = _cdiv(c * r * r, 64) * _cdiv(k, 64)
    sp = max(1, min(_cdiv(4 * sms, tiles), _cdiv(K, 64)))
    m = _cdiv(_cdiv(K, sp), 16) * 16
    splits = _cdiv(K, m)
    last = K - (splits - 1) * m
    if splits == 1:
        return "one split"
    return "split last-chunk-ragged" if last % 16 else "split"


def softmax_branch(shape, sms):
    """elementwise.cu softmax: one warp per row (lanes loop over cols > 32), 8 rows per block."""
    rows, cols = shape
    return ("lanes-loop" if cols > 32 else "one-pass") + (" partial-block" if rows % 8 else "")


def upsample_branch(shape, sms):
    n, c, h, w = shape
    return f"h={'odd' if h % 2 else 'even'} w={'odd' if w % 2 else 'even'}"


def channel_sum_branch(shape, sms):
    """simt_conv.cu channel_sum: one 256-thread block per channel striding n*h*w."""
    n, c, h, w = shape
    return f"strides={_cdiv(n * h * w, 256)}" + (" ragged" if n * h * w % 256 else "")


BRANCH_OF = {"loss": loss_branch, "sn": sn_branch, "adam": adam_branch, "adam_align": adam_align_branch,
             "adam_launch": adam_launch_branch, "bn": bn_branch, "ksplit": ksplit_branch, "wgrad": wgrad_branch,
             "softmax": softmax_branch, "upsample": upsample_branch, "channel_sum": channel_sum_branch}

# family -> [(shape, branch it must take, why)]
BRANCHES = {
    "loss": [  # (kind, rows, cols)
        (("bce", 8193, 1), "multi-block", "one element past a block: memset, then atomicAdd of 2 partials"),
        (("bce", 2097153, 1), "capped grid", "one element past 256 x 8192: block 0 strides a second chunk"),
        (("mse", 1700, 5), "multi-block", "5-wide code MSE at batch 1700 (> 1638)"),
        (("mse", 600001, 5), "capped grid", "3 M elements: every block strides past its chunk"),
        (("ce", 1024, 10), "one block", "CelebA's 1024 rows: each of 256 threads loops over 4 rows"),
        (("ce", 8193, 3), "multi-block", "rows select the grid of the cross-entropy kernels"),
        (("mi", 3000, 3), "multi-block", "9000 elements of the mutual-information loss"),
    ],
    "sn": [  # (rows, cols) of W viewed as a matrix
        ((128, 128), "small", "exactly 16384 weights"),
        ((128, 129), "multi split scalar", "one column past 16384 weights; cols % 4 != 0"),
        ((1, 4096), "small", "cols at the 4096 limit"),
        ((1, 4097), "multi splits=1 scalar dot-scalar", "cols 4097 > 4096 with 4097 weights; odd count"),
        ((1024, 16), "small", "rows at the 1024 limit, 16384 weights"),
        ((1025, 8), "multi split vec4 v-slice=1", "rows 1025 > 1024; rows > cols gives each sn_wv block one v"),
        ((8, 4100), "multi splits=1 vec4", "rows < 16: a single row range"),
        ((300, 75), "multi split scalar v-slice=1", "rows > cols, cols % 4 != 0"),
        ((63, 1027), "multi split scalar dot-scalar", "every scalar fallback, odd weight count"),
        ((512, 1000), "multi split vec4", "aligned multi-kernel reference"),
    ],
    "adam": [  # numel of one aligned tensor
        (1, "blocks=1 last=1 f4=0 tail=1", "scalar tail only"),
        (3, "blocks=1 last=3 f4=0 tail=3", "scalar tail only"),
        (16384, "blocks=1 last=16384 f4=16384 tail=0", "exactly one chunk"),
        (16385, "blocks=2 last=1 f4=0 tail=1", "one element past a chunk"),
        (16391, "blocks=2 last=7 f4=4 tail=3", "float4 and scalar tail inside the last chunk"),
        (3 * 16384 + 3, "blocks=4 last=3 f4=0 tail=3", "a last chunk of scalar tail only"),
    ],
    "adam_align": [  # element offset of the parameter in a flat buffer
        (1, "scalar", "4-byte misaligned slice"),
        (3, "scalar", "12-byte misaligned slice"),
    ],
    "adam_launch": [  # per-parameter step counts of one group, in order
        ((1,) * 50, "launches=2", "50 parameters: 48 + 2"),
        ((3, 2, 3, 3), "launches=3", "one parameter skipped a step: the group splits around it"),
    ],
    "bn": [  # (n, c, h, w, layout)
        ((2, 3, 45, 47, "nchw"), "kind0 jobs/plane=2 ragged", "a plane of 2115 spans two warp jobs, the last of 67"),
        ((3, 5, 64, 64, "nchw"), "kind0 jobs/plane=2", "a plane of exactly two warp jobs"),
        ((4, 96, 9, 11, "nhwc"), "kind1 cb=96 lanes=2 idle=64 passes=1", "c does not divide 256"),
        ((5, 3, 17, 13, "nhwc"), "kind1 cb=3 lanes=85 idle=1 passes=1", "3 channels: 85 pixel lanes"),
        ((3, 384, 5, 7, "nhwc"), "kind1 cb=256 lanes=1 idle=0 passes=2 partial", "c > 256: partial second pass"),
    ],
    "ksplit": [  # (direction, n, c, h, k, r, stride, pad) of the conv descriptor; square maps and kernels
        (("fprop", 5, 397, 1, 19, 1, 1, 0), "ksplit=4 K-tail", "Linear 397 -> 19: 25 k tiles, tail in CTA 3"),
        (("fprop", 7, 520, 1, 10, 1, 1, 0), "ksplit=8 empty-rank K-tail",
         "Linear 520 -> 10: 33 k tiles, per = 5, CTA 7 starts at tile 35 and only joins the cluster"),
        (("fprop", 4, 64, 3, 32, 3, 1, 1), "ksplit=8", "3x3 conv, pad 1, on a 3x3 map: padded gather"),
        (("dgrad", 4, 64, 3, 32, 3, 1, 1), "ksplit=4", "its input gradient: 18 k tiles"),
        (("dgrad", 3, 8, 4, 64, 4, 2, 1), "ksplit=8", "ConvTranspose 64 -> 8, stride 2: strided gather"),
    ],
    "wgrad": [  # (n, c, h, k, r, stride, pad)
        ((1000, 64, 1, 64, 1, 1, 0), "split last-chunk-ragged", "Linear at batch 1000: last split of 40 rows"),
        ((7, 8, 5, 16, 3, 1, 1), "split last-chunk-ragged", "3x3 conv, 175 pixels: last split of 47 rows"),
    ],
    "softmax": [((13, 75), "lanes-loop partial-block", "cols > 32 and rows % 8 != 0")],
    "upsample": [((2, 3, 5, 7), "h=odd w=odd", "odd map extents")],
    "channel_sum": [
        ((3, 5, 7, 11), "strides=1 ragged", "231 elements per channel"),
        ((2, 4, 10, 15), "strides=2 ragged", "300 elements per channel: one full stride and a tail"),
    ],
}


def _shapes(family):
    return [s for s, _, _ in BRANCHES[family]]


def _ids(shape):
    return "-".join(map(str, shape)) if isinstance(shape, tuple) else str(shape)


def _on_branch(family, shape, sms):
    want = next(b for s, b, _ in BRANCHES[family] if s == shape)
    got = BRANCH_OF[family](shape, sms)
    assert got == want, f"{family} {shape} takes '{got}' at {sms} SMs, not '{want}'"


def test_branch_table():
    """every table shape lands on its named branch at the B200's SM count (no GPU needed)"""
    for family, entries in BRANCHES.items():
        for shape, branch, _ in entries:
            assert BRANCH_OF[family](shape, B200_SMS) == branch, (family, shape, BRANCH_OF[family](shape, B200_SMS))


# ---- GPU tests -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sms(cuda):
    from eadgan_b200 import _lib
    return _lib.lib().eadgan_sm_count()


def _gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def _check(what, ours, ref32, ref64, tol=TOL):
    ok, errs = _ok(ours, ref32, ref64, tol)
    assert ok, f"{what}: error vs fp64 {errs[0]:.3g}, stock torch fp32 {errs[1]:.3g}"


def _loss_case(kind, rows, cols, g):
    """-> (inputs on the CPU, indices that take a gradient, our loss, torch's loss)"""
    import eadgan_b200.functional as Fn
    if kind == "bce":
        p = torch.rand(rows, cols, generator=g).clamp_(1e-4, 1 - 1e-4)
        t = (torch.rand(rows, cols, generator=g) > 0.5).float()
        p[::997] = t[::997]   # p exactly 0 or 1: log(0) is clamped at -100 and multiplied by a zero target
        return [p, t], [0], Fn.bce_loss, TF.binary_cross_entropy
    if kind == "mse":
        return [torch.randn(rows, cols, generator=g), torch.randn(rows, cols, generator=g)], [0, 1], Fn.mse_loss, \
            TF.mse_loss
    if kind == "ce":
        return [torch.randn(rows, cols, generator=g) * 2, torch.randint(0, cols, (rows,), generator=g)], [0], \
            Fn.cross_entropy, TF.cross_entropy
    q = torch.softmax(torch.randn(rows, cols, generator=g), 1)
    c = torch.softmax(torch.randn(rows, cols, generator=g), 1)
    ref = lambda q, c: (torch.mean(-torch.sum(torch.log(q + 1e-8) * c, dim=1)) +  # noqa: E731
                        torch.mean(-torch.sum(torch.log(c + 1e-8) * c, dim=1)))
    return [q, c], [0], Fn.mutual_info_loss, ref


@pytest.mark.gpu
@pytest.mark.parametrize("shape", _shapes("loss"), ids=_ids)
def test_loss_blocks(cuda, sms, shape):
    """loss value and input gradients (upstream gradient 0.7); BCE's fp64 reference clamps its logs at -100 too"""
    _on_branch("loss", shape, sms)
    args, gi, ours_fn, ref_fn = _loss_case(*shape, _gen(11))

    def run(dtype, fn):
        xs = [a.to(cuda, dtype) if a.is_floating_point() else a.to(cuda) for a in args]
        for i in gi:
            xs[i].requires_grad_()
        loss = fn(*xs)
        grads = torch.autograd.grad(loss, [xs[i] for i in gi], torch.tensor(0.7, device=cuda, dtype=dtype))
        return loss, grads

    (lo, go), (l32, g32), (l64, g64) = run(torch.float32, ours_fn), run(torch.float32, ref_fn), \
        run(torch.float64, ref_fn)
    _check("loss", lo, l32, l64)
    for i, (a, b, c) in enumerate(zip(go, g32, g64)):
        _check(f"grad {i}", a, b, c)


def _sn_ref(W, u, G, eps=1e-12):
    """torch.nn.utils.spectral_norm's training forward (one power iteration from u) and the backward of W / sigma
    with u, v held constant: dW / sigma - (<dW, W> / sigma^2) u v^T"""
    v = TF.normalize(torch.mv(W.t(), u), dim=0, eps=eps)
    Wv = torch.mv(W, v)
    u = TF.normalize(Wv, dim=0, eps=eps)
    sigma = torch.dot(u, Wv)
    dW = G / sigma - (torch.sum(G * W) / sigma ** 2) * torch.outer(u, v)
    return u, v, sigma, W / sigma, dW


@pytest.mark.gpu
@pytest.mark.parametrize("shape", _shapes("sn"), ids=_ids)
def test_spectral_norm_partials(cuda, sms, shape):
    """u, v, sigma, W / sigma and the weight gradient of a training forward, then the eval forward (no power iteration)
    from the updated u, v; the training pass twice on the same inputs is bitwise identical"""
    import eadgan_b200.functional as Fn
    _on_branch("sn", shape, sms)
    rows, cols = shape
    g = _gen(12)
    W = torch.randn(rows, cols, generator=g) * 0.1
    u0 = TF.normalize(torch.randn(rows, generator=g), dim=0)
    v0 = TF.normalize(torch.randn(cols, generator=g), dim=0)
    G = torch.randn(rows, cols, generator=g)

    def ours():
        w = W.to(cuda).requires_grad_()
        u, v = u0.to(cuda), v0.to(cuda)
        w_sn, sigma = Fn.spectral_norm_weight(w, u, v, True, 1e-12)
        (dw,) = torch.autograd.grad(w_sn, w, G.to(cuda))
        return u, v, sigma.reshape(()), w_sn.detach(), dw

    got = ours()
    r32 = _sn_ref(W.to(cuda), u0.to(cuda), G.to(cuda))
    r64 = _sn_ref(W.to(cuda, torch.float64), u0.to(cuda, torch.float64), G.to(cuda, torch.float64))
    for name, a, b, c in zip(("u", "v", "sigma", "W_sn", "dW"), got, r32, r64):
        _check(name, a, b, c)
    for name, a, b in zip(("u", "v", "sigma", "W_sn", "dW"), got, ours()):
        assert torch.equal(a, b), f"{name} differs between two runs on the same inputs"

    u, v = got[0].clone(), got[1].clone()
    w_sn, sigma = Fn.spectral_norm_weight(W.to(cuda), u, v, False, 1e-12)
    assert torch.equal(u, got[0]) and torch.equal(v, got[1]), "the eval forward changed u or v"
    s32 = torch.dot(u, torch.mv(W.to(cuda), v))
    s64 = torch.dot(u.double(), torch.mv(W.to(cuda, torch.float64), v.double()))
    _check("eval sigma", sigma.reshape(()), s32, s64)
    _check("eval W_sn", w_sn, W.to(cuda) / s32, W.to(cuda, torch.float64) / s64)


# ---- Adam --------------------------------------------------------------------------------------------------------
LR, BETAS, EPS = 2e-4, (0.5, 0.999), 1e-8


def _adam64(p, m, v, g, t, lr=LR, betas=BETAS, eps=EPS):
    """torch/optim/adam.py::_single_tensor_adam restated in fp64; returns the new (p, m, v)"""
    b1, b2 = betas
    m = b1 * m + (1 - b1) * g
    v = b2 * v + (1 - b2) * g * g
    p = p - lr / (1 - b1 ** t) * m / (v.sqrt() / math.sqrt(1 - b2 ** t) + eps)
    return p, m, v


def _adam_c(ps, gs, ms, vs, t, gscale=1.0, step_dev=None, lr=LR, betas=BETAS, eps=EPS):
    """one launch of eadgan_adam_step (host step count t) or eadgan_adam_step_dev (device step counter)"""
    from eadgan_b200 import _lib as L
    A = L.AdamTensors()
    for j, (p, g, m, v) in enumerate(zip(ps, gs, ms, vs)):
        A.p[j], A.g[j], A.m[j], A.v[j], A.numel[j] = p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel()
    A.count = len(ps)
    b1, b2 = betas
    if step_dev is None:
        L.call("eadgan_adam_step", C.byref(A), b1, b2, eps, lr / (1 - b1 ** t), math.sqrt(1 - b2 ** t), gscale,
               L.stream())
    else:
        L.call("eadgan_adam_step_dev", C.byref(A), b1, b2, eps, lr, C.c_void_p(step_dev.data_ptr()), gscale,
               L.stream())


def _adam_check(what, ours, theirs, ref64):
    """against torch fp32 at 2e-6 (SURVEY.md section 7.3-1 iii) and against the fp64 restatement by the referee rule"""
    assert rel_err(ours, theirs) <= 2e-6, (what, rel_err(ours, theirs))
    _check(what, ours, theirs, ref64, tol=2e-6)


def _adam_run(params, steps, cuda, seed):
    """our Adam and torch.optim.Adam(foreach=False) on copies of `params` (CPU tensors are copied to the device, a
    device leaf is stepped as is), each given the same gradients; steps[i] is the set of parameter indices that get a
    gradient at step i.  Checks p, m, v after every step; returns the parameters and the launches of every step."""
    from eadgan_b200 import _lib as L
    from eadgan_b200.optim import Adam
    po = [p if p.is_cuda else p.to(cuda).requires_grad_() for p in params]
    pr = [p.detach().clone().requires_grad_() for p in po]
    s64 = [[p.detach().double(), torch.zeros_like(p, dtype=torch.float64), torch.zeros_like(p, dtype=torch.float64), 0]
           for p in po]
    oo, orf = Adam(po, lr=LR, betas=BETAS), torch.optim.Adam(pr, lr=LR, betas=BETAS, foreach=False)
    g = _gen(seed)
    launches = []
    for it, active in enumerate(steps):
        for i, (a, b) in enumerate(zip(po, pr)):
            if i in active:
                gr = (torch.randn(a.shape, generator=g) * 10.0 ** (it - 1)).to(cuda)
                a.grad, b.grad = gr.clone(), gr.clone()
                st = s64[i]
                st[3] += 1
                st[0], st[1], st[2] = _adam64(st[0], st[1], st[2], gr.double(), st[3])
            else:
                a.grad = b.grad = None
        before = L.launches
        oo.step()
        launches.append(L.launches - before)
        orf.step()
        for i, (a, b) in enumerate(zip(po, pr)):
            _adam_check(f"p[{i}] step {it}", a, b, s64[i][0])
            _adam_check(f"m[{i}] step {it}", oo.state[a]["exp_avg"], orf.state[b]["exp_avg"], s64[i][1])
            _adam_check(f"v[{i}] step {it}", oo.state[a]["exp_avg_sq"], orf.state[b]["exp_avg_sq"], s64[i][2])
    return po, launches


@pytest.mark.gpu
@pytest.mark.parametrize("numel", _shapes("adam"), ids=_ids)
def test_adam_chunk_edges(cuda, sms, numel):
    _on_branch("adam", numel, sms)
    p = torch.randn(numel, generator=_gen(13))
    _adam_run([p], [{0}] * 3, cuda, seed=14)


@pytest.mark.gpu
@pytest.mark.parametrize("offset", _shapes("adam_align"), ids=_ids)
def test_adam_misaligned_slice(cuda, sms, offset):
    """a contiguous slice of a flat parameter buffer (scalar branch) in one launch with aligned tensors (float4)"""
    _on_branch("adam_align", offset, sms)
    g = _gen(15)
    n = 16391
    flat = torch.randn(offset + n, generator=g).to(cuda)
    sl = flat[offset:offset + n].requires_grad_()
    assert sl.data_ptr() % 16 != 0
    po, launches = _adam_run([torch.randn(16385, generator=g), sl, torch.randn(5, generator=g)], [{0, 1, 2}] * 3,
                             cuda, seed=16)
    assert launches == [1, 1, 1]
    assert po[1].data_ptr() == flat.data_ptr() + 4 * offset, "the slice was not stepped in place"


@pytest.mark.gpu
def test_adam_fifty_parameters(cuda, sms):
    _on_branch("adam_launch", (1,) * 50, sms)
    g = _gen(17)
    _, launches = _adam_run([torch.randn(1 + 37 * i, generator=g) for i in range(50)], [set(range(50))] * 2, cuda,
                            seed=18)
    assert launches == [2, 2]


@pytest.mark.gpu
def test_adam_skipped_step(cuda, sms):
    """parameter 1 gets no gradient at step 2: at step 3 it is at t = 2 while the others are at t = 3"""
    _on_branch("adam_launch", (3, 2, 3, 3), sms)
    g = _gen(19)
    _, launches = _adam_run([torch.randn(n, generator=g) for n in (16385, 7, 3, 16384)],
                            [{0, 1, 2, 3}, {0, 2, 3}, {0, 1, 2, 3}], cuda, seed=20)
    assert launches == [1, 1, 3]


@pytest.mark.gpu
def test_adam_grad_scale(cuda):
    """grad_scale = 0.5 (the data-parallel average over 2 ranks) through the C entry, against torch on 0.5 * g"""
    g = _gen(21)
    shapes = (16385, 7)
    ps = [torch.randn(n, generator=g).to(cuda) for n in shapes]
    ms, vs = [torch.zeros_like(p) for p in ps], [torch.zeros_like(p) for p in ps]
    pr = [p.clone().requires_grad_() for p in ps]
    s64 = [[p.double(), torch.zeros_like(p, dtype=torch.float64), torch.zeros_like(p, dtype=torch.float64)] for p in ps]
    orf = torch.optim.Adam(pr, lr=LR, betas=BETAS, foreach=False)
    for t in (1, 2):
        gs = [torch.randn(p.shape, generator=g).to(cuda) for p in ps]
        _adam_c(ps, gs, ms, vs, t, gscale=0.5)
        for b, gr in zip(pr, gs):
            b.grad = 0.5 * gr
        orf.step()
        for i in range(len(ps)):
            s64[i] = _adam64(*s64[i], 0.5 * gs[i].double(), t)
            _adam_check(f"p[{i}] t={t}", ps[i], pr[i], s64[i][0])
            _adam_check(f"m[{i}] t={t}", ms[i], orf.state[pr[i]]["exp_avg"], s64[i][1])
            _adam_check(f"v[{i}] t={t}", vs[i], orf.state[pr[i]]["exp_avg_sq"], s64[i][2])


@pytest.mark.gpu
def test_adam_device_step_counter(cuda):
    """eadgan_adam_step_dev (bias corrections formed on the device from the int64 counter that eadgan_adam_advance
    moves) is bitwise equal to the host entry and matches torch, for t = 1..4 and then t = 1000"""
    from eadgan_b200._lib import call, stream
    g = _gen(22)
    shapes = (16391, 3)
    init = [torch.randn(n, generator=g).to(cuda) for n in shapes]
    dev = [[p.clone(), torch.zeros_like(p), torch.zeros_like(p)] for p in init]
    host = [[p.clone(), torch.zeros_like(p), torch.zeros_like(p)] for p in init]
    pr = [p.clone().requires_grad_() for p in init]
    s64 = [[p.double(), torch.zeros_like(p, dtype=torch.float64), torch.zeros_like(p, dtype=torch.float64)]
           for p in init]
    orf = torch.optim.Adam(pr, lr=LR, betas=BETAS, foreach=False)
    counter = torch.zeros(1, device=cuda, dtype=torch.int64)
    for t in (1, 2, 3, 4, 1000):
        if t == 1000:
            counter.fill_(t)
            for b in pr:
                orf.state[b]["step"].fill_(t - 1)
        else:
            call("eadgan_adam_advance", C.c_void_p(counter.data_ptr()), stream())
        gs = [torch.randn(p.shape, generator=g).to(cuda) for p in init]
        _adam_c(*zip(*[(d[0], gr, d[1], d[2]) for d, gr in zip(dev, gs)]), t, step_dev=counter)
        _adam_c(*zip(*[(h[0], gr, h[1], h[2]) for h, gr in zip(host, gs)]), t)
        for b, gr in zip(pr, gs):
            b.grad = gr.clone()
        orf.step()
        assert int(counter) == t
        for i in range(len(init)):
            s64[i] = _adam64(*s64[i], gs[i].double(), t)
            for j, name in enumerate(("p", "m", "v")):
                assert torch.equal(dev[i][j], host[i][j]), f"{name}[{i}] t={t}: device-counter entry != host entry"
            _adam_check(f"p[{i}] t={t}", dev[i][0], pr[i], s64[i][0])
            _adam_check(f"m[{i}] t={t}", dev[i][1], orf.state[pr[i]]["exp_avg"], s64[i][1])
            _adam_check(f"v[{i}] t={t}", dev[i][2], orf.state[pr[i]]["exp_avg_sq"], s64[i][2])


# ---- BatchNorm fp32 ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", _shapes("bn"), ids=_ids)
def test_batchnorm_fp32_jobs(cuda, sms, shape):
    """training forward (y, running mean, unbiased running var), backward (dx, dgamma, dbeta), then eval forward and
    backward from the updated running statistics, through the C entries in the tensor's own layout"""
    import eadgan_b200.functional as Fn
    from eadgan_b200._lib import ACT_NONE, call, ptr, stream
    _on_branch("bn", shape, sms)
    n, c, h, w, layout = shape
    fmt = torch.channels_last if layout == "nhwc" else torch.contiguous_format
    g = _gen(23)
    eps, mom = 1e-5, 0.1
    x = torch.randn(n, c, h, w, generator=g) * 1.7 + 0.3
    dy = torch.randn(n, c, h, w, generator=g)
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g) * 0.2
    rm0, rv0 = torch.randn(c, generator=g) * 0.1, torch.rand(c, generator=g) + 0.5
    xd, dyd = x.to(cuda).contiguous(memory_format=fmt), dy.to(cuda).contiguous(memory_format=fmt)
    gd, bd, rm, rv = (t.to(cuda) for t in (gamma, beta, rm0, rv0))

    sums = torch.zeros(2 * c, device=cuda, dtype=torch.float64)
    call("eadgan_bn_stats", Fn._ref(xd), n, c, h, w, ptr(sums), stream())
    y = torch.empty_like(xd)
    mean, invstd, count, _ = Fn.bn_train_forward(xd, sums, gd, bd, rm, rv, mom, eps, ACT_NONE, 0.0, y)
    dx = torch.empty_like(xd)
    dgamma, dbeta, _ = Fn.bn_train_backward(dyd, xd, None, mean, invstd, gd, bd, ACT_NONE, 0.0, count,
                                            torch.zeros_like(sums), dx)
    ye = torch.empty_like(xd)
    call("eadgan_bn_eval", Fn._ref(xd), n, c, h, w, ptr(rm), ptr(rv), eps, ptr(gd), ptr(bd), ACT_NONE, 0.0,
         Fn._ref(ye), stream())
    dxe = torch.empty_like(xd)
    dge, dbe, _ = Fn.bn_eval_backward(dyd, xd, None, rm, rv, eps, gd, bd, ACT_NONE, 0.0, torch.zeros_like(sums), dxe)

    def ref(dtype):
        xs = xd.to(dtype).requires_grad_()
        ga, be = gd.to(dtype).requires_grad_(), bd.to(dtype).requires_grad_()
        rms, rvs = rm0.to(cuda, dtype), rv0.to(cuda, dtype)
        yr = TF.batch_norm(xs, rms, rvs, ga, be, True, mom, eps)
        grads = torch.autograd.grad(yr, (xs, ga, be), dyd.to(dtype))
        xe = xs.detach().requires_grad_()
        ga_e, be_e = ga.detach().requires_grad_(), be.detach().requires_grad_()
        yre = TF.batch_norm(xe, rms, rvs, ga_e, be_e, False, mom, eps)
        grads_e = torch.autograd.grad(yre, (xe, ga_e, be_e), dyd.to(dtype))
        return (yr, rms, rvs, *grads, yre, *grads_e)

    names = ("y", "running_mean", "running_var", "dx", "dgamma", "dbeta", "eval y", "eval dx", "eval dgamma",
             "eval dbeta")
    for name, a, b, c64 in zip(names, (y, rm, rv, dx, dgamma, dbeta, ye, dxe, dge, dbe), ref(torch.float32),
                               ref(torch.float64)):
        _check(name, a, b, c64)


# ---- SIMT convolution: split-K and split wgrad -------------------------------------------------------------------
def _desc(shape):
    from eadgan_b200._lib import ConvDesc
    _, n, c, h, k, r, stride, pad = shape
    p = (h + 2 * pad - r) // stride + 1
    return ConvDesc(n, c, h, h, k, r, r, p, p, stride, pad), p


@pytest.mark.gpu
@pytest.mark.parametrize("mask", [False, True], ids=["plain", "mask"])
@pytest.mark.parametrize("shape", _shapes("ksplit"), ids=_ids)
def test_simt_split_k(cuda, sms, shape, mask):
    """eadgan_conv_fprop / eadgan_conv_dgrad on launches that sum K over a thread-block cluster, with bias, and with
    the fused epilogue lrelu(acc + b, 0.1) * lrelu'(mask, 0.2) after the DSMEM reduction; two runs are bitwise equal
    (rank-order sum)"""
    from eadgan_b200._lib import ACT_LRELU, ACT_NONE, call, ptr, stream, t4
    _on_branch("ksplit", shape, sms)
    dirn, n, c, h, k, r, stride, pad = shape
    d, p = _desc(shape)
    g = _gen(24)
    w = torch.randn(k, c, r, r, generator=g) * 0.05
    if dirn == "fprop":
        a, out_shape, nb = torch.randn(n, c, h, h, generator=g), (n, k, p, p), k
        ref = lambda a, w, b: TF.conv2d(a, w, b, stride, pad)  # noqa: E731
    else:
        a, out_shape, nb = torch.randn(n, k, p, p, generator=g), (n, c, h, h), c
        op = h - ((p - 1) * stride - 2 * pad + r)
        ref = lambda a, w, b: TF.conv_transpose2d(a, w, b, stride, pad, output_padding=op)  # noqa: E731
    b = torch.randn(nb, generator=g)
    mk = torch.randn(out_shape, generator=g)
    ad, wd, bd, mkd = (t.to(cuda) for t in (a, w, b, mk))
    act, slope = (ACT_LRELU, 0.1) if mask else (ACT_NONE, 0.0)

    def run():
        out = torch.empty(out_shape, device=cuda)
        call("eadgan_conv_" + dirn, C.byref(d), C.byref(t4(ad)), ptr(wd), ptr(bd), act, slope, C.byref(t4(out)),
             C.byref(t4(mkd)) if mask else None, ACT_LRELU if mask else ACT_NONE, 0.2, stream())
        return out

    def reference(dtype):
        z = ref(ad.to(dtype), wd.to(dtype), bd.to(dtype))
        if mask:
            z = TF.leaky_relu(z, 0.1) * torch.where(mkd > 0, 1.0, 0.2).to(dtype)
        return z

    out = run()
    _check(dirn, out, reference(torch.float32), reference(torch.float64))
    assert torch.equal(out, run()), "split-K result differs between two runs"


@pytest.mark.gpu
@pytest.mark.parametrize("shape", _shapes("wgrad"), ids=_ids)
def test_simt_wgrad_split(cuda, sms, shape):
    """eadgan_conv_wgrad with the pixel reduction split over CTAs and summed by wgrad_sum_kernel in a fixed order"""
    import eadgan_b200.functional as Fn
    from eadgan_b200._lib import t4
    _on_branch("wgrad", shape, sms)
    n, c, h, k, r, stride, pad = shape
    d, p = _desc(("wgrad",) + shape)
    g = _gen(25)
    x, dy = torch.randn(n, c, h, h, generator=g).to(cuda), torch.randn(n, k, p, p, generator=g).to(cuda)

    def run():
        dw = torch.empty(k, c, r, r, device=cuda)
        Fn.conv_wgrad(d, t4(x), t4(dy), dw)
        return dw

    dw = run()
    ref = lambda dtype: torch.nn.grad.conv2d_weight(x.to(dtype), (k, c, r, r), dy.to(dtype), stride, pad)  # noqa: E731
    _check("dw", dw, ref(torch.float32), ref(torch.float64))
    assert torch.equal(dw, run()), "split wgrad differs between two runs"


# ---- softmax, upsample, channel_sum ------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", _shapes("softmax"), ids=_ids)
def test_softmax_lanes_loop(cuda, sms, shape):
    import eadgan_b200.functional as Fn
    _on_branch("softmax", shape, sms)
    g = _gen(26)
    x, go = (torch.randn(shape, generator=g) * 3).to(cuda), torch.randn(shape, generator=g).to(cuda)

    def run(fn, dtype):
        xs = x.to(dtype).requires_grad_()
        y = fn(xs)
        return y, torch.autograd.grad(y, xs, go.to(dtype))[0]

    ours, r32, r64 = run(Fn.softmax, torch.float32), run(lambda t: torch.softmax(t, 1), torch.float32), \
        run(lambda t: torch.softmax(t, 1), torch.float64)
    _check("y", ours[0], r32[0], r64[0])
    _check("dx", ours[1], r32[1], r64[1])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", _shapes("upsample"), ids=_ids)
def test_upsample_odd_map(cuda, sms, shape):
    import eadgan_b200.functional as Fn
    _on_branch("upsample", shape, sms)
    g = _gen(27)
    x = torch.randn(shape, generator=g).to(cuda).requires_grad_()
    go = torch.randn(shape[0], shape[1], 2 * shape[2], 2 * shape[3], generator=g).to(cuda)
    y = Fn.upsample2x(x)
    assert torch.equal(y, TF.interpolate(x, scale_factor=2))
    dx = torch.autograd.grad(y, x, go)[0]
    ref = lambda t: TF.avg_pool2d(t, 2) * 4  # noqa: E731   (the adjoint of the nearest 2x upsample)
    _check("dx", dx, ref(go), ref(go.double()))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", _shapes("channel_sum"), ids=_ids)
def test_channel_sum_ragged(cuda, sms, shape):
    import eadgan_b200.functional as Fn
    _on_branch("channel_sum", shape, sms)
    t = torch.randn(shape, generator=_gen(28)).to(cuda)
    _check("sum", Fn.channel_sum(t), t.sum((0, 2, 3)), t.double().sum((0, 2, 3)))
