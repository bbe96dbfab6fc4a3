"""-m gpu: the tcgen05/TMEM/TMA kernels (bf16 operands, fp32 accumulate) against torch fp32 on
bf16-ROUNDED inputs, so the only differences are accumulation order (and bf16 rounding of the
output when it is stored as bf16).  Tolerance: north_star's bf16 bound is 2e-2; these kernels
are held to 2e-3 (fp32 out) / 1e-2 (bf16 out)."""
import pytest
import torch
import torch.nn.functional as TF

from conftest import rel_err

pytestmark = pytest.mark.gpu


def _bf(x):
    return x.bfloat16().float()


@pytest.mark.parametrize("mnk", [(128, 128, 64), (256, 256, 512), (300, 128, 256), (1024, 512, 4096), (77, 64, 128),
                                 (128, 32, 64)])
def test_gemm(cuda, mnk):
    from eadgan_b200 import tc
    m, n, k = mnk
    torch.manual_seed(0)
    a = torch.randn(m, k, device=cuda).bfloat16()
    b = torch.randn(n, k, device=cuda).bfloat16()
    ref = a.float() @ b.float().t()
    out = tc.gemm(a, b)
    assert rel_err(out, ref) <= 1e-4


# (n, c_big, h_big, k_small)
GEOS = [(4, 128, 32, 256), (4, 256, 16, 512), (16, 512, 8, 1024), (3, 128, 32, 256), (8, 32, 32, 64),
        (5, 64, 8, 64), (2, 128, 64, 128), (8, 32, 64, 32), (6, 32, 32, 32), (3, 64, 16, 96)]

# ---- epilogue variants, on two ragged geometries (128 channels: the channel-major dgrad applies; 64 channels: it does
# not).  Forward epilogue activations, and the fused activation backward of an input gradient (mask = the producer's
# saved output) with or without the per-channel sums of the final value (stats_mode 2, include/eadgan.h).
EPI_GEOS = [(3, 128, 32, 256), (5, 64, 8, 64)]
MASKS = ("relu", "lrelu", "tanh", "sigmoid")
MASK_SLOPE = 0.2


def _act_id(name):
    from eadgan_b200 import _lib
    return {"none": _lib.ACT_NONE, "relu": _lib.ACT_RELU, "lrelu": _lib.ACT_LRELU, "tanh": _lib.ACT_TANH,
            "sigmoid": _lib.ACT_SIGMOID}[name]


def _act_ref(v, name, slope):
    if name == "relu":
        return torch.relu(v)
    if name == "lrelu":
        return TF.leaky_relu(v, slope)
    if name == "tanh":
        return torch.tanh(v)
    if name == "sigmoid":
        return torch.sigmoid(v)
    return v


def _saved_output(name, shape, dev):
    """a bf16 post-activation tensor as a producer of activation ``name`` saves it (exact zeros included for ReLU)"""
    return _bf(_act_ref(torch.randn(shape, device=dev), name, MASK_SLOPE))


def _act_grad_ref(y, name):
    """the activation derivative through its saved output y (fp64)"""
    y = y.double()
    if name == "relu":
        return (y > 0).double()
    if name == "lrelu":
        return torch.where(y > 0, 1.0, MASK_SLOPE).double()
    if name == "tanh":
        return 1 - y * y
    return y * (1 - y)


def _check_sums(sums, ref):
    """per-channel sums against fp64, relative to the largest per-channel sum of |value|"""
    want = ref.double().sum((0, 2, 3))
    assert float((sums - want).abs().max() / ref.double().abs().sum((0, 2, 3)).max()) <= 2e-3


def _mask_cases(geos, extra=((None, ""),)):
    return [pytest.param(g, m, s, e, id=f"mask_{m}-stats{s}{tag}-g{j}")
            for j, g in enumerate(geos) for m in MASKS for s in (0, 2) for e, tag in extra]


@pytest.mark.parametrize("geo,act,mask", [pytest.param(g, "lrelu", None, id=f"geo{i}") for i, g in enumerate(GEOS)] +
                         [pytest.param(g, a, None, id=f"act_{a}-g{j}") for j, g in enumerate(EPI_GEOS)
                          for a in ("relu", "tanh", "sigmoid")] +
                         [pytest.param(g, "none", (m, s), id=f"mask_{m}-stats{s}-g{j}") for j, g in enumerate(EPI_GEOS)
                          for m in MASKS for s in (0, 2)])
def test_fprop(cuda, geo, act, mask):
    """Conv2d(c,k,4,2,1) forward + bias + activation, padded NHWC bf16 in and out; and the same kernel as a
    ConvTranspose input gradient with the producer's activation backward fused (mask) and the per-channel sums."""
    from eadgan_b200 import tc
    n, c, h, k = geo
    torch.manual_seed(1)
    x = _bf(torch.randn(n, c, h, h, device=cuda))
    w = _bf(torch.randn(k, c, 4, 4, device=cuda) * 0.05)
    b = torch.randn(k, device=cuda)
    xp = tc.to_padded(x)
    assert torch.equal(tc.from_padded(xp), x)
    wpk = tc.pack_w(w, None, "fprop")
    if mask is not None:
        mname, stats_mode = mask
        y = _saved_output(mname, (n, k, h // 2, h // 2), cuda)
        ref = TF.conv2d(x.double(), w.double(), None, stride=2, padding=1) * _act_grad_ref(y, mname)
        sums = torch.zeros(k, device=cuda, dtype=torch.float64) if stats_mode else None
        out = tc.fprop(xp, wpk, None, k, mask=tc.to_padded(y), mask_mode=_act_id(mname), slope=MASK_SLOPE, stats=sums,
                       stats_mode=2)
        assert rel_err(tc.from_padded(out), ref) <= 1e-2
        if stats_mode:
            _check_sums(sums, ref)
        return
    slope = 0.1 if act == "lrelu" else 0.0
    ref = _act_ref(TF.conv2d(x, w, b, stride=2, padding=1), act, slope)
    out32 = tc.fprop(xp, wpk, b, k, _act_id(act), slope, out_f32_nchw=True)
    assert rel_err(out32, ref) <= 2e-3
    outp = tc.fprop(xp, wpk, b, k, _act_id(act), slope)
    assert rel_err(tc.from_padded(outp), ref) <= 1e-2
    # halo must still be zero
    assert float(outp[:, 0].abs().max()) == 0 and float(outp[:, :, 0].abs().max()) == 0
    assert float(outp[:, -1].abs().max()) == 0 and float(outp[:, :, -1].abs().max()) == 0


@pytest.mark.parametrize("geo,act", [pytest.param(g, "none", id=f"geo{i}") for i, g in enumerate(GEOS)] +
                         [pytest.param(g, a, id=f"act_{a}-g{j}") for j, g in enumerate(EPI_GEOS)
                          for a in ("relu", "tanh", "sigmoid")])
def test_dgrad(cuda, geo, act):
    """ConvTranspose2d(k,c,4,2,1) forward (= conv dgrad) + bias [+ activation], with fused BN statistics of the
    pre-activation value."""
    from eadgan_b200 import tc
    n, c, h, k = geo
    if k % 64 and k != 32:
        pytest.skip("tc dgrad needs k = 32 or k % 64 == 0")
    torch.manual_seed(2)
    y = _bf(torch.randn(n, k, h // 2, h // 2, device=cuda))
    w = _bf(torch.randn(k, c, 4, 4, device=cuda) * 0.05)
    b = torch.randn(c, device=cuda)
    pre = TF.conv_transpose2d(y, w, b, stride=2, padding=1)
    ref = _act_ref(pre, act, 0.0)
    yp = tc.to_padded(y)
    wpk = tc.pack_w(w, None, "dgrad")
    stats = torch.zeros(2 * c, device=cuda, dtype=torch.float64)
    out32 = tc.dgrad(yp, wpk, b, c, _act_id(act), out_f32_nchw=True, stats=stats)
    assert rel_err(out32, ref) <= 2e-3
    assert rel_err(stats[:c], pre.double().sum((0, 2, 3))) <= 2e-3
    assert rel_err(stats[c:], (pre.double() ** 2).sum((0, 2, 3))) <= 2e-3
    outp = tc.dgrad(yp, wpk, b, c, _act_id(act))
    assert rel_err(tc.from_padded(outp), ref) <= 1e-2


@pytest.mark.parametrize("geo,mask,stats_mode,dgradt",
                         [pytest.param(g, "lrelu", 0, None, id=f"geo{i}") for i, g in enumerate(GEOS)] +
                         _mask_cases(EPI_GEOS[:1], ((0, "-pixel_major"), (2, "-channel_major"))) +
                         _mask_cases(EPI_GEOS[1:], ((0, "-pixel_major"),)))
def test_dgrad_mask(cuda, monkeypatch, geo, mask, stats_mode, dgradt):
    """conv backward-data with the activation backward of the producer layer fused (mask), optionally with the
    per-channel sums of the result (the producer's bias gradient), on the pixel-major and channel-major kernels."""
    from eadgan_b200 import tc
    n, c, h, k = geo
    if k % 64 and k != 32:
        pytest.skip("tc dgrad needs k = 32 or k % 64 == 0")
    if dgradt is not None:
        monkeypatch.setenv("EADGAN_TC_DGRADT", str(dgradt))
    torch.manual_seed(3)
    dy = _bf(torch.randn(n, k, h // 2, h // 2, device=cuda))
    w = _bf(torch.randn(k, c, 4, 4, device=cuda) * 0.05)
    if dgradt is None:
        act_out = _bf(torch.randn(n, c, h, h, device=cuda))  # saved post-activation tensor of the producer
        ref = TF.conv_transpose2d(dy, w, None, stride=2, padding=1) * torch.where(act_out > 0, 1.0, 0.1)
        slope = 0.1
    else:
        act_out = _saved_output(mask, (n, c, h, h), cuda)
        ref = TF.conv_transpose2d(dy.double(), w.double(), None, stride=2, padding=1) * _act_grad_ref(act_out, mask)
        slope = MASK_SLOPE
    sums = torch.zeros(c, device=cuda, dtype=torch.float64) if stats_mode else None
    outp = tc.dgrad(tc.to_padded(dy), tc.pack_w(w, None, "dgrad"), None, c, mask=tc.to_padded(act_out),
                    mask_mode=_act_id(mask), slope=slope, stats=sums, stats_mode=2)
    assert rel_err(tc.from_padded(outp), ref) <= 1e-2
    if stats_mode:
        _check_sums(sums, ref)


@pytest.mark.parametrize("geo", GEOS)
def test_wgrad(cuda, geo):
    from eadgan_b200 import tc
    n, c, h, k = geo
    torch.manual_seed(4)
    x = _bf(torch.randn(n, c, h, h, device=cuda))
    dy = _bf(torch.randn(n, k, h // 2, h // 2, device=cuda))
    w = torch.zeros(k, c, 4, 4, device=cuda, requires_grad=True)
    ref = torch.autograd.grad(TF.conv2d(x, w, None, stride=2, padding=1), w, dy)[0]
    out = tc.wgrad(tc.to_padded(x), tc.to_padded(dy))
    assert rel_err(out, ref) <= 2e-3


def test_sigma_scaled_pack(cuda):
    from eadgan_b200 import tc
    torch.manual_seed(5)
    w = torch.randn(128, 64, 4, 4, device=cuda)
    sigma = torch.tensor([2.5], device=cuda)
    x = _bf(torch.randn(2, 64, 8, 8, device=cuda))
    ref = TF.conv2d(x, _bf(w / 2.5), None, stride=2, padding=1)
    out = tc.fprop(tc.to_padded(x), tc.pack_w(w, sigma, "fprop"), None, 128, out_f32_nchw=True)
    assert rel_err(out, ref) <= 2e-3


def test_channel_padded_image_layers(cuda):
    """3-channel image layers run with the big map zero-padded to 32 channels (c_real = 3)."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_TANH
    torch.manual_seed(6)
    n = 5
    # Conv2d(3,128,4,2,1) forward / wgrad / input-gradient
    x = _bf(torch.randn(n, 3, 64, 64, device=cuda))
    w = _bf(torch.randn(128, 3, 4, 4, device=cuda) * 0.1)
    b = torch.randn(128, device=cuda)
    xp = tc.to_padded(x, 32)
    ref = TF.conv2d(x, w, b, stride=2, padding=1)
    out = tc.fprop(xp, tc.pack_w(w, None, "fprop", 32), b, 128, out_f32_nchw=True)
    assert rel_err(out, ref) <= 2e-3
    dy = _bf(torch.randn(n, 128, 32, 32, device=cuda))
    wz = torch.zeros_like(w).requires_grad_()
    xr = x.clone().requires_grad_()
    gw = torch.autograd.grad(TF.conv2d(x, wz, None, stride=2, padding=1), wz, dy)[0]
    gx = torch.autograd.grad(TF.conv2d(xr, w, None, stride=2, padding=1), xr, dy)[0]
    dyp = tc.to_padded(dy)
    assert rel_err(tc.wgrad(xp, dyp, c_real=3), gw) <= 2e-3
    dx = tc.dgrad(dyp, tc.pack_w(w, None, "dgrad", 32), None, 32, out_f32_nchw=True, c_real=3)
    assert dx.shape == (n, 3, 64, 64) and rel_err(dx, gx) <= 2e-3
    # ConvTranspose2d(128,3,4,2,1) + bias + tanh forward
    bt = torch.randn(3, device=cuda)
    reft = torch.tanh(TF.conv_transpose2d(dy, w, bt, stride=2, padding=1))
    outt = tc.dgrad(dyp, tc.pack_w(w, None, "dgrad", 32), bt, 32, ACT_TANH, out_f32_nchw=True, c_real=3)
    assert rel_err(outt, reft) <= 2e-3


@pytest.mark.parametrize("n,mask,stats_mode", [pytest.param(n, "lrelu", 0, id=str(n)) for n in (8, 130, 200)] +
                         [pytest.param(130, m, s, id=f"130-mask_{m}-stats{s}") for m in MASKS for s in (0, 2)])
def test_dense_layers(cuda, n, mask, stats_mode):
    """ConvTranspose2d(218,1024,4,1,0) on 1x1 and Conv2d(1024,19,4,1,0) on 4x4 as batch GEMMs; the head's input
    gradient with the producer's activation backward fused, optionally with the per-channel sums of the result."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_LRELU
    torch.manual_seed(7)
    C = 1024
    # --- ConvT: z[n,218] -> [n,1024,4,4]
    z = _bf(torch.randn(n, 218, device=cuda))
    w = _bf(torch.randn(218, C, 4, 4, device=cuda) * 0.05)
    b = torch.randn(C, device=cuda)
    ref = TF.conv_transpose2d(z.view(n, 218, 1, 1), w, b, stride=1, padding=0)
    a = tc.pad_rows(z, 256)
    out = tc.dense_scatter(a, tc.dense_pack(w, 256, False), b, C)
    assert rel_err(tc.from_padded(out), ref) <= 1e-2
    assert float(out[:, 0].abs().max()) == 0 and float(out[:, :, 5].abs().max()) == 0
    g = _bf(torch.randn(n, C, 4, 4, device=cuda))
    wz = torch.zeros_like(w).requires_grad_()
    gw = torch.autograd.grad(TF.conv_transpose2d(z.view(n, 218, 1, 1), wz, None), wz, g)[0]
    assert rel_err(tc.dense_wgrad(a, tc.to_padded(g), 218), gw) <= 2e-3
    # --- head: y[n,1024,4,4] -> [n,19]
    y = _bf(torch.randn(n, C, 4, 4, device=cuda))
    wh = _bf(torch.randn(19, C, 4, 4, device=cuda) * 0.02)
    bh = torch.randn(19, device=cuda)
    yp = tc.to_padded(y)
    refh = TF.conv2d(y, wh, bh).view(n, 19)
    outh = tc.dense_gather(yp, tc.dense_pack(wh, 32, True), bh, 19)
    assert rel_err(outh, refh) <= 2e-3
    gh = _bf(torch.randn(n, 19, device=cuda))
    whz = torch.zeros_like(wh).requires_grad_()
    yr = y.clone().requires_grad_()
    gwh = torch.autograd.grad(TF.conv2d(y, whz, None).view(n, 19), whz, gh)[0]
    gy = torch.autograd.grad(TF.conv2d(yr, wh, None).view(n, 19), yr, gh)[0]
    ah = tc.pad_rows(gh, 64)
    assert rel_err(tc.dense_wgrad(ah, yp, 19), gwh) <= 2e-3
    if stats_mode == 0 and mask == "lrelu":
        dxp = tc.dense_scatter(ah, tc.dense_pack(wh, 64, False), None, C, mask=yp, mask_act=ACT_LRELU, slope=0.1)
        assert rel_err(tc.from_padded(dxp), gy * torch.where(y > 0, 1.0, 0.1)) <= 1e-2
    if n == 130 and mask is not None:
        # the masked input gradient against fp64 on the same bf16 operands
        ym = _saved_output(mask, (n, C, 4, 4), cuda)
        gyd = TF.conv_transpose2d(gh.double().view(n, 19, 1, 1), wh.double())
        ref = gyd * _act_grad_ref(ym, mask)
        sums = torch.zeros(C, device=cuda, dtype=torch.float64) if stats_mode else None
        dxp = tc.dense_scatter(ah, tc.dense_pack(wh, 64, False), None, C, mask=tc.to_padded(ym), mask_act=_act_id(mask),
                               slope=MASK_SLOPE, chan_sums=sums)
        assert rel_err(tc.from_padded(dxp), ref) <= 1e-2
        if stats_mode:
            _check_sums(sums, ref)


# ---- cta_group::2 (CTA pairs): forced on through EADGAN_TC_CG so that small, ragged cases exercise the pair protocol
# (odd numbers of M tiles -> the peer CTA of the last pair runs an all-out-of-range tile; one tile per pair; several)
@pytest.fixture
def pairs(monkeypatch):
    monkeypatch.setenv("EADGAN_TC_CG", "2")


PAIR_GEOS = [(4, 128, 32, 256), (3, 128, 32, 256), (9, 256, 16, 512), (16, 512, 8, 1024), (40, 256, 16, 256)]


@pytest.mark.parametrize("mnk", [(256, 256, 64), (384, 256, 512), (300, 128, 256), (8192, 512, 1024), (77, 256, 128)])
def test_gemm_cta_pairs(cuda, pairs, mnk):
    from eadgan_b200 import tc
    m, n, k = mnk
    torch.manual_seed(0)
    a = torch.randn(m, k, device=cuda).bfloat16()
    b = torch.randn(n, k, device=cuda).bfloat16()
    assert rel_err(tc.gemm(a, b), a.float() @ b.float().t()) <= 1e-4


@pytest.mark.parametrize("geo", PAIR_GEOS)
def test_conv_cta_pairs(cuda, pairs, geo):
    """fprop / dgrad (+ BatchNorm statistics, + fused mask) / wgrad through the cta_group::2 kernels."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_LRELU
    n, c, h, k = geo
    torch.manual_seed(8)
    x = _bf(torch.randn(n, c, h, h, device=cuda))
    w = _bf(torch.randn(k, c, 4, 4, device=cuda) * 0.05)
    bk, bc = torch.randn(k, device=cuda), torch.randn(c, device=cuda)
    ref = TF.leaky_relu(TF.conv2d(x, w, bk, stride=2, padding=1), 0.1)
    xp = tc.to_padded(x)
    out = tc.fprop(xp, tc.pack_w(w, None, "fprop"), bk, k, ACT_LRELU, 0.1, out_f32_nchw=True)
    assert rel_err(out, ref) <= 2e-3
    y = _bf(torch.randn(n, k, h // 2, h // 2, device=cuda))
    yp = tc.to_padded(y)
    reft = TF.conv_transpose2d(y, w, bc, stride=2, padding=1)
    stats = torch.zeros(2 * c, device=cuda, dtype=torch.float64)
    outt = tc.dgrad(yp, tc.pack_w(w, None, "dgrad"), bc, c, out_f32_nchw=True, stats=stats)
    assert rel_err(outt, reft) <= 2e-3
    assert rel_err(stats[:c], reft.double().sum((0, 2, 3))) <= 2e-3
    assert rel_err(stats[c:], (reft.double() ** 2).sum((0, 2, 3))) <= 2e-3
    refm = TF.conv_transpose2d(y, w, None, stride=2, padding=1) * torch.where(x > 0, 1.0, 0.1)
    outm = tc.dgrad(yp, tc.pack_w(w, None, "dgrad"), None, c, mask=xp, mask_mode=ACT_LRELU, slope=0.1)
    assert rel_err(tc.from_padded(outm), refm) <= 1e-2
    wz = torch.zeros(k, c, 4, 4, device=cuda, requires_grad=True)
    gw = torch.autograd.grad(TF.conv2d(x, wz, None, stride=2, padding=1), wz, y)[0]
    assert rel_err(tc.wgrad(xp, yp), gw) <= 2e-3


@pytest.mark.parametrize("geo", [(4, 128, 32, 256), (3, 128, 32, 256), (5, 128, 8, 64), (2, 128, 64, 128), (70, 128, 4, 192)])
def test_transposed_dgrad(cuda, monkeypatch, geo):
    """tc_dgradT_kernel (128 output channels as the MMA's M dimension), forced on for small / ragged cases: odd numbers
    of pixel tiles, several images per tile (4x4 small maps), plain / bias + BatchNorm statistics / fused mask + sums."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_LRELU
    monkeypatch.setenv("EADGAN_TC_DGRADT", "2")
    n, c, h, k = geo
    torch.manual_seed(9)
    y = _bf(torch.randn(n, k, h // 2, h // 2, device=cuda))
    w = _bf(torch.randn(k, c, 4, 4, device=cuda) * 0.05)
    b = torch.randn(c, device=cuda)
    yp, wpk = tc.to_padded(y), tc.pack_w(w, None, "dgrad")
    ref = TF.conv_transpose2d(y, w, b, stride=2, padding=1)
    stats = torch.zeros(2 * c, device=cuda, dtype=torch.float64)
    out = tc.dgrad(yp, wpk, b, c, stats=stats)
    assert rel_err(tc.from_padded(out), ref) <= 1e-2
    assert float(out[:, 0].abs().max()) == 0 and float(out[:, :, -1].abs().max()) == 0
    assert rel_err(stats[:c], ref.double().sum((0, 2, 3))) <= 2e-3
    assert rel_err(stats[c:], (ref.double() ** 2).sum((0, 2, 3))) <= 2e-3
    monkeypatch.setenv("EADGAN_TC_DGRADT", "0")
    old = tc.dgrad(yp, wpk, b, c)
    assert rel_err(tc.from_padded(out), tc.from_padded(old)) <= 8e-3      # both round the same fp32 values to bf16
    monkeypatch.setenv("EADGAN_TC_DGRADT", "2")
    act_out = _bf(torch.randn(n, c, h, h, device=cuda))
    sigma = torch.tensor([1.25], device=cuda)
    refm = TF.conv_transpose2d(y, w, None, stride=2, padding=1) / 1.25 * torch.where(act_out > 0, 1.0, 0.1)
    sums = torch.zeros(c, device=cuda, dtype=torch.float64)
    outm = tc.dgrad(yp, wpk, None, c, mask=tc.to_padded(act_out), mask_mode=ACT_LRELU, slope=0.1, stats=sums, stats_mode=2,
                    sigma=sigma)
    assert rel_err(tc.from_padded(outm), refm) <= 1e-2
    assert float((sums - refm.double().sum((0, 2, 3))).abs().max() / refm.double().abs().sum((0, 2, 3)).max()) <= 2e-3


@pytest.mark.parametrize("n", [5, 37])
def test_channel_major_thin_fprop(cuda, monkeypatch, n):
    """Conv2d(3,128,4,2,1) forward through the channel-major kernel (forced on for a ragged batch): bias + LeakyReLU +
    1/sigma, and the masked variant with per-channel sums, against torch."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_LRELU
    monkeypatch.setenv("EADGAN_TC_DGRADT", "2")
    torch.manual_seed(10)
    img = _bf(torch.rand(n, 3, 64, 64, device=cuda) * 2 - 1)
    w = torch.randn(128, 3, 4, 4, device=cuda) * 0.1
    b = torch.randn(128, device=cuda)
    sigma = torch.tensor([1.6], device=cuda)
    r = tc.thin_expand(img)
    ref = TF.leaky_relu(TF.conv2d(img, _bf(w), None, stride=2, padding=1) / 1.6 + b[None, :, None, None], 0.1)
    out = tc.thin_fprop(r, tc.thin_pack_w(w, "fprop"), b, 3, 128, ACT_LRELU, 0.1, sigma=sigma)
    assert rel_err(tc.from_padded(out), ref) <= 1e-2
    assert float(out[:, 0].abs().max()) == 0 and float(out[:, :, -1].abs().max()) == 0
    monkeypatch.setenv("EADGAN_TC_DGRADT", "0")
    old = tc.thin_fprop(r, tc.thin_pack_w(w, "fprop"), b, 3, 128, ACT_LRELU, 0.1, sigma=sigma)
    assert rel_err(tc.from_padded(out), tc.from_padded(old)) <= 8e-3
    monkeypatch.setenv("EADGAN_TC_DGRADT", "2")
    act_out = _bf(torch.randn(n, 128, 32, 32, device=cuda))
    refm = TF.conv2d(img, _bf(w), None, stride=2, padding=1) * torch.where(act_out > 0, 1.0, 0.1)
    sums = torch.zeros(128, device=cuda, dtype=torch.float64)
    outm = tc.thin_fprop(r, tc.thin_pack_w(w, "fprop"), None, 3, 128, mask=tc.to_padded(act_out), mask_mode=ACT_LRELU,
                         slope=0.1, stats=sums, stats_mode=2)
    assert rel_err(tc.from_padded(outm), refm) <= 1e-2
    assert float((sums - refm.double().sum((0, 2, 3))).abs().max() / refm.double().abs().sum((0, 2, 3)).max()) <= 2e-3


def test_pack_cache_goes_stale_per_parameter(cuda):
    """The bf16 operand packs are cached per parameter.  Our fused Adam updates weights through raw pointers, so it
    leaves a serial on exactly the parameters it stepped: their packs are rebuilt, everybody else's stay cached
    (phase G's optimiser step does not make D re-pack).  tc.prefetch_packs rebuilds the layouts used so far."""
    from eadgan_b200 import tc
    from eadgan_b200.optim import Adam
    torch.manual_seed(0)
    w1 = torch.nn.Parameter(torch.randn(64, 32, 4, 4, device=cuda))
    w2 = torch.nn.Parameter(torch.randn(64, 32, 4, 4, device=cuda))
    a1, b1 = tc.pack_w_cached(w1, "fprop", 32), tc.pack_w_cached(w2, "fprop", 32)
    b1d = tc.pack_w_cached(w2, "dgrad", 32)
    assert tc.pack_w_cached(w2, "fprop", 32) is b1
    opt = Adam([w2], lr=0.1)
    w2.grad = torch.ones_like(w2)
    opt.step()
    assert tc.pack_w_cached(w1, "fprop", 32) is a1              # not stepped: still cached
    tc.prefetch_packs(w2)                                       # rebuilds both layouts w2 was consumed in
    b2, b2d = tc.pack_w_cached(w2, "fprop", 32), tc.pack_w_cached(w2, "dgrad", 32)
    assert b2 is not b1 and b2d is not b1d
    assert torch.equal(b2, tc.pack_w(w2.detach(), None, "fprop", 32))
    assert torch.equal(b2d, tc.pack_w(w2.detach(), None, "dgrad", 32))
    assert not torch.equal(b2, b1)
    tc.invalidate_caches()
    assert tc.pack_w_cached(w1, "fprop", 32) is not a1          # wholesale invalidation still works
