"""-m gpu: the "thin" image-layer kernels (big map = a 1..4-channel image: D's first Conv2d(3,128), G's last
ConvTranspose2d(128,3), the dSprites Conv2d(1|3,32) / ConvTranspose2d(64,1|3)) against torch fp32 on bf16-ROUNDED
operands: row-expanded image buffer, thin fprop (one 64-wide k block), thin wgrad, and the GEMM + col2im
ConvTranspose forward.  Same tolerances as tests/test_tc_gpu.py."""
import pytest
import torch
import torch.nn.functional as TF

from conftest import rel_err

pytestmark = pytest.mark.gpu


def _bf(x):
    return x.bfloat16().float()


# (n, c_img, h_img, k_small)
GEOS = [(4, 3, 64, 128), (3, 1, 64, 64), (5, 3, 64, 32), (2, 3, 32, 128), (130, 3, 64, 128), (2, 4, 16, 64)]


@pytest.mark.parametrize("geo", [(4, 3, 64), (3, 1, 32), (2, 4, 16)])
def test_expand_layout(cuda, geo):
    from eadgan_b200 import tc
    n, c, h = geo
    torch.manual_seed(0)
    x = _bf(torch.randn(n, c, h, h, device=cuda))
    r = tc.thin_expand(x).float()                    # [n, h/2, h+2, ky, c4]
    xp = TF.pad(x, (1, 1, 1, 1))                      # [n, c, h+2, h+2]
    for ky in range(4):
        want = xp[:, :, ky:ky + h:2, :].permute(0, 2, 3, 1)   # rows 2*oy + ky -> [n, h/2, h+2, c]
        assert torch.equal(r[:, :, :, ky, :c], want), ky
        assert float(r[:, :, :, ky, c:].abs().max()) == 0 if c < 4 else True
    # fused activation backward: g * tanh'(y)
    y = torch.tanh(torch.randn_like(x))
    from eadgan_b200._lib import ACT_TANH
    r2 = tc.thin_expand(x, mask_y=y, act=ACT_TANH).float()
    want = _bf(x * (1 - y * y))
    assert torch.equal(r2[:, :, 1:-1, 1, :c], want[:, :, 0::2, :].permute(0, 2, 3, 1))


@pytest.mark.parametrize("geo,mask", [pytest.param(g, None, id=f"geo{i}") for i, g in enumerate(GEOS)] +
                         [pytest.param(g, (m, s, dt), id=f"mask_{m}-stats{s}-dgradt{dt}-g{j}")
                          for j, g in enumerate([(4, 3, 64, 128), (3, 1, 64, 32)]) for m in ("relu", "lrelu", "tanh", "sigmoid")
                          for s in (0, 2) for dt in ((0, 2) if g[3] == 128 else (0,))])
def test_thin_fprop(cuda, monkeypatch, geo, mask):
    """Conv2d(c<=4, k, 4, 2, 1) forward + bias + LeakyReLU (+ 1/sigma), padded NHWC bf16 out; and the same kernel as the
    input gradient of a ConvTranspose onto the image, with the producer's activation backward fused (mask) and the
    per-channel sums of the result, on the pixel-major and (128 channels) channel-major kernels."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_LRELU
    n, c, h, k = geo
    torch.manual_seed(1)
    x = _bf(torch.randn(n, c, h, h, device=cuda))
    w = _bf(torch.randn(k, c, 4, 4, device=cuda) * 0.1)
    b = torch.randn(k, device=cuda)
    sigma = torch.tensor([1.7], device=cuda)
    if mask is not None:
        from test_tc_gpu import MASK_SLOPE, _act_grad_ref, _act_id, _check_sums, _saved_output
        mname, stats_mode, dgradt = mask
        monkeypatch.setenv("EADGAN_TC_DGRADT", str(dgradt))
        y = _saved_output(mname, (n, k, h // 2, h // 2), cuda)
        ref = TF.conv2d(x.double(), w.double(), None, stride=2, padding=1) / 1.7 * _act_grad_ref(y, mname)
        sums = torch.zeros(k, device=cuda, dtype=torch.float64) if stats_mode else None
        out = tc.thin_fprop(tc.thin_expand(x), tc.thin_pack_w(w, "fprop"), None, c, k, mask=tc.to_padded(y),
                            mask_mode=_act_id(mname), slope=MASK_SLOPE, stats=sums, stats_mode=2, sigma=sigma)
        assert rel_err(tc.from_padded(out), ref) <= 1e-2
        if stats_mode:
            _check_sums(sums, ref)
        return
    ref = TF.leaky_relu(TF.conv2d(x, w / 1.7, b, stride=2, padding=1), 0.1)
    outp = tc.thin_fprop(tc.thin_expand(x), tc.thin_pack_w(w, "fprop"), b, c, k, ACT_LRELU, 0.1, sigma=sigma)
    assert rel_err(tc.from_padded(outp), ref) <= 1e-2
    assert float(outp[:, 0].abs().max()) == 0 and float(outp[:, :, -1].abs().max()) == 0


@pytest.mark.parametrize("geo", GEOS)
def test_thin_wgrad(cuda, geo):
    from eadgan_b200 import tc
    n, c, h, k = geo
    torch.manual_seed(2)
    x = _bf(torch.randn(n, c, h, h, device=cuda))
    dy = _bf(torch.randn(n, k, h // 2, h // 2, device=cuda))
    w = torch.zeros(k, c, 4, 4, device=cuda, requires_grad=True)
    TF.conv2d(x, w, None, stride=2, padding=1).backward(dy)
    dw = tc.thin_wgrad(tc.thin_expand(x), tc.to_padded(dy), c)
    assert dw.shape == w.grad.shape
    assert rel_err(dw, w.grad) <= 2e-3
    dw2 = tc.thin_wgrad(tc.thin_expand(x), tc.to_padded(dy), c)
    assert torch.equal(dw, dw2)          # split partials are summed in a fixed order


@pytest.mark.parametrize("geo", [g for g in GEOS if g[2] == 64 and g[1] <= 3])
@pytest.mark.parametrize("act", ["none", "tanh"])
def test_thin_dgrad(cuda, geo, act):
    """ConvTranspose2d(k, c<=3, 4, 2, 1) forward (= Conv2d input gradient): GEMM over input pixels + col2im epilogue."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_NONE, ACT_TANH
    n, c, h, k = geo
    torch.manual_seed(3)
    y = _bf(torch.randn(n, k, h // 2, h // 2, device=cuda))
    w = _bf(torch.randn(k, c, 4, 4, device=cuda) * 0.1)          # ConvTranspose layout [Cin = k, Cout = c, 4, 4]
    b = torch.randn(c, device=cuda) if act == "tanh" else None
    sigma = torch.tensor([0.8], device=cuda)
    ref = TF.conv_transpose2d(y, w / 0.8, b, stride=2, padding=1)
    if act == "tanh":
        ref = torch.tanh(ref)
    out = tc.thin_dgrad(tc.to_padded(y), tc.thin_pack_w(w, "dgrad"), b, c, ACT_TANH if act == "tanh" else ACT_NONE,
                        sigma=sigma)
    assert out.shape == ref.shape
    assert rel_err(out, ref) <= 2e-3
