"""-m gpu: parity IN THE BENCHMARKED REGIME (VERDICT r01 "what's weak" 1).

bench.py runs the CelebA step at 1024 images per GPU.  There every persistent tcgen05 kernel runs 4..28 tiles
per CTA: the TMEM accumulator double buffer flips phase (it >= 2), the shared-memory ring wraps across tiles, the
BatchNorm statistics fold across tiles of one channel block, and the wave-aware split of the weight-gradient
reduction picks its large-batch plan.  None of that is reached by the n <= 16 cases of tests/test_tc_gpu.py, so
every big-layer kernel, the thin image-layer kernels and the dense 1x1 <-> 4x4 GEMMs are run here at n = 1024 in
exactly the variants the step uses (celebA/EAD-GAN_celebA.py:75-92,109-122), against torch fp32 on bf16-rounded
operands (bounds as in test_tc_gpu.py: 2e-3 fp32 outputs, 1e-2 bf16 outputs), followed by one full CelebA step at
B = 1024 and one colored-dSprites step at B = 512 against the oracle on the GPU."""
import pytest
import torch
import torch.nn.functional as TF

pytestmark = pytest.mark.gpu
N = 1024
# the six 134-MMAC layers of CelebA's G and D share three conv-view geometries (c_big, h_big, k_small)
BIG = [(128, 32, 256), (256, 16, 512), (512, 8, 1024)]


def _bf(x):
    return x.bfloat16().float()


def err(a, b):
    """tensor-normalised max error, evaluated on the device (the tensors here have up to 134 M elements)"""
    return float((a.float() - b.float()).abs().max() / b.float().abs().max())


def _tiles_per_cta(m_rows, n_cols, bn, mt, parities=1):
    from eadgan_b200 import _lib
    sms = _lib.lib().eadgan_sm_count()
    return (m_rows // (128 * mt)) * (n_cols // bn) * parities / sms


@pytest.mark.parametrize("geo", BIG)
def test_fprop_discriminator_forward(cuda, geo):
    """SN-Conv2d(c,k,4,2,1) + bias + LeakyReLU(0.1), 1/sigma applied in the epilogue, bf16 padded NHWC out."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_LRELU
    c, h, k = geo
    torch.manual_seed(11)
    x = _bf(torch.randn(N, c, h, h, device=cuda))
    w = torch.randn(k, c, 4, 4, device=cuda) * 0.05
    b = torch.randn(k, device=cuda)
    sigma = torch.tensor([1.7], device=cuda)
    ref = TF.leaky_relu(TF.conv2d(x, _bf(w), None, stride=2, padding=1) / 1.7 + b[None, :, None, None], 0.1)
    assert _tiles_per_cta(N * (h // 2) ** 2, k, 256, 1) >= 3
    out = tc.fprop(tc.to_padded(x), tc.pack_w(w, None, "fprop"), b, k, ACT_LRELU, 0.1, sigma=sigma)
    assert err(tc.from_padded(out), ref) <= 1e-2
    assert float(out[:, 0].abs().max()) == 0 and float(out[:, :, -1].abs().max()) == 0     # halo untouched


@pytest.mark.parametrize("geo", BIG)
def test_dgrad_generator_forward_with_bn_statistics(cuda, geo):
    """ConvTranspose2d(k,c,4,2,1) + bias with the BatchNorm sums of x and x^2 folded across the tiles of a CTA."""
    from eadgan_b200 import tc
    c, h, k = geo
    torch.manual_seed(12)
    y = _bf(torch.randn(N, k, h // 2, h // 2, device=cuda))
    w = _bf(torch.randn(k, c, 4, 4, device=cuda) * 0.05)
    b = torch.randn(c, device=cuda)
    ref = TF.conv_transpose2d(y, w, b, stride=2, padding=1)
    stats = torch.zeros(2 * c, device=cuda, dtype=torch.float64)
    out = tc.dgrad(tc.to_padded(y), tc.pack_w(w, None, "dgrad"), b, c, stats=stats)
    assert err(tc.from_padded(out), ref) <= 1e-2
    assert err(stats[:c], ref.double().sum((0, 2, 3))) <= 2e-3
    assert err(stats[c:], (ref.double() ** 2).sum((0, 2, 3))) <= 2e-3


@pytest.mark.parametrize("geo", BIG)
def test_dgrad_discriminator_backward_mask_and_bias_sums(cuda, geo):
    """conv input gradient with the LeakyReLU backward of the producer fused (mask) and the per-channel sums of the
    result (= the producer's bias gradient) accumulated by the epilogue (stats_mode 2); 1/sigma in the epilogue."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_LRELU
    c, h, k = geo
    torch.manual_seed(13)
    dy = _bf(torch.randn(N, k, h // 2, h // 2, device=cuda))
    w = torch.randn(k, c, 4, 4, device=cuda) * 0.05
    act_out = _bf(torch.randn(N, c, h, h, device=cuda))
    sigma = torch.tensor([0.8], device=cuda)
    ref = TF.conv_transpose2d(dy, _bf(w), None, stride=2, padding=1) / 0.8 * torch.where(act_out > 0, 1.0, 0.1)
    sums = torch.zeros(c, device=cuda, dtype=torch.float64)
    out = tc.dgrad(tc.to_padded(dy), tc.pack_w(w, None, "dgrad"), None, c, mask=tc.to_padded(act_out),
                   mask_mode=ACT_LRELU, slope=0.1, stats=sums, stats_mode=2, sigma=sigma)
    assert err(tc.from_padded(out), ref) <= 1e-2
    assert err(sums, ref.double().sum((0, 2, 3))) <= 2e-3 * float(ref.abs().sum((0, 2, 3)).max() / ref.sum((0, 2, 3)).abs().max())


@pytest.mark.parametrize("geo", BIG)
def test_fprop_generator_backward(cuda, geo):
    """ConvTranspose2d input gradient = strided conv of dz with the same weights (no mask: the producer has a BN)."""
    from eadgan_b200 import tc
    c, h, k = geo
    torch.manual_seed(14)
    dz = _bf(torch.randn(N, c, h, h, device=cuda))
    w = _bf(torch.randn(k, c, 4, 4, device=cuda) * 0.05)
    ref = TF.conv2d(dz, w, None, stride=2, padding=1)
    out = tc.fprop(tc.to_padded(dz), tc.pack_w(w, None, "fprop"), None, k)
    assert err(tc.from_padded(out), ref) <= 1e-2


@pytest.mark.parametrize("geo", BIG)
def test_wgrad(cuda, geo):
    """dW over 1024 x p x q pixels: split reduction + fixed-order partial sums, run twice for determinism."""
    from eadgan_b200 import tc
    c, h, k = geo
    torch.manual_seed(15)
    x = _bf(torch.randn(N, c, h, h, device=cuda))
    dy = _bf(torch.randn(N, k, h // 2, h // 2, device=cuda))
    w = torch.zeros(k, c, 4, 4, device=cuda, requires_grad=True)
    ref = torch.autograd.grad(TF.conv2d(x, w, None, stride=2, padding=1), w, dy)[0]
    xp, dyp = tc.to_padded(x), tc.to_padded(dy)
    out = tc.wgrad(xp, dyp)
    assert err(out, ref) <= 2e-3
    assert torch.equal(out, tc.wgrad(xp, dyp))


def test_thin_image_layers(cuda):
    """D's Conv2d(3,128) and G's ConvTranspose2d(128,3) at n = 1024: forward, weight gradient, input gradient."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_LRELU, ACT_TANH
    torch.manual_seed(16)
    img = _bf(torch.rand(N, 3, 64, 64, device=cuda) * 2 - 1)
    w = torch.randn(128, 3, 4, 4, device=cuda) * 0.1
    b = torch.randn(128, device=cuda)
    sigma = torch.tensor([1.3], device=cuda)
    # D layer 1 forward
    r = tc.thin_expand(img)
    ref = TF.leaky_relu(TF.conv2d(img, _bf(w), None, stride=2, padding=1) / 1.3 + b[None, :, None, None], 0.1)
    out = tc.thin_fprop(r, tc.thin_pack_w(w, "fprop"), b, 3, 128, ACT_LRELU, 0.1, sigma=sigma)
    assert err(tc.from_padded(out), ref) <= 1e-2
    # its weight gradient and its input gradient (phase G: gradient w.r.t. the generated image)
    dy = _bf(torch.randn(N, 128, 32, 32, device=cuda))
    wz = torch.zeros(128, 3, 4, 4, device=cuda, requires_grad=True)
    gw = torch.autograd.grad(TF.conv2d(img, wz, None, stride=2, padding=1), wz, dy)[0]
    dyp = tc.to_padded(dy)
    assert err(tc.thin_wgrad(r, dyp, 3), gw) <= 2e-3
    gx = TF.conv_transpose2d(dy, _bf(w), None, stride=2, padding=1) / 1.3
    assert err(tc.thin_dgrad(dyp, tc.thin_pack_w(w, "dgrad"), None, 3, sigma=sigma), gx) <= 2e-3
    # G's last layer: ConvTranspose2d(128,3) + bias + tanh
    bt = torch.randn(3, device=cuda)
    wq = _bf(w)
    reft = torch.tanh(TF.conv_transpose2d(dy, wq, bt, stride=2, padding=1))
    assert err(tc.thin_dgrad(dyp, tc.thin_pack_w(wq, "dgrad"), bt, 3, ACT_TANH), reft) <= 2e-3
    # ... and its input gradient: conv of (dL/dimg * tanh') with the same weights
    g_img = _bf(torch.randn(N, 3, 64, 64, device=cuda))
    rg = tc.thin_expand(g_img, mask_y=reft, act=ACT_TANH)
    refg = TF.conv2d(_bf(g_img * (1 - reft * reft)), wq, None, stride=2, padding=1)
    outg = tc.thin_fprop(rg, tc.thin_pack_w(wq, "fprop"), None, 3, 128)
    assert err(tc.from_padded(outg), refg) <= 1e-2


def test_dense_layers(cuda):
    """ConvTranspose2d(218,1024,4,1,0) on 1x1 and the Conv2d(1024,19,4,1,0) head as batch GEMMs at n = 1024."""
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_LRELU
    torch.manual_seed(17)
    C = 1024
    z = _bf(torch.randn(N, 218, device=cuda))
    w = _bf(torch.randn(218, C, 4, 4, device=cuda) * 0.05)
    b = torch.randn(C, device=cuda)
    ref = TF.conv_transpose2d(z.view(N, 218, 1, 1), w, b)
    a = tc.pad_rows(z, 256)
    assert err(tc.from_padded(tc.dense_scatter(a, tc.dense_pack(w, 256, False), b, C)), ref) <= 1e-2
    g = _bf(torch.randn(N, C, 4, 4, device=cuda))
    wz = torch.zeros_like(w).requires_grad_()
    gw = torch.autograd.grad(TF.conv_transpose2d(z.view(N, 218, 1, 1), wz, None), wz, g)[0]
    assert err(tc.dense_wgrad(a, tc.to_padded(g), 218), gw) <= 2e-3
    y = _bf(torch.randn(N, C, 4, 4, device=cuda))
    wh = _bf(torch.randn(19, C, 4, 4, device=cuda) * 0.02)
    bh = torch.randn(19, device=cuda)
    yp = tc.to_padded(y)
    assert err(tc.dense_gather(yp, tc.dense_pack(wh, 32, True), bh, 19), TF.conv2d(y, wh, bh).view(N, 19)) <= 2e-3
    gh = _bf(torch.randn(N, 19, device=cuda))
    whz = torch.zeros_like(wh).requires_grad_()
    yr = y.clone().requires_grad_()
    gwh = torch.autograd.grad(TF.conv2d(y, whz, None).view(N, 19), whz, gh)[0]
    gy = torch.autograd.grad(TF.conv2d(yr, wh, None).view(N, 19), yr, gh)[0]
    ah = tc.pad_rows(gh, 64)
    assert err(tc.dense_wgrad(ah, yp, 19), gwh) <= 2e-3
    sums = torch.zeros(C, device=cuda, dtype=torch.float64)
    dxp = tc.dense_scatter(ah, tc.dense_pack(wh, 64, False), None, C, mask=yp, mask_act=ACT_LRELU, slope=0.1, chan_sums=sums)
    refx = gy * torch.where(y > 0, 1.0, 0.1)
    assert err(tc.from_padded(dxp), refx) <= 1e-2
    assert float((sums - refx.double().sum((0, 2, 3))).abs().max() / refx.double().abs().sum((0, 2, 3)).max()) <= 2e-3


def test_celeba_step_b1024_forced_gates(cuda):
    """ONE full CelebA step at the benchmarked batch (1024), three phases, against the oracle run on the GPU in fp32
    (cuDNN / cuBLAS with TF32 off; fp64 at this batch would only add minutes) on the gates of our run: the three
    losses and every gradient tensor of every phase to north_star's 2e-2."""
    import gates
    import step_util as U
    out = gates.forced_step("celeba", cuda, N, "bf16", oracle_dtypes=(torch.float32,))
    ref = out["forced"][0]
    assert out["flips"] <= 0.01 * out["gates"]
    names = U.grad_names(out["step"])
    worst = 0.0
    for k in ("g_loss", "d_loss", "info_loss"):
        assert abs(out["losses"][k] - ref["losses"][k]) <= 2e-2 * max(1.0, abs(ref["losses"][k])), (k, out["losses"])
        assert abs(out["losses"][k] - out["free"]["losses"][k]) <= 2e-2 * max(1.0, abs(ref["losses"][k])), k
    for ph in range(3):
        errs = U.phase_errors(names[ph], out["ours"][ph]["grads"], ref["phases"][ph]["grads"])
        for n, (mx, l2, cs) in errs.items():
            assert mx <= 2e-2, (ph, n, mx, l2)
            worst = max(worst, mx)
        # and UN-forced, against the oracle on its own gates: direction and size of every gradient
        free = U.phase_errors(names[ph], out["ours"][ph]["grads"], out["free"]["phases"][ph]["grads"])
        for n, (mx, l2, cs) in free.items():
            if isinstance(cs, float):
                assert cs >= 0.98 and l2 <= 0.15, (ph, n, cs, l2)
    print(f"B=1024: gate flips {out['flips']} of {out['gates']}; worst forced-gate gradient error {worst:.2e}")


def test_colored_step_b512(cuda):
    """BASELINE configs[2] at its full global batch (512) on one device: losses to 2e-2, gradients by direction / L2
    against the fp32 oracle on the GPU."""
    import step_util as U
    losses_k = ("d_loss", "g_loss", "cat_loss", "cont_loss", "affine_loss", "relative_cat_loss", "total")
    ref, rec, losses, st, ours = U.run_pair_colored(cuda, 512, "bf16", oracle_dtype=torch.float32)
    for k in losses_k:
        assert abs(losses[k] - ref["losses"][k]) <= 2e-2 * max(1.0, abs(ref["losses"][k])), (k, losses, ref["losses"])
    names = U.dsprites_grad_names(ours)
    for ph in range(2):
        errs = U.phase_errors(names[ph], rec[ph]["grads"], ref["phases"][ph]["grads"], U.DSPRITES_ZERO_GRAD)
        for n, (mx, l2, cs) in errs.items():
            if cs is None:
                assert mx <= 2e-2, (ph, n, mx)
            elif cs == "small":
                assert mx <= 0.15, (ph, n, mx)
            else:
                assert cs >= 0.95 and l2 <= 0.3, (ph, n, cs, l2)
