"""-m gpu: eadgan_b200.freeze on every reference network.

Every network gets random running statistics, gamma, beta and biases; spectral-normalised ones advance u / v by three
training-mode forwards first.  The frozen forward is held to the fp64 oracle's eval forward of the UNFOLDED network
(bf16: 2e-2; fp32: the per-operator rule), and, where the network's trunk runs on the bf16 chain, to the fp64 referee
of tests/bf16_emul.py run on the folded weights (1e-2).  Further: the original is left bit-identical, caches included;
the copy is a snapshot; its guards raise; and its forward launches no BatchNorm, spectral-norm or repeated pack kernel."""
import copy
import os
import re

import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu


def _img(c, hw):
    return lambda B, g: (torch.rand(B, c, hw, hw, generator=g) * 2 - 1,)


def _latent(dim, classes, code):
    def make(B, g):
        lab = torch.eye(classes)[torch.randint(0, classes, (B,), generator=g)]
        return torch.randn(B, dim, generator=g), lab, torch.rand(B, code, generator=g) * 2 - 1
    return make


def _rows(k):
    return lambda B, g: (torch.rand(B, k, generator=g) * 2 - 1,)


def _cases():
    from eadgan_b200.steps import celeba as CS, dsprites as DS, mnist as M
    from oracle import torch_oracle as O
    # name: (ours, oracle, inputs(B, generator), attribute of the trunk the bf16 chain runs or None, config batch)
    return {
        "celeba_G": (CS.Generator, O.CelebAGenerator, _latent(200, 10, 8), "conv_blocks", 1024),
        "celeba_D": (CS.Discriminator, O.CelebADiscriminator, _img(3, 64), "main", 1024),
        "dsprites_G": (lambda: DS.Generator(1, 4), lambda: O.DSpritesGenerator(3, 4, 1), _rows(7), "conv_block", 256),
        "dsprites_D": (lambda: DS.Discriminator(1), lambda: O.DSpritesDiscriminator(1), _img(1, 64), "conv_block", 256),
        "dsprites_E": (lambda: DS.Encoder(1, 4), lambda: O.DSpritesEncoder(3, 4, 1), _img(1, 64), "conv_block", 256),
        "dsprites_pxy": (lambda: DS.Encoder_pxy(1, 3), lambda: O.DSpritesEncoderPxy(1, 3), _img(1, 64), "conv_block",
                         128),
        "colored_G": (lambda: DS.Generator(3, 7), lambda: O.DSpritesGenerator(3, 7, 3), _rows(10), "conv_block", 512),
        "colored_D": (lambda: DS.Discriminator(3), lambda: O.DSpritesDiscriminator(3), _img(3, 64), "conv_block", 512),
        "colored_E": (lambda: DS.Encoder(3, 7), lambda: O.DSpritesEncoder(3, 7, 3), _img(3, 64), "conv_block", 512),
        "colored_pxy": (lambda: DS.Encoder_pxy(3, 6), lambda: O.DSpritesEncoderPxy(3, 6), _img(3, 64), "conv_block",
                        128),
        "mnist_G": (M.Generator, O.MnistGenerator, _latent(62, 10, 7), None, 64),
        "mnist_D": (M.Discriminator, O.MnistDiscriminator, _img(1, 32), "conv_blocks", 64),
        "mnist_E": (M.Encoder, O.MnistEncoder, _img(1, 32), None, 64),
        "approximator": (M.AffineApproximator, O.MnistAffineApproximator, _rows(6), None, 64),
    }


NAMES = ["celeba_G", "celeba_D", "dsprites_G", "dsprites_D", "dsprites_E", "dsprites_pxy", "colored_G", "colored_D",
         "colored_E", "colored_pxy", "mnist_G", "mnist_D", "mnist_E", "approximator"]
PARAMS = [(n, b) for n in NAMES for b in ("16", "config")]


def _randomise(net, gen):
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            c = m.num_features
            m.running_mean.copy_(torch.randn(c, generator=gen) * 0.3)
            m.running_var.copy_(torch.rand(c, generator=gen) + 0.5)
            m.weight.data.copy_(torch.rand(c, generator=gen) + 0.5)
            m.bias.data.copy_(torch.randn(c, generator=gen) * 0.2)
        elif isinstance(m, (torch.nn.Conv2d, torch.nn.ConvTranspose2d, torch.nn.Linear)) and m.bias is not None:
            m.bias.data.copy_(torch.randn(m.bias.shape, generator=gen) * 0.1)


def _inputs(name, B, dev, seed):
    return tuple(t.to(dev) for t in _cases()[name][2](B, torch.Generator().manual_seed(seed)))


def _build(name, dev, seed=0):
    """-> ours in eval mode: randomised, u / v advanced by three training-mode forwards"""
    os.environ["EADGAN_PRECISION"] = "bf16"
    make = _cases()[name][0]
    torch.manual_seed(seed)
    ours = make()
    _randomise(ours, torch.Generator().manual_seed(seed + 100))
    ours = ours.to(dev)
    if any(hasattr(m, "weight_u") for m in ours.modules()):
        ours.train()
        with torch.no_grad():
            for i in range(3):
                ours(*_inputs(name, 8, dev, seed + 200 + i))
    return ours.eval()


def _oracle(name, ours, dtype=torch.float64):
    ref = _cases()[name][1]().to(next(ours.parameters()).device)
    ref.load_state_dict(ours.state_dict())
    return ref.to(dtype).eval()


def _outs(y):
    return y if isinstance(y, tuple) else (y,)


def _worst(a, b):
    return max(rel_err(x, y) for x, y in zip(_outs(a), _outs(b)))


def _batch(name, which):
    return 16 if which == "16" else _cases()[name][4]


@pytest.mark.parametrize("name,which", PARAMS, ids=[f"{n}-B{b}" for n, b in PARAMS])
def test_frozen_bf16_forward(cuda, name, which):
    import bf16_emul
    import eadgan_b200
    B = _batch(name, which)
    ours = _build(name, cuda)
    ref = _oracle(name, ours)
    frozen = eadgan_b200.freeze(ours)
    x = _inputs(name, B, cuda, 1)
    trunk_name = _cases()[name][3]
    seen = []
    if trunk_name is not None:
        trunk = getattr(frozen, trunk_name)
        handle = trunk.register_forward_hook(lambda m, a, y: seen.append((a[0], y)))
    try:
        y = frozen(*x)
    finally:
        if trunk_name is not None:
            handle.remove()
    with torch.no_grad():
        want = ref(*(t.double() for t in x))
    err = _worst(y, want)
    print(name, "B", B, "frozen bf16 vs fp64 oracle (unfolded):", err)
    assert err <= 2e-2
    if trunk_name is not None:
        from eadgan_b200 import chain
        assert chain._plan(trunk) is not None, "the frozen trunk is not a chain stack"
        (xin, yout), = seen
        ref_trunk = copy.deepcopy(trunk).double()
        with torch.no_grad():
            emu = bf16_emul.emulate(trunk, ref_trunk, xin.double())
        e = rel_err(yout, emu)
        print(name, "B", B, "frozen trunk vs bf16 referee on the folded weights:", e)
        assert e <= 1e-2


def _per_op_ok(ours, ref64, stock32):
    """DESIGN section 2, per operator: within 1e-5 of fp64, or within 2x stock fp32's own error"""
    e, s = rel_err(ours, ref64), rel_err(stock32, ref64)
    return e <= 1e-5 or e <= 2 * s, (e, s)


@pytest.mark.parametrize("name,which", PARAMS, ids=[f"{n}-B{b}" for n, b in PARAMS])
def test_frozen_fp32_forward(cuda, name, which):
    import eadgan_b200
    B = _batch(name, which)
    ours = _build(name, cuda)
    ref = _oracle(name, ours)
    stock = _oracle(name, ours, torch.float32)
    x = _inputs(name, B, cuda, 2)
    os.environ["EADGAN_PRECISION"] = "fp32"
    try:
        frozen = eadgan_b200.freeze(ours)
        y = frozen(*x)
    finally:
        os.environ["EADGAN_PRECISION"] = "bf16"
    with torch.no_grad():
        want = ref(*(t.double() for t in x))
        s32 = stock(*x)
    for i, (a, b, s) in enumerate(zip(_outs(y), _outs(want), _outs(s32))):
        ok, es = _per_op_ok(a, b, s)
        print(name, "B", B, "output", i, "fp32 (ours, stock) vs fp64:", es)
        assert ok, (i, es)


def _caches(net):
    mods = {n: {k: m.__dict__[k] for k in ("_eadgan_plan", "_eadgan_sn_queue", "_eadgan_sn_src", "_eadgan_sigma")
                if k in m.__dict__} for n, m in net.named_modules()}
    params = {n: (getattr(p, "_eadgan_pack_uses", None), getattr(p, "_eadgan_stepped", None))
              for n, p in net.named_parameters()}
    return mods, params


@pytest.mark.parametrize("name", ["celeba_G", "celeba_D", "dsprites_E", "mnist_G", "mnist_E"])
def test_original_untouched(cuda, name):
    """state_dict, eval forward and the project's caches of the original are the same objects / bits after freeze and
    after running the copy; the copy shares none of them"""
    import eadgan_b200
    from eadgan_b200 import tc
    ours = _build(name, cuda)
    x = _inputs(name, 16, cuda, 3)
    with torch.no_grad():
        y0 = ours(*x)
    sd0 = {k: v.clone() for k, v in ours.state_dict().items()}
    mods0, params0 = _caches(ours)
    ids = {id(p) for p in ours.parameters()}
    packs0 = {k: v[2] for k, v in tc._pack_cache.items() if k[0] in ids}
    frozen = eadgan_b200.freeze(ours)
    assert all(torch.equal(v, sd0[k]) for k, v in ours.state_dict().items())
    frozen(*x)
    frozen(*x)
    assert all(torch.equal(v, sd0[k]) for k, v in ours.state_dict().items())
    with torch.no_grad():
        y1 = ours(*x)
    assert all(torch.equal(a, b) for a, b in zip(_outs(y0), _outs(y1)))
    mods1, params1 = _caches(ours)
    assert mods1.keys() == mods0.keys()
    for n in mods0:
        assert mods1[n].keys() == mods0[n].keys(), n
        assert all(mods1[n][k] is mods0[n][k] for k in mods0[n] if k == "_eadgan_plan"), n
    assert params1 == params0
    packs1 = {k: v[2] for k, v in tc._pack_cache.items() if k[0] in ids}
    assert packs1.keys() == packs0.keys() and all(packs1[k] is packs0[k] for k in packs0)
    # the copy: its own tensors, none of the private state of the original
    mine = set()
    for t in list(frozen.parameters()) + list(frozen.buffers()):
        assert not t.requires_grad and id(t) not in ids
        assert getattr(t, "_eadgan_stepped", None) is None
        mine.add(t.data_ptr())
    assert not mine & {t.data_ptr() for t in list(ours.parameters()) + list(ours.buffers())}
    for m in frozen.modules():
        assert not m.training
        assert not any(k in m.__dict__ for k in ("_eadgan_sn_queue", "_eadgan_sn_src", "_eadgan_sigma"))
        assert not hasattr(m, "weight_orig")


@pytest.mark.parametrize("name", ["celeba_G", "dsprites_E"])
def test_frozen_copy_is_a_snapshot(cuda, name):
    """an Adam step on the original does not reach the frozen copy; a second freeze() picks it up"""
    import eadgan_b200
    from eadgan_b200.optim import Adam
    ours = _build(name, cuda)
    x = _inputs(name, 16, cuda, 4)
    frozen = eadgan_b200.freeze(ours)
    y0 = frozen(*x)
    opt = Adam(ours.parameters(), lr=1e-2)
    for p in ours.parameters():
        p.grad = torch.randn_like(p)
    opt.step()
    y1 = frozen(*x)
    assert all(torch.equal(a, b) for a, b in zip(_outs(y0), _outs(y1)))
    again = eadgan_b200.freeze(ours)
    y2 = again(*x)
    assert _worst(y2, y0) > 1e-2
    with torch.no_grad():
        want = _oracle(name, ours)(*(t.double() for t in x))
    assert _worst(y2, want) <= 2e-2


def test_guards(cuda):
    import eadgan_b200
    ours = _build("celeba_D", cuda)
    frozen = eadgan_b200.freeze(ours)
    img = _inputs("celeba_D", 4, cuda, 5)[0]
    with pytest.raises(RuntimeError, match="inference-only"):
        frozen(img.clone().requires_grad_())
    with pytest.raises(RuntimeError, match="inference-only"):
        frozen.main(img.clone().requires_grad_())
    with pytest.raises(RuntimeError, match="training mode"):
        frozen.train()
    with pytest.raises(RuntimeError, match="training mode"):
        frozen.main[0].train()
    frozen.eval()       # train(False) is a no-op
    for sd in (ours.state_dict(), frozen.state_dict()):
        with pytest.raises(RuntimeError, match="state_dict"):
            frozen.load_state_dict(sd)
    assert not any(m.training for m in frozen.modules())
    frozen(img)


_BN = re.compile(r"(^|[^A-Za-z0-9_])bn_")
_SN = re.compile(r"(^|[^A-Za-z0-9_])sn_")
_PACK = re.compile(r"(^|[^A-Za-z0-9_])pack_w_")


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type.name == "CUDA"]


@pytest.mark.parametrize("name,B,absent", [("celeba_G", 1024, _BN), ("celeba_D", 64, _SN), ("dsprites_E", 64, _SN)],
                         ids=["celeba_G_no_bn", "celeba_D_no_sn", "dsprites_E_no_sn"])
def test_frozen_kernel_list(cuda, name, B, absent):
    import eadgan_b200
    ours = _build(name, cuda)
    x = _inputs(name, B, cuda, 6)
    with torch.no_grad():
        ours(*x)
        original = _kernels(lambda: ours(*x))
    assert any(absent.search(k) for k in original), "the original's eval forward should launch the folded work"
    frozen = eadgan_b200.freeze(ours)
    first = _kernels(lambda: frozen(*x))
    second = _kernels(lambda: frozen(*x))
    print(name, "frozen forward kernels:", second)
    assert not [k for k in first + second if absent.search(k)]
    assert not [k for k in second if _PACK.search(k)]
