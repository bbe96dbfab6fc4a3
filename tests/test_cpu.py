"""CPU suite (-m "not gpu"): the oracle against the golden vectors generated from the reference, the
oracle against the reference itself when a checkout of it is present ($EADGAN_REF), the host-side mirror (state_dict
layout, constructor parity, no-CPU-fallback errors), and the C-ABI library (loads, exports every
symbol include/eadgan.h declares)."""
import ctypes
import json
import os
import re
import warnings

import numpy as np
import pytest
import torch

from conftest import ROOT
from oracle import ref_runner

warnings.filterwarnings("ignore")
GOLDEN = os.path.join(ROOT, "tests", "golden")
# the upstream EAD-GAN scripts are not part of this repository: point EADGAN_REF at a checkout to run these
NEEDS_REFERENCE = pytest.mark.skipif(not ref_runner.available(), reason="needs a checkout of the reference ($EADGAN_REF)")


def _close(a, b, rtol, atol=1e-9):
    return abs(a - b) <= atol + rtol * max(abs(a), abs(b))


def _check_fp(t, fp, rtol):
    from oracle.torch_oracle import summarize
    s = summarize(t)
    scale = max(fp["absmax"], 1e-12)
    assert abs(s["l2"] - fp["l2"]) <= rtol * max(fp["l2"], 1e-12) + 1e-9
    assert abs(s["absmax"] - fp["absmax"]) <= rtol * scale + 1e-9
    for a, b in zip(s["probe"], fp["probe"]):
        assert abs(a - b) <= rtol * scale + 1e-9


@pytest.mark.parametrize("name", ["celeba_b4_seed0", "celeba_b6_seed3"])
def test_oracle_reproduces_reference_golden(name):
    """oracle/torch_oracle.py (the restatement that travels to the GPU box) vs fixtures produced by
    executing celebA/EAD-GAN_celebA.py itself (oracle/make_golden.py)."""
    from oracle import torch_oracle as O
    with open(os.path.join(GOLDEN, name + ".json")) as f:
        g = json.load(f)
    B, seed = g["batch"], g["seed"]
    torch.set_num_threads(8)
    st = O.build_celeba(seed=seed)
    rec = O.step_celeba(st, O.synth_celeba_images(B, seed), O.sample_celeba(np.random.RandomState(seed), B))
    for k, v in g["losses"].items():
        assert _close(rec["losses"][k], v, 1e-5), (k, rec["losses"][k], v)
    assert len(rec["phases"]) == len(g["phases"]) == 3
    # phase G and D start from identical weights: tight.  The info phase follows two Adam steps whose
    # first update is ~ lr*sign(g) (SURVEY.md section 7.3-1), so thread-count / ISA dependent rounding
    # can flip signs of near-zero gradients: gradients are still tight, post-step weights looser.
    for ph, gph, (rt_g, rt_p) in zip(rec["phases"], g["phases"], [(1e-4, 1e-4), (1e-4, 1e-4), (2e-3, 2e-3)]):
        assert len(ph["grads"]) == len(gph["grads"])
        for t, fp in zip(ph["grads"], gph["grads"]):
            _check_fp(t, fp, rt_g)
        for t, fp in zip(ph["params_after"], gph["params_after"]):
            _check_fp(t, fp, rt_p)


@pytest.mark.parametrize("name", ["dsprites_b6_seed0", "dsprites_b8_seed2"])
def test_dsprites_oracle_reproduces_reference_golden(name):
    """the dSprites stage-2 restatement vs fixtures produced by executing dSprites/rp.py itself."""
    from oracle import torch_oracle as O
    with open(os.path.join(GOLDEN, name + ".json")) as f:
        g = json.load(f)
    B, seed = g["batch"], g["seed"]
    torch.set_num_threads(8)
    st = O.build_dsprites(seed=seed)
    rec = O.step_dsprites(st, O.synth_dsprites_images(B, seed), O.sample_dsprites(np.random.RandomState(seed), B))
    for k, v in g["losses"].items():
        assert _close(rec["losses"][k], v, 1e-5), (k, rec["losses"][k], v)
    assert len(rec["phases"]) == len(g["phases"]) == 2
    for ph, gph in zip(rec["phases"], g["phases"]):
        assert len(ph["grads"]) == len(gph["grads"])
        for t, fp in zip(ph["grads"], gph["grads"]):
            _check_fp(t, fp, 1e-4)
        for t, fp in zip(ph["params_after"], gph["params_after"]):
            _check_fp(t, fp, 1e-4)


@pytest.mark.parametrize("name", ["colored_b6_seed0", "colored_b8_seed1"])
def test_colored_oracle_reproduces_reference_golden(name):
    """the colored-dSprites stage-2 restatement vs fixtures produced by executing colored_dSprites/rp_color.py."""
    from oracle import torch_oracle as O
    with open(os.path.join(GOLDEN, name + ".json")) as f:
        g = json.load(f)
    B, seed = g["batch"], g["seed"]
    torch.set_num_threads(8)
    st = O.build_dsprites(seed=seed, colored=True)
    rec = O.step_colored(st, O.synth_dsprites_images(B, seed), O.sample_colored(np.random.RandomState(seed), B))
    for k, v in g["losses"].items():
        assert _close(rec["losses"][k], v, 1e-5), (k, rec["losses"][k], v)
    assert len(rec["phases"]) == len(g["phases"]) == 2
    for ph, gph in zip(rec["phases"], g["phases"]):
        assert len(ph["grads"]) == len(gph["grads"])
        for t, fp in zip(ph["grads"], gph["grads"]):
            _check_fp(t, fp, 1e-4)
        for t, fp in zip(ph["params_after"], gph["params_after"]):
            _check_fp(t, fp, 1e-4)


@pytest.mark.parametrize("name", ["mnist_b8_seed0", "mnist_b64_seed1"])
def test_mnist_oracle_reproduces_reference_golden(name):
    """BASELINE configs[0]: the MNIST restatement vs fixtures produced by executing MNIST/EAD-GAN_rpqmnxy.py
    (batch 64 is the configuration's own batch size)."""
    from oracle import torch_oracle as O
    with open(os.path.join(GOLDEN, name + ".json")) as f:
        g = json.load(f)
    B, seed = g["batch"], g["seed"]
    torch.set_num_threads(8)
    st = O.build_mnist(seed=seed)
    rec = O.step_mnist(st, O.synth_mnist_images(B, seed), O.sample_mnist(np.random.RandomState(seed), B))
    for k, v in g["losses"].items():
        assert _close(rec["losses"][k], v, 1e-5), (k, rec["losses"][k], v)
    assert len(rec["phases"]) == len(g["phases"]) == 3
    for ph, gph, rt in zip(rec["phases"], g["phases"], (1e-4, 1e-4, 2e-3)):
        assert len(ph["grads"]) == len(gph["grads"])
        for t, fp in zip(ph["grads"], gph["grads"]):
            if (t is None) != (fp is None):
                raise AssertionError("gradient presence differs from the reference run")
            if t is not None:
                _check_fp(t, fp, rt)
        for t, fp in zip(ph["params_after"], gph["params_after"]):
            _check_fp(t, fp, rt)


def test_mnist_affine_glue_matches_oracle():
    from eadgan_b200 import affine
    from oracle import torch_oracle as O
    g = torch.Generator().manual_seed(7)
    c1, c2 = torch.rand(32, 7, generator=g) * 2 - 1, torch.rand(32, 7, generator=g) * 2 - 1
    assert (affine.mnist_matrix23(c1) - O.mnist_get_matrix(c1)[:, 0:2]).abs().max() <= 1e-6
    rel = O.mnist_get_matrix(c2) @ torch.inverse(O.mnist_get_matrix(c1))
    assert (affine.mnist_relative_rows_torch(c1, c2) - torch.cat((rel[:, 0], rel[:, 1]), dim=1)).abs().max() <= 1e-5
    A = O.MnistAffineApproximator()
    want = O.mnist_affine_regularizer(c1, c2, A)
    got = affine.mnist_code_from_params(A(affine.mnist_relative_rows_torch(c1, c2)))
    assert (got - want).abs().max() <= 1e-4


@pytest.mark.parametrize("name,colored", [("pxy_b8_seed0", False), ("pxy_color_b8_seed0", True)])
def test_pxy_oracle_reproduces_reference_golden(name, colored):
    """stage 1 (dSprites/pxy.py, colored_dSprites/pxy_color.py) restatement vs the scripts' own outputs"""
    from eadgan_b200 import affine
    from oracle import torch_oracle as O
    with open(os.path.join(GOLDEN, name + ".json")) as f:
        g = json.load(f)
    B, seed = g["batch"], g["seed"]
    st = O.build_pxy(seed=seed, colored=colored)
    rec = O.step_pxy(st, O.synth_dsprites_images(B, seed), O.sample_pxy(np.random.RandomState(seed), B, colored))
    assert _close(rec["losses"]["affine_loss"], g["losses"]["affine_loss"], 1e-5)
    for t, fp in zip(rec["phases"][0]["grads"], g["phases"][0]["grads"]):
        _check_fp(t, fp, 1e-4)
    for t, fp in zip(rec["phases"][0]["params_after"], g["phases"][0]["params_after"]):
        _check_fp(t, fp, 1e-4)
    # device-side glue vs the oracle's matrix form
    gen = torch.Generator().manual_seed(3)
    k = 6 if colored else 3
    c1, c2 = torch.rand(16, k, generator=gen) * 2 - 1, torch.rand(16, k, generator=gen) * 2 - 1
    assert (affine.pxy_matrix23(c1) - O.pxy_get_matrix(c1)[:, 0:2]).abs().max() <= 1e-6
    assert (affine.pxy_relative_code(c1, c2) - O.pxy_affine_regularizer(c1, c2)).abs().max() <= 1e-4


def test_colored_affine_glue_matches_oracle():
    """device-side restatement (eadgan_b200/affine.py) of affine_color_regularzier vs the oracle's (which is
    pinned to colored_dSprites/rp_color.py through the golden fixtures above)."""
    from eadgan_b200 import affine
    from oracle import torch_oracle as O
    g = torch.Generator().manual_seed(5)
    c1, c2 = torch.rand(32, 7, generator=g) * 2 - 1, torch.rand(32, 7, generator=g) * 2 - 1
    assert (affine.colored_relative_code_torch(c1, c2) - O.colored_affine_color_regularizer(c1, c2)).abs().max() <= 1e-4


def test_celeba_and_dsprites_affine_glue_matches_oracle():
    """the product's closed-form affine glue (eadgan_b200/affine.py) vs the oracle's matrix form, which the golden
    fixtures pin to the reference's utils_*.py through the losses and gradients of whole steps (the tests below
    compare with utils_*.py directly when a checkout of the reference is present)."""
    from eadgan_b200 import affine
    from oracle import torch_oracle as O
    g = torch.Generator().manual_seed(1)
    c1, c2, c3 = (torch.rand(9, k, generator=g) * 2 - 1 for k in (4, 4, 3))
    assert (affine.dsprites_matrix23(c1) - O.dsprites_get_matrix(c1)[:, 0:2]).abs().max() <= 1e-6
    assert (affine.dsprites_align_inverse(c3) - torch.inverse(O.dsprites_align_matrix(c3))[:, 0:2]).abs().max() <= 1e-6
    assert (affine.dsprites_relative_code_torch(c1, c2) - O.dsprites_affine_regularizer(c1, c2)).abs().max() <= 1e-4
    c1, c2 = torch.rand(9, 8, generator=g) * 2 - 1, torch.rand(9, 8, generator=g) * 2 - 1
    assert (affine.celeba_matrix(c1[:, :5]) - O.celeba_get_matrix(c1[:, :5])).abs().max() <= 1e-6
    assert (affine.celeba_relative_code_torch(c1, c2) - O.celeba_affine_regularizer(c1, c2)).abs().max() <= 1e-4


@NEEDS_REFERENCE
def test_oracle_classes_equal_reference_classes():
    """key-for-key, bit-for-bit equality of the restated modules with the AST-extracted reference classes."""
    from oracle import ref_runner as R, torch_oracle as O
    ns = R.extract_defs("celeba")
    torch.manual_seed(5)
    G_ref, D_ref = ns["Generator"](), ns["Discriminator"]()
    torch.manual_seed(5)
    G, D = O.CelebAGenerator(), O.CelebADiscriminator()
    for a, b in ((G_ref, G), (D_ref, D)):
        sa, sb = a.state_dict(), b.state_dict()
        assert list(sa.keys()) == list(sb.keys())
        for k in sa:
            assert sa[k].shape == sb[k].shape and sa[k].dtype == sb[k].dtype and torch.equal(sa[k], sb[k]), k
    z, lab, code = torch.randn(3, 200), torch.eye(10)[:3], torch.rand(3, 8)
    assert torch.equal(G_ref(z, lab, code), G(z, lab, code))
    x = torch.randn(3, 3, 64, 64)
    for a, b in zip(D_ref(x), D(x)):
        assert torch.equal(a, b)


@NEEDS_REFERENCE
def test_reference_affine_glue_matches():
    import importlib.util
    import sys
    from oracle import ref_runner as R, torch_oracle as O
    from eadgan_b200 import affine
    saved = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        spec = importlib.util.spec_from_file_location("ref_utils_rpqxy", os.path.join(R.REF_ROOT, "celebA", "utils_rpqxy.py"))
        U = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(U)
        torch.manual_seed(0)
        c1, c2 = torch.rand(9, 8) * 2 - 1, torch.rand(9, 8) * 2 - 1
        m_ref = U.get_matrix(c1[:, :5])
        r_ref = U.affine_regularzier(c1, c2)
    finally:
        torch.Tensor.cuda = saved
    for impl_m, impl_r in ((O.celeba_get_matrix, O.celeba_affine_regularizer),
                           (affine.celeba_matrix, affine.celeba_relative_code_torch)):
        assert (impl_m(c1[:, :5]) - m_ref).abs().max() <= 1e-6
        assert (impl_r(c1, c2) - r_ref).abs().max() <= 1e-4


@NEEDS_REFERENCE
def test_reference_dsprites_affine_glue_matches():
    """dSprites/utils_pxy.py + utils_rp.py executed as is vs the oracle restatement and the device-side
    closed-form glue of the product (eadgan_b200/affine.py)."""
    import importlib.util
    from oracle import ref_runner as R, torch_oracle as O
    from eadgan_b200 import affine
    saved = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        mods = {}
        for name in ("utils_pxy", "utils_rp"):
            spec = importlib.util.spec_from_file_location("ref_" + name, os.path.join(R.REF_ROOT, "dSprites", name + ".py"))
            mods[name] = importlib.util.module_from_spec(spec)
            mods[name].np = np          # utils_rp.py uses np without importing it (the scripts star-import numpy first)
            spec.loader.exec_module(mods[name])
        torch.manual_seed(1)
        c1, c2, c3 = torch.rand(9, 4) * 2 - 1, torch.rand(9, 4) * 2 - 1, torch.rand(9, 3) * 2 - 1
        m_ref = mods["utils_rp"].get_matrix_D(c1)
        m2_ref = mods["utils_rp"].get_matrix(c1)
        al_ref = torch.inverse(mods["utils_pxy"].get_matrix_pxy_align(c3))
        r_ref = mods["utils_rp"].affine_regularzier(c1, c2)
    finally:
        torch.Tensor.cuda = saved
    assert torch.equal(m_ref, m2_ref)
    assert (O.dsprites_get_matrix(c1) - m_ref).abs().max() <= 1e-6
    assert (affine.dsprites_matrix23(c1) - m_ref[:, 0:2]).abs().max() <= 1e-6
    assert (torch.inverse(O.dsprites_align_matrix(c3)) - al_ref).abs().max() <= 1e-6
    assert (affine.dsprites_align_inverse(c3) - al_ref[:, 0:2]).abs().max() <= 1e-6
    assert (O.dsprites_affine_regularizer(c1, c2) - r_ref).abs().max() <= 1e-5
    assert (affine.dsprites_relative_code_torch(c1, c2) - r_ref).abs().max() <= 1e-4


def test_product_modules_mirror_reference_layout():
    """eadgan_b200 modules: same keys / shapes / seeded init as the stock-torch oracle, both directions of
    load_state_dict, legacy spectral-norm metadata."""
    from eadgan_b200.steps.celeba import Discriminator, Generator
    from oracle import torch_oracle as O
    torch.manual_seed(11)
    G, D = Generator(), Discriminator()
    torch.manual_seed(11)
    Gr, Dr = O.CelebAGenerator(), O.CelebADiscriminator()
    for a, b in ((G, Gr), (D, Dr)):
        sa, sb = a.state_dict(), b.state_dict()
        assert list(sa.keys()) == list(sb.keys())
        assert all(torch.equal(sa[k], sb[k]) for k in sa)
        assert sa._metadata == sb._metadata
        b.load_state_dict(sa)
        a.load_state_dict(sb)
    assert sum(p.numel() for p in G.parameters()) == 14591619
    assert sum(p.numel() for p in D.parameters()) == 11329427
    names = [type(m).__name__ for m in G.modules()]
    assert any("Conv" in n for n in names) and any("BatchNorm" in n for n in names)  # weights_init_normal keys


def test_no_cpu_fallback():
    import eadgan_b200.nn as enn
    from eadgan_b200.optim import Adam
    with pytest.raises(RuntimeError, match="no CPU"):
        enn.Conv2d(3, 4, 4, 2, 1)(torch.zeros(1, 3, 8, 8))
    with pytest.raises(RuntimeError, match="no CPU"):
        enn.BCELoss()(torch.rand(4), torch.ones(4))
    p = torch.nn.Parameter(torch.zeros(3))
    p.grad = torch.ones(3)
    with pytest.raises(RuntimeError, match="CUDA"):
        Adam([p], lr=1e-3).step()


def test_patch_rebinds_and_restores():
    import eadgan_b200
    import eadgan_b200.nn as enn
    stock = torch.nn.Conv2d
    eadgan_b200.patch()
    try:
        assert torch.nn.Conv2d is enn.Conv2d and torch.optim.Adam is eadgan_b200.optim.Adam
        assert torch.nn.utils.spectral_norm is enn.spectral_norm
        m = torch.nn.utils.spectral_norm(torch.nn.Conv2d(3, 8, 4, 2, 1))
        assert list(m.state_dict().keys()) == ["bias", "weight_orig", "weight_u", "weight_v"]
    finally:
        eadgan_b200.unpatch()
    assert torch.nn.Conv2d is stock


def test_c_abi_exports_every_declared_symbol():
    from eadgan_b200 import _lib
    import __graft_entry__ as ge
    ge.build()
    hdr = open(os.path.join(ROOT, "include", "eadgan.h")).read()
    declared = set(re.findall(r"\b(eadgan_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"eadgan_status", "eadgan_dtype", "eadgan_act"}
    lib = ctypes.CDLL(_lib.LIB_PATH)
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, missing
    assert declared == set(_lib.EXPORTED), declared ^ set(_lib.EXPORTED)
    assert lib.eadgan_version() == 100


def test_sass_is_blackwell_native():
    """tcgen05.mma / tcgen05.ld / TMA must be in the built library (UTC*MMA / LDTM / UTMALDG SASS)."""
    import shutil
    import subprocess
    from eadgan_b200 import _lib
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    sass = subprocess.run(["cuobjdump", "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    for mnemonic in ("UTCHMMA", "LDTM", "UTMALDG"):
        assert mnemonic in sass, mnemonic


def _kernel_plan(seq, in_shape):
    """the bf16 chain executor's plan of a conv stack, one line per stage:
    "forward / weight-gradient / input-gradient family, big-map channels:allocated, small-map channels,
    input > output buffer format[, fuse]" -- and the stack's output shape"""
    from eadgan_b200 import chain
    stages = chain._plan(seq)
    assert stages is not None
    plans = chain._plan_kernels(stages, in_shape)
    return ([f"{p.fwd}/{p.wgrad}/{p.dx} c{p.d.c}:{p.ca} k{p.d.k} {p.in_fmt}>{p.out_fmt}" + (" fuse" if p.fuse else "")
             for p in plans], plans[-1].out_shape)


def test_chain_plans_route_every_celeba_and_dsprites_layer_to_a_tensor_core_kernel():
    """host logic of the bf16 chain executor (no kernels run): which kernel family runs the forward, the weight
    gradient and the input gradient of each layer of the reference networks.  Guards the geometry rules (_tc_ok /
    _thin_ok / dense) against regressions that would silently push a hot layer back to the SIMT kernels."""
    from eadgan_b200.steps import celeba, dsprites, mnist

    torch.manual_seed(0)
    got, shape = _kernel_plan(celeba.Generator().conv_blocks, (8, 218, 1, 1))
    assert got == ["dense_T/dense/simt c1024:1024 k218 ext>pad",
                   "tc/tc/tc c512:512 k1024 pad>pad",
                   "tc/tc/tc c256:256 k512 pad>pad",
                   "tc/tc/tc c128:128 k256 pad>pad",
                   "thin/thin/thin c3:3 k128 pad>ext"] and shape == (8, 3, 64, 64), got
    got, shape = _kernel_plan(celeba.Discriminator().main, (8, 3, 64, 64))
    assert got == ["thin/thin/thin c3:3 k128 ext>pad",
                   "tc/tc/tc c128:128 k256 pad>pad fuse",
                   "tc/tc/tc c256:256 k512 pad>pad fuse",
                   "tc/tc/tc c512:512 k1024 pad>pad fuse",
                   "dense_C/dense/dense c1024:1024 k19 pad>ext fuse"] and shape == (8, 19, 1, 1), got
    for ch in (1, 3):
        got, shape = _kernel_plan(dsprites.Generator(ch, 4 if ch == 1 else 7).conv_block, (8, 64, 4, 4))
        assert got == ["tc/tc/tc c64:64 k64 pad>pad"] * 3 + [f"thin/thin/thin c{ch}:{ch} k64 pad>ext"], got
        assert shape == (8, ch, 64, 64)
        # k = 32 layers: zero-filled 64-wide TMA boxes in both backward directions
        trunk = [f"thin/thin/thin c{ch}:{ch} k32 ext>pad", "tc/tc/tc c32:32 k32 pad>pad fuse",
                 "tc/tc/tc c32:32 k64 pad>pad fuse", "tc/tc/tc c64:64 k64 pad>ext fuse"]
        for net in (dsprites.Discriminator(ch), dsprites.Encoder(ch), dsprites.Encoder_pxy(ch)):
            got, shape = _kernel_plan(net.conv_block, (8, ch, 64, 64))
            assert got == trunk and shape == (8, 64, 4, 4), (type(net).__name__, got)
    # 3x3 stride-2 convs: no tensor-core kernel covers them
    got, shape = _kernel_plan(mnist.Discriminator().conv_blocks, (8, 1, 32, 32))
    assert got == ["simt/simt/simt c1:1 k16 ext>pad", "simt/simt/simt c16:16 k32 pad>pad fuse",
                   "simt/simt/simt c32:32 k64 pad>pad fuse", "simt/simt/simt c64:64 k128 pad>ext fuse"], got
    assert shape == (8, 128, 2, 2)


def test_chain_plans_of_small_and_channel_padded_stacks():
    """the plan of the stacks tests/test_chain_gpu.py runs, and of layers whose big map has 5..31 channels (zero-padded
    to 32 on the tensor-core path), which no reference network has"""
    import eadgan_b200.nn as enn
    from test_chain_gpu import SMALL, _build

    plans = {name: _kernel_plan(_build(enn, spec), shape) for name, spec, shape in SMALL}
    assert plans["dsprites_trunk"] == (["tc/tc/tc c32:32 k32 pad>pad", "tc/tc/tc c32:32 k64 pad>pad fuse",
                                        "tc/tc/tc c64:64 k64 pad>ext fuse"], (6, 64, 4, 4))
    # a 16-wide image is not the 32-wide one of the thin input-gradient kernel: the tensor-core path pads 1 -> 32
    assert plans["dsprites_G"] == (["tc/tc/tc c64:64 k64 pad>pad"] * 2 + ["tc/tc/tc c1:32 k64 pad>ext"], (6, 1, 32, 32))
    # first stage: the input gradient has zero-padded channels too, written by the fp32 NCHW epilogue
    seq = enn.Sequential(enn.Conv2d(16, 64, 4, 2, 1), enn.LeakyReLU(0.2), enn.Conv2d(64, 64, 4, 2, 1))
    assert _kernel_plan(seq, (8, 16, 32, 32)) == (["tc/tc/tc c16:32 k64 pad>pad", "tc/tc/tc c64:64 k64 pad>ext fuse"],
                                                  (8, 64, 8, 8))
    # last stage: the forward writes fp32 NCHW; the weight gradient's channel-padded copy of dz feeds the input gradient
    seq = enn.Sequential(enn.ConvTranspose2d(64, 64, 4, 2, 1), enn.ReLU(), enn.ConvTranspose2d(64, 16, 4, 2, 1))
    assert _kernel_plan(seq, (8, 64, 8, 8)) == (["tc/tc/tc c64:64 k64 pad>pad", "tc/tc/tc c16:32 k64 pad>ext fuse"],
                                                (8, 16, 32, 32))
    # not last: a ConvTranspose onto 16 channels runs on SIMT into a 16-channel buffer; the tensor-core conv after it
    # reads that map channel-padded to 32 (the executor copies it), and its input gradient runs on SIMT
    seq = enn.Sequential(enn.ConvTranspose2d(64, 16, 4, 2, 1), enn.LeakyReLU(0.2), enn.Conv2d(16, 64, 4, 2, 1))
    assert _kernel_plan(seq, (8, 64, 8, 8)) == (["simt/simt/simt c16:16 k64 ext>pad", "tc/tc/simt c16:32 k64 pad>ext fuse"],
                                                (8, 64, 8, 8))
    # a bias or BatchNorm statistics on more than 1024 output channels do not fit the fused epilogues: SIMT
    seq = enn.Sequential(enn.Conv2d(64, 2048, 4, 2, 1), enn.LeakyReLU(0.2), enn.Conv2d(2048, 64, 4, 2, 1))
    assert _kernel_plan(seq, (8, 64, 8, 8)) == (["simt/simt/simt c64:64 k2048 ext>pad",
                                                 "tc/tc/tc c2048:2048 k64 pad>ext fuse"], (8, 64, 2, 2))
    seq = enn.Sequential(enn.Conv2d(64, 2048, 4, 2, 1, bias=False), enn.LeakyReLU(0.2), enn.Conv2d(2048, 64, 4, 2, 1))
    assert _kernel_plan(seq, (8, 64, 8, 8))[0][0] == "tc/tc/tc c64:64 k2048 pad>pad"


# Every (forward, weight gradient, input gradient, input format, output format, fused mask, channel-padded) row and every
# (BatchNorm, activation) pair that tests/test_chain_stages_gpu.py runs against its fp64 referee.  A planner rule that
# adds a row makes this test fail until a catalogue entry reaches it.
CATALOGUE_ROWS = {
    ("dense_C", "dense", "dense", "pad", "ext", True, False),
    ("dense_T", "dense", "simt", "ext", "pad", False, False),
    ("simt", "simt", "simt", "ext", "pad", False, False),
    ("simt", "simt", "simt", "pad", "ext", True, False),
    ("simt", "simt", "simt", "pad", "pad", True, False),
    ("tc", "simt", "tc", "pad", "pad", False, False),
    ("tc", "tc", "simt", "pad", "ext", False, True),
    ("tc", "tc", "simt", "pad", "pad", True, False),
    ("tc", "tc", "simt", "pad", "pad", True, True),
    ("tc", "tc", "tc", "pad", "ext", False, False),
    ("tc", "tc", "tc", "pad", "ext", False, True),
    ("tc", "tc", "tc", "pad", "ext", True, False),
    ("tc", "tc", "tc", "pad", "ext", True, True),
    ("tc", "tc", "tc", "pad", "pad", False, False),
    ("tc", "tc", "tc", "pad", "pad", False, True),
    ("tc", "tc", "tc", "pad", "pad", True, False),
    ("thin", "thin", "simt", "ext", "pad", False, False),
    ("thin", "thin", "simt", "pad", "pad", True, False),
    ("thin", "thin", "thin", "ext", "pad", False, False),
    ("thin", "thin", "thin", "pad", "ext", False, False),
    ("thin", "thin", "thin", "pad", "ext", True, False),
}


def test_stage_catalogue_covers_every_plan_row():
    from eadgan_b200 import chain
    from eadgan_b200._lib import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_TANH
    import eadgan_b200.nn as enn
    from test_chain_stages_gpu import STAGES, build

    rows, pairs, fused_masks = set(), set(), set()
    for name, spec, shape in STAGES:
        stages = chain._plan(build(enn, spec))
        assert stages is not None, name
        plans = chain._plan_kernels(stages, shape)
        for si, (st, p) in enumerate(zip(stages, plans)):
            rows.add((p.fwd, p.wgrad, p.dx, p.in_fmt, p.out_fmt, p.fuse, p.ca != p.d.c))
            pairs.add((st.bn is not None, st.act[0]))
            if p.fuse:
                fused_masks.add((p.dx, stages[si - 1].act[0]))
    assert rows == CATALOGUE_ROWS, (rows - CATALOGUE_ROWS, CATALOGUE_ROWS - rows)
    acts = {ACT_NONE, ACT_RELU, ACT_LRELU, ACT_TANH, ACT_SIGMOID}
    assert pairs == {(bn, a) for bn in (False, True) for a in acts}, pairs
    # every activation's backward fused into a tensor-core input gradient
    assert {a for dx, a in fused_masks if dx == "tc"} == acts - {ACT_NONE}, fused_masks


def test_header_is_plain_c():
    """the drop-in boundary is a C ABI: include/eadgan.h must compile as C (no C++-isms, no torch types)"""
    import shutil
    import subprocess
    import tempfile
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "abi.c")
        with open(src, "w") as f:
            f.write('#include "eadgan.h"\nint main(void) { return (int)sizeof(eadgan_tc_desc) == 0; }\n')
        r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(root, "include"), src],
                           capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_reference_arm_prints_one_json_line():
    """bench.py --impl reference: the reference CPU path timed on the host cores; stdout carries exactly ONE JSON line
    with the driver's keys (a bounded sample: 1 step of batch 2 here)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-batch", "2"], capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_run_module_patches_before_running_the_script(tmp_path):
    """python -m eadgan_b200.run <script>: the script sees the replacement classes under the stock torch names
    (CPU: only the rebinding is checked, no kernel runs).  Regression test: the package re-exports the function
    ``patch``, which shadowed the submodule inside run.py."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "probe.py"
    script.write_text(
        "import sys, torch, torch.nn as nn, torch.nn.functional as F\n"
        "from torch.nn.utils import spectral_norm\n"
        "names = [nn.Conv2d.__module__, nn.Sequential.__module__, torch.optim.Adam.__module__, spectral_norm.__module__,\n"
        "         F.sigmoid.__module__, sys.argv[1]]\n"
        "print('PROBE', *names)\n")
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "eadgan_b200.run", str(script), "--flag"], capture_output=True, text=True,
                       timeout=300, cwd=str(tmp_path), env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("PROBE")][0].split()[1:]
    assert line == ["eadgan_b200.nn", "eadgan_b200.nn", "eadgan_b200.optim", "eadgan_b200.nn", "eadgan_b200.patch", "--flag"]
    r = subprocess.run([sys.executable, "-m", "eadgan_b200.run"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 2


@pytest.mark.parametrize("c,k", [(3, 8), (1, 5), (4, 6)])
def test_thin_layer_layout_algebra(c, k):
    """oracle/thin_layout.py (numpy restatement of the thin kernels' data layout: row-expanded image buffer,
    (kx, ky, c) patch order, weight packs, col2im ownership rule) against torch's conv2d / conv_transpose2d in fp64."""
    import torch.nn.functional as TF
    from oracle import thin_layout as T
    rs = np.random.RandomState(7)
    x = rs.randn(2, c, 8, 12)
    w = rs.randn(k, c, 4, 4)
    dy = rs.randn(2, k, 4, 6)
    xt, wt, dyt = (torch.tensor(a) for a in (x, w, dy))
    r = T.expand(x)
    assert r.shape == (2, 4, 14, 4, 4)
    assert np.array_equal(r[:, 1, 3, 2, :c], x[:, :, 2 * 1 + 2 - 1, 3 - 1])            # R[n][oy][X][ky][c] = Xpad[2 oy + ky][X]
    assert np.abs(T.fprop(x, w) - TF.conv2d(xt, wt, stride=2, padding=1).numpy()).max() < 1e-12
    wref = torch.zeros_like(wt, requires_grad=True)
    TF.conv2d(xt, wref, stride=2, padding=1).backward(dyt)
    assert np.abs(T.wgrad(x, dy) - wref.grad.numpy()).max() < 1e-12
    if c <= 3:
        ref = TF.conv_transpose2d(dyt, wt, stride=2, padding=1).numpy()                  # weight read as [Cin = k, Cout = c]
        assert np.abs(T.dgrad(dy, w) - ref).max() < 1e-12


def test_tc_operand_layout_algebra():
    """oracle/tc_layout.py (numpy restatement of the wide tcgen05 kernels' operand layouts: (a, b, dy, dx, c) K order of
    the space-to-depth fprop, parity decomposition + Wd pack of dgrad, wgrad column permutation) vs torch in fp64."""
    import torch.nn.functional as TF
    from oracle import tc_layout as T
    rs = np.random.RandomState(3)
    x, w, dy = rs.randn(2, 5, 8, 12), rs.randn(7, 5, 4, 4), rs.randn(2, 7, 4, 6)
    xt, wt, dyt = (torch.tensor(a) for a in (x, w, dy))
    assert np.abs(T.fprop(x, w) - TF.conv2d(xt, wt, stride=2, padding=1).numpy()).max() < 1e-12
    wref = torch.zeros_like(wt, requires_grad=True)
    TF.conv2d(xt, wref, stride=2, padding=1).backward(dyt)
    assert np.abs(T.wgrad(x, dy) - wref.grad.numpy()).max() < 1e-12
    assert np.abs(T.dgrad(dy, w) - TF.conv_transpose2d(dyt, wt, stride=2, padding=1).numpy()).max() < 1e-12


def test_benchmark_input_generator_equals_the_oracles():
    from eadgan_b200 import synthetic
    from oracle import torch_oracle as O
    for seed in (0, 1, 7):
        assert torch.equal(synthetic.celeba_images(5, seed), O.synth_celeba_images(5, seed))
        assert torch.equal(synthetic.dsprites_images(6, seed), O.synth_dsprites_images(6, seed))
        mine = synthetic.sample_celeba(np.random.RandomState(seed), 4)
        ref = O.sample_celeba(np.random.RandomState(seed), 4)
        assert all(torch.equal(a, ref[k]) for a, k in zip(mine, ("z", "code", "labels")))
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")).read()
    main_arm = src[src.index("def _main():"):]
    # the product arm of the benchmark touches the oracle only inside cpu_reference() (the cpu_baseline leg) and
    # parity_block() (the checker of the timed configuration, outside the timed region)
    assert "from oracle" not in main_arm and "import oracle" not in main_arm


def test_philox_restatement_known_answers():
    """oracle/philox_ref.py against the known-answer vectors of Philox4x32-10 (Random123 kat_vectors)."""
    from oracle.philox_ref import philox4x32_10
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in kat:
        got = philox4x32_10(np.array([ctr], dtype=np.uint32), key)[0]
        assert tuple(int(x) for x in got) == want


def test_affine_product_entry_points_have_no_cpu_fallback():
    from eadgan_b200 import affine
    c = torch.zeros(4, 7)
    for fn in (affine.celeba_relative_code, affine.dsprites_relative_code, affine.mnist_relative_rows,
               affine.colored_relative_code):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn(c, c)


def test_approximator_oracle_reproduces_reference_golden():
    """MNIST/approximate_rpqmnxy.py (pre-training of the affine approximator MLP): the restatement vs the fixture
    produced by executing the script itself for 3 iterations (oracle/ref_runner.run_approximator)."""
    from oracle import torch_oracle as O
    with open(os.path.join(GOLDEN, "approximator_it3_seed0.json")) as f:
        g = json.load(f)
    st = O.build_approximator(seed=g["seed"])
    rs = np.random.RandomState(g["seed"])
    recs = [O.step_approximator(st, O.sample_approximator(rs, g["batch"])) for _ in range(g["iterations"])]
    assert _close(recs[-1]["loss"], g["losses"]["affine_loss"], 1e-6)
    for rec, gph in zip(recs, g["phases"]):
        for t, fp in zip(rec["grads"], gph["grads"]):
            _check_fp(t, fp, 1e-5)
        for t, fp in zip(rec["params_after"], gph["params_after"]):
            _check_fp(t, fp, 1e-5)


@NEEDS_REFERENCE
def test_approximator_oracle_equals_the_executed_script():
    from oracle import ref_runner as R, torch_oracle as O
    ns, log = R.run_approximator(3, seed=1)
    st = O.build_approximator(seed=1)
    rs = np.random.RandomState(1)
    for e in log:
        rec = O.step_approximator(st, O.sample_approximator(rs, 128))
        for a, b in zip(rec["params_after"], e["params_after"]):
            assert torch.equal(a, b)
    assert rec["loss"] == float(ns["affine_loss"])
