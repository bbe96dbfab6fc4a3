"""-m gpu: one full CelebA training step (three phases, three Adams; celebA/EAD-GAN_celebA.py:296-401)
through the drop-in modules vs the oracle restatement on identical seeded inputs and identical seeded
random-init weights.

Protocol (SURVEY.md section 7.3-1): the torch fp64 oracle is the referee; every phase of OUR run starts
from the oracle's post-phase state (tests/step_util.py), so Adam's lr*sign(g) noise does not cascade;
gradients are compared per tensor with the tensor-normalised max error max|a-b|/max|b| (conv biases in
front of a train-mode BatchNorm -- mathematically zero gradient -- use their weight's scale); Adam is
tested in isolation on identical gradients in tests/test_ops_gpu.py.
"""
import pytest
import torch

import step_util as U
from conftest import rel_err

pytestmark = pytest.mark.gpu


def test_celeba_step_fp32(cuda):
    ref, rec, losses, st, ours = U.run_pair(cuda, 8, "fp32")
    for k in ("g_loss", "d_loss", "info_loss"):
        assert abs(losses[k] - ref["losses"][k]) <= 2e-5 * max(1.0, abs(ref["losses"][k])), (k, losses, ref["losses"])
    # A single ReLU/LeakyReLU gate flip (a pre-activation within fp32 rounding of 0) moves every upstream
    # gradient by 4e-4..1.4e-3 in the reference run against ITSELF in fp64 (SURVEY.md section 7.3-1), so the
    # step-level bound is 1e-2 max / 5e-3 median; the 1e-5 bound is carried by the per-operator tests.
    names = U.grad_names(ours)
    for ph in range(3):
        errs = U.phase_errors(names[ph], rec[ph]["grads"], ref["phases"][ph]["grads"])
        mx = sorted(v[0] for v in errs.values())
        assert mx[-1] <= 1e-2, (ph, errs)
        assert mx[len(mx) // 2] <= 5e-3, (ph, errs)
    # BN running statistics and spectral-norm vectors after the whole step
    so, sr = ours.G.state_dict(), st["G"].state_dict()
    for k in sr:
        if "running" in k:
            assert rel_err(so[k], sr[k]) <= 1e-4, k
        if "num_batches" in k:
            assert int(so[k]) == int(sr[k]) == 2
    so, sr = ours.D.state_dict(), st["D"].state_dict()
    for k in sr:
        if k.endswith("_u") or k.endswith("_v"):
            assert rel_err(so[k], sr[k]) <= 1e-3, k


def test_celeba_step_fp32_post_step_weights(cuda):
    """post-step weights against torch fp32 + torch.optim.Adam.  Adam's first step is lr*g/(|g|+1e-8): where
    the gradient is well above eps and above the two runs' own disagreement, the updated weights must agree
    to 2e-3 of one step; nowhere may they differ by more than the full step size."""
    ref, rec, losses, st, ours = U.run_pair(cuda, 8, "fp32", oracle_dtype=torch.float32)
    checked = 0
    for ph, lr in ((0, 1e-3), (1, 2e-4), (2, 2e-4)):
        for a, b, go, gr in zip(rec[ph]["params_after"], ref["phases"][ph]["params_after"], rec[ph]["grads"],
                                ref["phases"][ph]["grads"]):
            d = (a.double() - b.double()).abs()
            assert float(d.max()) <= 2.001 * lr
            ok = (gr.abs() > 1e-5) & (gr.abs() > 100 * (go - gr).abs())
            if bool(ok.any()):
                checked += int(ok.sum())
                assert float(d[ok].max()) <= 2e-3 * lr + 1e-7 * float(b.abs().max()), float(d[ok].max())
    assert checked > 1_000_000


def test_celeba_state_dict_roundtrip(cuda):
    from eadgan_b200.steps.celeba import CelebAStep
    from oracle import torch_oracle as O
    ours = CelebAStep(seed=1, device=cuda)
    st = O.build_celeba(seed=2, device=cuda)
    st["G"].load_state_dict(ours.G.state_dict())
    st["D"].load_state_dict(ours.D.state_dict())
    ours.G.load_state_dict(st["G"].state_dict())
    ours.D.load_state_dict(st["D"].state_dict())
    assert list(ours.D.state_dict().keys()) == list(st["D"].state_dict().keys())
    assert list(ours.G.state_dict().keys()) == list(st["G"].state_dict().keys())


@pytest.mark.parametrize("B", [16, 64])
def test_celeba_step_bf16(cuda, B):
    """bf16 tcgen05 chain, UN-forced: losses to north_star's 2e-2; gradients by direction and L2 against the fp64
    oracle on its own branch (any two bf16 evaluations of these nets flip ~0.1-0.3 % of the LeakyReLU(0.1) / ReLU
    gates against fp64; the per-tensor 2e-2 bound is asserted by test_celeba_step_bf16_forced_gates below, where
    both runs are on the same piecewise-linear branch)."""
    ref, rec, losses, st, ours = U.run_pair(cuda, B, "bf16")
    for k in ("g_loss", "d_loss", "info_loss"):
        assert abs(losses[k] - ref["losses"][k]) <= 2e-2 * max(1.0, abs(ref["losses"][k])), (k, losses, ref["losses"])
    names = U.grad_names(ours)
    for ph in range(3):
        errs = U.phase_errors(names[ph], rec[ph]["grads"], ref["phases"][ph]["grads"])
        for n, (mx, l2, cs) in errs.items():
            if cs is None:
                assert mx <= 2e-2, (ph, n, mx)      # zero-gradient biases: closed form, exact
            elif cs == "small":
                assert mx <= 0.15, (ph, n, mx)      # [3]-element bias, normalised by its layer's weight gradient
            else:
                assert cs >= 0.95, (ph, n, cs)
                # measured: 0.153 for G's first layer (every gate flip of 7 gated layers lies upstream of it), the same at
                # B = 16 and 64 -- at random init the per-sample gradients are mutually incoherent, so signal and flip
                # noise both shrink like 1/sqrt(B); <= 0.10 for every other tensor
                assert l2 <= 0.2, (ph, n, l2)
    so, sr = ours.G.state_dict(), st["G"].state_dict()
    for k in sr:
        if "running" in k:
            assert rel_err(so[k], sr[k]) <= 2e-2, k


def _assert_forced(out, tol, what):
    ours_names = U.grad_names(out["step"])
    ref = out["forced"][0]
    for k in ("g_loss", "d_loss", "info_loss"):
        assert abs(out["losses"][k] - ref["losses"][k]) <= tol * max(1.0, abs(ref["losses"][k])), (what, k)
    worst = 0.0
    for ph in range(3):
        errs = U.phase_errors(ours_names[ph], out["ours"][ph]["grads"], ref["phases"][ph]["grads"])
        for n, (mx, l2, cs) in errs.items():
            assert mx <= tol, (what, ph, n, mx, l2)
            worst = max(worst, mx)
    return worst


@pytest.mark.parametrize("B", [16, 64])
def test_celeba_step_bf16_forced_gates(cuda, B):
    """north_star's bf16 bound on EVERY gradient tensor of EVERY phase: max|ours - oracle| / max|oracle| <= 2e-2
    with the fp64 oracle evaluated on the activation gates of our run (tests/gates.py)."""
    import gates
    out = gates.forced_step("celeba", cuda, B, "bf16")
    assert out["flips"] <= 0.01 * out["gates"]          # the forced branch is the oracle's own up to ~0.1-0.3 %
    worst = _assert_forced(out, 2e-2, f"bf16 B={B}")
    print(f"bf16 B={B}: gate flips {out['flips']} of {out['gates']}, worst tensor-normalised gradient error {worst:.2e}")


def test_celeba_step_fp32_relative_to_stock_fp32(cuda):
    """SURVEY.md section 7.3-1 (ii): with fp64 as referee, OUR fp32 error may not exceed 3x stock torch fp32's own
    error (cuDNN / cuBLAS, TF32 off) on the same inputs, tensor by tensor -- all three runs on the same gates."""
    import gates
    out = gates.forced_step("celeba", cuda, 8, "fp32", oracle_dtypes=(torch.float64, torch.float32))
    ref64, ref32 = out["forced"]
    for k in ("g_loss", "d_loss", "info_loss"):
        assert abs(out["losses"][k] - ref64["losses"][k]) <= 2e-5 * max(1.0, abs(ref64["losses"][k])), k
    names = U.grad_names(out["step"])
    for ph in range(3):
        e_ours = U.phase_errors(names[ph], out["ours"][ph]["grads"], ref64["phases"][ph]["grads"])
        e_ref = U.phase_errors(names[ph], ref32["phases"][ph]["grads"], ref64["phases"][ph]["grads"])
        for n in e_ours:
            assert e_ours[n][0] <= max(3.0 * e_ref[n][0], 1e-5), (ph, n, e_ours[n][0], e_ref[n][0])


def test_phase_g_skips_discriminator_weight_gradients(cuda):
    """phase G differentiates through D with D frozen (SURVEY.md section 7.3-8): D's parameters receive no gradient
    there, the generator's gradients are unchanged, and D is trainable again in phases D / info."""
    import os
    import numpy as np
    from eadgan_b200.steps.celeba import CelebAStep
    from oracle import torch_oracle as O
    os.environ["EADGAN_PRECISION"] = "bf16"
    step = CelebAStep(seed=0, device=cuda)
    imgs = O.synth_celeba_images(8, 0).to(cuda)
    d = O.sample_celeba(np.random.RandomState(0), 8)
    seen = {}

    def after(i):
        seen[i] = [p.grad is None for p in step.D.parameters()]

    rec = []
    step(imgs, d["z"].to(cuda), d["code"].to(cuda), d["labels"].to(cuda), record=rec, after_phase=after)
    assert all(seen[0])                      # after phase G: no D gradient was produced
    assert not any(seen[1])                  # after phase D: every D parameter has one
    assert all(p.requires_grad for p in step.D.parameters())
    assert all(g is not None for g in rec[2]["grads"])      # the info phase owns G and D


@pytest.mark.parametrize("defer_D", [False, True])
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
def test_deferred_optimizer_steps_equal_the_literal_order(cuda, prec, defer_D):
    """CelebAStep defers opt_G.step() past phase D and -- under data parallelism, forced here -- opt_D.step() past the
    info phase's G forward (nothing reads the weights in between; the gradient all-reduces hide behind that work), and
    re-packs the GEMM operands / runs the spectral-norm iterations ahead of time on a side stream.  Two iterations in
    the deferred order must leave exactly the losses, weights, BatchNorm statistics and spectral-norm vectors of the
    reference's literal order (kept whenever a test hook is attached)."""
    import os
    import numpy as np
    from eadgan_b200.steps.celeba import CelebAStep
    from oracle import torch_oracle as O
    os.environ["EADGAN_PRECISION"] = prec
    a, b = CelebAStep(seed=5, device=cuda), CelebAStep(seed=5, device=cuda)
    a._defer_D = defer_D
    for it in range(3):
        imgs = O.synth_celeba_images(16, it).to(cuda)
        d = O.sample_celeba(np.random.RandomState(it), 16)
        args = (imgs, d["z"].to(cuda), d["code"].to(cuda), d["labels"].to(cuda))
        la = a(*args)                                   # deferred
        lb = b(*args, after_phase=lambda i: None)       # literal
        for k in la:
            assert float(la[k]) == float(lb[k]), (it, k)
    for net_a, net_b in ((a.G, b.G), (a.D, b.D)):
        for (k, va), (_, vb) in zip(net_a.state_dict().items(), net_b.state_dict().items()):
            assert torch.equal(va, vb), k
