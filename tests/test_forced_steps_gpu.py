"""-m gpu: the dSprites, colored-dSprites, MNIST and Encoder_pxy training steps tensor by tensor, against the oracle
evaluated on the activation gates -- and, for the stage-2 dSprites steps, the frozen Encoder_pxy code -- of our run
(tests/gates.py).  test_step_gpu.py does the same for CelebA.

On common gates nothing but rounding of smooth arithmetic separates the two runs, so the bounds are the project's
own: losses and every gradient tensor of every phase to 2e-2 in bf16; in fp32, every gradient tensor's error against
fp64 to at most 3x stock torch fp32's error (cuDNN / cuBLAS, TF32 off, same gates, same Encoder_pxy code), with a
floor of 1e-5 for tensors where stock fp32 happens to be exact.  The oracle-on-its-own-gates tests
(test_dsprites_gpu.py, ...) stay: they check agreement on the branch the oracle picks itself."""
import pytest
import torch

import gates
import step_util as U
from conftest import rel_err

pytestmark = pytest.mark.gpu


def _names(config, step):
    """-> (per-phase parameter names, zero-gradient sibling map) of a configuration's optimisers"""
    if config == "celeba":
        return U.grad_names(step), U.ZERO_GRAD
    if config in ("dsprites", "colored"):
        return U.dsprites_grad_names(step), U.DSPRITES_ZERO_GRAD
    if config == "mnist":
        return U.mnist_grad_names(step), U.MNIST_ZERO_GRAD
    return [["E." + n for n, _ in step.E.named_parameters()]], {}


def _grad_errors(config, step, phases, ref):
    """-> {(phase, name): tensor-normalised max error} of the per-phase gradients ``phases`` against ``ref``.
    A parameter gets a gradient in ``phases`` exactly when it gets one in ``ref`` (MNIST's E.noise_layer gets none)."""
    names, zero_grad = _names(config, step)
    out = {}
    for ph, nm in enumerate(names):
        og, rg = phases[ph]["grads"], ref["phases"][ph]["grads"]
        assert len(og) == len(rg) == len(nm), ph
        assert [g is None for g in og] == [g is None for g in rg], (ph, [n for n, g in zip(nm, rg) if g is None])
        keep = [i for i, g in enumerate(rg) if g is not None]
        errs = U.phase_errors([nm[i] for i in keep], [og[i] for i in keep], [rg[i] for i in keep], zero_grad)
        out.update({(ph, n): v[0] for n, v in errs.items()})
    return out


def _buffers(state, ref, keys, pick):
    """-> {(net, buffer): rel_err} of the buffers selected by ``pick`` of ``state`` against ``ref`` (both
    {net: state_dict}); BatchNorm batch counters must agree exactly"""
    out = {}
    for key in keys:
        if key not in ref:
            continue
        for k, v in ref[key].items():
            if pick(k):
                out[(key, k)] = rel_err(state[key][k], v)
            if "num_batches" in k:
                assert int(state[key][k]) == int(v), (key, k)
    return out


def _sn(k):
    return k.endswith("weight_u") or k.endswith("weight_v")


def _running(k):
    return "running" in k


def _check(config, out, tol, stock=None, sn_nets=("D", "E")):
    """every bound of a forced-gate step; ``stock`` = stock torch fp32's forced record (fp32 mode); ``sn_nets``: the
    networks whose spectral-norm u / v are compared with the oracle's -> worst values"""
    step, ref = out["step"], out["forced"][0]
    assert out["gates"] > 0 and out["flips"] <= 0.01 * out["gates"], (out["flips"], out["gates"])
    code_err = 0.0
    if "Epxy" in gates.NETS[config]:
        assert len(out["codes"]) == len(ref["codes"]) == 2
        code_err = max(U.tensor_err(a, b) for a, b in zip(out["codes"], ref["codes"]))
        assert code_err <= tol, code_err
    loss_err = 0.0
    for k, want in ref["losses"].items():
        e = abs(out["losses"][k] - want) / max(1.0, abs(want))
        assert e <= tol, (k, out["losses"][k], want)
        loss_err = max(loss_err, e)

    def bounds(ours, theirs):
        if stock is None:
            return {k: tol for k in ours}
        return {k: max(3.0 * theirs[k], 1e-5) for k in ours}

    grads = _grad_errors(config, step, out["ours"], ref)
    g_bound = bounds(grads, stock and _grad_errors(config, step, stock["phases"], ref))
    bad = {k: (v, g_bound[k]) for k, v in grads.items() if v > g_bound[k]}
    assert not bad, bad
    # spectral-norm u / v depend on fp32 weights only (never on activations): 1e-5 in both precisions
    ours = gates.net_states(step, config)
    sn = _buffers(ours, ref["state"], sn_nets, _sn)
    assert all(v <= 1e-5 for v in sn.values()), sn
    bn = _buffers(ours, ref["state"], ("G", "E"), _running)
    bn_bound = bounds(bn, stock and _buffers(stock["state"], ref["state"], ("G", "E"), _running))
    bad = {k: (v, bn_bound[k]) for k, v in bn.items() if v > bn_bound[k]}
    assert not bad, bad
    worst = max(grads, key=grads.get)
    return {"flips": out["flips"], "gates": out["gates"], "grad": grads[worst], "grad_at": worst, "loss": loss_err,
            "code": code_err, "sn": max(sn.values(), default=0.0), "bn": max(bn.values(), default=0.0)}


def _report(what, w):
    print(f"{what}: gate flips {w['flips']} of {w['gates']}; worst gradient error {w['grad']:.2e} at {w['grad_at']}, "
          f"loss {w['loss']:.1e}, Encoder_pxy code {w['code']:.1e}, spectral-norm u/v {w['sn']:.1e}, "
          f"BatchNorm running stats {w['bn']:.1e}")


@pytest.mark.parametrize("config,B", [("dsprites", 32), ("colored", 32), ("mnist", 64), ("pxy", 128),
                                      ("pxy_color", 128)])
def test_forced_step_bf16(cuda, config, B):
    out = gates.forced_step(config, cuda, B, "bf16")
    _report(f"{config} bf16 B={B}", _check(config, out, 2e-2))


@pytest.mark.parametrize("config,B", [("dsprites", 32), ("colored", 32), ("mnist", 16), ("pxy", 16),
                                      ("pxy_color", 16)])
def test_forced_step_fp32_relative_to_stock_fp32(cuda, config, B):
    out = gates.forced_step(config, cuda, B, "fp32", oracle_dtypes=(torch.float64, torch.float32))
    _report(f"{config} fp32 B={B}", _check(config, out, 2e-5, stock=out["forced"][1]))


@pytest.mark.parametrize("config,B", [("dsprites", 256), ("colored", 512)])
def test_forced_step_bf16_benchmarked_batch(cuda, config, B):
    """the batches bench.py runs (colored: its global batch on one device), against the oracle on the GPU in fp32
    (TF32 off; fp64 at this batch would only add minutes) on the gates of our run"""
    out = gates.forced_step(config, cuda, B, "bf16", oracle_dtypes=(torch.float32,))
    _report(f"{config} bf16 B={B}", _check(config, out, 2e-2))
