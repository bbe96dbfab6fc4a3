"""-m gpu: every configuration's whole step captured in a CUDA graph replays to the same results as eager execution."""
import os

import numpy as np
import pytest
import torch

import gates

pytestmark = pytest.mark.gpu

CONFIGS = ("celeba", "dsprites", "colored", "mnist", "pxy", "pxy_color")
BATCH = {"celeba": 16, "dsprites": 32, "colored": 32, "mnist": 64, "pxy": 128, "pxy_color": 128}


def _has_batchnorm(step, config):
    return any(isinstance(m, torch.nn.BatchNorm2d) for k in gates.NETS[config] for m in getattr(step, k).modules())


def _diffs(a, b):
    """-> {name: (max |a - b|, mean |a - b|)} over the networks' state and the Adam moments of two training_states;
    the Adam step mirrors must agree exactly"""
    out = {}
    for key, sd in a["nets"].items():
        for k, v in sd.items():
            w = b["nets"][key][k]
            if v.is_floating_point():
                d = (v.double() - w.double()).abs()
                out[f"{key}.{k}"] = (float(d.max()), float(d.mean()))
            else:
                assert torch.equal(v, w), (key, k)
    for name, per in a["opts"].items():
        for i, (s, t) in enumerate(zip(per, b["opts"][name])):
            assert (s is None) == (t is None), (name, i)
            if s is None:
                continue
            assert s["step"] == t["step"], (name, i, s["step"], t["step"])
            for k in ("exp_avg", "exp_avg_sq"):
                d = (s[k].double() - t[k].double()).abs()
                out[f"{name}.{i}.{k}"] = (float(d.max()), float(d.mean()))
    return out


def _adam_ratio(t, beta1=0.5, beta2=0.999):
    """a bound on |m^ / sqrt(v^)| of Adam at step t for ANY gradient sequence (Cauchy-Schwarz on the two moment sums:
    |sum a_i g_i| <= sqrt(sum a_i^2 / b_i) sqrt(sum b_i g_i^2)); 1 at t = 1, 1.33 at t = 5"""
    s = sum((beta1 ** 2 / beta2) ** k for k in range(t))
    return (1 - beta1) / (1 - beta1 ** t) * (s * (1 - beta2 ** t) / (1 - beta2)) ** 0.5


def _lr_sum(step):
    """the largest sum of learning rates over the optimisers that share one parameter"""
    total = {}
    for opt in step.optimizers():
        for grp in opt.param_groups:
            for p in grp["params"]:
                total[id(p)] = total.get(id(p), 0.0) + grp["lr"]
    return max(total.values())


@pytest.mark.parametrize("config", CONFIGS)
@pytest.mark.parametrize("prec", ["bf16", "fp32"])
def test_graphed_step_matches_eager(cuda, prec, config):
    """the graphed and the eager step object run in lockstep on the same batches; losses and the whole training state
    (weights, BatchNorm statistics and counters, spectral-norm u / v, Adam moments and step counts) are compared after
    every step"""
    os.environ["EADGAN_PRECISION"] = prec
    from eadgan_b200.graph import GraphedStep
    B, W, K = BATCH[config], 2, 3
    eager, graphed = gates.make_step(config, cuda), gates.make_step(config, cuda)
    # Sources of run-to-run nondeterminism.  The only float atomics the steps run are the fp64 atomics that sum the
    # BatchNorm statistics (csrc/bn.cu, the tcgen05 GEMM epilogue): the tcgen05 kernels use no other float atomics,
    # the SIMT split-K and wgrad sum their partials in a fixed order, the spectral-norm reductions are fixed-order, the
    # losses here fit one block each, and no step differentiates an image through the STN (whose backward atomics
    # are the only other ones).  Without BatchNorm (the Encoder_pxy steps) the two runs must be bitwise identical.
    exact = not _has_batchnorm(eager, config)
    gs = GraphedStep(graphed, gates.batch(config, cuda, B, 0)[0], warmup=W)    # W eager warm-up steps inside
    for _ in range(W):
        eager(*gates.batch(config, cuda, B, 0)[0])
    torch.cuda.synchronize()
    worst_loss, worst = 0.0, {}
    for i in range(1, K + 1):
        x = gates.batch(config, cuda, B, 10 + i)[0]
        le = {k: float(v) for k, v in eager(*x).items()}
        lg = {k: float(v) for k, v in gs(*x).items()}
        torch.cuda.synchronize()
        a, b = gates.training_state(eager, config), gates.training_state(graphed, config)
        d = _diffs(a, b)
        for k in le:
            worst_loss = max(worst_loss, abs(le[k] - lg[k]) / max(1.0, abs(le[k])))
        for k, v in d.items():
            worst[k] = max(worst.get(k, (0.0, 0.0)), v)
        if exact:
            assert le == lg, (i, le, lg)
            assert not {k: v for k, v in d.items() if v[0] != 0.0}, (i, {k: v for k, v in d.items() if v[0] != 0.0})
        else:
            # A different commit order of the fp64 atomics moves a BatchNorm sum by ~1e-16 relative; that is visible
            # only where it moves the fp32 mean / variance across a rounding boundary, by one fp32 ulp in one channel.
            # Losses then move at that rounding level (6e-8): bound 1e-6 in both precisions.  Smooth state moves at
            # the same level; what can move further is Adam's update of an element whose gradient is at the level of
            # that noise (at t = 1 the update is lr * sign(g)) and of the zero-gradient biases in front of a
            # BatchNorm, whose gradient is nothing but noise: at most twice the largest update per step, sum over
            # steps of 2 r_t lr (r_t below), capped at 6e-3 (what this test held CelebA to before).  Such elements are
            # few, so the mean stays at 2e-5 in both precisions.  Adam's moments follow the gradients themselves and
            # are compared bitwise above only; their step counts are compared exactly.
            for k in le:
                assert abs(le[k] - lg[k]) <= 1e-6 * max(1.0, abs(le[k])), (i, k, le, lg)
            bound = min(6e-3, 2 * _lr_sum(graphed) * sum(_adam_ratio(t) for t in range(1, W + i + 1)))
            for k, (mx, mean) in d.items():
                if k.startswith("opt"):
                    continue
                assert mx <= bound and mean <= 2e-5, (i, k, mx, mean, bound)
        # python-side step mirrors follow the device counter
        for opt in graphed.optimizers():
            steps = {opt.state[p]["step"] for p in gates.opt_params(opt) if opt.state.get(p)}
            assert steps == {W + i} and int(opt._step_dev) == W + i, (steps, int(opt._step_dev))
    top = sorted(worst.items(), key=lambda kv: -kv[1][0])[:4]
    print(f"{config} {prec}: {'bitwise' if exact else 'BatchNorm atomics'}; worst loss {worst_loss:.1e}; "
          f"worst state max/mean " + ", ".join(f"{k} {v[0]:.1e}/{v[1]:.1e}" for k, v in top))
    assert gs.kernels_per_replay > (100 if config == "celeba" else 10)


def test_prefetch_pipeline_gives_the_same_steps(cuda):
    """GraphedStep(..., prefetch=next batch): the next step's host->device copy runs on a copy stream during the
    current replay; results must equal feeding the same batches without the pipeline."""
    os.environ["EADGAN_PRECISION"] = "bf16"
    from eadgan_b200.graph import GraphedStep
    from eadgan_b200.steps.celeba import CelebAStep
    from oracle.torch_oracle import sample_celeba, synth_celeba_images
    B = 16

    def host_batch(i):
        d = sample_celeba(np.random.RandomState(20 + i), B)
        return [t.contiguous().pin_memory() for t in (synth_celeba_images(B, i), d["z"], d["code"], d["labels"])]

    batches = [host_batch(i) for i in range(4)]
    dev0 = [t.to(cuda) for t in batches[0]]
    plain = GraphedStep(CelebAStep(seed=0, device=cuda), dev0, warmup=1)
    piped = GraphedStep(CelebAStep(seed=0, device=cuda), dev0, warmup=1)
    for i in range(4):
        a = {k: float(v) for k, v in plain(*batches[i]).items()}
        b = {k: float(v) for k, v in piped(*batches[i], prefetch=batches[(i + 1) % 4]).items()}
        assert a == b, (i, a, b)
