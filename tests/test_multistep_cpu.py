"""Host-side check of the training-state transfer behind tests/test_multistep_gpu.py, on the CPU: our step objects and
the oracle's states (build_*) are only constructed, no kernel is launched.  A transfer that missed an optimiser, paired
parameters in a different order, or dropped a moment, a step count or a network buffer would start the oracle from a
state other than ours, and the multi-step tests would compare two different trainings."""
import pytest
import torch

import gates

CONFIGS = sorted(gates.NETS)


def _oracle(config, seed, dtype):
    from oracle import torch_oracle as O
    if config == "celeba":
        return O.build_celeba(seed=seed, dtype=dtype)
    if config in ("dsprites", "colored"):
        return O.build_dsprites(seed=seed, dtype=dtype, colored=config == "colored")
    if config == "mnist":
        return O.build_mnist(seed=seed, dtype=dtype)
    return O.build_pxy(seed=seed, dtype=dtype, colored=config == "pxy_color")


def _listing(holder, config, name):
    """[(qualified name, shape)] of an optimiser's parameters, in param_groups order"""
    member = holder[name] if isinstance(holder, dict) else getattr(holder, name)
    named = {id(p): f"{k}.{n}" for k in gates.NETS[config]
             for n, p in (holder[k] if isinstance(holder, dict) else getattr(holder, k)).named_parameters()}
    return [(named[id(p)], tuple(p.shape)) for p in gates.opt_params(member)]


@pytest.mark.parametrize("config", CONFIGS)
def test_optimisers_pair_up_parameter_by_parameter(config):
    """gates.OPTS names every optimiser of both sides; ours and the oracle's of the same name list parameters of equal
    qualified name and shape in the same order"""
    ours, st = gates.make_step(config, "cpu"), _oracle(config, 0, torch.float32)
    assert list(ours.optimizers()) == [getattr(ours, n) for n in gates.OPTS[config]]
    assert sorted(k for k in st if k.startswith("opt")) == sorted(gates.OPTS[config])
    for name in gates.OPTS[config]:
        mine, theirs = _listing(ours, config, name), _listing(st, config, name)
        assert mine and mine == theirs, (name, [(a, b) for a, b in zip(mine, theirs) if a != b][:3])


@pytest.mark.parametrize("config", CONFIGS)
def test_fabricated_training_state_survives_a_round_trip(config):
    """a fabricated training state (distinct step counts and moments per parameter, some parameters without state,
    perturbed weights and buffers) goes ours -> fp64 oracle -> a fresh step object of ours unchanged"""
    ours = gates.make_step(config, "cpu")
    gen = torch.Generator().manual_seed(7)
    for k in gates.NETS[config]:
        for v in getattr(ours, k).state_dict().values():
            if v.is_floating_point():
                v.add_(torch.randn(v.shape, generator=gen, dtype=v.dtype))
            else:
                v.add_(5)
    for j, name in enumerate(gates.OPTS[config]):
        opt = getattr(ours, name)
        for i, p in enumerate(gates.opt_params(opt)):
            if i % 3 == 1:
                continue                                 # no gradient yet: no state
            opt.state[p] = {"step": 2 + i + 10 * j, "exp_avg": torch.randn(p.shape, generator=gen),
                            "exp_avg_sq": torch.rand(p.shape, generator=gen)}
    a = gates.training_state(ours, config)

    st = _oracle(config, 1, torch.float64)
    gates.load_training_state(st, config, a)
    for name in gates.OPTS[config]:
        opt = st[name]
        for p, s in zip(gates.opt_params(opt), a["opts"][name]):
            assert p.dtype == torch.float64
            if s is None:
                assert p not in opt.state
            else:                                        # torch.optim.Adam's own layout: a tensor step count
                assert torch.is_tensor(opt.state[p]["step"]) and float(opt.state[p]["step"]) == s["step"]
                assert opt.state[p]["exp_avg"].dtype == torch.float64
    b = gates.training_state(st, config)

    back = gates.make_step(config, "cpu", seed=2)
    gates.load_training_state(back, config, b)
    c = gates.training_state(back, config)
    for key, sd in a["nets"].items():
        assert list(sd) == list(c["nets"][key])
        for k, v in sd.items():
            assert c["nets"][key][k].dtype == v.dtype and torch.equal(c["nets"][key][k], v), (key, k)
    for name, per in a["opts"].items():
        assert len(per) == len(c["opts"][name])
        for i, (s, t) in enumerate(zip(per, c["opts"][name])):
            assert (s is None) == (t is None), (name, i)
            if s is not None:
                assert type(t["step"]) is int and t["step"] == s["step"], (name, i)
                assert torch.equal(t["exp_avg"], s["exp_avg"]) and torch.equal(t["exp_avg_sq"], s["exp_avg_sq"])
