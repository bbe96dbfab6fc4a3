"""Host-side structure of the forced-gate harness (tests/gates.py), on the CPU: our networks and the oracle's are only
constructed (and the oracle's run once), no kernel is launched.  A harness that matched no Sequential, or an oracle
network that applied a ReLU / LeakyReLU where no ForcedGate can replace it, would force nothing and let the
forced-gate GPU tests pass on the oracle's own gates."""
import pytest
import torch
import torch.nn as tnn
from torch.overrides import TorchFunctionMode

import gates

CONFIGS = sorted(gates.NETS)


def _nets(config):
    """-> (our networks, the oracle's), {key: module} for the keys of gates.NETS[config]"""
    from oracle import torch_oracle as O
    if config == "celeba":
        from eadgan_b200.steps.celeba import CelebAStep
        ours, st = CelebAStep(seed=0, device="cpu"), O.build_celeba(seed=0)
    elif config in ("dsprites", "colored"):
        from eadgan_b200.steps.colored import ColoredDSpritesStep
        from eadgan_b200.steps.dsprites import DSpritesStep
        colored = config == "colored"
        step = ColoredDSpritesStep if colored else DSpritesStep
        ours = step(seed=0, device="cpu", pxy_state=O.dsprites_pxy_state(0, colored=colored))
        st = O.build_dsprites(seed=0, colored=colored)
    elif config == "mnist":
        from eadgan_b200.steps.mnist import MnistStep
        ours, st = MnistStep(seed=0, device="cpu", approximator_state=O.mnist_approximator_state(0)), O.build_mnist(seed=0)
    else:
        from eadgan_b200.steps.pxy import PxyStep
        colored = config == "pxy_color"
        ours, st = PxyStep(seed=0, device="cpu", colored=colored), O.build_pxy(seed=0, colored=colored)
    keys = gates.NETS[config]
    return {k: getattr(ours, k) for k in keys}, {k: st[k] for k in keys}


def _inputs(config, key, B=2):
    """a forward argument tuple of the oracle network ``key``"""
    ch = 3 if config in ("celeba", "colored", "pxy_color") else 1
    if config == "celeba":
        return (torch.randn(B, 200), torch.eye(10)[:B], torch.randn(B, 8)) if key == "G" else \
            (torch.randn(B, 3, 64, 64),)
    if config == "mnist":
        return {"A": (torch.randn(B, 6),), "G": (torch.randn(B, 62), torch.eye(10)[:B], torch.randn(B, 7))}.get(
            key, (torch.randn(B, 1, 32, 32),))
    if key == "G":
        return (torch.rand(B, 3 + (7 if config == "colored" else 4)),)
    return (torch.rand(B, ch, 64, 64),)


@pytest.mark.parametrize("config", CONFIGS)
def test_every_oracle_gate_has_a_logged_twin(config):
    """each oracle ReLU / LeakyReLU sits directly in a Sequential whose qualified name exists on our side, with the
    same number of gated stages there, and no Sequential of ours logs masks that no oracle gate would consume"""
    ours, ref = _nets(config)
    mods = {f"{key}.{name}": m for key, net in ref.items() for name, m in net.named_modules()}
    for qn, m in mods.items():
        if isinstance(m, gates.GATED):
            parent = qn.rsplit(".", 1)[0]
            assert isinstance(mods.get(parent), tnn.Sequential), qn
    theirs = {qn: n for qn, n in gates.oracle_gates(ref).items() if n}
    mine = {qn: n for qn, n in gates.our_gates(ours).items() if n}
    assert theirs and theirs == mine, (theirs, mine)
    if config == "celeba":
        assert theirs == {"G.conv_blocks": 3, "D.main": 4}


class _CountGates(TorchFunctionMode):
    """counts the ReLU-family functions applied, whichever module or function applies them"""

    def __init__(self):
        super().__init__()
        self.calls = 0

    def __torch_function__(self, func, types, args=(), kwargs=None):
        name = getattr(func, "__name__", "")
        if "relu" in name or "threshold" in name:
            self.calls += 1
        return func(*args, **(kwargs or {}))


@pytest.mark.parametrize("config", CONFIGS)
def test_no_oracle_gate_outside_a_sequential(config):
    """one forward of every oracle network applies exactly one ReLU-family function per call of a ReLU / LeakyReLU
    child of a Sequential: nothing a ForcedGate cannot reach (a functional relu in a forward, a gate module outside a
    Sequential) gates the oracle"""
    _, ref = _nets(config)
    torch.manual_seed(0)
    for key, net in ref.items():
        seen = []
        hooks = [m.register_forward_hook(lambda *a: seen.append(1))
                 for seq in gates.sequentials({key: net}).values() for m in seq.children()
                 if isinstance(m, gates.GATED)]
        count = _CountGates()
        with torch.no_grad(), count:
            net(*_inputs(config, key))
        for h in hooks:
            h.remove()
        assert seen and count.calls == len(seen), (key, count.calls, len(seen))
