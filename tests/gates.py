"""Test helper: forced activation gates (VERDICT r01 "what's weak" 2; SURVEY.md section 7.3-1).

A ReLU / LeakyReLU network is piecewise linear in its parameters' gradients: a single gate that differs between
two evaluations (a pre-activation within rounding of 0) moves EVERY upstream gradient by a finite amount, whatever
the quality of the kernels.  To hold every gradient tensor of a bf16 tensor-core step to north_star's 2e-2, the
oracle is therefore evaluated on the SAME piecewise-linear branch as our run:

  1. our step runs with ``eadgan_b200.chain.gate_log`` switched on: every Sequential records, per ReLU / LeakyReLU
     stage and per call, the mask ``output > 0`` -- for a chain stack the very bits its fused backward kernels read;
  2. the oracle's ``nn.ReLU`` / ``nn.LeakyReLU`` modules are replaced by ``ForcedGate`` modules that consume the
     masks logged by the Sequential of the same qualified name (``G.conv_block``, ``D.fc1``, ``A.fc_block``, ...),
     in call order: y = where(mask, x, slope * x).  Where the oracle's own gate agrees (all but ~0.1 % of the
     elements) this IS ReLU / LeakyReLU; where it does not, |x| is within bf16 rounding of 0, so the forward value
     moves by less than one bf16 ulp of the activation scale.

The frozen Encoder_pxy of the dSprites steps sets the alignment grid of every real image; its code is forced too
(the oracle's own code is kept for comparison), so that a rounding-level difference of that code does not move the
sampled sprite edges under D and E.  What is left between the two runs is rounding of smooth arithmetic, which the
2e-2 bound is about."""
import os

import numpy as np
import torch
import torch.nn as tnn

GATED = (tnn.ReLU, tnn.LeakyReLU)

# the networks of each configuration's step, by attribute name (ours) == state key (oracle)
NETS = {"celeba": ("G", "D"), "dsprites": ("Epxy", "E", "D", "G"), "colored": ("Epxy", "E", "D", "G"),
        "mnist": ("A", "G", "D", "E"), "pxy": ("E",), "pxy_color": ("E",)}


class ForcedGate(tnn.Module):
    def __init__(self, slope, queue):
        super().__init__()
        self.slope, self.queue = float(slope), queue
        self.flips = 0
        self.total = 0

    def forward(self, x):
        mask = self.queue.pop(0)
        self.flips += int(((x > 0) != mask).sum())
        self.total += mask.numel()
        return torch.where(mask, x, x * self.slope)


def install(seq, queue):
    """replace every ReLU / LeakyReLU of the torch Sequential ``seq`` by a ForcedGate fed from ``queue``"""
    gates = []
    for name, m in list(seq._modules.items()):
        if isinstance(m, tnn.LeakyReLU):
            seq._modules[name] = ForcedGate(m.negative_slope, queue)
        elif isinstance(m, tnn.ReLU):
            seq._modules[name] = ForcedGate(0.0, queue)
        else:
            continue
        gates.append(seq._modules[name])
    return gates


def sequentials(nets):
    """{qualified name: Sequential} over ``nets`` = {key: module}, e.g. 'G.conv_block', 'D.fc1'"""
    return {f"{key}.{name}": m for key, net in nets.items() for name, m in net.named_modules()
            if isinstance(m, tnn.Sequential)}


def oracle_gates(nets):
    """{qualified name: number of ReLU / LeakyReLU children} of the oracle's Sequentials"""
    return {qn: sum(isinstance(m, GATED) for m in seq.children()) for qn, seq in sequentials(nets).items()}


def our_gates(nets):
    """{qualified name: number of gated stages} of our Sequentials: one logged mask per ReLU / LeakyReLU per call"""
    from eadgan_b200 import nn as enn
    from eadgan_b200._lib import ACT_LRELU, ACT_RELU
    return {qn: sum(isinstance(m, enn._Act) and m.act()[0] in (ACT_RELU, ACT_LRELU) for m in seq.children())
            for qn, seq in sequentials(nets).items()}


def make_step(config, dev, seed=0):
    """-> our step object of ``config``, with seeded weights (and the seeded frozen Encoder_pxy / approximator)"""
    from oracle import torch_oracle as O
    if config == "celeba":
        from eadgan_b200.steps.celeba import CelebAStep
        return CelebAStep(seed=seed, device=dev)
    if config in ("dsprites", "colored"):
        from eadgan_b200.steps.colored import ColoredDSpritesStep
        from eadgan_b200.steps.dsprites import DSpritesStep
        colored = config == "colored"
        return (ColoredDSpritesStep if colored else DSpritesStep)(
            seed=seed, device=dev, pxy_state=O.dsprites_pxy_state(seed, colored=colored))
    if config == "mnist":
        from eadgan_b200.steps.mnist import MnistStep
        return MnistStep(seed=seed, device=dev, approximator_state=O.mnist_approximator_state(seed))
    if config in ("pxy", "pxy_color"):
        from eadgan_b200.steps.pxy import PxyStep
        return PxyStep(seed=seed, device=dev, colored=config == "pxy_color")
    raise ValueError(config)


def batch(config, dev, B, seed):
    """-> (our step's positional inputs, the oracle's (images, draws)) of one seeded batch of ``config``"""
    from oracle import torch_oracle as O
    rs = np.random.RandomState(seed)
    if config == "celeba":
        imgs, d = O.synth_celeba_images(B, seed).to(dev), O.sample_celeba(rs, B)
        return (imgs, d["z"].to(dev), d["code"].to(dev), d["labels"].to(dev)), (imgs, d)
    if config in ("dsprites", "colored"):
        imgs = O.synth_dsprites_images(B, seed).to(dev)
        d = O.sample_colored(rs, B) if config == "colored" else O.sample_dsprites(rs, B)
        extra = (d["color"].to(dev),) if config == "colored" else ()
        return (imgs, *extra, d["code_d"].to(dev), d["labels_d"].to(dev), d["code_info"].to(dev),
                d["labels_info"].to(dev)), (imgs, d)
    if config == "mnist":
        imgs, d = O.synth_mnist_images(B, seed).to(dev), O.sample_mnist(rs, B)
        return (imgs, d["z"].to(dev), d["code"].to(dev), d["labels"].to(dev)), (imgs, d)
    if config in ("pxy", "pxy_color"):
        imgs, d = O.synth_dsprites_images(B, seed).to(dev), O.sample_pxy(rs, B, config == "pxy_color")
        extra = (d["color"].to(dev),) if config == "pxy_color" else ()
        return (imgs, d["code"].to(dev), *extra), (imgs, d)
    raise ValueError(config)


def _setup(config, dev, B, seed, data_seed):
    """-> (build(dtype) -> oracle state, run_oracle(st, dtype, after_phase) -> record, our step,
    run_ours(step, record, after_phase) -> losses, the phases after which both runs restart from the free oracle)"""
    from oracle import torch_oracle as O
    args, (imgs, d) = batch(config, dev, B, data_seed)
    if config == "celeba":
        return (lambda dt: O.build_celeba(seed=seed, device=dev, dtype=dt),
                lambda st, dt, after: O.step_celeba(st, imgs.to(dt), d, after_phase=after),
                lambda ours, rec, after: ours(*args, record=rec, after_phase=after), (0, 1))
    if config in ("dsprites", "colored"):
        colored = config == "colored"
        step_fn = O.step_colored if colored else O.step_dsprites
        return (lambda dt: O.build_dsprites(seed=seed, device=dev, dtype=dt, colored=colored),
                lambda st, dt, after: step_fn(st, imgs, d, after_phase=after),
                lambda ours, rec, after: ours(*args, record=rec, after_phase=after), (0,))
    if config == "mnist":
        return (lambda dt: O.build_mnist(seed=seed, device=dev, dtype=dt),
                lambda st, dt, after: O.step_mnist(st, imgs, d, after_phase=after),
                lambda ours, rec, after: ours(*args, record=rec, after_phase=after), (0, 1))
    if config in ("pxy", "pxy_color"):
        colored = config == "pxy_color"
        return (lambda dt: O.build_pxy(seed=seed, device=dev, dtype=dt, colored=colored),
                lambda st, dt, after: O.step_pxy(st, imgs, d),
                lambda ours, rec, after: ours(*args, record=rec), ())
    raise ValueError(config)


def _cast(sd, dt):
    return {k: v.to(dt) if v.is_floating_point() else v for k, v in sd.items()}


def _state(nets):
    return {key: {k: v.detach().clone() for k, v in net.state_dict().items()} for key, net in nets.items()}


def net_states(step, config):
    """{net: state_dict} of our step's networks, keyed as the forced records' ``state``"""
    return _state({k: getattr(step, k) for k in NETS[config]})


# the optimisers of each configuration's step, by attribute name (ours) == state key (oracle)
OPTS = {"celeba": ("opt_G", "opt_D", "opt_info"), "dsprites": ("opt_D", "opt_info"), "colored": ("opt_D", "opt_info"),
        "mnist": ("opt_G", "opt_D", "opt_info"), "pxy": ("opt_E",), "pxy_color": ("opt_E",)}


def _member(holder, key):
    """a network / optimiser of our step object (attribute) or of an oracle state (build_*: dict entry)"""
    return holder[key] if isinstance(holder, dict) else getattr(holder, key)


def opt_params(opt):
    return [p for g in opt.param_groups for p in g["params"]]


def training_state(step, config):
    """-> {"nets": {net: state_dict}, "opts": {optimiser: [per parameter in param_groups order: None (no state yet)
    or {"step": int, "exp_avg", "exp_avg_sq"}]}}: a copy of everything one training step hands to the next, taken from
    our step object or from an oracle state (build_*)"""
    opts = {}
    for name in OPTS[config]:
        opt = _member(step, name)
        per = []
        for p in opt_params(opt):
            s = opt.state.get(p)
            per.append({"step": int(s["step"]), "exp_avg": s["exp_avg"].detach().clone(),
                        "exp_avg_sq": s["exp_avg_sq"].detach().clone()} if s else None)
        opts[name] = per
    return {"nets": _state({k: _member(step, k) for k in NETS[config]}), "opts": opts}


def load_training_state(step, config, state):
    """put ``state`` (training_state) into our step object or an oracle state (build_*), floating-point tensors cast to
    the receiving parameters' dtype.  torch.optim.Adam keeps ``step`` as a tensor, our Adam as an int; a parameter
    without state is left without state (it has not had a gradient yet: MNIST's E.noise_layer never gets one)."""
    for key, sd in state["nets"].items():
        net = _member(step, key)
        net.load_state_dict(_cast(sd, next(net.parameters()).dtype))
    for name, per in state["opts"].items():
        opt = _member(step, name)
        ps = opt_params(opt)
        assert len(ps) == len(per), (name, len(ps), len(per))
        for p, s in zip(ps, per):
            opt.state.pop(p, None)
            if s is None:
                continue
            assert s["exp_avg"].shape == s["exp_avg_sq"].shape == p.shape, (name, tuple(p.shape))
            opt.state[p] = {"step": torch.tensor(float(s["step"])) if isinstance(opt, torch.optim.Adam) else s["step"],
                            "exp_avg": s["exp_avg"].to(p.device, p.dtype).clone(memory_format=torch.contiguous_format),
                            "exp_avg_sq": s["exp_avg_sq"].to(p.device, p.dtype).clone(
                                memory_format=torch.contiguous_format)}


def forced_step(config, dev, B, precision="bf16", seed=0, oracle_dtypes=(torch.float64,), start=None, ours=None,
                data_seed=None):
    """-> dict(forced=[oracle record per dtype in ``oracle_dtypes``], ours=our per-phase record, losses=our losses,
    free=free oracle record (first dtype; None with ``start``), flips=..., gates=..., step=our step object,
    codes=[our Encoder_pxy outputs]).  Each forced record also carries ``state`` (its nets' state after the step) and,
    for the dSprites configurations, ``codes`` (the oracle's own Encoder_pxy outputs on the forced gates).

    Runs on identical seeded inputs (batch ``data_seed``, default ``seed``) and weights: the free oracle (its
    post-phase states are the common starting point of every later phase of every run), OUR step (gates logged), then
    the oracle with OUR gates -- and our Encoder_pxy code -- forced, once per requested dtype (fp64 = the referee;
    fp32 = stock torch's own rounding error on the same branch).

    ``start`` (training_state): both runs begin from that training state instead of the seeded initial one, and no
    phase is restarted.  Restarts exist because Adam's first update, at t = 1 with zero moments, is lr * sign(g):
    a gradient element at rounding level of 0 moves its weight by a full step either way.  From t = 2 on the update
    m^/(sqrt(v^)+eps) is a smooth function of the gradient, so the phases may run on as the step runs them.  (The
    zero-gradient biases of the ZERO_GRAD maps are still noise-driven, but the train-mode BatchNorm right after each
    removes their update exactly.)  ``ours``: a step object to run instead of a freshly seeded one -- with ``start``
    it is NOT reloaded (``start`` must be its own training_state), so the bf16 packs, prefetched spectral-norm results
    and frozen / trainable flags it carries over from its earlier steps are what this step runs on."""
    from eadgan_b200 import chain
    os.environ["EADGAN_PRECISION"] = precision
    build, run_oracle, run_ours, restarts = _setup(config, dev, B, seed, seed if data_seed is None else data_seed)
    if ours is None:
        ours = make_step(config, dev, seed)
        if start is not None:
            load_training_state(ours, config, start)
    keys = NETS[config]
    dt0 = oracle_dtypes[0]

    def build_from(dt):
        st = build(dt)
        if start is not None:
            load_training_state(st, config, start)
        return st

    free = None if start is not None else run_oracle(build(dt0), dt0, None)
    states = {i: free["phases"][i]["state_after"] for i in restarts} if free is not None else {}

    def restart(nets, dt):
        def after_phase(i):
            if i in states:
                for key, sd in states[i].items():
                    nets[key].load_state_dict(_cast(sd, dt))
        return after_phase

    our_nets = {k: getattr(ours, k) for k in keys}
    codes = []
    hooks = [ours.Epxy.register_forward_hook(lambda m, a, out: codes.append(out.detach().clone()))] \
        if "Epxy" in keys else []
    rec = []
    chain.gate_log = []
    try:
        losses = run_ours(ours, rec, restart(our_nets, torch.float32))
        log = chain.gate_log
    finally:
        chain.gate_log = None
        for h in hooks:
            h.remove()
    names = {id(seq): qn for qn, seq in sequentials(our_nets).items()}
    masks = {}
    for seq, ms in log:
        masks.setdefault(names[id(seq)], []).extend(ms)

    forced, flips, total = [], 0, 0
    for dt in oracle_dtypes:
        st = build_from(dt)
        nets = {k: st[k] for k in keys}
        queues = {qn: list(ms) for qn, ms in masks.items()}
        gates = []
        for qn, seq in sequentials(nets).items():
            gates += install(seq, queues.setdefault(qn, []))
        assert not [m for net in nets.values() for m in net.modules() if isinstance(m, GATED)], "unforced gate"
        own, code_q = [], list(codes)
        if "Epxy" in keys:
            def force_code(m, a, out, _dt=dt):
                own.append(out.detach().clone())
                return code_q.pop(0).to(_dt)
            st["Epxy"].register_forward_hook(force_code)
        r = run_oracle(st, dt, restart(nets, dt))
        assert not any(queues.values()), {qn: len(q) for qn, q in queues.items() if q}
        assert not code_q
        r["state"], r["codes"] = _state(nets), own
        r["flips"], r["gates"] = sum(g.flips for g in gates), sum(g.total for g in gates)
        if dt == dt0:
            flips, total = r["flips"], r["gates"]
        forced.append(r)
        del st, nets
    return {"forced": forced, "ours": rec, "losses": {k: float(v) for k, v in losses.items()}, "free": free,
            "flips": flips, "gates": total, "step": ours, "codes": codes}


def celeba_forced(dev, B, precision="bf16", seed=0, oracle_dtypes=(torch.float64,)):
    """the CelebA step of ``forced_step`` (bench.py's parity block calls it by this name)"""
    return forced_step("celeba", dev, B, precision, seed, oracle_dtypes)
