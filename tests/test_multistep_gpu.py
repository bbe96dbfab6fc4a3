"""-m gpu: the training state one step hands to the next, held to the fp64 oracle for every configuration.

Every other oracle-refereed step test checks ONE step from the seeded initial state: Adam at t = 1 with zero moments,
and each phase restarted from the oracle's post-phase state (which also reloads u / v and drops every cached pack).
Here three production steps run first -- eagerly (CelebA in its deferred order), or as GraphedStep (one eager warm-up
step, then two replays) -- on three different seeded batches.  Their training state (weights, BatchNorm running
statistics and batch counters, spectral-norm u / v, every Adam moment and step count) is then snapshotted and step 4
runs through the forced-gate harness from that snapshot (tests/gates.py, ``start=``): our step object carries on with
whatever it holds (bf16 packs rebuilt after the last optimiser step, prefetched power iterations, frozen / trainable
flags), the oracle starts from the snapshot, and no phase is restarted -- from t = 2 on Adam's update is a smooth
function of the gradient.

Bounds are the project's existing rules (test_forced_steps_gpu.py ``_check``: every gradient tensor of every phase to
2e-2 in bf16, to max(3 x stock torch fp32's error, 1e-5) in fp32; gate flips <= 1 %; spectral-norm u / v to 1e-5;
BatchNorm running statistics to the gradient rule) or are derived below from Adam's formulas."""
import os

import pytest
import torch

import gates
from conftest import rel_err
from test_forced_steps_gpu import _check, _report

pytestmark = pytest.mark.gpu

CONFIGS = ("celeba", "dsprites", "colored", "mnist", "pxy", "pxy_color")
# the batches of test_step_gpu.py (CelebA) and test_forced_steps_gpu.py (the others)
BATCH = {"bf16": {"celeba": 16, "dsprites": 32, "colored": 32, "mnist": 64, "pxy": 128, "pxy_color": 128},
         "fp32": {"celeba": 8, "dsprites": 32, "colored": 32, "mnist": 16, "pxy": 16, "pxy_color": 16}}
K = 3                       # production steps before the refereed one

# Adam in fp32 against its formulas in fp64, from OUR recorded tensors (g = the phase's recorded gradient, m3 / v3 /
# p_before from the snapshot or the previous phase's params_after, m4 / v4 / p_after as our step left them).  u is the
# unit roundoff of fp32; every operation of adam_kernel is one correctly rounded fp32 operation (relative error <= u);
# beta1 = 0.5, so 1 - beta1 and 1 - (1 - beta1) are exact in fp32:
#   m4 = beta1 m3 + (1-beta1) g:  g - m3 rounded, then g - 0.5 (g - m3) rounded   -> |err| <= u (|g| + |m3|); bound 2u
#   v4 = beta2 v3 + (1-beta2) g^2:  beta2 and 1-beta2 rounded to fp32, 2 products into the first term, 3 into the
#        second, all terms >= 0, one final add                                   -> |err| <= 4u v4;  bound 5u v4
#   p_after = p_before - D,  D = lr/bc1 * m4 / (sqrt(v4)/sqrt(bc2) + eps):  lr/bc1, sqrt(bc2), eps rounded to fp32,
#        sqrt, divide, add eps (denominator <= 4u relative), product with lr/bc1 (2u), divide (u) -> D within 7u;
#        the final add rounds to u |p_after|                                     -> bound u (|p_ref| + 9 |D|)
# plus FLT_MIN everywhere for results in the subnormal range.
U32 = 2.0 ** -24
FLT_MIN = 2.0 ** -126


# forwards per step of each spectral-normalised network, each running one power iteration (eadgan_b200/steps):
# (on the weights the step starts from, after the network's own optimiser stepped it within the step).  Where the
# second count is 0, u / v depend on the snapshot alone and must match the oracle's to 1e-5.  Otherwise the last
# iterations run on weights that already carry one Adam update computed from OUR gradients -- bf16 ones differ from
# the oracle's by up to 2e-2, and so do the updates -- so their referee is the same power iteration in fp64 on our
# own start weights and our own recorded params_after, again to 1e-5.
SN_FORWARDS = {"celeba": {"D": (3, 3)}, "dsprites": {"D": (2, 1), "E": (3, 0)}, "colored": {"D": (2, 1), "E": (3, 0)},
               "mnist": {"D": (3, 0), "E": (3, 0)}, "pxy": {}, "pxy_color": {}}


def _sn_referee(config, step, start, rec):
    """-> {(net, buffer): rel_err} of our u / v after the step against fp64 power iterations (torch's legacy
    spectral_norm: v = normalize(W^T u), u = normalize(W v)) from the snapshot's u / v, on the snapshot's weights and
    then on the params_after of the first phase that stepped them, for the networks of SN_FORWARDS with forwards after
    that phase"""
    named = {id(p): (k, n) for k in gates.NETS[config] for n, p in getattr(step, k).named_parameters()}
    stepped = {}
    for r in rec:
        for p, a in zip(gates.opt_params(getattr(step, "opt_" + r["name"])), r["params_after"]):
            stepped.setdefault(named[id(p)], a)
    ours, out = gates.net_states(step, config), {}
    for key, (n0, n1) in SN_FORWARDS[config].items():
        if n1 == 0:
            continue
        sd = start["nets"][key]
        for k in [k for k in sd if k.endswith("weight_u")]:
            pre = k[:-len("weight_u")]
            u, v = sd[k].double(), sd[pre + "weight_v"].double()
            for w, n in ((sd[pre + "weight_orig"], n0), (stepped[(key, pre + "weight_orig")], n1)):
                mat = w.double().reshape(w.shape[0], -1)
                for _ in range(n):
                    v = torch.nn.functional.normalize(mat.t() @ u, dim=0, eps=1e-12)
                    u = torch.nn.functional.normalize(mat @ v, dim=0, eps=1e-12)
            out[(key, k)] = rel_err(ours[key][k], u)
            out[(key, pre + "weight_v")] = rel_err(ours[key][pre + "weight_v"], v)
    return out


def _no_prefetch_left(step, config):
    """every power iteration prefetched by a step was consumed by that step: a leftover queue entry means u / v
    advanced by an iteration that the reference never runs"""
    left = [f"{k}.{n}" for k in gates.NETS[config] for n, m in getattr(step, k).named_modules()
            if m.__dict__.get("_eadgan_sn_queue")]
    assert not left, left


def _counters(step, config, want, graph):
    """the python step mirror of every parameter with Adam state -- and, after graph replays, the device counter --
    equal ``want``; exactly the parameters that ever had a gradient have state"""
    for name in gates.OPTS[config]:
        opt = getattr(step, name)
        steps = [opt.state[p]["step"] for p in gates.opt_params(opt) if opt.state.get(p)]
        assert steps and all(s == want for s in steps), (name, sorted(set(steps)), want)
        if graph:
            assert int(opt._step_dev) == want, (name, int(opt._step_dev), want)


def _adam(config, step, start, rec):
    """-> worst (error / bound) of m4, v4 and p_after over every optimiser, parameter and element (see the table at
    the top); parameters without a gradient must be left bit-identical and without state"""
    named = {id(p): (k, n) for k in gates.NETS[config] for n, p in getattr(step, k).named_parameters()}
    cur = {}                    # parameter -> its value before the current phase, fp64
    for p in (p for name in gates.OPTS[config] for p in gates.opt_params(getattr(step, name))):
        k, n = named[id(p)]
        cur[id(p)] = start["nets"][k][n].double()
    worst = {"m": 0.0, "v": 0.0, "p": 0.0}
    assert [r["name"] for r in rec] == [name[4:] for name in gates.OPTS[config]], [r["name"] for r in rec]
    for r in rec:
        name = "opt_" + r["name"]
        opt = getattr(step, name)
        (group,) = opt.param_groups
        (b1, b2), lr, eps = group["betas"], group["lr"], group["eps"]
        assert b1 == 0.5, b1                    # the exactness the m4 bound relies on
        ps = gates.opt_params(opt)
        assert len(ps) == len(r["grads"]) == len(r["params_after"]) == len(start["opts"][name])
        for p, g, after, s0 in zip(ps, r["grads"], r["params_after"], start["opts"][name]):
            before = cur[id(p)]
            if g is None:
                assert s0 is None and not opt.state.get(p), (name, named[id(p)])
                assert torch.equal(after.double(), before), (name, named[id(p)])
                continue
            st = opt.state[p]
            t = s0["step"] + 1
            assert st["step"] == t == K + 1, (name, named[id(p)], st["step"])
            g, m3, v3 = g.double(), s0["exp_avg"].double(), s0["exp_avg_sq"].double()
            m4, v4 = st["exp_avg"].double(), st["exp_avg_sq"].double()
            em = (m4 - (b1 * m3 + (1 - b1) * g)).abs() / (2 * U32 * (g.abs() + m3.abs()) + FLT_MIN)
            v_ref = b2 * v3 + (1 - b2) * g * g
            ev = (v4 - v_ref).abs() / (5 * U32 * v_ref + FLT_MIN)
            d = lr / (1 - b1 ** t) * m4 / (v4.sqrt() / (1 - b2 ** t) ** 0.5 + eps)
            p_ref = before - d
            after = after.double()
            ep = (after - p_ref).abs() / (U32 * (p_ref.abs() + 9 * d.abs()) + FLT_MIN)
            for key, e in (("m", em), ("v", ev), ("p", ep)):
                worst[key] = max(worst[key], float(e.max()))
                assert float(e.max()) <= 1.0, (name, named[id(p)], key, float(e.max()))
            cur[id(p)] = after
    for p_id, want in cur.items():          # the last phase's params_after is what the networks hold
        k, n = named[p_id]
        assert torch.equal(dict(getattr(step, k).named_parameters())[n].double(), want), (k, n)
    return worst


@pytest.mark.parametrize("driver", ["eager", "graph"])
@pytest.mark.parametrize("prec", ["bf16", "fp32"])
@pytest.mark.parametrize("config", CONFIGS)
def test_forced_step_after_training(cuda, config, prec, driver):
    os.environ["EADGAN_PRECISION"] = prec
    B = BATCH[prec][config]
    step = gates.make_step(config, cuda)
    batches = [gates.batch(config, cuda, B, 1 + i)[0] for i in range(K)]
    if driver == "eager":
        for x in batches:
            step(*x)
            _no_prefetch_left(step, config)
    else:
        from eadgan_b200.graph import GraphedStep
        gs = GraphedStep(step, batches[0], warmup=1)        # step 1 runs eagerly inside, then the capture
        _no_prefetch_left(step, config)
        for x in batches[1:]:
            gs(*x)
            _no_prefetch_left(step, config)
    torch.cuda.synchronize()
    _counters(step, config, K, driver == "graph")
    start = gates.training_state(step, config)

    dts = (torch.float64,) if prec == "bf16" else (torch.float64, torch.float32)
    out = gates.forced_step(config, cuda, B, prec, oracle_dtypes=dts, start=start, ours=step, data_seed=K + 1)
    _no_prefetch_left(step, config)
    _counters(step, config, K + 1, driver == "graph")
    assert set(SN_FORWARDS[config]) == {k for k, sd in start["nets"].items() if any(n.endswith("_u") for n in sd)}
    direct = tuple(k for k, (_, n1) in SN_FORWARDS[config].items() if n1 == 0)
    w = _check(config, out, 2e-2 if prec == "bf16" else 2e-5, stock=out["forced"][1] if prec == "fp32" else None,
               sn_nets=direct)
    sn = _sn_referee(config, step, start, out["ours"])
    assert all(v <= 1e-5 for v in sn.values()), sn
    # a BatchNorm counts one batch per train-mode forward: the oracle's count over step 4 is the reference's number
    # of such forwards per step, ours must be K and K + 1 times it
    after = gates.net_states(step, config)
    for key, sd in start["nets"].items():
        for k, v in sd.items():
            if k.endswith("num_batches_tracked"):
                per_step = int(out["forced"][0]["state"][key][k]) - int(v)
                assert per_step > 0 and int(v) == K * per_step and int(after[key][k]) == (K + 1) * per_step, \
                    (key, k, int(v), per_step, int(after[key][k]))
    adam = _adam(config, step, start, out["ours"])
    _report(f"{config} {prec} {driver} B={B} step {K + 1}", w)
    print(f"  Adam error / bound: m {adam['m']:.2f}, v {adam['v']:.2f}, p {adam['p']:.2f}; spectral-norm u/v against "
          f"fp64 power iterations on our weights {max(sn.values(), default=0.0):.1e}")
