"""-m gpu: BatchNorm2d in eval mode, forward and backward, on the bf16 chain and on the fp32 per-operator path.

``EVAL_STAGES`` are the BatchNorm-bearing entries of tests/test_chain_stages_gpu.py plus a tensor-core Conv2d and a thin
Conv2d in front of a BatchNorm.  Each runs with every BatchNorm in eval mode (random running statistics, gamma and beta)
through the chain with its gates logged, and through the fp64 referee of tests/bf16_emul.py with the same gates forced:
output, input gradient and every parameter gradient within STAGE_MAX.  The conv bias in front of an eval BatchNorm has a
real gradient (gamma * rsqrt(running_var + eps) * sum dz) and is compared like any other tensor.  The running statistics
and num_batches_tracked must not move."""
import copy
import os

import pytest
import torch

from conftest import rel_err
from test_chain_stages_gpu import SAME_MAX, STAGE_MAX, STAGES, _zero_grad_biases, build

pytestmark = pytest.mark.gpu

EVAL_STAGES = [e for e in STAGES if any(it[0] == "bn" for it in e[1])] + [
    # tensor-core Conv2d (fprop forward, dgrad input gradient) + BatchNorm(128, nhwc8) + LeakyReLU
    ("tc_conv_bn128_lrelu", [("conv", 32, 128, 4, 2, 1), ("bn", 128), ("lrelu", 0.2), ("conv", 128, 32, 4, 2, 1)],
     (5, 32, 16, 16)),
    # thin Conv2d on the image + BatchNorm(64) + ReLU, then a tc conv without a bias
    ("thin_conv_bn64_relu", [("conv", 3, 64, 4, 2, 1), ("bn", 64), ("relu",), ("conv", 64, 64, 4, 2, 1, False)],
     (3, 3, 32, 32)),
]
EVAL_IDS = [name for name, _, _ in EVAL_STAGES]


def _randomise_bn(seq, gen):
    for m in seq.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            c = m.num_features
            m.running_mean.copy_(torch.randn(c, generator=gen) * 0.3)
            m.running_var.copy_(torch.rand(c, generator=gen) + 0.5)
            m.weight.data.copy_(torch.rand(c, generator=gen) + 0.5)
            m.bias.data.copy_(torch.randn(c, generator=gen) * 0.2)


def _set_modes(seq, train_idx):
    """every BatchNorm of ``seq`` in eval mode except those at the Sequential positions in ``train_idx``"""
    for i, m in enumerate(seq._modules.values()):
        if isinstance(m, torch.nn.BatchNorm2d):
            m.train(i in train_idx)


def _run(ours, x, go, names):
    from eadgan_b200 import chain
    chain.gate_log = []
    try:
        xo = x.clone().requires_grad_()
        yo = ours(xo)
        log = chain.gate_log
    finally:
        chain.gate_log = None
    assert len(log) == 1 and log[0][0] is ours, "the stack did not run through the chain executor"
    params = [p for _, p in ours.named_parameters()]
    gs = torch.autograd.grad(yo, [xo] + params, go)
    return yo, dict(zip(names, gs)), log[0][1]


def run_eval_entry(spec, shape, dev, seed=0, train_idx=()):
    """-> ({tensor: error against the fp64 referee}, {tensor: error of the frozen / no-input-gradient runs against the
    full run}, {buffer: bit-identical before and after})"""
    import eadgan_b200.nn as enn
    import bf16_emul
    os.environ["EADGAN_PRECISION"] = "bf16"
    torch.manual_seed(seed)
    gen = torch.Generator().manual_seed(seed + 100)
    ours = build(enn, spec)
    _randomise_bn(ours, gen)
    ours = ours.to(dev)
    ref = build(torch.nn, spec).to(dev).double()
    ref.load_state_dict(ours.state_dict())
    _set_modes(ours, train_idx)
    _set_modes(ref, train_idx)
    sd0 = copy.deepcopy(ours.state_dict())
    x = torch.randn(*shape, device=dev)
    names = ["x"] + [n for n, _ in ours.named_parameters()]

    from eadgan_b200 import chain
    out_shape = chain._plan_kernels(chain._plan(ours), tuple(shape))[-1].out_shape
    go = torch.randn(*out_shape, device=dev)
    yo, gso, gates = _run(ours, x, go, names)
    after = ours.state_dict()
    unchanged = {}
    for i, m in enumerate(spec):
        if m[0] == "bn" and i not in train_idx:
            for b in ("running_mean", "running_var", "num_batches_tracked"):
                unchanged[f"{i}.{b}"] = torch.equal(after[f"{i}.{b}"], sd0[f"{i}.{b}"])

    xe = x.double().requires_grad_()
    ye = bf16_emul.emulate(ours, ref, xe, update_running=True, gates=gates, round_grads=True, sn_epilogue=True)
    gse = torch.autograd.grad(ye, [xe] + [p for _, p in ref.named_parameters()], go.double())
    errs = {"y": rel_err(yo, ye)}
    ref_g = dict(zip(names, gse))
    # a conv bias in front of a TRAINING-mode BatchNorm has a mathematically zero gradient: measured against its
    # sibling weight gradient, as tests/test_chain_stages_gpu.py does.  In front of an eval-mode one it is a real value.
    zero = {n: w for n, w in _zero_grad_biases(spec).items() if int(n.split(".")[0]) + 1 in train_idx}
    for n, b in zip(names, gse):
        a = gso[n]
        assert a is not None and a.shape == b.shape, n
        errs["d" + n] = (float((a.double() - b).abs().max()) / float(ref_g[zero[n]].abs().max()) if n in zero
                         else rel_err(a, b))
    sd_r = ref.state_dict()
    for i in train_idx:
        for b in ("running_mean", "running_var"):
            errs[f"{i}.{b}"] = rel_err(after[f"{i}.{b}"], sd_r[f"{i}.{b}"])

    same = {}
    ours.load_state_dict(sd0)
    chain.set_trainable(ours, False)
    try:
        x2 = x.clone().requires_grad_()
        y2 = ours(x2)
        y2.backward(go)
        same["y|frozen"] = rel_err(y2, yo)
        same["dx|frozen"] = rel_err(x2.grad, gso["x"])
        assert all(p.grad is None for p in ours.parameters()), "a frozen parameter received a gradient"
    finally:
        chain.set_trainable(ours, True)
    ours.load_state_dict(sd0)
    x3 = x.clone()
    y3 = ours(x3)
    y3.backward(go)
    assert x3.grad is None
    same["y|no_dx"] = rel_err(y3, yo)
    for n, p in ours.named_parameters():
        assert p.grad is not None, n
        same[f"d{n}|no_dx"] = (float((p.grad - gso[n]).abs().max()) / float(gso[zero[n]].abs().max()) if n in zero
                               else rel_err(p.grad, gso[n]))
    return errs, same, unchanged


# The stage catalogue's bound.  Worst max-normalised error per entry measured on a B200 (1000 W), seed 0:
# dense_T_bn64_c3last 1.8e-4, bn64_tanh_thinT_c3k64 5.6e-4, bn96_lrelu_fprop_mask 9.6e-4, bn384_c16last 3.6e-4,
# c16first_sigmoid_bn 9.6e-4, simt16_bn_to_tc 3.2e-7, tc_conv_bn128_lrelu 2.1e-6, thin_conv_bn64_relu 8.0e-7.
# CelebA generator inversion on forced gates: worst tensor 5.5e-3 at B = 16 and at B = 1024.
EVAL_MAX = STAGE_MAX


@pytest.mark.parametrize("name,spec,shape", EVAL_STAGES, ids=EVAL_IDS)
def test_eval_stage_against_fp64_referee(cuda, name, spec, shape):
    errs, same, unchanged = run_eval_entry(spec, shape, cuda)
    print(name, "worst", max(errs.values()))
    bad = {k: v for k, v in errs.items() if not v <= EVAL_MAX}
    assert not bad, (name, bad)
    bad = {k: v for k, v in same.items() if not v <= SAME_MAX}
    assert not bad, (name, bad)
    assert unchanged and all(unchanged.values()), (name, unchanged)


def test_mixed_train_and_eval_batchnorm_in_one_stack(cuda):
    """BatchNorm(64) at position 1 in training mode, BatchNorm(96) at position 4 in eval mode"""
    spec = [("convT", 64, 64, 4, 2, 1), ("bn", 64), ("relu",), ("convT", 64, 96, 4, 2, 1), ("bn", 96), ("lrelu", 0.2),
            ("conv", 96, 32, 4, 2, 1)]
    errs, same, unchanged = run_eval_entry(spec, (4, 64, 4, 4), cuda, train_idx=(1,))
    assert "1.running_mean" in errs and "4.running_mean" not in errs
    bad = {k: v for k, v in errs.items() if not v <= EVAL_MAX}
    assert not bad, bad
    bad = {k: v for k, v in same.items() if not v <= SAME_MAX}
    assert not bad, bad
    assert set(unchanged) == {"4.running_mean", "4.running_var", "4.num_batches_tracked"} and all(unchanged.values())


def test_mode_toggle_between_forward_and_backward(cuda):
    """the backward follows the forward's plan: .train() after an eval forward changes no gradient bit"""
    import eadgan_b200.nn as enn
    os.environ["EADGAN_PRECISION"] = "bf16"
    spec = [("convT", 64, 128, 4, 2, 1), ("bn", 128), ("relu",), ("convT", 128, 96, 4, 2, 1), ("bn", 96), ("tanh",),
            ("conv", 96, 32, 4, 2, 1)]
    torch.manual_seed(3)
    seq = build(enn, spec)
    _randomise_bn(seq, torch.Generator().manual_seed(3))
    seq = seq.to(cuda).eval()
    x = torch.randn(4, 64, 8, 8, device=cuda)
    sd0 = copy.deepcopy(seq.state_dict())
    params = list(seq.parameters())
    grads = []
    for toggle in (False, True):
        seq.eval()
        xo = x.clone().requires_grad_()
        y = seq(xo)
        if toggle:
            seq.train()
        go = torch.ones_like(y)
        grads.append(torch.autograd.grad(y, [xo] + params, go))
        seq.eval()
        for k, v in seq.state_dict().items():
            assert torch.equal(v, sd0[k]), k
    for a, b in zip(*grads):
        assert torch.equal(a, b)


def _celeba_inputs(B, dev, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    z = torch.randn(B, 200, generator=g).to(dev)
    lab = torch.eye(10)[torch.randint(0, 10, (B,), generator=g)].to(dev)
    code = (torch.rand(B, 8, generator=g) * 2 - 1).to(dev)
    target = (torch.rand(B, 3, 64, 64, generator=g) * 2 - 1).to(dev)
    return z, lab, code, target


def _celeba_eval_pair(dev, seed):
    from eadgan_b200.steps import celeba as CS
    from oracle import torch_oracle as O
    torch.manual_seed(seed)
    ref = O.CelebAGenerator()
    _randomise_bn(ref, torch.Generator().manual_seed(seed))
    ref = ref.to(dev)
    ours = CS.Generator().to(dev)
    ours.load_state_dict(ref.state_dict())
    return ours.eval(), ref.eval()


@pytest.mark.parametrize("B", [16, 1024])
def test_celeba_generator_inversion_gradients(cuda, B):
    """latent-space projection through a frozen-statistics generator: MSE(G(z, lab, code), target) differentiated
    w.r.t. z, code and every parameter of G, against the fp64 oracle on our forced gates"""
    import eadgan_b200.nn as enn
    from eadgan_b200 import chain
    import gates as GT
    os.environ["EADGAN_PRECISION"] = "bf16"
    ours, ref = _celeba_eval_pair(cuda, 5)
    sd0 = {k: v.clone() for k, v in ours.state_dict().items()}
    z, lab, code, target = _celeba_inputs(B, cuda, 5)
    zo, co = z.clone().requires_grad_(), code.clone().requires_grad_()
    chain.gate_log = []
    try:
        loss = enn.MSELoss()(ours(zo, lab, co), target)
        log = chain.gate_log
    finally:
        chain.gate_log = None
    assert len(log) == 1 and log[0][0] is ours.conv_blocks and len(log[0][1]) == 3, "G did not run through the chain"
    names = ["z", "code"] + [n for n, _ in ours.named_parameters()]
    go = torch.autograd.grad(loss, [zo, co] + [p for _, p in ours.named_parameters()])
    assert all(torch.equal(v, sd0[k]) for k, v in ours.state_dict().items())

    ref = ref.double()
    queue = list(log[0][1])
    GT.install(ref.conv_blocks, queue)
    zr, cr = z.double().requires_grad_(), code.double().requires_grad_()
    lr = torch.nn.functional.mse_loss(ref(zr, lab.double(), cr), target.double())
    gr = torch.autograd.grad(lr, [zr, cr] + [p for _, p in ref.named_parameters()])
    assert not queue
    errs = {n: rel_err(a, b) for n, a, b in zip(names, go, gr)}
    print("B", B, "worst", max(errs.values()), errs)
    bad = {k: v for k, v in errs.items() if not v <= 2e-2}
    assert not bad, bad


def test_celeba_generator_eval_forward_b1024_matches_fp32(cuda):
    ours, _ = _celeba_eval_pair(cuda, 6)
    z, lab, code, _ = _celeba_inputs(1024, cuda, 6)
    outs = {}
    for prec in ("bf16", "fp32"):
        os.environ["EADGAN_PRECISION"] = prec
        with torch.no_grad():
            outs[prec] = ours(z, lab, code)
    os.environ["EADGAN_PRECISION"] = "bf16"
    err = rel_err(outs["bf16"], outs["fp32"])
    print("bf16 vs fp32 eval forward, B = 1024:", err)
    assert err <= 2e-2


def _per_op_ok(ours, ref64, stock32):
    """DESIGN section 2, per operator: within 1e-5 of fp64, or within 2x stock fp32's own error"""
    e, s = rel_err(ours, ref64), rel_err(stock32, ref64)
    return e <= 1e-5 or e <= 2 * s, (e, s)


@pytest.mark.parametrize("shape", [(4, 16, 8, 8), (32, 64, 1, 1)], ids=["nchw", "n_c_1_1"])
@pytest.mark.parametrize("act", ["none", "relu", "lrelu", "tanh"])
def test_fp32_per_op_eval_batchnorm_backward(cuda, shape, act):
    import torch.nn.functional as TF
    from eadgan_b200 import functional as Fn
    from eadgan_b200._lib import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_TANH
    kind, slope = {"none": (ACT_NONE, 0.0), "relu": (ACT_RELU, 0.0), "lrelu": (ACT_LRELU, 0.2),
                   "tanh": (ACT_TANH, 0.0)}[act]
    torch.manual_seed(7)
    c = shape[1]
    x = torch.randn(*shape, device=cuda)
    gamma, beta = torch.rand(c, device=cuda) + 0.5, torch.randn(c, device=cuda) * 0.2
    rm, rv = torch.randn(c, device=cuda) * 0.3, torch.rand(c, device=cuda) + 0.5
    go = torch.randn(*shape, device=cuda)
    rm0, rv0 = rm.clone(), rv.clone()

    def torch_bn(dt):
        xs, gs, bs = (t.to(dt).requires_grad_() for t in (x, gamma, beta))
        y = TF.batch_norm(xs, rm.to(dt), rv.to(dt), gs, bs, training=False, momentum=0.1, eps=1e-5)
        y = {"none": lambda v: v, "relu": torch.relu, "lrelu": lambda v: TF.leaky_relu(v, 0.2),
             "tanh": torch.tanh}[act](y)
        return (y,) + torch.autograd.grad(y, [xs, gs, bs], go.to(dt))

    xs, gs, bs = (t.clone().requires_grad_() for t in (x, gamma, beta))
    y = Fn.batch_norm(xs, gs, bs, rm, rv, False, 0.1, 1e-5, kind, slope)
    ours = (y,) + torch.autograd.grad(y, [xs, gs, bs], go)
    ref, stock = torch_bn(torch.float64), torch_bn(torch.float32)
    for name, a, b, s in zip(("y", "dx", "dgamma", "dbeta"), ours, ref, stock):
        ok, es = _per_op_ok(a, b, s)
        assert ok, (name, es)
    assert torch.equal(rm, rm0) and torch.equal(rv, rv0)


def test_mnist_generator_eval_gradients_per_op(cuda):
    """the MNIST generator (Upsample + 3x3 convs: the per-operator path in both precision modes) in eval mode"""
    from eadgan_b200.steps import mnist as M
    from oracle import torch_oracle as O
    os.environ["EADGAN_PRECISION"] = "fp32"
    try:
        torch.manual_seed(8)
        ref = O.MnistGenerator()
        ref.apply(O.mnist_weights_init_normal)
        _randomise_bn(ref, torch.Generator().manual_seed(8))
        ref = ref.to(cuda)
        ours = M.Generator().to(cuda)
        ours.load_state_dict(ref.state_dict())
        ours.eval(), ref.eval()
        z = torch.randn(16, 62, device=cuda)
        lab = torch.eye(10, device=cuda)[torch.randint(0, 10, (16,), device=cuda)]
        code = torch.rand(16, 7, device=cuda) * 2 - 1
        go = torch.randn(16, 1, 32, 32, device=cuda)

        def grads(net, dt):
            zz, cc = z.to(dt).requires_grad_(), code.to(dt).requires_grad_()
            y = net(zz, lab.to(dt), cc)
            return [y] + list(torch.autograd.grad(y, [zz, cc] + list(net.parameters()), go.to(dt)))

        mine = grads(ours, torch.float32)
        stock = grads(ref, torch.float32)
        r64 = copy.deepcopy(ref).double()
        full = grads(r64, torch.float64)
        names = ["y", "z", "code"] + [n for n, _ in ours.named_parameters()]
        bad = {}
        for n, a, b, s in zip(names, mine, full, stock):
            ok, es = _per_op_ok(a, b, s)
            if not ok:
                bad[n] = es
        assert not bad, bad
    finally:
        os.environ["EADGAN_PRECISION"] = "bf16"


def _padded(n, h, w, c, dev, fill=None):
    from eadgan_b200 import tc
    t = tc.alloc_padded(n, h, w, c, dev)
    if fill is not None:
        tc.interior(t).copy_(fill)
    return t


@pytest.mark.parametrize("c", [64, 128, 96, 384])
@pytest.mark.parametrize("act", ["relu", "tanh", "none"])
def test_eval_bwd_kernel_in_place_and_write_bounds(cuda, c, act):
    """eadgan_bn_eval_bwd on padded bf16 buffers (c = 64, 128: the nhwc8 kernel; 96, 384: the generic one): the in-place
    result equals the out-of-place one, and neither writes outside the interior of its output"""
    import ctypes as C
    from eadgan_b200 import tc
    from eadgan_b200._lib import ACT_NONE, ACT_RELU, ACT_TANH, call, ptr, stream, t4
    from test_guard_gpu import _check, _guarded
    kind = {"relu": ACT_RELU, "tanh": ACT_TANH, "none": ACT_NONE}[act]
    torch.manual_seed(c)
    n, h, w = 5, 8, 8
    x = torch.randn(n, c, h, w, device=cuda).bfloat16().float()
    rm, rv = torch.randn(c, device=cuda) * 0.3, torch.rand(c, device=cuda) + 0.5
    gamma, beta = torch.rand(c, device=cuda) + 0.5, torch.randn(c, device=cuda) * 0.2
    dy = torch.randn(n, c, h, w, device=cuda)
    xp, yp = _padded(n, h, w, c, cuda, x), _padded(n, h, w, c, cuda)
    # the y a forward wrote: the stored gate is what the backward must reproduce
    call("eadgan_bn_eval", C.byref(t4(tc.interior(xp))), n, c, h, w, ptr(rm), ptr(rv), 1e-5, ptr(gamma), ptr(beta),
         kind, 0.0, C.byref(t4(tc.interior(yp))), stream())

    def launch(dy_buf, dx_buf):
        sums = torch.zeros(2 * c, device=cuda, dtype=torch.float64)
        small = torch.empty(3 * c, device=cuda)
        call("eadgan_bn_eval_bwd", C.byref(t4(tc.interior(dy_buf))), C.byref(t4(tc.interior(xp))),
             C.byref(t4(tc.interior(yp))), n, c, h, w, ptr(rm), ptr(rv), 1e-5, ptr(gamma), ptr(beta), kind, 0.0,
             ptr(sums), C.byref(t4(tc.interior(dx_buf))), ptr(small[:c]), ptr(small[c:2 * c]), ptr(small[2 * c:]),
             stream())
        return small

    ref_dx = _padded(n, h, w, c, cuda)
    dyp = _padded(n, h, w, c, cuda, dy)
    small_ref = launch(dyp, ref_dx)
    # out of place into a guarded buffer
    big, out = _guarded((n, h + 2, w + 2, c), torch.bfloat16, cuda)
    small = launch(dyp, out)
    _check(big, out, ref_dx, halo=True)
    torch.testing.assert_close(small, small_ref, rtol=1e-6, atol=0)
    # in place: dx overwrites dy, which lives in a guarded buffer
    big, buf = _guarded((n, h + 2, w + 2, c), torch.bfloat16, cuda)
    tc.interior(buf).copy_(dy)
    small = launch(buf, buf)
    _check(big, buf, ref_dx, halo=True)
    torch.testing.assert_close(small, small_ref, rtol=1e-6, atol=0)
    # and the values: dx = dy * act'(y) * gamma * rsqrt(rv + eps)
    ys = tc.interior(yp).float()
    gate = {"relu": (ys > 0).float(), "tanh": 1 - ys * ys, "none": torch.ones_like(ys)}[act]
    dz = dy.bfloat16().float() * gate
    is_ = torch.rsqrt(rv + 1e-5)
    want = dz * (gamma * is_)[None, :, None, None]
    assert rel_err(tc.interior(ref_dx), want) <= 1e-2
    xhat = (x - rm[None, :, None, None]) * is_[None, :, None, None]
    assert rel_err(small_ref[:c], (dz * xhat).sum((0, 2, 3))) <= 1e-4        # dgamma
    assert rel_err(small_ref[c:2 * c], dz.sum((0, 2, 3))) <= 1e-4            # dbeta
    assert rel_err(small_ref[2 * c:], gamma * is_ * dz.sum((0, 2, 3))) <= 1e-4   # conv-bias gradient


def test_no_collective_in_eval(cuda):
    """SyncBN does not communicate in eval mode: with an all-reduce hook installed, an eval forward + backward makes no
    call; the same stack in training mode makes one per BatchNorm in each direction"""
    import eadgan_b200.nn as enn
    from eadgan_b200 import functional as Fn
    os.environ["EADGAN_PRECISION"] = "bf16"
    spec = [("convT", 64, 64, 4, 2, 1), ("bn", 64), ("relu",), ("convT", 64, 96, 4, 2, 1), ("bn", 96), ("lrelu", 0.2),
            ("conv", 96, 32, 4, 2, 1)]
    torch.manual_seed(9)
    seq = build(enn, spec).to(cuda)
    x = torch.randn(4, 64, 4, 4, device=cuda, requires_grad=True)
    calls = []
    saved = (Fn._allreduce_sum, Fn._world_size)
    Fn.set_allreduce(lambda t: calls.append(t.numel()), 1)
    try:
        seq.eval()
        seq(x).sum().backward()
        n_eval = len(calls)
        seq.train()
        seq(x).sum().backward()
        n_train = len(calls) - n_eval
    finally:
        Fn.set_allreduce(*saved)
    assert n_eval == 0, calls
    assert n_train == 4, calls
