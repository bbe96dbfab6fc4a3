"""Host logic of the bf16 chain executor for eval-mode BatchNorm (no kernels run): an eval-mode stack is planned with
the same kernel families as in training mode, and the eval catalogue of tests/test_eval_gpu.py reaches every forward
family that can precede a BatchNorm, both BatchNorm kernel layouts and every activation after an eval BatchNorm."""
import torch


def _plans(seq, in_shape):
    from eadgan_b200 import chain
    stages = chain._plan(seq)
    assert stages is not None
    return chain._plan_kernels(stages, in_shape)


def _fields(p):
    return {k: getattr(p, k) for k in p.__slots__ if k != "bn"}


def test_eval_plans_equal_training_plans():
    from eadgan_b200.steps import celeba, dsprites

    torch.manual_seed(0)
    trunks = [(celeba.Generator().conv_blocks, (8, 218, 1, 1))]
    for ch, code in ((1, 4), (3, 7)):         # dSprites and colored dSprites
        trunks.append((dsprites.Generator(ch, code).conv_block, (8, 64, 4, 4)))
    for seq, shape in trunks:
        n_bn = sum(isinstance(m, torch.nn.BatchNorm2d) for m in seq.modules())
        assert n_bn == 3
        seq.train()
        train = _plans(seq, shape)
        seq.eval()
        ev = _plans(seq, shape)
        assert [p.bn for p in train].count("train") == n_bn
        assert [p.bn for p in ev].count("eval") == n_bn
        assert [p.bn is None for p in train] == [p.bn is None for p in ev]
        for a, b in zip(train, ev):
            fa, fb = _fields(a), _fields(b)
            fa["d"], fb["d"] = tuple(getattr(a.d, f) for f, _ in a.d._fields_), tuple(getattr(b.d, f) for f, _ in b.d._fields_)
            assert fa == fb


def test_eval_catalogue_covers_every_family_in_front_of_a_batchnorm():
    from eadgan_b200 import chain
    from eadgan_b200._lib import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_TANH
    import eadgan_b200.nn as enn
    from test_chain_stages_gpu import build
    from test_eval_gpu import EVAL_STAGES

    fwd, layouts, acts = set(), set(), set()
    for name, spec, shape in EVAL_STAGES:
        seq = build(enn, spec)
        seq.eval()
        plans = _plans(seq, shape)
        stages = chain._plan(seq)
        assert any(p.bn == "eval" for p in plans), name
        for st, p in zip(stages, plans):
            if p.bn is None:
                continue
            assert p.bn == "eval"
            fwd.add((p.fwd, st.kind))
            c = p.out_shape[1]
            # bn.cu nhwc8_ok: the vectorised kernels take c % 8 == 0 with c / 8 dividing 256
            layouts.add("nhwc8" if c % 8 == 0 and c <= 1024 and 256 % (c // 8) == 0 else "generic")
            acts.add(st.act[0])
    assert fwd == {("tc", "convT"), ("tc", "conv"), ("thin", "conv"), ("simt", "convT")}, fwd
    assert layouts == {"nhwc8", "generic"}, layouts
    assert acts == {ACT_NONE, ACT_RELU, ACT_LRELU, ACT_TANH, ACT_SIGMOID}, acts

