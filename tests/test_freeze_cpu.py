"""eadgan_b200.freeze's planner on every reference network (no kernels run): which layers fold a BatchNorm, which fold
their spectral norm's sigma, and which BatchNorm layers stay; and freeze() of a CPU module raises."""
import pytest
import torch


def _nets():
    from eadgan_b200.steps import celeba, dsprites, mnist
    torch.manual_seed(0)
    return {
        "celeba_G": celeba.Generator(), "celeba_D": celeba.Discriminator(),
        "dsprites_G": dsprites.Generator(1, 4), "dsprites_D": dsprites.Discriminator(1),
        "dsprites_E": dsprites.Encoder(1, 4), "dsprites_pxy": dsprites.Encoder_pxy(1, 3),
        "colored_G": dsprites.Generator(3, 7), "colored_D": dsprites.Discriminator(3),
        "colored_E": dsprites.Encoder(3, 7), "colored_pxy": dsprites.Encoder_pxy(3, 6),
        "mnist_G": mnist.Generator(), "mnist_D": mnist.Discriminator(), "mnist_E": mnist.Encoder(),
        "approximator": mnist.AffineApproximator(),
    }


def _sn(*names):
    return [(n, None, True) for n in names]


_DSPRITES_D = _sn("conv_block.0", "conv_block.2", "conv_block.4", "conv_block.6", "fc1.0")
_DSPRITES_E = _sn("conv_block.0", "conv_block.2", "conv_block.4", "conv_block.6", "fc1.0", "fc2.0", "cat_layer.0",
                  "cont_layer.0")
_DSPRITES_G = [("conv_block.0", "conv_block.1", False), ("conv_block.3", "conv_block.4", False),
               ("conv_block.6", "conv_block.7", False)]

# (folds as (layer, folded BatchNorm, sigma folded), BatchNorm layers kept)
EXPECTED = {
    "celeba_G": ([("conv_blocks.1", "conv_blocks.2", False), ("conv_blocks.4", "conv_blocks.5", False),
                  ("conv_blocks.7", "conv_blocks.8", False)], []),
    "celeba_D": (_sn("main.0", "main.2", "main.4", "main.6"), []),
    "dsprites_G": (_DSPRITES_G, []), "dsprites_D": (_DSPRITES_D, []), "dsprites_E": (_DSPRITES_E, []),
    "dsprites_pxy": ([], []),
    "colored_G": (_DSPRITES_G, []), "colored_D": (_DSPRITES_D, []), "colored_E": (_DSPRITES_E, []),
    "colored_pxy": ([], []),
    # the leading BatchNorm2d(128) of the generator precedes the Upsample; the Encoder's follow a LeakyReLU
    "mnist_G": ([("conv_blocks.2", "conv_blocks.3", False), ("conv_blocks.6", "conv_blocks.7", False)],
                ["conv_blocks.0"]),
    "mnist_D": (_sn("conv_blocks.0", "conv_blocks.2", "conv_blocks.4", "conv_blocks.6", "adv_layer.0"), []),
    "mnist_E": (_sn("conv_blocks.0", "conv_blocks.2", "conv_blocks.5", "conv_blocks.8", "aux_layer.0",
                    "latent_layer.0", "noise_layer.0"), ["conv_blocks.4", "conv_blocks.7", "conv_blocks.10"]),
    "approximator": ([], []),
}


@pytest.mark.parametrize("name", sorted(EXPECTED))
def test_plan_of_every_reference_network(name):
    from eadgan_b200 import frozen
    folds, kept = frozen.plan(_nets()[name])
    want_folds, want_kept = EXPECTED[name]
    assert [tuple(f) for f in folds] == want_folds
    assert kept == want_kept


def test_plan_is_the_same_on_stock_torch_modules():
    """the rules read the module tree only: the oracle's stock-torch networks plan exactly like ours"""
    from eadgan_b200 import frozen
    from oracle import torch_oracle as O
    ours = _nets()
    for name, ref in (("celeba_G", O.CelebAGenerator()), ("celeba_D", O.CelebADiscriminator()),
                      ("dsprites_E", O.DSpritesEncoder(3, 4, 1)), ("mnist_G", O.MnistGenerator()),
                      ("mnist_E", O.MnistEncoder())):
        assert frozen.plan(ref) == frozen.plan(ours[name]), name


def test_plan_conditions():
    """a BatchNorm folds only when it directly follows the layer, has running statistics and an affine transform, and
    neither module carries a hook"""
    from eadgan_b200 import frozen
    import eadgan_b200.nn as enn

    def seq(*mods):
        return enn.Sequential(*mods)

    def names(s):
        folds, kept = frozen.plan(s)
        return [tuple(f) for f in folds], kept

    assert names(seq(enn.Conv2d(3, 8, 3), enn.BatchNorm2d(8), enn.ReLU())) == ([("0", "1", False)], [])
    assert names(seq(enn.Linear(4, 8), enn.BatchNorm2d(8))) == ([("0", "1", False)], [])
    assert names(seq(enn.Conv2d(3, 8, 3), enn.ReLU(), enn.BatchNorm2d(8))) == ([], ["2"])
    assert names(seq(enn.Conv2d(3, 8, 3), enn.BatchNorm2d(8, affine=False))) == ([], ["1"])
    assert names(seq(enn.Conv2d(3, 8, 3), enn.BatchNorm2d(8, track_running_stats=False))) == ([], ["1"])
    hooked = seq(enn.Conv2d(3, 8, 3), enn.BatchNorm2d(8))
    hooked[0].register_forward_hook(lambda *a: None)
    assert names(hooked) == ([], ["1"])
    hooked = seq(enn.Conv2d(3, 8, 3), enn.BatchNorm2d(8))
    hooked[1].register_forward_pre_hook(lambda *a: None)
    assert names(hooked) == ([], ["1"])
    # ConvTranspose2d: the output channels are dim 1 of its weight; a spectral norm and a BatchNorm combine
    assert names(seq(enn.ConvTranspose2d(8, 4, 4, 2, 1), enn.BatchNorm2d(4))) == ([("0", "1", False)], [])
    assert names(seq(enn.spectral_norm(enn.Conv2d(3, 8, 3)), enn.BatchNorm2d(8))) == ([("0", "1", True)], [])


def test_freeze_of_a_cpu_module_raises():
    import eadgan_b200
    from eadgan_b200.steps import celeba
    with pytest.raises(RuntimeError, match="CUDA"):
        eadgan_b200.freeze(celeba.Generator())
