"""CPU checks of define_D's 'pixel' discriminator and of the PatchGAN at every depth (reference models/networks.py:163-206,:555-753):
module sequences, checkpoint layouts, parameter counts and the initialisation stream, against plain-torch restatements."""
import functools

import pytest
import torch
import torch.nn as nn
from torch.nn import init

from healthivert_gan_b200 import _lib, networks

PIXEL_LAYOUT = {
    "batch": (["net.0.weight", "net.0.bias", "net.2.weight", "net.3.weight", "net.3.bias", "net.3.running_mean", "net.3.running_var",
               "net.3.num_batches_tracked", "net.5.weight"], 8_704),
    "instance": (["net.0.weight", "net.0.bias", "net.2.weight", "net.2.bias", "net.5.weight", "net.5.bias"], 8_577),
    "none": (["net.0.weight", "net.0.bias", "net.2.weight", "net.5.weight"], 8_448),
}
NORM_KIND = {"batch": "BatchNorm2d", "instance": "InstanceNorm2d", "none": "Identity"}


def _norm(norm, c):
    return {"batch": lambda: nn.BatchNorm2d(c, affine=True, track_running_stats=True),
            "instance": lambda: nn.InstanceNorm2d(c, affine=False, track_running_stats=False),
            "none": lambda: nn.Identity()}[norm]()


def _init(net):
    """init_weights('normal', 0.02) written out (same RNG consumption order: module order)"""
    for m in net.modules():
        if isinstance(m, nn.Conv2d):
            init.normal_(m.weight.data, 0.0, 0.02)
            if m.bias is not None:
                init.constant_(m.bias.data, 0.0)
        elif isinstance(m, nn.BatchNorm2d):
            init.normal_(m.weight.data, 1.0, 0.02)
            init.constant_(m.bias.data, 0.0)
    return net


def _plain_pixel(norm, seed, ndf=64):
    torch.manual_seed(seed)
    bias = norm == "instance"
    return _init(nn.Sequential(nn.Conv2d(1, ndf, 1, 1, 0), nn.LeakyReLU(0.2, True),
                               nn.Conv2d(ndf, 2 * ndf, 1, 1, 0, bias=bias), _norm(norm, 2 * ndf), nn.LeakyReLU(0.2, True),
                               nn.Conv2d(2 * ndf, 1, 1, 1, 0, bias=bias)))


def _plain_patchgan(norm, n_layers, seed, ndf=64):
    torch.manual_seed(seed)
    bias = norm == "instance"
    seq = [nn.Conv2d(1, ndf, 4, 2, 1), nn.LeakyReLU(0.2, True)]
    mult = 1
    for n in range(1, n_layers):
        prev, mult = mult, min(2 ** n, 8)
        seq += [nn.Conv2d(ndf * prev, ndf * mult, 4, 2, 1, bias=bias), _norm(norm, ndf * mult), nn.LeakyReLU(0.2, True)]
    prev, mult = mult, min(2 ** n_layers, 8)
    seq += [nn.Conv2d(ndf * prev, ndf * mult, 4, 1, 1, bias=bias), _norm(norm, ndf * mult), nn.LeakyReLU(0.2, True)]
    seq += [nn.Conv2d(ndf * mult, 1, 4, 1, 1)]
    return _init(nn.Sequential(*seq))


def _same_state(sd, ref_sd, prefix):
    rsd = {prefix + k: v for k, v in ref_sd.items()}
    assert list(sd) == list(rsd)
    for k in sd:
        assert sd[k].shape == rsd[k].shape, k
        assert torch.equal(sd[k], rsd[k]), k


@pytest.mark.parametrize("norm", ["batch", "instance", "none"])
def test_pixel_layout_and_initialisation(norm):
    torch.manual_seed(5)
    net = networks.define_D(1, 64, "pixel", 3, norm, "normal", 0.02, [])
    assert isinstance(net, networks.PixelDiscriminator)
    assert net.precision == "fp32"
    assert [type(m).__name__ for m in net.net] == ["Conv2d", "LeakyReLU", "Conv2d", NORM_KIND[norm], "LeakyReLU", "Conv2d"]
    assert [(m.in_channels, m.out_channels, m.kernel_size, m.stride, m.padding) for m in net.net if isinstance(m, nn.Conv2d)] == [
        (1, 64, (1, 1), (1, 1), (0, 0)), (64, 128, (1, 1), (1, 1), (0, 0)), (128, 1, (1, 1), (1, 1), (0, 0))]
    keys, count = PIXEL_LAYOUT[norm]
    sd = net.state_dict()
    assert list(sd) == keys
    assert sum(p.numel() for p in net.parameters()) == count
    _same_state(sd, _plain_pixel(norm, 5).state_dict(), "net.")
    net2 = networks.define_D(1, 64, "pixel", 3, norm, "normal", 0.02, [])
    net2.load_state_dict(sd)                          # strict round trip
    assert all(torch.equal(a, b) for a, b in zip(net2.state_dict().values(), sd.values()))


def test_pixel_other_widths_follow_the_reference():
    net = networks.define_D(3, 32, "pixel", 3, "batch", "normal", 0.02, [])
    convs = [m for m in net.net if isinstance(m, nn.Conv2d)]
    assert [(m.in_channels, m.out_channels) for m in convs] == [(3, 32), (32, 64), (64, 1)]
    assert net.net[3].num_features == 64


@pytest.mark.parametrize("norm", ["batch", "instance", "none"])
@pytest.mark.parametrize("n_layers", [1, 2, 4, 5])
def test_n_layers_layout_and_initialisation(n_layers, norm):
    torch.manual_seed(11)
    net = networks.define_D(1, 64, "n_layers", n_layers, norm, "normal", 0.02, [])
    ref = _plain_patchgan(norm, n_layers, 11)
    assert [type(m).__name__ for m in net.model] == [type(m).__name__ if not isinstance(m, nn.Identity) else "Identity" for m in ref]
    assert [(m.in_channels, m.out_channels, m.stride) for m in net.model if isinstance(m, nn.Conv2d)] == \
        [(m.in_channels, m.out_channels, m.stride) for m in ref if isinstance(m, nn.Conv2d)]
    _same_state(net.state_dict(), ref.state_dict(), "model.")
    networks.define_D(1, 64, "n_layers", n_layers, norm, "normal", 0.02, []).load_state_dict(net.state_dict())


def test_unknown_discriminator_names_still_raise():
    for bad in ("pixelgan", "Pixel", "unet", ""):
        with pytest.raises(NotImplementedError, match=r"Discriminator model name \[%s\] is not recognized" % bad):
            networks.define_D(1, 64, bad, 3, "batch", "normal", 0.02, [])


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_pixel_without_cuda_raises(precision):
    net = networks.define_D(1, 64, "pixel", 3, "none", "normal", 0.02, [])
    net.precision = precision
    with pytest.raises(_lib.HvError, match="PixelDiscriminator needs CUDA tensors"):
        net(torch.zeros(1, 1, 4, 4))


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("flags", [dict(affine=True), dict(track_running_stats=True)])
def test_pixel_rejects_instance_norms_it_does_not_build(flags, precision):
    """an InstanceNorm2d that get_norm_layer('instance') does not make (affine, or with running statistics) is refused on both paths
    before any kernel runs, instead of being applied without its parameters"""
    norm_layer = functools.partial(nn.InstanceNorm2d, **{"affine": False, "track_running_stats": False, **flags})
    net = networks.PixelDiscriminator(1, 64, norm_layer=norm_layer)
    net.precision = precision
    with pytest.raises(NotImplementedError, match="InstanceNorm2d is built as get_norm_layer"):
        net(torch.zeros(1, 1, 4, 4))
