"""CPU checks of the PatchGAN discriminator's normalisation options (reference models/networks.py:30-47,:555-602): the module sequence,
the checkpoint layout and the initialisation stream of define_D(..., norm) for norm in {'instance', 'none'}."""
import functools

import pytest
import torch
import torch.nn as nn
from torch.nn import init

from healthivert_gan_b200 import networks

LAYOUT = {
    "instance": ([f"model.{i}.{p}" for i in (0, 2, 5, 8, 11) for p in ("weight", "bias")], 2_762_689),
    "none": (["model.0.weight", "model.0.bias", "model.2.weight", "model.5.weight", "model.8.weight", "model.11.weight", "model.11.bias"],
             2_761_793),
    "batch": ([f"model.{i}.{p}" for i in (0, 11) for p in ("weight", "bias")] + [f"model.{i}.weight" for i in (2, 5, 8)]
              + [f"model.{i}.{p}" for i in (3, 6, 9) for p in ("weight", "bias", "running_mean", "running_var", "num_batches_tracked")],
              2_763_585),
}


def _plain_reference(norm, seed):
    """The reference's layout written out with plain torch modules, initialised as init_weights('normal', 0.02) does."""
    torch.manual_seed(seed)
    bias = norm == "instance"
    mk = {"instance": lambda c: nn.InstanceNorm2d(c, affine=False, track_running_stats=False), "none": lambda c: nn.Identity()}[norm]
    seq = [nn.Conv2d(1, 64, 4, 2, 1), nn.LeakyReLU(0.2, True)]
    for cin, cout, s in ((64, 128, 2), (128, 256, 2), (256, 512, 1)):
        seq += [nn.Conv2d(cin, cout, 4, s, 1, bias=bias), mk(cout), nn.LeakyReLU(0.2, True)]
    seq += [nn.Conv2d(512, 1, 4, 1, 1)]
    net = nn.Sequential(*seq)
    for m in net.modules():
        if isinstance(m, nn.Conv2d):
            init.normal_(m.weight.data, 0.0, 0.02)
            if m.bias is not None:
                init.constant_(m.bias.data, 0.0)
    return net


@pytest.mark.parametrize("norm", ["instance", "none"])
def test_define_d_layout_and_initialisation(norm):
    torch.manual_seed(3)
    net = networks.define_D(1, 64, "basic", 3, norm, "normal", 0.02, [])
    kinds = [type(m).__name__ for m in net.model]
    n = "InstanceNorm2d" if norm == "instance" else "Identity"
    assert kinds == ["Conv2d", "LeakyReLU"] + ["Conv2d", n, "LeakyReLU"] * 3 + ["Conv2d"]
    for i in (3, 6, 9):
        m = net.model[i]
        if norm == "instance":
            assert not m.affine and not m.track_running_stats and m.eps == 1e-5
        else:
            assert isinstance(m, networks.Identity)
            x = torch.randn(2, 3)
            assert m(x) is x
    for i in (2, 5, 8):
        assert (net.model[i].bias is not None) == (norm == "instance")
    keys, count = LAYOUT[norm]
    sd = net.state_dict()
    assert list(sd) == keys
    assert sum(p.numel() for p in net.parameters()) == count
    ref = _plain_reference(norm, 3)
    rsd = {"model." + k: v for k, v in ref.state_dict().items()}
    assert list(rsd) == keys
    for k in keys:
        assert sd[k].shape == rsd[k].shape, k
        assert torch.equal(sd[k], rsd[k]), k          # no RNG draw for the norm layers: the same conv weights as the reference
    net2 = networks.define_D(1, 64, "basic", 3, norm, "normal", 0.02, [])
    net2.load_state_dict(sd)                          # strict round trip


def test_batch_layout_is_unchanged():
    net = networks.define_D(1, 64, "basic", 3, "batch", "normal", 0.02, [])
    keys, count = LAYOUT["batch"]
    assert sorted(net.state_dict()) == sorted(keys)
    assert sum(p.numel() for p in net.parameters()) == count


def test_norm_layer_factories():
    f = networks.get_norm_layer("instance")
    assert isinstance(f, functools.partial) and f.func is nn.InstanceNorm2d
    assert f.keywords == {"affine": False, "track_running_stats": False}
    assert isinstance(networks.get_norm_layer("none")(64), networks.Identity)
    for bad in ("bogus", "group", "layer"):
        with pytest.raises(NotImplementedError):
            networks.get_norm_layer(bad)
    with pytest.raises(NotImplementedError):
        networks.define_D(1, 64, "basic", 3, "bogus", "normal", 0.02, [])
