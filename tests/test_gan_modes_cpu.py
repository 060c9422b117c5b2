"""CPU checks of the reference's GAN objectives and learning-rate policies (models/networks.py:39-65,:212-278): get_scheduler on
FusedAdam against the same torch schedulers on torch.optim.Adam, BaseModel.update_learning_rate, and the constructors' error messages."""
import pytest
import torch
from torch.optim import lr_scheduler

from healthivert_gan_b200 import networks, train_ops as T
from healthivert_gan_b200.pix2pix_model import BaseModel
from oracle import synth

LR = 2e-4


def _reference_scheduler(optimizer, opt):
    """the reference's get_scheduler (models/networks.py:39-65), written out on its own"""
    if opt.lr_policy == "linear":
        return lr_scheduler.LambdaLR(
            optimizer, lambda e: 1.0 - max(0, e + opt.epoch_count - opt.n_epochs) / float(opt.n_epochs_decay + 1))
    if opt.lr_policy == "step":
        return lr_scheduler.StepLR(optimizer, step_size=opt.lr_decay_iters, gamma=0.1)
    if opt.lr_policy == "plateau":
        return lr_scheduler.ReduceLROnPlateau(optimizer, mode="min", factor=0.2, threshold=0.01, patience=5)
    return lr_scheduler.CosineAnnealingLR(optimizer, T_max=opt.n_epochs, eta_min=0)


def _pair(opt):
    ours = T.FusedAdam([torch.nn.Parameter(torch.zeros(4))], lr=LR, betas=(0.5, 0.999))
    ref = torch.optim.Adam([torch.nn.Parameter(torch.zeros(4))], lr=LR, betas=(0.5, 0.999))
    return ours, networks.get_scheduler(ours, opt), ref, _reference_scheduler(ref, opt)


def _lrs(policy, epochs, metrics=None, **over):
    opt = synth.train_options(lr_policy=policy, **over)
    ours, s_ours, ref, s_ref = _pair(opt)
    got, want = [ours.param_groups[0]["lr"]], [ref.param_groups[0]["lr"]]
    for e in range(epochs):
        ours.step()                      # no gradients: the step is a no-op, but keeps torch's call-order check quiet
        ref.step()
        if policy == "plateau":
            s_ours.step(metrics[e])
            s_ref.step(metrics[e])
        else:
            s_ours.step()
            s_ref.step()
        got.append(ours.param_groups[0]["lr"])
        want.append(ref.param_groups[0]["lr"])
    return got, want


@pytest.mark.parametrize("policy,over", [
    ("linear", dict(epoch_count=1, n_epochs=4, n_epochs_decay=6)),
    ("linear", dict(epoch_count=3, n_epochs=5, n_epochs_decay=9)),
    ("step", dict(lr_decay_iters=3, n_epochs=7)),
    ("step", dict(lr_decay_iters=1, n_epochs=7)),
    ("cosine", dict(n_epochs=7)),
    ("cosine", dict(n_epochs=10)),
])
def test_lr_policies_match_torch(policy, over):
    """three periods of the cosine (T_max = n_epochs) and several step decays; the lr after every step is compared with =="""
    epochs = 3 * max(over.get("n_epochs", 1), over.get("lr_decay_iters", 1), over.get("n_epochs", 0) + over.get("n_epochs_decay", 0))
    got, want = _lrs(policy, epochs, **over)
    assert got == want
    assert len(set(got)) > 2                 # the lr actually moves


@pytest.mark.parametrize("metrics", [
    [0.0] * 40,                                                             # BaseModel.metric's value unless a driver sets it
    [1.0 / (1 + e) for e in range(40)],                                     # decreasing
    [1.0 + 0.3 * float(torch.sin(torch.tensor(1.7 * e))) for e in range(40)],   # noisy
])
def test_plateau_matches_torch(metrics):
    got, want = _lrs("plateau", len(metrics), metrics)
    assert got == want
    if metrics[0] == 0.0:
        assert got[-1] < LR                  # a constant metric is a plateau: the lr is reduced


def test_linear_is_the_closed_form():
    """'linear' reproduces lr * (1 - max(0, e + epoch_count - n_epochs) / (n_epochs_decay + 1)) bit for bit"""
    for ec, n, nd in ((1, 4, 6), (3, 5, 9), (1, 200, 800)):
        opt = synth.train_options(lr_policy="linear", epoch_count=ec, n_epochs=n, n_epochs_decay=nd)
        ours = T.FusedAdam([torch.nn.Parameter(torch.zeros(4))], lr=LR)
        sched = networks.get_scheduler(ours, opt)
        for e in range(1, n + nd + 3):
            ours.step()
            sched.step()
            assert ours.param_groups[0]["lr"] == LR * (1.0 - max(0, e + ec - n) / float(nd + 1)), (ec, n, nd, e)


def _base_model(policy, **over):
    opt = synth.train_options(gpu_ids=[], lr_policy=policy, **over)
    m = BaseModel(opt)
    m.optimizers = [T.FusedAdam([torch.nn.Parameter(torch.zeros(4))], lr=LR) for _ in range(2)]
    m.setup(opt)
    return m


def test_update_learning_rate_plateau_passes_the_metric(capsys):
    m = _base_model("plateau")
    seen = []
    for s in m.schedulers:
        real = s.step
        s.step = lambda *a, real=real: (seen.append(a), real(*a))
    m.metric = 0.25
    m.update_learning_rate()
    assert seen == [(0.25,), (0.25,)]
    assert capsys.readouterr().out == "learning rate %.7f -> %.7f\n" % (LR, LR)
    assert isinstance(m.schedulers[0], lr_scheduler.ReduceLROnPlateau)
    assert m.metric == 0.25
    assert BaseModel(synth.train_options(gpu_ids=[])).metric == 0


def test_update_learning_rate_step(capsys):
    m = _base_model("step", lr_decay_iters=1)
    m.update_learning_rate()
    assert [o.param_groups[0]["lr"] for o in m.optimizers] == [LR * 0.1] * 2
    assert capsys.readouterr().out == "learning rate %.7f -> %.7f\n" % (LR, LR * 0.1)


def test_gan_loss_and_scheduler_construction():
    for mode in ("vanilla", "lsgan", "wgangp"):
        crit = networks.GANLoss(mode)
        assert crit.gan_mode == mode
        assert float(crit.real_label) == 1.0 and float(crit.fake_label) == 0.0
    crit = networks.GANLoss("lsgan", target_real_label=0.9, target_fake_label=0.1)
    assert float(crit.real_label) == pytest.approx(0.9) and float(crit.fake_label) == pytest.approx(0.1)
    for bad in ("hinge", "wgan", "LSGAN"):
        with pytest.raises(NotImplementedError, match=r"^gan mode %s not implemented$" % bad):
            networks.GANLoss(bad)
    ours = T.FusedAdam([torch.nn.Parameter(torch.zeros(4))], lr=LR)
    assert isinstance(ours, torch.optim.Optimizer)
    for bad in ("exponential", "Linear", "none"):
        with pytest.raises(NotImplementedError, match=r"^learning rate policy \[%s\] is not implemented$" % bad):
            networks.get_scheduler(ours, synth.train_options(lr_policy=bad))
