"""GPU checks of the reference's LSGAN and WGAN objectives (models/networks.py:212-278) on the loss kernels (hv_reduce_scalar kinds 3
and 5, hv_loss_grad kinds 2 and 3), through GANLoss, through one Pix2PixModel training step in both precisions, and of a scheduled
learning rate reaching the Adam kernel.  The references are float64 torch.

'wgangp' is the reference's objective as its pix2pix model uses it: -mean(D(x)) against real, mean(D(x)) against fake, with no
gradient penalty (the model never calls cal_gradient_penalty) and no weight clipping."""
import copy

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from healthivert_gan_b200 import _lib, networks, train_ops as T
from healthivert_gan_b200._lib import ptr
from healthivert_gan_b200.pix2pix_model import Pix2PixModel
from oracle import synth

pytestmark = pytest.mark.gpu

MODES = ("vanilla", "lsgan", "wgangp")
SHAPES = [(16, 1, 30, 30), (2, 1, 30, 30), (3, 1, 7, 5), (1 << 20,)]   # the 2^20 vector takes all 1024 partial blocks


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def f32(x):
    """the value a kernel receives for a Python float (a C float argument)"""
    return float(np.float32(x))


def loss64(p, is_real, mode, labels=(1.0, 0.0)):
    """the reference's GANLoss(mode)(p, is_real) in float64 (its labels are float32 buffers)"""
    if mode == "wgangp":
        return -p.mean() if is_real else p.mean()
    t = torch.full_like(p, f32(labels[0] if is_real else labels[1]))
    if mode == "lsgan":
        return F.mse_loss(p, t)
    return F.binary_cross_entropy_with_logits(p, t)


def _logits(shape, seed):
    # an offset keeps the WGAN mean away from 0, so that its relative error measures the kernel, not the cancellation
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * 1.5 + 0.7


def _scales(dev):
    """(S as the kernel applies it, device pointer, scale_is_reciprocal)"""
    s = torch.tensor([7.0], device=dev)
    return [(1.0, None, 0), (7.0, ptr(s), 0), (1.0 / 7.0, ptr(s), 1)], s


def _loss_grad(a, t, kind, g, sp, recip, out=None):
    da = torch.empty_like(a) if out is None else out
    _lib.check(_lib.lib().hv_loss_grad(ptr(a), None, float(t), kind, float(g), sp, recip, ptr(da), int(out is not None), a.numel(),
                                       _lib.stream()))
    return da


@pytest.mark.parametrize("t", [1.0, 0.0, 0.9])
@pytest.mark.parametrize("shape", SHAPES)
def test_lsgan_kernels_against_float64(shape, t):
    """value: kind 5, scale * sum (a - t)^2; gradient: kind 2, g * S * 2 (a - t), plain and accumulated"""
    x = _logits(shape, len(shape) * 31 + shape[-1])
    xd = x.cuda()
    d64 = x.double() - f32(t)
    for scale in (1.0 / x.numel(), 1.0, -0.5):
        v = T.reduce_scalar(xd, None, 5, scale, t)
        want = f32(scale) * float((d64 * d64).sum())
        assert abs(float(v) - want) <= 1e-5 * abs(want), (scale, float(v), want)
    scales, keep = _scales(xd.device)
    for g in (1.0, 0.5 / x.numel(), -1.0 / 6, 3.0):
        for s, sp, recip in scales:
            want = f32(g) * s * 2 * d64
            assert rel(_loss_grad(xd, t, 2, g, sp, recip), want) <= 1e-6, (g, s)
    base = torch.randn(shape, generator=torch.Generator().manual_seed(5))
    acc = _loss_grad(xd, t, 2, 0.25, None, 0, out=base.cuda())
    assert rel(acc, base.double() + f32(0.25) * 2 * d64) <= 1e-6
    torch.cuda.synchronize()
    del keep


@pytest.mark.parametrize("shape", SHAPES)
def test_wgan_kernels_against_float64(shape):
    """value: kind 3 (sum a) with scale -+1/count; gradient: kind 3, the constant g * S (the sign rides in g)"""
    x = _logits(shape, len(shape) * 17 + shape[-1])
    xd = x.cuda()
    for sign in (-1.0, 1.0):
        v = T.reduce_scalar(xd, None, 3, sign / x.numel())
        want = sign * float(x.double().mean())
        assert abs(float(v) - want) <= 1e-5 * abs(want), (sign, float(v), want)
    scales, keep = _scales(xd.device)
    for g in (1.0, -0.5 / x.numel(), 1.0 / 6, -3.0):
        for s, sp, recip in scales:
            got = _loss_grad(xd, 0.0, 3, g, sp, recip)
            assert rel(got, torch.full(shape, f32(g) * s, dtype=torch.float64)) <= 1e-6, (g, s)
    base = torch.randn(shape, generator=torch.Generator().manual_seed(6))
    acc = _loss_grad(xd, 0.0, 3, -0.125, None, 0, out=base.cuda())
    assert rel(acc, base.double() - 0.125) <= 1e-6
    torch.cuda.synchronize()
    del keep


def test_out_of_range_kinds_are_rejected_before_any_launch():
    L = _lib.lib()
    x = torch.randn(64, device="cuda")
    out = torch.empty(1, device="cuda")
    scratch = torch.empty(1024, device="cuda")
    da = torch.empty_like(x)
    before = _lib.launch_count()
    for kind in (-1, 6, 100):
        rc = L.hv_reduce_scalar(ptr(x), ptr(x), 0.0, kind, x.numel(), 1.0, ptr(out), ptr(scratch), _lib.stream())
        assert rc < 0 and b"kind" in L.hv_last_error(), (kind, rc, L.hv_last_error())
    for kind in (-1, 4, 100):
        rc = L.hv_loss_grad(ptr(x), ptr(x), 0.0, kind, 1.0, None, 0, ptr(da), 0, x.numel(), _lib.stream())
        assert rc < 0 and b"kind" in L.hv_last_error(), (kind, rc, L.hv_last_error())
    assert _lib.launch_count() == before
    with pytest.raises(_lib.HvError, match="kind"):
        T.reduce_scalar(x, None, 6, 1.0)


@pytest.mark.parametrize("labels", [(1.0, 0.0), (0.9, 0.1)])
@pytest.mark.parametrize("is_real", [True, False])
@pytest.mark.parametrize("mode", MODES)
def test_gan_loss_module_against_float64(mode, is_real, labels):
    crit = networks.GANLoss(mode, *labels).cuda()
    for shape in SHAPES[:3]:
        x = _logits(shape, shape[0] + 3 * is_real)
        for g in (1.0, 0.5, 1.0 / 6):
            v = crit(x.cuda(), is_real)
            d = crit.grad(x.cuda(), is_real, g)
            assert v.shape == () and v.is_cuda and d.shape == x.shape
            p = x.double().requires_grad_()
            ref = loss64(p, is_real, mode, labels)
            (g * ref).backward()
            assert abs(float(v) - float(ref)) <= 1e-5 * abs(float(ref)), (shape, float(v), float(ref))
            assert rel(d, p.grad) <= 1e-6, (shape, g)


class _no_tf32:
    """torch's fp32 reference runs in true fp32 (no TF32 tensor-core rounding)"""

    def __enter__(self):
        self.saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False

    def __exit__(self, *exc):
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.saved


def _model(tmp_path, **over):
    opt = synth.train_options(gpu_ids=[0], checkpoints_dir=str(tmp_path), **over)
    torch.manual_seed(0)
    m = Pix2PixModel(opt)
    m.setup(opt)
    m.netG.load_state_dict(synth.synthetic_generator_state_dict())
    m.train()
    m.set_input(synth.synthetic_train_batch(n=2, seed=7))
    return m


def _record(monkeypatch):
    """wraps GANLoss.__call__ / .grad: (logits, is_real, value) and (logits, is_real, g, seed) of every call, in order"""
    values, seeds = [], []
    call, grad = networks.GANLoss.__call__, networks.GANLoss.grad

    def rec_call(self, prediction, target_is_real):
        v = call(self, prediction, target_is_real)
        values.append((prediction.detach().clone(), target_is_real, v))
        return v

    def rec_grad(self, prediction, target_is_real, g=1.0):
        d = grad(self, prediction, target_is_real, g)
        seeds.append((prediction.detach().clone(), target_is_real, g, d))
        return d

    monkeypatch.setattr(networks.GANLoss, "__call__", rec_call)
    monkeypatch.setattr(networks.GANLoss, "grad", rec_grad)
    return values, seeds


@pytest.mark.parametrize("norm", ["batch", "none"])
@pytest.mark.parametrize("gan_mode", ["lsgan", "wgangp"])
def test_training_step(gan_mode, norm, tmp_path, monkeypatch):
    """One optimize_parameters() at n = 2 in fp32 mode with the bars of test_gpu_dnorm.test_training_step: each discriminator's
    losses and gradient against float64 autograd of 0.5 * (L(D(fake), False) + L(D(real), True)) on the model's own inputs with the
    pre-step weights, each tensor within max(1e-3, 2 x the error of torch's own fp32 autograd on the GPU).  The logit conv's bias
    gradient (one number) is bounded absolutely by 2^-20 * sum|dL/dlogit|: with WGAN it is 0 in exact arithmetic (the fake and
    real passes contribute +0.5 and -0.5), so only rounding is left to compare.  The G phase: the seeds GANLoss.grad hands to the
    tape of D_1 and D_3, and loss_G_GAN, against float64 on the logits the step produced.  Then the bf16 step: losses within 1 % of
    the fp32 step, whole-gradient cosine per net >= 0.999 (>= 0.998 where the fp32 gradient itself is more than 1e-4 from float64).

    WGAN with BatchNorm is held to less.  Its seed dL/dlogit is the same number everywhere, and a batch-statistics BatchNorm maps
    every input to outputs of zero mean, so its backward removes that uniform part exactly: the discriminator's gradient is the small
    remainder of much larger terms.  Its value then moves with the forward's activations far more than under LSGAN, where the seed
    varies with the logit.  The bf16 forward rounds those activations to 8 mantissa bits, and the cosine of the whole gradient to the
    fp32 step comes out 0.97975 for D_1 and 0.99790 for D_3 (LSGAN, same nets and batch: 0.99945 and 0.99932; D_2, whose fp32
    gradient is within 1e-5 of float64, 0.99970).  Those two nets, the ones whose fp32 gradient is more than 1e-4 from float64, are held
    to cosine >= 0.97; every other net of that step to the rule above."""
    nets = ("netD_1", "netD_2", "netD_3")
    m = _model(tmp_path, gan_mode=gan_mode, norm=norm)
    assert m.criterionGAN.gan_mode == gan_mode
    values, seeds = _record(monkeypatch)
    pre = {a: copy.deepcopy(getattr(m, a)).cpu() for a in nets}
    m.optimize_parameters()
    torch.cuda.synchronize()
    pairs = {"netD_1": (m.fake_B, m.real_B), "netD_2": (m.fake_B_mask_raw, m.real_B_mask), "netD_3": (m.fake_B_local, m.real_B_local)}
    worst32 = {}
    for k, a in enumerate(nets, start=1):
        grads, logits = {}, {}
        for dt in (torch.float64, torch.float32):
            dev = "cpu" if dt == torch.float64 else "cuda"
            ref = copy.deepcopy(pre[a].model).to(device=dev, dtype=dt)
            fake, real = (t.detach().to(device=dev, dtype=dt) for t in pairs[a])
            with _no_tf32():
                pf, pr = ref(fake), ref(real)
            pf.retain_grad()
            pr.retain_grad()
            lf, lr = loss64(pf, False, gan_mode), loss64(pr, True, gan_mode)
            with _no_tf32():
                (0.5 * (lf + lr)).backward()
            grads[dt] = {"model." + n_: p.grad.cpu() for n_, p in ref.named_parameters()}
            logits[dt] = (pf.grad.cpu(), pr.grad.cpu(), lf.detach().cpu(), lr.detach().cpu())
        pfg, prg, lf, lr = logits[torch.float64]
        assert abs(float(getattr(m, "loss_D_fake_%d" % k)) - float(lf)) <= 1e-5, (a, "fake", float(getattr(m, "loss_D_fake_%d" % k)), float(lf))
        assert abs(float(getattr(m, "loss_D_real_%d" % k)) - float(lr)) <= 1e-5, (a, "real", float(getattr(m, "loss_D_real_%d" % k)), float(lr))
        got = {n_: p.grad.cpu() for n_, p in getattr(m, a).named_parameters()}
        for key, want in grads[torch.float64].items():
            if want.numel() == 1:
                bound = 2.0 ** -20 * float(pfg.abs().sum() + prg.abs().sum())
                assert abs(float(got[key]) - float(want)) <= bound, (a, key, float(got[key]), float(want), bound)
            else:
                e, e32 = rel(got[key], want), rel(grads[torch.float32][key], want)
                print(f"{gan_mode} {norm} {a} {key}: relative error {e:.2e} (torch fp32 on the GPU: {e32:.2e})")
                worst32[a] = max(worst32.get(a, 0.0), e32)
                assert e <= max(1e-3, 2 * e32), (a, key, e, e32)
    # the G phase: D_1(fake_B), D_2(fake_B_mask_raw), D_3(fake_B_local), all against True, in that order
    g_values = values[-3:]
    assert [r for _, r, _ in g_values] == [True] * 3
    want = sum(float(loss64(p.double().cpu(), True, gan_mode)) for p, _, _ in g_values) / 6
    assert abs(float(m.loss_G_GAN) - want) <= 1e-5, (float(m.loss_G_GAN), want)
    g_seeds = seeds[-2:]                         # D_1's and D_3's tapes; D_2's input is thresholded, so it seeds nothing
    assert [(r, g) for _, r, g, _ in g_seeds] == [(True, 1.0 / 6)] * 2
    assert torch.equal(g_seeds[0][0], g_values[0][0]) and torch.equal(g_seeds[1][0], g_values[2][0])
    for p, _, _, d in g_seeds:
        p64 = p.double().cpu().requires_grad_()
        (loss64(p64, True, gan_mode) / 6).backward()
        assert rel(d, p64.grad) <= 1e-6, rel(d, p64.grad)
    # the tensor-core training mode, same weights and batch
    monkeypatch.undo()
    try:
        m16 = _model(tmp_path, gan_mode=gan_mode, norm=norm, precision="bf16")
        m16.optimize_parameters()
        torch.cuda.synchronize()
    finally:
        T.BACKWARD_PRECISION = T.FORWARD_PRECISION = "fp32"
    l32, l16 = m.get_current_losses(), m16.get_current_losses()
    ref = np.array(list(l32.values()))
    got = np.array([l16[k] for k in l32])
    assert np.abs(got - ref).max() <= 1e-2 * np.maximum(1.0, np.abs(ref)).max(), dict(zip(l32, zip(got, ref)))
    cos = {}
    for a in nets + ("netG",):
        ga = torch.cat([p.grad.double().flatten() for p in getattr(m16, a).parameters()])
        ra = torch.cat([p.grad.double().flatten() for p in getattr(m, a).parameters()])
        cos[a] = float(ga @ ra / (ga.norm() * ra.norm()))
        print(f"{gan_mode} {norm}: bf16 step {a}: whole-gradient cosine {cos[a]:.6f}, norm ratio {float(ga.norm() / ra.norm()):.5f}")
    for a, c in cos.items():
        ill = worst32.get(a, 0.0) > 1e-4
        floor = (0.97 if gan_mode == "wgangp" and norm == "batch" else 0.998) if ill else 0.999
        assert c >= floor, (a, c, worst32.get(a))


def test_scheduled_lr_reaches_the_adam_kernel(tmp_path, capsys):
    """lr_policy='step' with lr_decay_iters=1: one update_learning_rate() multiplies every optimiser's lr by 0.1, and D_1's first
    Adam step (lr * g / (|g| + eps) = lr * sign(g) where |g| >> eps) moves its weights 0.1 times as far as without the update.  The
    comparison keeps weights below 2^-6 in magnitude, where the fp32 rounding of the stored weight is below 3e-5 of the step."""
    base = _model(tmp_path, lr_policy="step", lr_decay_iters=1)
    sched = _model(tmp_path, lr_policy="step", lr_decay_iters=1)
    sched.update_learning_rate()
    lr = sched.opt.lr
    assert capsys.readouterr().out == "learning rate %.7f -> %.7f\n" % (lr, lr * 0.1)
    assert [o.param_groups[0]["lr"] for o in sched.optimizers] == [lr * 0.1] * 4
    assert [o.param_groups[0]["lr"] for o in base.optimizers] == [lr] * 4
    w0 = {n_: p.detach().clone() for n_, p in base.netD_1.named_parameters()}
    assert all(torch.equal(w0[n_], p) for n_, p in sched.netD_1.named_parameters())
    base.optimize_parameters()
    sched.optimize_parameters()
    torch.cuda.synchronize()
    checked = 0
    for (n_, pb), (_, ps) in zip(base.netD_1.named_parameters(), sched.netD_1.named_parameters()):
        db, ds = (pb.detach() - w0[n_]).double(), (ps.detach() - w0[n_]).double()
        keep = (pb.grad.abs() > 1e-5) & (ps.grad.abs() > 1e-5) & (w0[n_].abs() < 2.0 ** -6)
        assert bool((db[keep].abs() > 0.5 * lr).all()), n_
        err = ((ds[keep] - 0.1 * db[keep]).abs() / (0.1 * db[keep].abs())).max() if bool(keep.any()) else 0.0
        assert float(err) <= 1e-4, (n_, float(err))
        checked += int(keep.sum())
    assert checked > 100_000, checked
