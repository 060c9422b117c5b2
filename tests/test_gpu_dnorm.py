"""GPU checks of the PatchGAN discriminator with norm='instance' and norm='none' (reference models/networks.py:555-602): the fused
InstanceNorm + LeakyReLU kernels (hv_in_lrelu_fwd / _bwd), the discriminator in both precisions and one Pix2PixModel training step,
against float64 torch autograd.

Bias gradients before an InstanceNorm are zero in exact arithmetic (each normalised plane's gradient sums to zero); the kernels return
fp32 rounding noise, as the reference does.  They are bounded absolutely per channel by n * hw * 2^-20 * max|g|, where g is the
per-element gradient the bias sums (the gradient w.r.t. the normalised layer's input), and are never compared relatively."""
import copy

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from healthivert_gan_b200 import networks, train_ops as T
from healthivert_gan_b200.pix2pix_model import Pix2PixModel
from oracle import synth

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def bias_bound(g):
    """per-channel bound on a pre-InstanceNorm bias gradient; g: [n, c, h, w] gradient the bias sums"""
    n, c, h, w = g.shape
    return n * h * w * 2.0 ** -20 * g.detach().abs().amax(dim=(0, 2, 3)).double().cpu()


@pytest.mark.parametrize("with_bias", [False, True])
@pytest.mark.parametrize("shape", [(16, 128, 64, 64), (16, 256, 32, 32), (16, 512, 31, 31), (2, 128, 75, 75), (3, 8, 5, 7)])
def test_in_lrelu_kernels_against_float64_autograd(shape, with_bias):
    """(16,128,64,64) / (16,256,32,32) / (16,512,31,31) are the batch-16 discriminator's planes (16-byte and scalar loads); 75 x 75 is
    above the on-chip plane size (the streaming variant); 5 x 7 is ragged.  The float64 reference takes the LeakyReLU's branch from the
    kernel's own y: where |xhat| is within fp32 rounding of 0 the two could pick different branches, and each such element would move
    dx by 0.8 |dy| invstd (about 3e-4 relative L2 for one flip in 8M elements) without either being wrong."""
    n, c, h, w = shape
    g = torch.Generator().manual_seed(n * c + h)
    x = torch.randn(shape, generator=g) * 3 + 0.5
    dy = torch.randn(shape, generator=g)
    bias = torch.randn(c, generator=g) if with_bias else None
    xv = T.Var(x.cuda())
    bp = nn.Parameter(bias.cuda()) if with_bias else None
    tape = T.Tape()
    out = T.in_lrelu(tape, xv, bp, 0.2, 1e-5)
    out.grad = dy.cuda()
    tape.backward()
    torch.cuda.synchronize()
    yk = out.data.cpu()

    x64 = x.double().requires_grad_()
    b64 = bias.double().requires_grad_() if with_bias else None
    pre = x64 + b64.view(1, c, 1, 1) if with_bias else x64
    xhat = F.instance_norm(pre, eps=1e-5)
    assert rel(yk, F.leaky_relu(xhat, 0.2).detach()) <= 1e-5
    y_branch = xhat * torch.where(yk > 0, 1.0, 0.2).double()
    y_branch.backward(dy.double())
    assert rel(xv.grad, x64.grad) <= 1e-5
    if with_bias:
        db = bp.grad.double().cpu()
        assert float(b64.grad.abs().max()) <= 1e-9                   # zero in exact arithmetic
        assert bool((db.abs() <= bias_bound(x64.grad)).all()), float((db.abs() / bias_bound(x64.grad)).max())


def _net(norm, seed=3, random_bias=True):
    torch.manual_seed(seed)
    net = networks.define_D(1, 64, "basic", 3, norm, "normal", 0.02, [])
    if random_bias:       # the reference initialises biases to 0; random ones exercise the bias paths (they cancel in the norm)
        with torch.no_grad():
            for m in net.model:
                if isinstance(m, nn.Conv2d) and m.bias is not None:
                    m.bias.normal_(0.0, 0.05)
    return net


def _keep_output(store, idx):
    """forward hook: keep the module's output (one per call) with its gradient retained"""
    def hook(mod, inp, out):
        out.retain_grad()
        store.setdefault(idx, []).append(out)
    return hook


def _torch_ref(net, x, train):
    """float64 autograd of the same module objects on CPU copies; returns logits, input gradient, parameter gradients and the
    gradients w.r.t. the outputs of the convs that feed an InstanceNorm (for the bias bound)."""
    ref = copy.deepcopy(net.model).cpu().double().train(train)
    for p in ref.parameters():
        p.grad = None
    conv_out = {}
    for i, m in enumerate(ref):
        if isinstance(m, nn.InstanceNorm2d):
            ref[i - 1].register_forward_hook(_keep_output(conv_out, i - 1))
    x64 = x.double().requires_grad_()
    y = ref(x64)
    F.binary_cross_entropy_with_logits(y, torch.ones_like(y)).backward()
    grads = {"model." + k: p.grad for k, p in ref.named_parameters()}
    return y.detach(), x64.grad, grads, {"model.%d.bias" % i: o[0].grad for i, o in conv_out.items()}


def _run(net, x):
    crit = networks.GANLoss("vanilla").cuda()
    for p in net.parameters():
        p.grad = None
    tape = T.Tape()
    xv = T.Var(x.cuda())
    out = net.run(xv, tape)
    out.grad = crit.grad(out.data, True, 1.0)
    tape.backward()
    torch.cuda.synchronize()
    return out.data.cpu(), xv.grad.cpu(), {k: p.grad.cpu() for k, p in net.named_parameters()}


def _check_grads(got, want, conv_out_grads, tol):
    for k, g in want.items():
        if k in conv_out_grads:
            assert bool((got[k].double().abs() <= bias_bound(conv_out_grads[k])).all()), k
        else:
            assert rel(got[k], g) <= tol, (k, rel(got[k], g))


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("norm", ["instance", "none"])
def test_discriminator_fp32_against_float64_autograd(norm, train):
    """fp32 parity mode (SIMT convs; 'none' fuses the LeakyReLU into the conv) with the bars of the BatchNorm discriminator's test."""
    net = _net(norm).cuda().train(train)
    x = torch.randn(2, 1, 256, 256, generator=torch.Generator().manual_seed(8))
    y, dx, grads = _run(net, x)
    ry, rdx, rgrads, conv_out = _torch_ref(net, x, train)
    assert y.shape == (2, 1, 30, 30)
    assert rel(y, ry) <= 1e-4
    assert rel(dx, rdx) <= 1e-3
    _check_grads(grads, rgrads, conv_out, 1e-3)


def _f64(t):
    return t.detach().double().cpu()


@pytest.mark.parametrize("norm", ["instance", "none"])
def test_discriminator_bf16_takes_the_tensor_cores(norm, monkeypatch):
    """bf16 mode: layers 2-4 run on T.conv2d_tc.  Each of the three convs is pinned to float64 on its own bf16-rounded operands (the
    fp32 input the kernel received, rounded to bf16 as its im2col does, and the bf16-rounded weight), and the logits to a float64 run
    of the remaining modules from the last tensor-core conv's own output.  A float64 restatement that rounds from its OWN upstream
    values instead drifts by 3.5e-4 ('none') to 5.0e-4 ('instance') relative L2 in the logits: a 1e-7 difference upstream moves a
    few 1e-5 of the operands across a bf16 rounding boundary (2^-8 each), and those moves grow from layer to layer.  Against this
    library's fp32 mode the whole gradient keeps cosine >= 0.999 and its norm within 1 %."""
    calls = []
    real = T.conv2d_tc

    def counting(tape, x, weight, stride, *a, **k):
        out = real(tape, x, weight, stride, *a, **k)
        calls.append((x.data.clone(), weight.clone(), stride, out.data.clone()))
        return out

    monkeypatch.setattr(T, "conv2d_tc", counting)
    x = torch.randn(2, 1, 256, 256, generator=torch.Generator().manual_seed(9))
    net = _net(norm).cuda().train()
    _, _, g32 = _run(net, x)
    assert not calls
    net.precision = "bf16"
    y16, _, g16 = _run(net, x)
    assert [tuple(c[1].shape[:2]) for c in calls] == [(128, 64), (256, 128), (512, 256)]
    bf = lambda t: _f64(t.float().to(torch.bfloat16))
    for xin, w, stride, yk in calls:
        want = F.conv2d(bf(xin), bf(w), None, stride, 1)
        assert rel(yk, want) <= 1e-4, rel(yk, want)
    tail = copy.deepcopy(net.model).cpu().double()
    h = _f64(calls[-1][3])
    if tail[8].bias is not None:                # added on load by the norm kernel
        h = h + tail[8].bias.view(1, -1, 1, 1)
    for m in list(tail)[9:]:
        h = m(h)
    assert rel(y16, h.detach()) <= 1e-4
    a = torch.cat([g16[k].double().flatten() for k in g32])
    b = torch.cat([g32[k].double().flatten() for k in g32])
    cos = float(a @ b / (a.norm() * b.norm()))
    print(f"bf16 discriminator ({norm}): whole-gradient cosine {cos:.6f}, norm ratio {float(a.norm() / b.norm()):.5f}")
    assert cos >= 0.999 and abs(float(a.norm() / b.norm()) - 1.0) <= 0.01


class _no_tf32:
    """torch's fp32 reference runs in true fp32 (no TF32 tensor-core rounding)"""

    def __enter__(self):
        self.saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False

    def __exit__(self, *exc):
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.saved


def _model(norm, tmp_path, **over):
    opt = synth.train_options(gpu_ids=[0], norm=norm, checkpoints_dir=str(tmp_path), **over)
    torch.manual_seed(0)
    m = Pix2PixModel(opt)
    m.setup(opt)
    m.netG.load_state_dict(synth.synthetic_generator_state_dict())
    m.train()
    m.set_input(synth.synthetic_train_batch(n=2, seed=7))
    return m


@pytest.mark.parametrize("norm", ["instance", "none"])
def test_training_step(norm, tmp_path):
    """One optimize_parameters() at n = 2 in fp32 mode: each discriminator's gradient against float64 autograd of
    0.5 * (BCE(D(fake), 0) + BCE(D(real), 1)) on the model's own inputs with the pre-step weights; the bf16 mode's step against it;
    the checkpoint round trip.  The logit conv's bias gradient (one number) is the sum of both passes' logit gradients, which nearly
    cancel when D sees similar inputs: for D_2 (thresholded fake mask vs real mask) it is -1.15e-5 from terms summing to ~0.5 in
    magnitude, so fp32 summation alone moves it by 1.3e-3 relative (observed, 'none').  It is bounded absolutely instead, by
    2^-20 * sum|d loss / d logit|.  With InstanceNorm, fp32 arithmetic itself is off by more than 1e-3 here: D_3's first-layer weight
    gradient comes out 3.5e-3 from float64 both from these kernels and from torch's own fp32 autograd of the same modules on the GPU
    (cudnn, TF32 off; the two agree to the printed digits; torch on the CPU accumulates fp32 sums in fp64 and stays near 1e-6).  So each
    tensor is held to 1e-3 or to twice the error of torch's fp32 GPU autograd, whichever is larger, and both errors are printed.
    The same conditioning shows in the bf16 step: its whole-gradient cosine to the fp32 step is 0.99891 for D_1 and 0.99841 for D_3 with
    'instance' (0.9998 / 0.9999 for D_2 / G, >= 0.99976 for every net with 'none').  A net whose fp32 gradient is itself more than 1e-4
    from float64 is held to cosine >= 0.998, every other net to 0.999."""
    nets = ("netD_1", "netD_2", "netD_3")
    m = _model(norm, tmp_path)
    pre = {a: copy.deepcopy(getattr(m, a)).cpu() for a in nets}
    m.optimize_parameters()
    torch.cuda.synchronize()
    pairs = {"netD_1": (m.fake_B, m.real_B), "netD_2": (m.fake_B_mask_raw, m.real_B_mask), "netD_3": (m.fake_B_local, m.real_B_local)}
    worst32 = {}                                     # per net: the largest error of torch's own fp32 GPU autograd against float64
    for k, a in enumerate(nets, start=1):
        grads, logits, conv_out = {}, {}, {}
        for dt in (torch.float64, torch.float32):
            dev = "cpu" if dt == torch.float64 else "cuda"
            ref = copy.deepcopy(pre[a].model).to(device=dev, dtype=dt)
            for i, mod in enumerate(ref):
                if isinstance(mod, nn.Conv2d) and i + 1 < len(ref) and isinstance(ref[i + 1], nn.InstanceNorm2d) and dt == torch.float64:
                    ref[i].register_forward_hook(_keep_output(conv_out, i))
            fake, real = (t.detach().to(device=dev, dtype=dt) for t in pairs[a])
            with _no_tf32():
                pf, pr = ref(fake), ref(real)
            pf.retain_grad()
            pr.retain_grad()
            lf = F.binary_cross_entropy_with_logits(pf, torch.zeros_like(pf))
            lr = F.binary_cross_entropy_with_logits(pr, torch.ones_like(pr))
            with _no_tf32():
                (0.5 * (lf + lr)).backward()
            grads[dt] = {"model." + n_: p.grad.cpu() for n_, p in ref.named_parameters()}
            logits[dt] = (pf.grad.cpu(), pr.grad.cpu(), lf.cpu(), lr.cpu())
        pfg, prg, lf, lr = logits[torch.float64]
        assert abs(float(getattr(m, "loss_D_fake_%d" % k)) - float(lf)) <= 1e-5, (a, "fake")
        assert abs(float(getattr(m, "loss_D_real_%d" % k)) - float(lr)) <= 1e-5, (a, "real")
        got = {n_: p.grad.cpu() for n_, p in getattr(m, a).named_parameters()}
        for key, want in grads[torch.float64].items():
            idx = int(key.split(".")[1])
            if idx in conv_out and key.endswith("bias"):
                g = torch.cat([o.grad for o in conv_out[idx]])          # the bias sums over both passes
                assert bool((got[key].double().abs() <= bias_bound(g)).all()), (a, key)
            elif want.numel() == 1:
                bound = 2.0 ** -20 * float(pfg.abs().sum() + prg.abs().sum())
                assert abs(float(got[key]) - float(want)) <= bound, (a, key, float(got[key]), float(want), bound)
            else:
                e, e32 = rel(got[key], want), rel(grads[torch.float32][key], want)
                print(f"{norm} {a} {key}: relative error {e:.2e} (torch fp32 on the GPU: {e32:.2e})")
                worst32[a] = max(worst32.get(a, 0.0), e32)
                assert e <= max(1e-3, 2 * e32), (a, key, e, e32)
    # the tensor-core training mode, same weights and batch
    try:
        m16 = _model(norm, tmp_path, precision="bf16")
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
        print(f"{norm}: bf16 step {a}: whole-gradient cosine {cos[a]:.6f}, norm ratio {float(ga.norm() / ra.norm()):.5f}")
    for a, c in cos.items():
        assert c >= (0.998 if worst32.get(a, 0.0) > 1e-4 else 0.999), (a, c, worst32.get(a))
    # checkpoints: save_networks writes the reference layout, load_networks reads it back strictly
    m.save_networks("latest")
    saved = {a: {k: v.clone() for k, v in getattr(m, a).state_dict().items()} for a in nets}
    m2 = _model(norm, tmp_path)
    m2.load_networks("latest")
    for a in nets:
        sd = getattr(m2, a).state_dict()
        assert list(sd) == list(saved[a])
        assert all(torch.equal(sd[k], saved[a][k]) for k in sd), a
