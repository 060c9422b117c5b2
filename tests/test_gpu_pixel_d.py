"""GPU checks of the PixelDiscriminator (netD='pixel', reference models/networks.py:604-753) in both precisions, and of one training
step with the PatchGAN at depths 1, 2, 4 and 5 (netD='n_layers').

Parity mode (the layer kernels) is held to float64 autograd of the same modules with the bounds of the PatchGAN's test
(test_gpu_dnorm.py), including its per-channel absolute bound for a bias gradient before an InstanceNorm (zero in exact arithmetic).

The fused tensor-core kernels are held to a float64 restatement of their own roundings: h1 = lrelu(fp32(w1 x + b1)) bit for bit, h1 and
W2 rounded to bf16 in the forward, dh2, W2 and h1 rounded to bf16 in the backward, everything else float64.  Logits, the norm statistics
and the gradients that do not pass through dh2 (w3, b3, gamma, beta) meet 1e-5 relative L2.  dx, W2, w1 and b1 pass through
bf16(dh2): the kernel rounds its fp32 dh2, the restatement its float64 dh2, and the two differ by a few 1e-7 relative, so about 1e-4 of
the dh2 elements land on the other side of a bf16 rounding boundary (2^-8 relative).  That moves these tensors by about 4e-5 relative
L2 without either side being wrong; dx is held to 1e-4.  The weight gradients of W2, w1 and b1 sum products of dh2 (or of dh1 = dh2 W2)
over pixels, and a norm's backward leaves dh2 with (nearly, for BatchNorm over the batch; exactly, for InstanceNorm per plane) zero
mean, so their entries are small differences of large terms and the same flips show larger there.  Measured on a B200 at batch 16 x
256^2 and at 3 x 37 x 53: 2e-5 to 7e-5 (batch), 1.2e-4 to 2.2e-4 (instance) relative L2.  They are held to 5e-4."""
import copy

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from healthivert_gan_b200 import _lib, networks, train_ops as T
from healthivert_gan_b200._lib import ptr
from healthivert_gan_b200.pix2pix_model import Pix2PixModel
from oracle import synth

pytestmark = pytest.mark.gpu

NORMS = ["batch", "instance", "none"]


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def bias_bound(g):
    """per-channel bound on a pre-InstanceNorm bias gradient; g: [n, c, h, w] gradient the bias sums"""
    n, c, h, w = g.shape
    return n * h * w * 2.0 ** -20 * g.detach().abs().amax(dim=(0, 2, 3)).double().cpu()


def _net(norm, seed=4):
    torch.manual_seed(seed)
    net = networks.define_D(1, 64, "pixel", 3, norm, "normal", 0.02, [])
    with torch.no_grad():      # random biases and BatchNorm affine exercise every parameter path
        for m in net.net:
            if isinstance(m, nn.Conv2d):
                m.weight.normal_(0.0, 0.2)
                if m.bias is not None:
                    m.bias.normal_(0.0, 0.1)
            elif isinstance(m, nn.BatchNorm2d):
                m.weight.normal_(1.0, 0.2)
                m.bias.normal_(0.0, 0.2)
                m.running_mean.normal_(0.0, 0.1)
                m.running_var.uniform_(0.5, 1.5)
    return net.cuda().train()


def _inputs(shape, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g).clamp(-3, 3)
    dy = torch.randn(shape[0], 1, shape[2], shape[3], generator=g) / (shape[0] * shape[2] * shape[3]) ** 0.5
    return x.cuda(), dy.cuda()


def _run(net, x, dy, param_grads=True, want_dx=True):
    for p in net.parameters():
        p.grad = None
    tape = T.Tape()
    xv = T.Var(x.clone(), requires_grad=want_dx)
    out = net.run(xv, tape, param_grads=param_grads)
    out.grad = dy
    tape.backward()
    torch.cuda.synchronize()
    grads = {k: p.grad.clone() for k, p in net.named_parameters() if p.grad is not None}
    return out.data.clone(), (xv.grad.clone() if want_dx else None), grads


@pytest.mark.parametrize("shape", [(16, 1, 256, 256), (3, 1, 37, 53)])
@pytest.mark.parametrize("norm", NORMS)
def test_parity_mode_against_float64_autograd(norm, shape):
    net = _net(norm)
    x, dy = _inputs(shape, 1)
    ref = copy.deepcopy(net.net).double()
    y, dx, grads = _run(net, x, dy)
    conv_out = []

    def keep(mod, inp, out):
        out.retain_grad()
        conv_out.append(out)

    if norm == "instance":
        ref[2].register_forward_hook(keep)
    x64 = x.double().requires_grad_()
    ry = ref(x64)
    ry.backward(dy.double())
    assert y.shape == (shape[0], 1, shape[2], shape[3])
    assert rel(y, ry) <= 1e-4
    assert rel(dx, x64.grad) <= 1e-3
    for k, p in ref.named_parameters():
        key = "net." + k
        if norm == "instance" and key == "net.2.bias":
            assert bool((grads[key].double().cpu().abs() <= bias_bound(conv_out[0].grad)).all()), key
        else:
            assert rel(grads[key], p.grad) <= 1e-3, (key, rel(grads[key], p.grad))
    if norm == "batch":
        assert rel(net.net[3].running_mean, ref[3].running_mean) <= 1e-4
        assert rel(net.net[3].running_var, ref[3].running_var) <= 1e-4
        assert int(net.net[3].num_batches_tracked) == 1


def _bf(t):
    return t.float().to(torch.bfloat16).double()


def _restate(net, x, dy, norm):
    """float64 restatement of the fused kernels' own roundings: (logits, dx, parameter gradients, (mean, biased var))"""
    c1, c2, c3 = net.net[0], net.net[2], net.net[5]
    w1, b1 = c1.weight.detach().view(1, 64, 1, 1), c1.bias.detach().view(1, 64, 1, 1)
    pre1 = (x.double() * w1.double() + b1.double()).float()                  # fmaf: the exact product-sum rounded once
    h1 = torch.where(pre1 > 0, pre1, pre1 * 0.2)                              # fp32 LeakyReLU, as the kernel
    h1b = _bf(h1)
    w2b = _bf(c2.weight.detach().view(128, 64))
    h2 = torch.einsum("nchw,dc->ndhw", h1b, w2b)
    if c2.bias is not None:
        h2 = h2 + c2.bias.detach().double().view(1, 128, 1, 1)
    dims = (0, 2, 3) if norm == "batch" else (2, 3)
    stats = None
    if norm == "none":
        xhat, z = None, h2
    else:
        mu = h2.mean(dims, keepdim=True)
        var = ((h2 - mu) ** 2).mean(dims, keepdim=True)
        eps = net.net[3].eps
        inv = 1.0 / torch.sqrt(var + eps)
        xhat = (h2 - mu) * inv
        if norm == "batch":
            gam = net.net[3].weight.detach().double().view(1, 128, 1, 1)
            z = gam * xhat + net.net[3].bias.detach().double().view(1, 128, 1, 1)
        else:
            gam = torch.ones(1, 128, 1, 1, dtype=torch.float64, device=x.device)
            z = xhat
        stats = (mu, var)
    a = torch.where(z > 0, z, 0.2 * z)
    w3 = c3.weight.detach().double().view(1, 128, 1, 1)
    y = (a * w3).sum(1, keepdim=True)
    if c3.bias is not None:
        y = y + c3.bias.detach().double()
    g = dy.double()
    grads = {"net.5.weight": (g * a).sum((0, 2, 3)).view(1, 128, 1, 1)}
    if c3.bias is not None:
        grads["net.5.bias"] = g.sum().view(1)
    dz = g * w3 * torch.where(z > 0, 1.0, 0.2)
    if norm == "none":
        dh2 = dz
    else:
        s1 = dz.sum(dims, keepdim=True)
        s2 = (dz * xhat).sum(dims, keepdim=True)
        m = h2.numel() // 128 if norm == "batch" else h2.shape[2] * h2.shape[3]
        dh2 = inv * (gam * dz - gam * s1 / m - xhat * gam * s2 / m)
        if norm == "batch":
            grads["net.3.weight"] = s2.view(128)
            grads["net.3.bias"] = s1.view(128)
    if c2.bias is not None:
        grads["net.2.bias"] = dh2.sum((0, 2, 3))
    dh2b = _bf(dh2)
    grads["net.2.weight"] = torch.einsum("ndhw,nchw->dc", dh2b, h1b).view(128, 64, 1, 1)
    dh1 = torch.einsum("ndhw,dc->nchw", dh2b, w2b)
    dpre1 = dh1 * torch.where(pre1 > 0, 1.0, 0.2)
    grads["net.0.weight"] = (dpre1 * x.double()).sum((0, 2, 3)).view(64, 1, 1, 1)
    grads["net.0.bias"] = dpre1.sum((0, 2, 3))
    dx = (dpre1 * w1.double()).sum(1, keepdim=True)
    return y, dx, grads, stats, dh2


def _check_fused(net, x, dy, norm, param_grads=True, want_dx=True):
    rm0 = net.net[3].running_mean.clone() if norm == "batch" else None
    rv0 = net.net[3].running_var.clone() if norm == "batch" else None
    y, dx, grads = _run(net, x, dy, param_grads, want_dx)
    ry, rdx, rgrads, stats, dh2 = _restate(net, x, dy, norm)
    assert rel(y, ry) <= 1e-5, rel(y, ry)
    if want_dx:
        assert rel(dx, rdx) <= 1e-4, rel(dx, rdx)
        print(f"{norm} {tuple(x.shape)}: dx relative L2 {rel(dx, rdx):.2e}")
    else:
        assert dx is None
    if not param_grads:
        assert not grads
    else:
        assert set(grads) == set(rgrads), set(grads) ^ set(rgrads)
        for k, want in rgrads.items():
            if k == "net.2.bias":      # before InstanceNorm: zero up to rounding
                assert bool((grads[k].double().cpu().abs() <= bias_bound(dh2)).all()), k
                continue
            tol = 1e-5 if k in ("net.5.weight", "net.5.bias", "net.3.weight", "net.3.bias") else 5e-4
            e = rel(grads[k], want.view(grads[k].shape))
            print(f"{norm} {tuple(x.shape)} {k}: relative L2 {e:.2e}")
            assert e <= tol, (k, e)
    if norm == "batch":
        mom = net.net[3].momentum
        mu, var = stats
        cnt = x.numel()
        m_impl = (net.net[3].running_mean.double() - (1 - mom) * rm0.double()) / mom
        v_impl = (net.net[3].running_var.double() - (1 - mom) * rv0.double()) / mom
        assert rel(m_impl, mu.view(128)) <= 1e-5, rel(m_impl, mu.view(128))
        assert rel(v_impl, var.view(128) * cnt / (cnt - 1)) <= 1e-5


@pytest.mark.parametrize("shape", [(16, 1, 256, 256), (3, 1, 37, 53)])
@pytest.mark.parametrize("norm", NORMS)
def test_fused_against_float64_restatement(norm, shape):
    net = _net(norm)
    net.precision = "bf16"
    x, dy = _inputs(shape, 2)
    _check_fused(net, x, dy, norm)


@pytest.mark.parametrize("norm", NORMS)
def test_fused_without_parameter_gradients_or_dx(norm):
    net = _net(norm)
    net.precision = "bf16"
    x, dy = _inputs((2, 1, 40, 45), 3)
    _check_fused(net, x, dy, norm, param_grads=False, want_dx=True)
    _check_fused(net, x, dy, norm, param_grads=True, want_dx=False)


@pytest.mark.parametrize("spread", ["wide", "narrow"])
@pytest.mark.parametrize("norm", ["batch", "instance"])
def test_fused_statistics(norm, spread):
    """the per-channel (batch) or per-(sample, channel) (instance) mean and inverse standard deviation the forward saves.  'narrow':
    b1 near 3 and w1 near 0 make every channel's mean about 300 times its standard deviation, where a one-pass E[h^2] - E[h]^2 in fp32
    loses the variance; the kernels' shifted sums must still meet 1e-5."""
    net = _net(norm)
    if spread == "narrow":
        with torch.no_grad():
            net.net[0].weight.normal_(0.0, 0.01)
            net.net[0].bias.normal_(3.0, 0.1)
    x, _ = _inputs((3, 1, 37, 53), 5)
    n, _, h, w = x.shape
    c1, c2, c3, nm = net.net[0], net.net[2], net.net[5], net.net[3]
    kind = 1 if norm == "batch" else 2
    d = lambda t: t.detach().contiguous() if t is not None else None
    L = _lib.lib()
    ws = torch.empty(L.hv_pixel_d_workspace_bytes(n, h, w), device="cuda", dtype=torch.uint8)
    y = torch.empty(n, 1, h, w, device="cuda")
    k = 128 * (n if kind == 2 else 1)
    mean, invstd = torch.empty(k, device="cuda"), torch.empty(k, device="cuda")
    gamma, beta = (d(nm.weight), d(nm.bias)) if kind == 1 else (None, None)
    _lib.check(L.hv_pixel_d_fwd_bf16(ptr(x), ptr(d(c1.weight)), ptr(d(c1.bias)), ptr(d(c2.weight)), ptr(d(c2.bias)), ptr(gamma),
                                     ptr(beta), ptr(d(c3.weight)), ptr(d(c3.bias)), None, None, ptr(y), ptr(mean), ptr(invstd), n, 1, 64,
                                     h, w, kind, 0.1, 1e-5, 0.2, ptr(ws), _lib.stream()))
    torch.cuda.synchronize()
    _, _, _, (mu, var), _ = _restate(net, x, torch.zeros_like(y), norm)
    ratio = float((mu.abs() / var.sqrt()).median())
    print(f"{norm} {spread}: median |mean| / std {ratio:.1f}, invstd relative L2 {rel(invstd, (1.0 / torch.sqrt(var + 1e-5)).reshape(-1)):.2e}")
    assert spread == "wide" or ratio > 100
    assert rel(mean, mu.reshape(-1)) <= 1e-5
    assert rel(invstd, (1.0 / torch.sqrt(var + 1e-5)).reshape(-1)) <= 1e-5


def test_fused_rejects_unbuilt_geometries():
    L = _lib.lib()
    x = torch.zeros(1, 1, 8, 8, device="cuda")
    for cin, ndf, norm, what in ((3, 64, 0, "input_nc"), (1, 32, 0, "ndf"), (1, 64, 3, "norm")):
        with pytest.raises(_lib.HvError, match=what):
            _lib.check(L.hv_pixel_d_fwd_bf16(ptr(x), ptr(x), ptr(x), ptr(x), None, None, None, ptr(x), None, None, None, ptr(x), ptr(x),
                                             ptr(x), 1, cin, ndf, 8, 8, norm, 0.1, 1e-5, 0.2, ptr(x), _lib.stream()))


def test_other_widths_take_the_layer_path(monkeypatch):
    torch.manual_seed(1)
    net = networks.define_D(1, 32, "pixel", 3, "instance", "normal", 0.02, []).cuda().train()
    net.precision = "bf16"
    monkeypatch.setattr(T, "pixel_d", lambda *a, **k: pytest.fail("the fused kernels take ndf = 64 only"))
    x, dy = _inputs((2, 1, 16, 16), 6)
    y, _, _ = _run(net, x, dy)
    assert rel(y, copy.deepcopy(net.net).double()(x.double())) <= 1e-4


def test_eval_mode_batchnorm_raises():
    for prec in ("fp32", "bf16"):
        net = _net("batch").eval()
        net.precision = prec
        with pytest.raises(NotImplementedError):
            net.run(torch.zeros(1, 1, 8, 8, device="cuda"))


@pytest.mark.parametrize("norm", NORMS)
def test_fused_is_deterministic(norm):
    net = _net(norm)
    net.precision = "bf16"
    x, dy = _inputs((16, 1, 256, 256), 7)
    a = _run(net, x, dy)
    b = _run(net, x, dy)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert all(torch.equal(a[2][k], b[2][k]) for k in a[2])


def _peak(net, x, dy):
    _run(net, x, dy)          # warm-up: workspaces and allocator blocks of the first call
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    _run(net, x, dy)
    return torch.cuda.max_memory_allocated() - base


def test_fused_keeps_the_maps_on_chip():
    x, dy = _inputs((16, 1, 256, 256), 8)
    net = _net("batch")
    net.precision = "bf16"
    fused = _peak(net, x, dy)
    net.precision = "fp32"
    layers = _peak(net, x, dy)
    print(f"peak extra memory of one forward + backward at 16 x 256^2: fused {fused / 2**20:.1f} MiB, layer path {layers / 2**20:.1f} MiB")
    assert fused <= 64 * 2 ** 20
    assert layers > 2 ** 30


def _model(tmp_path, **over):
    opt = synth.train_options(gpu_ids=[0], checkpoints_dir=str(tmp_path), **over)
    torch.manual_seed(0)
    m = Pix2PixModel(opt)
    m.setup(opt)
    m.netG.load_state_dict(synth.synthetic_generator_state_dict())
    m.train()
    m.set_input(synth.synthetic_train_batch(n=2, seed=7))
    return m


class _no_tf32:
    """torch's fp32 reference runs in true fp32 (no TF32 tensor-core rounding)"""

    def __enter__(self):
        self.saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False

    def __exit__(self, *exc):
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.saved


NETS = ("netD_1", "netD_2", "netD_3")


def _pairs(m):
    return {"netD_1": (m.fake_B, m.real_B), "netD_2": (m.fake_B_mask_raw, m.real_B_mask), "netD_3": (m.fake_B_local, m.real_B_local)}


def _seq(net):
    return net.net if isinstance(net, networks.PixelDiscriminator) else net.model


def _fp32_conditioning(pre, pairs):
    """per discriminator: the largest relative L2 error, over its weight tensors, of torch's own fp32 autograd on the GPU (TF32 off)
    against float64 autograd, for 0.5 * (BCE(D(fake), 0) + BCE(D(real), 1)) on the step's inputs with the pre-step weights - the measure
    test_gpu_dnorm.py and test_gpu_gan_modes.py use to tell an ill-conditioned net.  Single numbers (the logit bias) and the biases in
    front of an InstanceNorm (zero in exact arithmetic) are left out, as there."""
    worst = {}
    for a in NETS:
        grads = {}
        for dt, dev in ((torch.float64, "cpu"), (torch.float32, "cuda")):
            ref = copy.deepcopy(_seq(pre[a])).to(device=dev, dtype=dt).train()
            fake, real = (t.detach().to(device=dev, dtype=dt) for t in pairs[a])
            with _no_tf32():
                pf, pr = ref(fake), ref(real)
                loss = 0.5 * (F.binary_cross_entropy_with_logits(pf, torch.zeros_like(pf))
                              + F.binary_cross_entropy_with_logits(pr, torch.ones_like(pr)))
                loss.backward()
            skip = {"%d.bias" % i for i in range(len(ref) - 1) if isinstance(ref[i + 1], nn.InstanceNorm2d)}
            grads[dt] = {k: p.grad.cpu() for k, p in ref.named_parameters() if k not in skip and p.numel() > 1}
        worst[a] = max(rel(grads[torch.float32][k], grads[torch.float64][k]) for k in grads[torch.float64])
    return worst


def _fused_vs_rounding_model(pre16, pairs16, norm, m32):
    """each pixel discriminator's bf16 gradient of the step, recomputed from the pre-step weights and the bf16 step's own inputs, against
    the float64 restatement of the fused kernels' roundings (_restate).  Returns, per net, (relative L2 of the whole gradient between the
    kernels and their rounding model, cosine of the rounding model's gradient to the fp32 step's)."""
    crit = networks.GANLoss("vanilla").cuda()
    out = {}
    for a in NETS:
        net = copy.deepcopy(pre16[a]).cuda().train()
        net.precision = "bf16"
        got, want = {}, {}
        for x, real in zip(pairs16[a], (False, True)):
            x = x.detach().clone()
            dy = crit.grad(net.run(x).data, real, 0.5)
            _, _, grads = _run(net, x, dy, want_dx=False)
            _, _, rgrads, _, _ = _restate(net, x, dy, norm)
            for k, g in grads.items():
                got[k] = got.get(k, 0) + g.double()
                want[k] = want.get(k, 0) + rgrads[k].view(g.shape)
        keys = sorted(got)
        ga = torch.cat([got[k].flatten() for k in keys]).cpu()
        wa = torch.cat([want[k].flatten() for k in keys]).cpu()
        ra = torch.cat([getattr(m32, a).get_parameter(k).grad.double().flatten() for k in keys]).cpu()
        out[a] = (rel(ga, wa), float(wa @ ra / (wa.norm() * ra.norm())))
    return out


def _step_pair(tmp_path, **over):
    """one optimize_parameters() in fp32 and in bf16 from the same weights and batch, held to the tensor-core rule of the other
    training-step tests: losses within 1 %, each net's whole gradient with cosine >= 0.999 to the fp32 step's and its norm within 1 %.
    As in test_gpu_dnorm.py / test_gpu_gan_modes.py, a discriminator whose fp32 gradient is itself more than 1e-4 from float64
    (_fp32_conditioning, measured here on the step's own inputs) is held to cosine >= 0.998; every other net keeps 0.999.

    For the pixel discriminator, each net's fused bf16 gradient is also recomputed from the pre-step weights and the bf16 step's inputs and
    held to the float64 restatement of the kernels' own roundings (relative L2 <= 5e-4, the bound of the restatement test for
    gradients that pass through bf16(dh2)).  Where that rounding model is itself below the cosine bar against the fp32 step, the bar
    becomes the model's own cosine (less 1e-5) with the norm within 3 %: measured on a B200, 'batch' D_3 (the masked centre crop) sits
    at 0.980261 and 'none' D_1 at 0.997442, the fused kernels match the model there to 1.3e-6 relative L2 and their cosine equals the
    model's to six digits, while torch's fp32 autograd on the same inputs is within 5e-5 of float64.  The deviation is the bf16 rounding
    of h1, W2 and dh2 that this mode specifies, not the kernels.

    The PatchGAN at depths 4 and 5 is held to cosine >= 0.995 and norm within 1.5 % per discriminator (measured on a B200: 0.99539 to
    0.99974, norm ratios within 1.31 %; fp32 autograd within 5e-6 of float64 there).  Its tensor-core convolutions at every geometry
    these depths add are pinned to float64 on their own bf16 operands, forward and both gradients, by
    test_patchgan_tensor_core_convs_at_every_depth; no whole-net rounding model of the PatchGAN is checked."""
    pixel = over.get("netD") == "pixel"
    deep = over.get("netD") == "n_layers" and over.get("n_layers_D", 3) >= 4
    try:
        m = _model(tmp_path, **over)
        pre = {a: copy.deepcopy(getattr(m, a)).cpu() for a in NETS}
        m.optimize_parameters()
        m16 = _model(tmp_path, precision="bf16", **over)
        pre16 = {a: copy.deepcopy(getattr(m16, a)) for a in NETS}
        m16.optimize_parameters()
        torch.cuda.synchronize()
    finally:
        T.BACKWARD_PRECISION = T.FORWARD_PRECISION = "fp32"
    l32, l16 = m.get_current_losses(), m16.get_current_losses()
    assert all(np.isfinite(v) for v in l32.values()) and all(np.isfinite(v) for v in l16.values())
    ref = np.array(list(l32.values()))
    got = np.array([l16[k] for k in l32])
    assert np.abs(got - ref).max() <= 1e-2 * np.maximum(1.0, np.abs(ref)).max(), dict(zip(l32, zip(got, ref)))
    worst32 = _fp32_conditioning(pre, _pairs(m))
    model = _fused_vs_rounding_model(pre16, _pairs(m16), over.get("norm", "batch"), m) if pixel else {}
    bad = []
    for a in NETS + ("netG",):
        ga = torch.cat([p.grad.double().flatten() for p in getattr(m16, a).parameters()])
        ra = torch.cat([p.grad.double().flatten() for p in getattr(m, a).parameters()])
        cos, ratio = float(ga @ ra / (ga.norm() * ra.norm())), float(ga.norm() / ra.norm())
        c_min = 0.998 if worst32.get(a, 0.0) > 1e-4 else 0.999
        if a in model and model[a][1] < c_min:
            # the rounding model itself is that far from the fp32 step: the fused kernels must reproduce the model's direction
            c_min = model[a][1] - 1e-5
            r_tol = 0.03
        elif deep and a != "netG":
            c_min, r_tol = 0.995, 0.015
        else:
            r_tol = 0.01
        line = f"{over}: bf16 step {a}: whole-gradient cosine {cos:.6f}, norm ratio {ratio:.5f}"
        if a in worst32:
            line += f"; fp32 autograd vs float64 {worst32[a]:.2e}"
        if a in model:
            line += f"; fused vs its rounding model {model[a][0]:.2e}, rounding model's cosine to the fp32 step {model[a][1]:.6f}"
            if model[a][0] > 5e-4:
                bad.append((a, "fused vs rounding model", model[a][0]))
        print(line)
        if not (cos >= c_min and abs(ratio - 1.0) <= r_tol):
            bad.append((a, cos, ratio, worst32.get(a)))
    assert not bad, bad
    return m, m16


@pytest.mark.parametrize("norm", NORMS)
def test_training_step_pixel(norm, tmp_path):
    m, m16 = _step_pair(tmp_path, netD="pixel", norm=norm)
    assert m.netD_1.net[0].weight.shape == (64, 1, 1, 1)
    m.save_networks("latest")
    m2 = _model(tmp_path, netD="pixel", norm=norm)
    m2.load_networks("latest")
    for a in ("netD_1", "netD_2", "netD_3"):
        assert all(torch.equal(u, v) for u, v in zip(getattr(m2, a).state_dict().values(), getattr(m, a).state_dict().values()))


@pytest.mark.parametrize("cin,cout,stride,size", [(64, 128, 1, 128), (128, 256, 1, 64), (256, 512, 2, 32), (512, 512, 1, 16),
                                                   (512, 512, 2, 16), (512, 512, 1, 8)])
def test_patchgan_tensor_core_convs_at_every_depth(cin, cout, stride, size):
    """the 4x4 tensor-core convolutions that the PatchGAN's depths 1, 2, 4 and 5 add at 256^2 (batch 2), against float64 on their own
    bf16-rounded operands: y from bf16(x), bf16(w); dw from bf16(dy), bf16(x); dx = col2im of the per-tap products bf16(w)^T bf16(dy),
    which the data-gradient GEMM stores in bf16 before col2im adds the 16 taps (hv_dconv_bwd_bf16).  That intermediate rounding is
    applied by the kernel to its fp32 sums and by the restatement to its float64 ones, so a few 1e-5 of the products round the other
    way; dx is held to 1e-4.  dw sums up to 2 x 127^2 pixel products in fp32 (1.8e-5 relative L2 measured on a B200 at 127 x 127) and
    is held to 1e-4, y (K = cin * 16 terms) to 1e-5."""
    g = torch.Generator(device="cuda").manual_seed(cin + cout + stride + size)
    x = torch.randn(2, cin, size, size, device="cuda", generator=g)
    w = torch.randn(cout, cin, 4, 4, device="cuda", generator=g) * 0.02
    xv = T.Var(x.clone())
    tape = T.Tape()
    dws = []
    out = T.conv2d_tc(tape, xv, w, stride, lambda dw, db: dws.append(dw))
    dy = torch.randn(out.data.shape, device="cuda", generator=g)
    out.grad = dy
    tape.backward()
    torch.cuda.synchronize()
    xb, wb, dyb = _bf(x), _bf(w), _bf(dy)
    want = F.conv2d(xb, wb, None, stride, 1)
    assert rel(out.data, want) <= 1e-5, rel(out.data, want)
    n, _, ho, wo = dy.shape
    dcol = _bf(torch.einsum("ok,nop->nkp", wb.reshape(cout, cin * 16), dyb.reshape(n, cout, ho * wo)))
    dx = F.fold(dcol, (size, size), 4, padding=1, stride=stride)
    dw = torch.nn.grad.conv2d_weight(xb, w.shape, dyb, stride, 1)
    assert rel(xv.grad, dx) <= 1e-4, rel(xv.grad, dx)
    assert rel(dws[0], dw) <= 1e-4, rel(dws[0], dw)


@pytest.mark.parametrize("n_layers", [1, 2, 4, 5])
def test_training_step_n_layers(n_layers, tmp_path):
    m, _ = _step_pair(tmp_path, netD="n_layers", n_layers_D=n_layers)
    side = {1: 126, 2: 62, 4: 14, 5: 6}[n_layers]
    assert m.netD_1.run(m.real_B).data.shape == (2, 1, side, side)
