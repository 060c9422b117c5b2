"""Drop-in mirror of the hot-path parts of the reference's ``models/networks.py`` on hand-written kernels:
``NLayerDiscriminator`` (:555-602), ``PixelDiscriminator`` (in :604-753), ``GANLoss`` (:212-278: 'vanilla', 'lsgan', 'wgangp' without a gradient penalty),
``define_D`` (:163-206), ``get_norm_layer`` (:30-47: 'batch', 'instance', 'none'), ``Identity`` (:25-27),
``init_weights`` / ``init_net`` (:68-117), ``get_scheduler`` (:39-65: 'linear', 'step', 'plateau', 'cosine', torch's own
schedulers on ``train_ops.FusedAdam``).

The torch ``nn.Conv2d`` / ``nn.BatchNorm2d`` objects are parameter CONTAINERS only (identical ``state_dict`` keys and identical
initialisation streams); all arithmetic runs in libhv_b200.so.  Discriminator layouts by norm:
'batch' ``model.{0,2,3,5,6,8,9,11}.*``; 'instance' ``model.{0,2,5,8,11}.{weight,bias}`` (InstanceNorm2d(affine=False) has no
state, the convs before it have a bias); 'none' ``model.{0,11}.{weight,bias}`` + ``model.{2,5,8}.weight``.  PixelDiscriminator:
'batch' ``net.{0,2,3,5}.*`` (no bias on convs 2 and 5); 'instance' ``net.{0,2,5}.{weight,bias}``; 'none' ``net.0.{weight,bias}`` +
``net.{2,5}.weight``.
"""
import functools

import torch
import torch.nn as nn
from torch.nn import init
from torch.optim import lr_scheduler

from . import _lib, train_ops as T
from ._lib import HV_SRC_DIRECT


class Identity(nn.Module):
    def forward(self, x):
        return x


def get_norm_layer(norm_type="batch"):
    if norm_type == "batch":
        return functools.partial(nn.BatchNorm2d, affine=True, track_running_stats=True)
    if norm_type == "instance":
        return functools.partial(nn.InstanceNorm2d, affine=False, track_running_stats=False)
    if norm_type == "none":
        def norm_layer(x):
            return Identity()
        return norm_layer
    raise NotImplementedError("normalization layer [%s] is not found" % norm_type)


def _use_bias(norm_layer):
    if type(norm_layer) == functools.partial:
        return norm_layer.func == nn.InstanceNorm2d
    return norm_layer == nn.InstanceNorm2d


def run_blocks(net, seq, x, tape=None, param_grads=True):
    """The layer path of both discriminators: walk ``seq`` as the reference's blocks conv [-> BatchNorm2d | InstanceNorm2d | Identity]
    [-> LeakyReLU(0.2)] on the hand-written kernels (SIMT convs, or T.conv2d_tc for the normalised 4x4 convs when net.precision is
    'bf16').  x: tensor or tape Var; returns a Var."""
    name = type(net).__name__
    if not isinstance(x, T.Var):
        x = T.Var(x.to(torch.float32).contiguous(), requires_grad=False)
    if not x.data.is_cuda:
        raise _lib.HvError("hv_b200 %s needs CUDA tensors (no CPU fallback)" % name)
    mods = list(seq)
    i = 0
    while i < len(mods):
        m = mods[i]
        if not isinstance(m, nn.Conv2d):
            raise NotImplementedError("unexpected module in the %s sequence: %r" % (name, m))
        j = i + 1
        norm = mods[j] if j < len(mods) and isinstance(mods[j], (nn.BatchNorm2d, nn.InstanceNorm2d, Identity)) else None
        j += norm is not None
        lrelu = j < len(mods) and isinstance(mods[j], nn.LeakyReLU)
        if isinstance(norm, nn.InstanceNorm2d) and (norm.affine or norm.track_running_stats or not lrelu):
            raise NotImplementedError("hv_b200 %s: InstanceNorm2d is built as get_norm_layer('instance') makes it" % name)
        inorm = isinstance(norm, nn.InstanceNorm2d)
        bare_lrelu = lrelu and not isinstance(norm, (nn.BatchNorm2d, nn.InstanceNorm2d))   # conv [-> Identity] -> LeakyReLU
        w = m.weight.detach()
        b = m.bias.detach() if m.bias is not None else None

        def on_grad(dw, db, m=m):
            T.accumulate_param(m.weight, dw)
            if db is not None and m.bias is not None:
                T.accumulate_param(m.bias, db)

        h, wd = x.data.shape[2], x.data.shape[3]
        # the tensor cores take the normalised or norm-free 4x4 convs (64->128, 128->256, 256->512: 97 % of the PatchGAN's FLOPs); a
        # bias before InstanceNorm goes into the norm kernel
        tc = (net.precision == "bf16" and norm is not None and (b is None or inorm) and m.kernel_size == (4, 4)
              and m.padding == (1, 1) and m.dilation == (1, 1) and m.stride[0] in (1, 2) and m.in_channels % 8 == 0
              and m.out_channels % 128 == 0)
        if tc:
            x = T.conv2d_tc(tape, x, w.contiguous(), m.stride[0], on_grad, param_grads)
            if bare_lrelu:
                x = T.lrelu(tape, x)
        else:
            x = T.conv2d(tape, [(x, HV_SRC_DIRECT)], w, b, m.kernel_size[0], m.stride[0], m.padding[0], m.dilation[0],
                         "lrelu" if bare_lrelu else "none", (h, wd), on_grad, param_grads)
        if isinstance(norm, nn.BatchNorm2d):
            if not net.training:
                raise NotImplementedError("hv_b200 %s: eval-mode BatchNorm is not on the training path" % name)
            x = T.bn_lrelu(tape, x, norm, 0.2, param_grads)
        elif inorm:
            x = T.in_lrelu(tape, x, m.bias if tc else None, 0.2, norm.eps, param_grads)
        i = j + 1 if lrelu else j
    return x


class NLayerDiscriminator(nn.Module):
    """PatchGAN discriminator (reference models/networks.py:555-602): conv4x4 s2 + LReLU, (conv4x4 s2 + norm + LReLU) x2,
    conv4x4 s1 + norm + LReLU, conv4x4 s1 -> 1-channel logits.  norm: BatchNorm2d (train mode only), InstanceNorm2d(affine=False)
    (fused with the LeakyReLU, train and eval) or Identity (the LeakyReLU is fused into the conv)."""

    def __init__(self, input_nc, ndf=64, n_layers=3, norm_layer=nn.BatchNorm2d):
        super().__init__()
        use_bias = _use_bias(norm_layer)
        kw, padw = 4, 1
        sequence = [nn.Conv2d(input_nc, ndf, kernel_size=kw, stride=2, padding=padw), nn.LeakyReLU(0.2, True)]
        nf_mult = 1
        for n in range(1, n_layers):
            nf_mult_prev, nf_mult = nf_mult, min(2 ** n, 8)
            sequence += [nn.Conv2d(ndf * nf_mult_prev, ndf * nf_mult, kernel_size=kw, stride=2, padding=padw, bias=use_bias),
                         norm_layer(ndf * nf_mult), nn.LeakyReLU(0.2, True)]
        nf_mult_prev, nf_mult = nf_mult, min(2 ** n_layers, 8)
        sequence += [nn.Conv2d(ndf * nf_mult_prev, ndf * nf_mult, kernel_size=kw, stride=1, padding=padw, bias=use_bias),
                     norm_layer(ndf * nf_mult), nn.LeakyReLU(0.2, True)]
        sequence += [nn.Conv2d(ndf * nf_mult, 1, kernel_size=kw, stride=1, padding=padw)]
        self.model = nn.Sequential(*sequence)
        # 'fp32': SIMT parity kernels everywhere; 'bf16': the three 4x4 convs between the first and the last (64->128, 128->256,
        # 256->512: 97 % of the discriminator's FLOPs) run on the tensor cores with bf16 operands and fp32 accumulation
        # (train_ops.conv2d_tc)
        self.precision = "fp32"

    def run(self, x, tape=None, param_grads=True):
        """Forward through the hand-written kernels.  x: tensor or tape Var; returns a Var (logits [N,1,30,30])."""
        return run_blocks(self, self.model, x, tape, param_grads)

    def forward(self, input):
        return self.run(input).data


class PixelDiscriminator(nn.Module):
    """1x1 PatchGAN (pixelGAN) discriminator (reference models/networks.py:604-753): conv1x1 input_nc->ndf + LReLU, conv1x1
    ndf->2ndf + norm + LReLU, conv1x1 2ndf->1 logits [N,1,H,W].

    'fp32': the layer path (run_blocks).  'bf16': at ndf = 64 and input_nc = 1 the whole net is one fused computation
    (train_ops.pixel_d: the 64->128 product on the tensor cores with bf16 operands, the 64- and 128-channel maps never leave the
    chip); other geometries take the layer path."""

    def __init__(self, input_nc, ndf=64, norm_layer=nn.BatchNorm2d):
        super().__init__()
        use_bias = _use_bias(norm_layer)
        self.net = nn.Sequential(
            nn.Conv2d(input_nc, ndf, kernel_size=1, stride=1, padding=0), nn.LeakyReLU(0.2, True),
            nn.Conv2d(ndf, ndf * 2, kernel_size=1, stride=1, padding=0, bias=use_bias), norm_layer(ndf * 2), nn.LeakyReLU(0.2, True),
            nn.Conv2d(ndf * 2, 1, kernel_size=1, stride=1, padding=0, bias=use_bias))
        self.precision = "fp32"

    def run(self, x, tape=None, param_grads=True):
        """Forward through the hand-written kernels.  x: tensor or tape Var; returns a Var (logits [N,1,H,W])."""
        norm = self.net[3]
        if isinstance(norm, nn.InstanceNorm2d) and (norm.affine or norm.track_running_stats):
            raise NotImplementedError("hv_b200 PixelDiscriminator: InstanceNorm2d is built as get_norm_layer('instance') makes it")
        if self.precision == "bf16" and T.pixel_d_supported(self):
            if isinstance(norm, nn.BatchNorm2d) and not self.training:
                raise NotImplementedError("hv_b200 PixelDiscriminator: eval-mode BatchNorm is not on the training path")
            return T.pixel_d(tape, x, self, param_grads)
        return run_blocks(self, self.net, x, tape, param_grads)

    def forward(self, input):
        return self.run(input).data


class GANLoss(nn.Module):
    """reference models/networks.py:212-278.  'vanilla': BCEWithLogitsLoss and 'lsgan': MSELoss against the constant real / fake
    label; 'wgangp': -mean(prediction) against real, mean(prediction) against fake.  The reference's pix2pix model never calls
    cal_gradient_penalty, so 'wgangp' has no gradient penalty (and no weight clipping) here either.

    ``__call__`` returns the loss as a 0-dim device tensor; ``grad(prediction, target_is_real, g)`` returns d(g * loss)/d prediction."""

    def __init__(self, gan_mode, target_real_label=1.0, target_fake_label=0.0):
        super().__init__()
        self.register_buffer("real_label", torch.tensor(target_real_label))
        self.register_buffer("fake_label", torch.tensor(target_fake_label))
        self.gan_mode = gan_mode
        if gan_mode not in T.GAN_KINDS:
            raise NotImplementedError("gan mode %s not implemented" % gan_mode)
        # the kernels take the target by value: kept as Python floats, so no call reads the buffers back from the device
        self._labels = (float(target_fake_label), float(target_real_label))

    def _target(self, target_is_real):
        """(t, sign) of train_ops.gan_loss"""
        if self.gan_mode == "wgangp":
            return 0.0, (-1.0 if target_is_real else 1.0)
        return self._labels[bool(target_is_real)], 1.0

    def __call__(self, prediction, target_is_real):
        t, sign = self._target(target_is_real)
        return T.gan_loss(prediction, self.gan_mode, t, sign)[0]

    def grad(self, prediction, target_is_real, g=1.0):
        t, sign = self._target(target_is_real)
        return T.gan_loss_grad(prediction.contiguous(), self.gan_mode, t, g, sign)


def init_weights(net, init_type="normal", init_gain=0.02):
    """reference models/networks.py:68-99 (same RNG consumption order: net.apply)."""
    def init_func(m):
        classname = m.__class__.__name__
        if hasattr(m, "weight") and (classname.find("Conv") != -1 or classname.find("Linear") != -1):
            if init_type == "normal":
                init.normal_(m.weight.data, 0.0, init_gain)
            elif init_type == "xavier":
                init.xavier_normal_(m.weight.data, gain=init_gain)
            elif init_type == "kaiming":
                init.kaiming_normal_(m.weight.data, a=0, mode="fan_in")
            elif init_type == "orthogonal":
                init.orthogonal_(m.weight.data, gain=init_gain)
            else:
                raise NotImplementedError("initialization method [%s] is not implemented" % init_type)
            if hasattr(m, "bias") and m.bias is not None:
                init.constant_(m.bias.data, 0.0)
        elif classname.find("BatchNorm2d") != -1:
            init.normal_(m.weight.data, 1.0, init_gain)
            init.constant_(m.bias.data, 0.0)
    net.apply(init_func)


def init_net(net, init_type="normal", init_gain=0.02, gpu_ids=[]):
    """reference :102-117.  No nn.DataParallel wrapper: multi-GPU is one process per GPU (SURVEY §5), so the
    state_dict keys are the unwrapped ones that save_networks writes anyway (base_model.py:152-173)."""
    if len(gpu_ids) > 0:
        net.to(torch.device("cuda", gpu_ids[0]))
    init_weights(net, init_type, init_gain=init_gain)
    return net


def define_D(input_nc, ndf, netD, n_layers_D=3, norm="batch", init_type="normal", init_gain=0.02, gpu_ids=[]):
    """reference models/networks.py:163-206 ('basic' and 'n_layers' are the PatchGAN variants, 'pixel' the 1x1 PixelDiscriminator)."""
    norm_layer = get_norm_layer(norm_type=norm)
    if netD == "basic":
        net = NLayerDiscriminator(input_nc, ndf, n_layers=3, norm_layer=norm_layer)
    elif netD == "n_layers":
        net = NLayerDiscriminator(input_nc, ndf, n_layers_D, norm_layer=norm_layer)
    elif netD == "pixel":
        net = PixelDiscriminator(input_nc, ndf, norm_layer=norm_layer)
    else:
        raise NotImplementedError("Discriminator model name [%s] is not recognized" % netD)
    return init_net(net, init_type, init_gain, gpu_ids)


def get_scheduler(optimizer, opt):
    """reference models/networks.py:39-65: torch's own schedulers (train_ops.FusedAdam is a torch.optim.Optimizer).  'plateau' is
    stepped with the model's metric (BaseModel.update_learning_rate); opt.lr_decay_iters is read by 'step' alone."""
    if opt.lr_policy == "linear":
        def lambda_rule(epoch):
            return 1.0 - max(0, epoch + opt.epoch_count - opt.n_epochs) / float(opt.n_epochs_decay + 1)
        return lr_scheduler.LambdaLR(optimizer, lr_lambda=lambda_rule)
    if opt.lr_policy == "step":
        return lr_scheduler.StepLR(optimizer, step_size=opt.lr_decay_iters, gamma=0.1)
    if opt.lr_policy == "plateau":
        return lr_scheduler.ReduceLROnPlateau(optimizer, mode="min", factor=0.2, threshold=0.01, patience=5)
    if opt.lr_policy == "cosine":
        return lr_scheduler.CosineAnnealingLR(optimizer, T_max=opt.n_epochs, eta_min=0)
    raise NotImplementedError("learning rate policy [%s] is not implemented" % opt.lr_policy)
