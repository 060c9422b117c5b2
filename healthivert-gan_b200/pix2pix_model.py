"""Drop-in mirror of the reference's ``models/pix2pix_model.py`` (+ the ``BaseModel`` contract of
``models/base_model.py``) on hand-written sm_100a kernels: G forward / backward, height-adaptive stitching, three PatchGAN
discriminator updates, the G losses (GAN/6 + masked L1 + 2 Dice + edge MSE + height) and four fused Adam optimisers,
sequenced exactly like ``optimize_parameters`` (reference :356-382).

torch is used for device memory, parameter containers and (optionally) ``torch.distributed`` gradient all-reduces; every
number on the gradient path comes from libhv_b200.so.  There is no CPU fallback.
"""
import os
from collections import OrderedDict

import torch

from . import _lib, mask_ops, networks, train_ops as T
from ._lib import check, ptr
from .edge_operator import Sobel, edge_mse_loss
from .inpaint_networks import Generator


class BaseModel:
    """The subset of the reference's BaseModel (models/base_model.py:8-243) that the train / eval drivers call."""

    def __init__(self, opt):
        self.opt = opt
        self.gpu_ids = opt.gpu_ids
        self.isTrain = opt.isTrain
        self.device = torch.device("cuda:{}".format(self.gpu_ids[0])) if self.gpu_ids else torch.device("cuda")
        # every kernel launches on the CURRENT device's current stream and hv_generator_create allocates on the current device:
        # make gpu_ids[0] current, as the reference does in its option parsing (options/base_options.py:137-139)
        if self.gpu_ids and torch.cuda.is_available():
            torch.cuda.set_device(self.device)
        self.save_dir = os.path.join(opt.checkpoints_dir, opt.name)
        self.loss_names, self.model_names, self.visual_names, self.optimizers, self.image_paths = [], [], [], [], []
        self.metric = 0

    def setup(self, opt):
        if self.isTrain:
            self.schedulers = [networks.get_scheduler(o, opt) for o in self.optimizers]
        if not self.isTrain or opt.continue_train:
            self.load_networks("iter_%d" % opt.load_iter if opt.load_iter > 0 else opt.epoch)

    def eval(self):
        for name in self.model_names:
            getattr(self, "net" + name).eval()

    def train(self):
        for name in self.model_names:
            getattr(self, "net" + name).train()

    def test(self):
        with torch.no_grad():
            self.forward()

    def get_image_paths(self):
        return self.image_paths

    def update_learning_rate(self):
        old_lr = self.optimizers[0].param_groups[0]["lr"]
        for s in self.schedulers:
            if self.opt.lr_policy == "plateau":
                s.step(self.metric)
            else:
                s.step()
        lr = self.optimizers[0].param_groups[0]["lr"]
        print("learning rate %.7f -> %.7f" % (old_lr, lr))

    def get_current_visuals(self):
        return OrderedDict((n, getattr(self, n)) for n in self.visual_names if isinstance(n, str) and hasattr(self, n))

    def get_current_losses(self):
        return OrderedDict((n, float(getattr(self, "loss_" + n))) for n in self.loss_names if isinstance(n, str))

    def save_networks(self, epoch):
        os.makedirs(self.save_dir, exist_ok=True)
        for name in self.model_names:
            path = os.path.join(self.save_dir, "%s_net_%s.pth" % (epoch, name))
            torch.save({k: v.cpu() for k, v in getattr(self, "net" + name).state_dict().items()}, path)

    def load_networks(self, epoch):
        for name in self.model_names:
            path = os.path.join(self.save_dir, "%s_net_%s.pth" % (epoch, name))
            getattr(self, "net" + name).load_state_dict(torch.load(path, map_location=str(self.device)))

    def set_requires_grad(self, nets, requires_grad=False):
        if not isinstance(nets, list):
            nets = [nets]
        for net in nets:
            if net is not None:
                for p in net.parameters():
                    p.requires_grad = requires_grad


class Pix2PixModel(BaseModel):
    """reference models/pix2pix_model.py:41-382"""

    def __init__(self, opt):
        BaseModel.__init__(self, opt)
        self.loss_names = ["G_GAN", "G_maskL1", "G_Dice", "coarse_Dice", "edge",
                           "D_real_1", "D_fake_1", "D_real_2", "D_fake_2", "D_real_3", "D_fake_3", "h"]
        self.visual_names = ["real_A", "fake_B", "fake_B_mask_raw", "normal_vert", "coarse_seg_binary",
                             "fake_B_coarse", "real_B", "mask", "fake_B_raw", "real_B_mask", "CAM", "real_edges", "fake_B_local"]
        self.model_names = ["G", "D_1", "D_2", "D_3"] if self.isTrain else ["G"]
        if self.device.type != "cuda":
            raise _lib.HvError("hv_b200 Pix2PixModel needs a CUDA device (no CPU fallback)")
        self.netG = Generator({"input_dim": 1, "ngf": 16}, True).to(self.device)
        self.sobel_edge = Sobel(requires_grad=False).to(self.device)
        self._buckets = {}
        self.world_size = 1          # set by the launcher for data-parallel training (gradient all-reduce, SURVEY §8e)
        if self.isTrain:
            mk = lambda: networks.define_D(opt.input_nc, opt.ndf, opt.netD, opt.n_layers_D, opt.norm, opt.init_type,
                                           opt.init_gain, self.gpu_ids).to(self.device)
            self.netD_1, self.netD_2, self.netD_3 = mk(), mk(), mk()
            # opt.precision: 'fp32' = parity mode (SIMT kernels, gradients within 1e-4 of autograd); 'bf16' = tensor-core training mode:
            # the discriminators' convolutions (forward, data and weight gradients) and the generator's conv backward run as tcgen05
            # GEMMs with bf16 operands and fp32 accumulation, and the generator's conv forward runs on the tcgen05 conv kernel
            # (opt.g_forward_precision = 'fp32' keeps that part on the SIMT kernels).  opt.d_precision overrides the discriminator part
            # alone.
            self.precision = getattr(opt, "precision", "fp32")
            T.BACKWARD_PRECISION = self.precision
            T.FORWARD_PRECISION = getattr(opt, "g_forward_precision", self.precision)
            self.d_precision = getattr(opt, "d_precision", self.precision)
            for net in (self.netD_1, self.netD_2, self.netD_3):
                net.precision = self.d_precision
            self.criterionGAN = networks.GANLoss(opt.gan_mode).to(self.device)
            adam = lambda net: T.FusedAdam(net.parameters(), lr=opt.lr, betas=(opt.beta1, 0.999))
            self.optimizer_G, self.optimizer_D_1 = adam(self.netG), adam(self.netD_1)
            self.optimizer_D_2, self.optimizer_D_3 = adam(self.netD_2), adam(self.netD_3)
            self.optimizers += [self.optimizer_G, self.optimizer_D_1, self.optimizer_D_2, self.optimizer_D_3]

    # ------------------------------------------------------------------------------------------ input
    def set_input(self, input):
        AtoB = self.opt.direction == "AtoB"
        dev = self.device
        f32 = lambda t: t.to(device=dev, dtype=torch.float32).contiguous()
        self.real_B = f32(input["B" if AtoB else "A"])
        self.real_B_mask = f32(input["A_mask"])
        self.real_A = f32(input["A" if AtoB else "B"])
        self.CAM = f32(input["CAM"])
        self.normal_vert = f32(input["normal_vert"])
        self.height = input["height"].to(dev)
        self.mask = f32(input["mask"])
        self.slice_ratio = input["slice_ratio"].to(dev)
        self.x1 = input["x1"].to(dev)
        self.x2 = input["x2"].to(dev)
        self.maxheight = input["h2"].to(dev)
        # the stitch / height-loss kernels take ONE maxheight for the batch (the dataset's h2 is the constant 40,
        # data/aligned_dataset.py:202); it is read here, from the collated host tensor, not per forward on the device
        h2 = input["h2"].reshape(-1)
        self._maxh = int(h2[0]) if h2.numel() else 40
        if h2.numel() and not bool((h2 == h2[0]).all()):
            raise _lib.HvError("hv_b200 Pix2PixModel: per-sample maxheight (h2) values differ within the batch; "
                               "the device-side stitch takes one value per batch")
        self.image_paths = input["A_paths" if AtoB else "B_paths"]

    # ------------------------------------------------------------------------------------------ forward
    def forward(self):
        """reference :180-264.  Records the generator on a tape when gradients are enabled (training)."""
        train = self.isTrain and torch.is_grad_enabled() and self.netG.training
        self._tape = T.Tape() if train else None
        n = self.real_A.shape[0]
        cam_temp = torch.empty_like(self.CAM)   # 1 - CAM (:184)
        check(_lib.lib().hv_affine(-1.0, ptr(self.CAM), 1.0, ptr(cam_temp), cam_temp.numel(), _lib.stream()))
        if train:
            out = self.netG.forward_tape(self._tape, self.real_A, self.mask, cam_temp, self.slice_ratio)
            cs, fs, x1v, x2v, flow, p1, p2 = out
            self._vars = dict(coarse_seg=cs, fine_seg=fs, x_stage1=x1v, x_stage2=x2v, pred1_h=p1, pred2_h=p2)
            cs, fs, x1t, x2t, p1t, p2t = cs.data, fs.data, x1v.data, x2v.data, p1.data, p2.data
        else:
            with torch.no_grad():
                cs, fs, x1t, x2t, flow, p1t, p2t = self.netG(self.real_A, self.mask, cam_temp, self.slice_ratio)
        self.coarse_seg_sigmoid, self.fake_B_mask_sigmoid, self.x_stage1, self.fake_B_raw, self.offset_flow = cs, fs, x1t, x2t, flow
        self._pred1_raw, self._pred2_raw = p1t, p2t                  # sigmoid outputs in (0, 1), [N, 1]
        maxh = self._maxh
        w = self.mask.shape[-1]
        self._center = (w // 2 - 35, w // 2 + 35)                    # :254-260
        # :201-264 + the edge loss of :349 in ONE pass (hv_post_forward): thresholds, both height-adaptive stitches (device-side row
        # arithmetic, no .item() syncs), the masked centre crops, both Sobel maps and the XOR-count edge loss
        h = self.mask.shape[-2]
        dev = cs.device
        new = lambda: torch.empty(n, 1, h, w, device=dev, dtype=torch.float32)
        (self.fake_B_mask_raw, self.coarse_seg_binary, self.fake_B, self.fake_B_coarse, self.fake_B_local, self.real_B_local,
         self.real_edges, self.fake_edges) = (new() for _ in range(8))
        self._rows_fine = torch.empty(n, 4, device=dev, dtype=torch.int32)
        self._rows_coarse = torch.empty(n, 4, device=dev, dtype=torch.int32)
        self._edge_xor = torch.empty(1, device=dev, dtype=torch.int64)
        self._edge_loss_dev = torch.empty(1, device=dev, dtype=torch.float32)
        i32 = lambda t: t.to(device=dev, dtype=torch.int32).contiguous()
        x1d, x2d, hd = i32(self.x1), i32(self.x2), i32(self.height)
        p1c, p2c = p1t.reshape(-1).contiguous(), p2t.reshape(-1).contiguous()
        check(_lib.lib().hv_post_forward(
            ptr(fs.contiguous()), ptr(cs.contiguous()), ptr(x2t.contiguous()), ptr(x1t.contiguous()), ptr(self.real_B), ptr(self.real_B_mask),
            ptr(self.mask), ptr(p2c), ptr(p1c), ptr(x1d), ptr(x2d), ptr(hd), int(maxh), self._center[0], self._center[1],
            ptr(self.fake_B_mask_raw), ptr(self.coarse_seg_binary), ptr(self.fake_B), ptr(self.fake_B_coarse), ptr(self.fake_B_local),
            ptr(self.real_B_local), ptr(self.real_edges), ptr(self.fake_edges), ptr(self._rows_fine), ptr(self._rows_coarse),
            ptr(self._edge_xor), ptr(self._edge_loss_dev), n, h, w, _lib.stream()))

    def _local(self, x):
        out = torch.empty_like(x)
        c0, c1 = self._center
        check(_lib.lib().hv_masked_center(ptr(x), ptr(self.mask), ptr(out), x.shape[-1], c0, c1, x.numel(), _lib.stream()))
        return out

    # ------------------------------------------------------------------------------------------ D updates
    def _allreduce(self, params, tag="G"):
        """Data-parallel gradient exchange: ONE all-reduce per net on a flat gradient bucket (4 per step: D_1, D_2, D_3, G; NCCL over
        NVLink when launched under torchrun), averaged on the way back (train_ops.GradientBucket)."""
        if self.world_size <= 1:
            return
        import torch.distributed as dist
        bucket = self._buckets.setdefault(tag, T.GradientBucket())
        bucket.allreduce_mean_([p.grad for p in params if p.grad is not None], self.world_size, dist.all_reduce)

    def _backward_D(self, netD, fake, real, idx):
        """reference backward_D_k (:267-314): 0.5 * (L(D(fake.detach()), False) + L(D(real), True)) with L = criterionGAN (any
        gan_mode), gradients into netD."""
        tape = T.Tape()
        pf = netD.run(fake, tape)
        loss_fake = self.criterionGAN(pf.data, False)
        pf.grad = self.criterionGAN.grad(pf.data, False, 0.5)
        tape.backward()
        tape = T.Tape()
        pr = netD.run(real, tape)
        loss_real = self.criterionGAN(pr.data, True)
        pr.grad = self.criterionGAN.grad(pr.data, True, 0.5)
        tape.backward()
        setattr(self, "loss_D_fake_%d" % idx, loss_fake)
        setattr(self, "loss_D_real_%d" % idx, loss_real)
        setattr(self, "loss_D_%d" % idx, (loss_fake + loss_real) * 0.5)

    def backward_D_1(self):
        self._backward_D(self.netD_1, self.fake_B, self.real_B, 1)

    def backward_D_2(self):
        self._backward_D(self.netD_2, self.fake_B_mask_raw, self.real_B_mask, 2)

    def backward_D_3(self):
        self._backward_D(self.netD_3, self.fake_B_local, self.real_B_local, 3)

    # ------------------------------------------------------------------------------------------ G update
    def backward_G(self):
        """reference :317-354"""
        L = _lib.lib()
        st = _lib.stream()
        v = self._vars
        n = self.real_A.shape[0]
        # --- GAN terms: D_1(fake_B), D_2(fake_B_mask_raw) (thresholded: value only), D_3(fake_B_local); weights frozen
        tape1, tape3 = T.Tape(), T.Tape()
        fb = T.Var(self.fake_B)
        fl = T.Var(self.fake_B_local)
        p_ct = self.netD_1.run(fb, tape1, param_grads=False)
        p_mask = self.netD_2.run(self.fake_B_mask_raw, None, param_grads=False)
        p_loc = self.netD_3.run(fl, tape3, param_grads=False)
        g_ct = self.criterionGAN(p_ct.data, True)
        g_mask = self.criterionGAN(p_mask.data, True)
        g_loc = self.criterionGAN(p_loc.data, True)
        self.loss_G_GAN = (g_ct + g_mask + g_loc) / 6
        p_ct.grad = self.criterionGAN.grad(p_ct.data, True, 1.0 / 6)
        p_loc.grad = self.criterionGAN.grad(p_loc.data, True, 1.0 / 6)
        tape1.backward()
        tape3.backward()
        d_fake_B = fb.grad                                            # d loss / d fake_B through D_1
        d_loc = self._local(fl.grad)                                  # ... through D_3 (mask * center is its own adjoint)
        check(L.hv_axpby(1.0, ptr(d_loc), 1.0, ptr(d_fake_B), d_fake_B.numel(), st))
        # --- masked L1 (:336-338): (L1(fake_B) + L1(fake_B_coarse)) * 0.5 * lambda * (W*W / count_nonzero(mask)) * 2
        cnt = T.reduce_scalar(self.mask, None, 2, 1.0)
        w = self.mask.shape[-1]
        lam = float(self.opt.lambda_L1) * w * w
        l1_f = T.l1_mean(self.fake_B, self.real_B)
        l1_c = T.l1_mean(self.fake_B_coarse, self.real_B)
        self.loss_G_maskL1 = ((l1_f + l1_c) * 0.5 * lam / cnt * 2)[0]
        g_l1 = T.l1_grad(self.fake_B, self.real_B, lam, cnt, True)
        check(L.hv_axpby(1.0, ptr(g_l1), 1.0, ptr(d_fake_B), d_fake_B.numel(), st))
        d_fake_B_coarse = T.l1_grad(self.fake_B_coarse, self.real_B, lam, cnt, True)
        # --- through the stitch: only the generated rows carry gradient
        d_x2 = torch.empty_like(d_fake_B)
        check(L.hv_stitch_bwd(ptr(d_fake_B), ptr(self._rows_fine), ptr(d_x2), n, d_x2.shape[2], d_x2.shape[3], st))
        d_x1 = torch.empty_like(d_fake_B)
        check(L.hv_stitch_bwd(ptr(d_fake_B_coarse), ptr(self._rows_coarse), ptr(d_x1), n, d_x1.shape[2], d_x1.shape[3], st))
        # --- Dice (:344-346)
        dice_c, sums_c = T.dice(self.coarse_seg_sigmoid, self.normal_vert)
        dice_f, sums_f = T.dice(self.fake_B_mask_sigmoid, self.real_B_mask)
        self.loss_coarse_Dice = ((1 - dice_c) * 10)[0]
        self.loss_G_Dice = ((1 - dice_f) * 15)[0]
        d_cs = T.dice_grad(self.normal_vert, sums_c, -10.0 / n)
        d_fs = T.dice_grad(self.real_B_mask, sums_f, -15.0 / n)
        # --- edge loss (:349): MSE of Sobel maps of thresholded masks -> integer XOR count, no gradient (SURVEY F3)
        self.loss_edge = self._edge_loss()
        # --- height loss (:350): mean(40 |40 p1 - h| / h + 40 |40 p2 - h| / h)
        self.loss_h, d_p1, d_p2 = self._height_loss()
        # --- seed the tape and run the generator backward
        T.accumulate(v["x_stage2"], d_x2)
        T.accumulate(v["x_stage1"], d_x1)
        T.accumulate(v["coarse_seg"], d_cs)
        T.accumulate(v["fine_seg"], d_fs)
        T.accumulate(v["pred1_h"], d_p1)
        T.accumulate(v["pred2_h"], d_p2)
        self.loss_G = self.loss_G_GAN + self.loss_G_maskL1 + self.loss_G_Dice + self.loss_edge + self.loss_coarse_Dice + self.loss_h
        self._tape.backward()

    def _edge_loss(self):
        return self._edge_loss_dev[0]      # computed by hv_post_forward together with the edge maps

    def _height_loss(self):
        """loss_h (:350) and its gradients w.r.t. the two sigmoid height outputs, one small kernel."""
        n = self._pred1_raw.shape[0]
        h = self.height.to(torch.float32).reshape(n).contiguous()
        p1, p2 = self._pred1_raw.reshape(n).contiguous(), self._pred2_raw.reshape(n).contiguous()
        loss = torch.empty(1, device=h.device, dtype=torch.float32)
        d1, d2 = torch.empty(n, 1, device=h.device, dtype=torch.float32), torch.empty(n, 1, device=h.device, dtype=torch.float32)
        check(_lib.lib().hv_height_loss(ptr(p1), ptr(p2), ptr(h), float(self._maxh), n, ptr(loss), ptr(d1), ptr(d2), _lib.stream()))
        return loss[0], d1, d2

    # ------------------------------------------------------------------------------------------ step
    def optimize_parameters(self):
        """reference :356-382"""
        self.forward()
        for k, (net, opt_, bwd) in enumerate(((self.netD_1, self.optimizer_D_1, self.backward_D_1),
                                              (self.netD_2, self.optimizer_D_2, self.backward_D_2),
                                              (self.netD_3, self.optimizer_D_3, self.backward_D_3))):
            self.set_requires_grad(net, True)
            opt_.zero_grad()
            bwd()
            self._allreduce(net.parameters(), "D_%d" % (k + 1))
            opt_.step()
        self.set_requires_grad([self.netD_1, self.netD_2, self.netD_3], False)
        self.optimizer_G.zero_grad()
        self.backward_G()
        self._allreduce(self.netG.parameters(), "G")
        self.optimizer_G.step()
