"""Reverse-mode tape over the hand-written training kernels (C ABI: include/hv_b200.h, "Training step").

The reference relies on torch.autograd (models/pix2pix_model.py:286,:300,:314,:354); here every forward op records a
closure that calls the matching hand-written backward kernel, and ``Tape.backward()`` replays the closures in reverse.
torch supplies device memory (``torch.empty``) and parameter containers only - no torch arithmetic on the gradient path.
"""
import torch

from . import _lib
from ._lib import HV_ACT, HV_SRC_DIRECT, HV_SRC_SCALAR, HV_SRC_SUB2, HV_SRC_UP2, check, ptr


# 'fp32': SIMT parity kernels for the conv backward (hv_conv2d_dgrad / _wgrad); 'bf16': im2col + tcgen05 GEMMs with bf16 operands and
# fp32 accumulation (hv_conv2d_dgrad_bf16 / _wgrad_bf16).  Set by Pix2PixModel from opt.precision; a process-wide switch because the
# tape closures of every net consult it when they run.
BACKWARD_PRECISION = "fp32"
# 'bf16': the generator's convolution FORWARD runs on the tcgen05 kernel too (hv_conv2d_bf16: operands and the stored activation rounded
# to bf16, fp32 accumulation); the single-filter output heads (conv17 / conv18, allconv17 / allconv18) stay fp32 so that the images and
# masks the losses read are not quantised to 8 mantissa bits.
FORWARD_PRECISION = "fp32"
_WS = {}


def _workspace(nbytes, dev):
    """One grow-only scratch buffer per device for the tensor-core backward (up to ~1 GB at batch 16: the im2col operands)."""
    key = (dev.type, dev.index)
    buf = _WS.get(key)
    if buf is None or buf.numel() < nbytes:
        _WS[key] = buf = torch.empty(int(nbytes * 1.25) + 4096, device=dev, dtype=torch.uint8)
    return buf


class Var:
    """A tensor on the tape: ``data`` plus an accumulated gradient (None until something flows back)."""
    __slots__ = ("data", "grad", "requires_grad")

    def __init__(self, data, requires_grad=True):
        self.data = data
        self.grad = None
        self.requires_grad = requires_grad

    @property
    def shape(self):
        return self.data.shape


def _L():
    return _lib.lib()


def accumulate(var, g):
    """var.grad += g (first contribution is adopted without a copy)."""
    if not var.requires_grad:
        return
    if var.grad is None:
        var.grad = g
    else:
        check(_L().hv_axpby(1.0, ptr(g), 1.0, ptr(var.grad), g.numel(), _lib.stream()))


def accumulate_param(p, g):
    if p.grad is None:
        p.grad = g
    else:
        check(_L().hv_axpby(1.0, ptr(g), 1.0, ptr(p.grad), g.numel(), _lib.stream()))


class Tape:
    def __init__(self):
        self.ops = []
        self.keep = []   # tensors that must outlive the enqueued kernels of the forward
        self.finalizers = []   # run once after the last recorded op's backward (batched per-net work, e.g. the spectral-norm adjoint)

    def record(self, fn):
        self.ops.append(fn)

    def backward(self):
        for fn in reversed(self.ops):
            fn()
        for fn in self.finalizers:
            fn()
        self.ops = []
        self.keep = []
        self.finalizers = []


def _desc(sources, cin, cout, k, stride, pad, dil, act, hin, win, n):
    d = _lib.hv_conv_desc()
    keep = []
    for i, (t, mode) in enumerate(sources):
        t = t.contiguous()
        keep.append(t)
        d.src[i].ptr = ptr(t)
        d.src[i].channels = 1 if mode == HV_SRC_SCALAR else t.shape[1]
        d.src[i].mode = mode
    d.n, d.cin, d.cout, d.hin, d.win = n, cin, cout, hin, win
    d.k, d.stride, d.pad, d.dil, d.act, d.nsrc = k, stride, pad, dil, HV_ACT[act], len(sources)
    return d, keep


def conv2d(tape, sources, weight, bias, k, stride, pad, dil, act, extent, on_weight_grad, param_grads=True, dw_buffer=None):
    """act(conv2d(cat(sources), weight) + bias) with the fused source gather of hv_conv2d_fwd.

    sources: [(Var | tensor, hv_src_mode)]; plain tensors are constants.  weight: effective weight TENSOR [cout,cin,k,k];
    on_weight_grad(dw, db): receives the gradients w.r.t. weight / bias (skipped when param_grads is False); dw_buffer: tensor the weight
    gradient is written to (default: a fresh one)."""
    srcs = [((s.data if isinstance(s, Var) else s), m) for s, m in sources]
    first = srcs[0][0]
    n = first.shape[0]
    hin, win = extent
    cin = sum(1 if m == HV_SRC_SCALAR else t.shape[1] for t, m in srcs)
    cout = weight.shape[0]
    eff = (k - 1) * dil + 1
    hout, wout = (hin + 2 * pad - eff) // stride + 1, (win + 2 * pad - eff) // stride + 1
    d, keep = _desc(srcs, cin, cout, k, stride, pad, dil, act, hin, win, n)
    y = torch.empty(n, cout, hout, wout, device=first.device, dtype=torch.float32)
    tc_fwd = (FORWARD_PRECISION == "bf16" and k in (3, 5) and pad == (k - 1) // 2 * dil and 8 <= cout <= 64
              and (stride == 1 or (stride == 2 and k == 3 and dil == 1 and hin % 2 == 0 and win % 2 == 0)))
    if tc_fwd:
        check(_L().hv_conv2d_bf16(d, ptr(weight), ptr(bias), ptr(y), None, 0, _lib.stream()))
    else:
        check(_L().hv_conv2d_fwd(d, ptr(weight), ptr(bias), ptr(y), None, _lib.stream()))
    out = Var(y)
    if tape is None:
        return out
    tape.keep.append(keep)

    def bwd():
        if out.grad is None:
            return
        L = _L()
        st = _lib.stream()
        dpre = out.grad
        tc = BACKWARD_PRECISION == "bf16"
        db = torch.empty(cout, device=y.device, dtype=torch.float32) if (bias is not None and param_grads) else None
        db_done = False
        if act != "none":
            dpre = torch.empty_like(y)
            if db is not None and tc:      # pre-activation gradient and its channel sums (the bias gradient) in one pass
                check(L.hv_act_bwd_bias(ptr(y), ptr(out.grad), ptr(dpre), ptr(db), HV_ACT[act], n, cout, hout * wout, st))
                db_done = True
            else:
                check(L.hv_act_bwd(ptr(y), ptr(out.grad), ptr(dpre), HV_ACT[act], y.numel(), st))
        dd, keep2 = _desc(srcs, cin, cout, k, stride, pad, dil, "none", hin, win, n)
        if param_grads:
            dw = dw_buffer if dw_buffer is not None else torch.empty_like(weight)
            if tc:
                ws = _workspace(L.hv_conv2d_wgrad_bf16_workspace_bytes(dd), y.device)
                check(L.hv_conv2d_wgrad_bf16(dd, ptr(dpre), ptr(dw), None if db_done else ptr(db), ptr(ws), st))
            else:
                check(L.hv_conv2d_wgrad(dd, ptr(dpre), ptr(dw), ptr(db), st))
            on_weight_grad(dw, db)
        need = [isinstance(s, Var) and s.requires_grad for s, _ in sources]
        per_source = (tc and cin > 64 and stride == 1 and k in (3, 5) and pad == (k - 1) // 2 * dil
                      and all((m in (HV_SRC_DIRECT, HV_SRC_UP2) and t.shape[1] <= 64) or not nd for (_, m), (t, _), nd in zip(sources, srcs, need)))
        if any(need) and per_source:
            # more input channels than the conv-form data gradient writes at once (64): one convolution per SOURCE that needs a
            # gradient, over that source's slice of the filters (conv20: only the 64 upsampled channels of its 65; allconv11: 64 + 64)
            c0 = 0
            for (s, m), (t, _), nd in zip(sources, srcs, need):
                ch = 1 if m == HV_SRC_SCALAR else t.shape[1]
                if nd:
                    sub, keep3 = _desc([(t, HV_SRC_DIRECT)], ch, cout, k, stride, pad, dil, "none", hin, win, n)
                    sub.src[0].ptr = None        # the data gradient does not read the source
                    wsub = weight[:, c0:c0 + ch].contiguous()
                    dxs = torch.empty(n, ch, hin, win, device=y.device, dtype=torch.float32)
                    ws = _workspace(L.hv_conv2d_dgrad_bf16_workspace_bytes(sub), y.device)
                    check(L.hv_conv2d_dgrad_bf16(sub, ptr(wsub), ptr(dpre), ptr(dxs), ptr(ws), st))
                    if m == HV_SRC_UP2:
                        g = torch.empty_like(t)
                        check(L.hv_upsample2_bwd(ptr(dxs), ptr(g), n, ch, hin // 2, win // 2, ch, 0, st))
                    else:
                        g = dxs
                    accumulate(s, g)
                c0 += ch
        elif any(need):
            dx = torch.empty(n, cin, hin, win, device=y.device, dtype=torch.float32)
            if tc:
                ws = _workspace(L.hv_conv2d_dgrad_bf16_workspace_bytes(dd), y.device)
                check(L.hv_conv2d_dgrad_bf16(dd, ptr(weight), ptr(dpre), ptr(dx), ptr(ws), st))
            else:
                ws = torch.empty(cin * cout * k * k, device=y.device, dtype=torch.float32)
                check(L.hv_conv2d_dgrad(dd, ptr(weight), ptr(dpre), ptr(dx), ptr(ws), st))
            c0 = 0
            for (s, m), (t, _), nd in zip(sources, srcs, need):
                ch = 1 if m == HV_SRC_SCALAR else t.shape[1]
                if nd:
                    if m == HV_SRC_DIRECT:
                        g = dx if (c0 == 0 and ch == cin) else dx[:, c0:c0 + ch].contiguous()
                    elif m == HV_SRC_UP2:
                        g = torch.empty_like(t)
                        check(L.hv_upsample2_bwd(ptr(dx), ptr(g), n, ch, hin // 2, win // 2, cin, c0, st))
                    else:
                        raise NotImplementedError("gradient through a sub-sampled / scalar source")
                    accumulate(s, g)
                c0 += ch
        del keep2

    tape.record(bwd)
    return out


def conv2d_tc(tape, x, weight, stride, on_weight_grad, param_grads=True):
    """4x4 / padding-1 convolution without bias or activation (the BatchNorm-followed PatchGAN layers, models/networks.py:583-597) on
    the tensor cores: bf16 operands, fp32 accumulation (hv_dconv_fwd_bf16 / hv_dconv_bwd_bf16).  x: Var [n,cin,h,w]; weight: fp32
    [cout,cin,4,4].  The backward recomputes the im2col operand from x instead of keeping it alive."""
    n, cin, h, w = x.data.shape
    cout = weight.shape[0]
    ho, wo = (h + 2 - 4) // stride + 1, (w + 2 - 4) // stride + 1
    L = _L()
    dev = x.data.device
    nbytes = L.hv_dconv_workspace_bytes(n, cin, cout, h, w, stride)
    if nbytes == 0:
        raise _lib.HvError(f"conv2d_tc: unsupported geometry cin={cin} cout={cout} stride={stride}")
    ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
    y = torch.empty(n, cout, ho, wo, device=dev, dtype=torch.float32)
    check(L.hv_dconv_fwd_bf16(ptr(x.data), ptr(weight), ptr(y), n, cin, cout, h, w, stride, ptr(ws), _lib.stream()))
    out = Var(y)
    if tape is None:
        return out

    def bwd():
        if out.grad is None:
            return
        need_dx = x.requires_grad
        if not (need_dx or param_grads):
            return
        ws2 = torch.empty(nbytes, device=dev, dtype=torch.uint8)
        dx = torch.empty_like(x.data) if need_dx else None
        dw = torch.empty_like(weight) if param_grads else None
        check(L.hv_dconv_bwd_bf16(ptr(x.data), ptr(weight), ptr(out.grad.contiguous()), ptr(dx), ptr(dw), n, cin, cout, h, w, stride,
                                  ptr(ws2), _lib.stream()))
        if param_grads:
            on_weight_grad(dw, None)
        if need_dx:
            accumulate(x, dx)

    tape.record(bwd)
    return out


def gap_fc_sigmoid(tape, x, fc):
    """sigmoid(fc(mean_HW(x))) (reference inpaint_networks.py:90-93,:211-214); fc: nn.Linear(c, 1)."""
    n, c, h, w = x.data.shape
    out = torch.empty(n, 1, device=x.data.device, dtype=torch.float32)
    fw, fb = fc.weight.detach().contiguous(), fc.bias.detach().contiguous()
    check(_L().hv_gap_fc_sigmoid(ptr(x.data), ptr(fw), ptr(fb), ptr(out), n, c, h * w, _lib.stream()))
    res = Var(out)
    if tape is None:
        return res

    def bwd():
        if res.grad is None:
            return
        dx = torch.empty_like(x.data)
        dfw = torch.empty_like(fw)
        dfb = torch.empty_like(fb)
        check(_L().hv_gap_fc_sigmoid_bwd(ptr(x.data), ptr(out), ptr(res.grad.contiguous()), ptr(fw), ptr(dx), 0, ptr(dfw),
                                         ptr(dfb), n, c, h * w, _lib.stream()))
        accumulate(x, dx)
        accumulate_param(fc.weight, dfw.reshape(fc.weight.shape))
        accumulate_param(fc.bias, dfb.reshape(fc.bias.shape))

    tape.record(bwd)
    return res


def ctx_attention(tape, f, mask, scale, fuse, per_sample_mask, want_flow=True):
    """ContextualAttention.forward(f, f, mask) with its hand-written adjoint (fp32 tensors; in the tensor-core training mode the six
    dense contractions run on tcgen05 with bf16-rounded operands: hv_ctx_attn_fwd_tc / hv_ctx_attn_bwd_tc)."""
    n, c, h, w = f.data.shape
    L = _L()
    tc = BACKWARD_PRECISION == "bf16" and (c * 9) % 64 == 0
    fwd, bwd_fn = (L.hv_ctx_attn_fwd_tc, L.hv_ctx_attn_bwd_tc) if tc else (L.hv_ctx_attn_fwd, L.hv_ctx_attn_bwd)
    dev = f.data.device
    y = torch.empty_like(f.data)
    offsets = torch.empty(n, 2, h // 2, w // 2, device=dev, dtype=torch.int32)
    flow = torch.empty(n, 3, 4 * h, 4 * w, device=dev, dtype=torch.float32) if want_flow else None
    ws = torch.empty(L.hv_ctx_attn_workspace_bytes(n, c, h, w), device=dev, dtype=torch.uint8)
    mask = mask.contiguous()
    check(fwd(ptr(f.data), ptr(mask), ptr(y), ptr(offsets), ptr(flow), n, c, h, w, float(scale), int(bool(fuse)),
              int(per_sample_mask), ptr(ws), _lib.stream()))
    out = Var(y)
    if tape is not None:
        def bwd():
            if out.grad is None:
                return
            bws = torch.empty(L.hv_ctx_attn_bwd_workspace_bytes(n, c, h, w), device=dev, dtype=torch.uint8)
            df = torch.empty_like(f.data)
            check(bwd_fn(ptr(out.grad.contiguous()), ptr(df), n, c, h, w, float(scale), int(bool(fuse)), ptr(ws),
                         ptr(bws), _lib.stream()))
            accumulate(f, df)

        tape.record(bwd)
    return out, flow, offsets


def bn_lrelu(tape, x, bn, slope=0.2, param_grads=True):
    """BatchNorm2d (batch statistics, running stats updated) + LeakyReLU(slope) (reference networks.py:583-597)."""
    n, c, h, w = x.data.shape
    dev = x.data.device
    y = torch.empty_like(x.data)
    mean = torch.empty(c, device=dev, dtype=torch.float32)
    invstd = torch.empty(c, device=dev, dtype=torch.float32)
    gamma, beta = bn.weight.detach(), bn.bias.detach()
    check(_L().hv_bn_lrelu_fwd(ptr(x.data), ptr(gamma), ptr(beta), ptr(bn.running_mean), ptr(bn.running_var), ptr(y), ptr(mean),
                               ptr(invstd), n, c, h * w, float(bn.momentum), float(bn.eps), float(slope), _lib.stream()))
    bn.num_batches_tracked += 1
    out = Var(y)
    if tape is None:
        return out

    def bwd():
        if out.grad is None:
            return
        dx = torch.empty_like(x.data)
        dg = torch.empty_like(gamma)
        db = torch.empty_like(beta)
        check(_L().hv_bn_lrelu_bwd(ptr(x.data), ptr(y), ptr(out.grad.contiguous()), ptr(gamma), ptr(mean), ptr(invstd), ptr(dx),
                                   ptr(dg), ptr(db), n, c, h * w, float(slope), _lib.stream()))
        if param_grads:
            accumulate_param(bn.weight, dg)
            accumulate_param(bn.bias, db)
        accumulate(x, dx)

    tape.record(bwd)
    return out


def in_lrelu(tape, x, bias=None, slope=0.2, eps=1e-5, param_grads=True):
    """InstanceNorm2d(affine=False) + LeakyReLU(slope) (reference networks.py:583-597 with norm='instance'), instance statistics in
    train and eval.  bias: the preceding convolution's bias parameter, added on load (the tensor-core conv has no bias epilogue); its
    gradient, zero up to rounding, is accumulated into bias.grad when param_grads."""
    n, c, h, w = x.data.shape
    dev = x.data.device
    y = torch.empty_like(x.data)
    mean = torch.empty(n * c, device=dev, dtype=torch.float32)
    invstd = torch.empty(n * c, device=dev, dtype=torch.float32)
    b = bias.detach() if bias is not None else None
    check(_L().hv_in_lrelu_fwd(ptr(x.data), ptr(b), ptr(y), ptr(mean), ptr(invstd), n, c, h * w, float(eps), float(slope),
                               _lib.stream()))
    out = Var(y)
    if tape is None:
        return out

    def bwd():
        if out.grad is None:
            return
        dx = torch.empty_like(x.data)
        db = torch.empty(c, device=dev, dtype=torch.float32) if (b is not None and param_grads) else None
        check(_L().hv_in_lrelu_bwd(ptr(x.data), ptr(b), ptr(out.grad.contiguous()), ptr(mean), ptr(invstd), ptr(dx), ptr(db), n, c,
                                   h * w, float(slope), _lib.stream()))
        if db is not None:
            accumulate_param(bias, db)
        accumulate(x, dx)

    tape.record(bwd)
    return out


PIXEL_D_NORM = {"Identity": 0, "BatchNorm2d": 1, "InstanceNorm2d": 2}


def pixel_d_supported(net):
    """True when PixelDiscriminator ``net`` has the geometry the fused kernels are built for (ndf = 64, input_nc = 1)."""
    c1, c2 = net.net[0], net.net[2]
    return c1.in_channels == 1 and c1.out_channels == 64 and c2.out_channels == 128


def pixel_d(tape, x, net, param_grads=True):
    """The whole PixelDiscriminator ``net`` (models/networks.py:604-753) as ONE tape op on the fused tensor-core kernels
    (hv_pixel_d_fwd_bf16 / _bwd_bf16): logits [n,1,h,w].  The forward keeps only x and the norm statistics; the backward recomputes the
    64- and 128-channel maps on chip.  BatchNorm running statistics and num_batches_tracked are updated on every call."""
    if not isinstance(x, Var):
        x = Var(x.to(torch.float32).contiguous(), requires_grad=False)
    xd = x.data.contiguous()
    if not xd.is_cuda:
        raise _lib.HvError("hv_b200 PixelDiscriminator needs CUDA tensors (no CPU fallback)")
    n, _, h, w = xd.shape
    c1, norm_mod, c2, c3 = net.net[0], net.net[3], net.net[2], net.net[5]
    kind = PIXEL_D_NORM[type(norm_mod).__name__]
    dev = xd.device
    L = _L()
    d = lambda t: t.detach().contiguous() if t is not None else None
    w1, b1, w2, b2, w3, b3 = d(c1.weight), d(c1.bias), d(c2.weight), d(c2.bias), d(c3.weight), d(c3.bias)
    bn = norm_mod if kind == 1 else None
    gamma, beta = (d(bn.weight), d(bn.bias)) if bn is not None else (None, None)
    ws = torch.empty(L.hv_pixel_d_workspace_bytes(n, h, w), device=dev, dtype=torch.uint8)
    y = torch.empty(n, 1, h, w, device=dev, dtype=torch.float32)
    nstat = 128 * (n if kind == 2 else 1)
    mean = torch.empty(nstat, device=dev, dtype=torch.float32) if kind else None
    invstd = torch.empty(nstat, device=dev, dtype=torch.float32) if kind else None
    eps = float(norm_mod.eps) if kind else 1e-5
    check(L.hv_pixel_d_fwd_bf16(ptr(xd), ptr(w1), ptr(b1), ptr(w2), ptr(b2), ptr(gamma), ptr(beta), ptr(w3), ptr(b3),
                                ptr(bn.running_mean) if bn is not None else None, ptr(bn.running_var) if bn is not None else None,
                                ptr(y), ptr(mean), ptr(invstd), n, 1, 64, h, w, kind, float(bn.momentum) if bn is not None else 0.0,
                                eps, 0.2, ptr(ws), _lib.stream()))
    if bn is not None:
        bn.num_batches_tracked += 1
    out = Var(y)
    if tape is None:
        return out

    def bwd():
        if out.grad is None:
            return
        need_dx = x.requires_grad
        if not (need_dx or param_grads):
            return
        e = lambda t: torch.empty_like(t) if (param_grads and t is not None) else None
        dx = torch.empty_like(xd) if need_dx else None
        dw1, db1, dw2, db2, dw3, db3 = e(w1), e(b1), e(w2), e(b2), e(w3), e(b3)
        dg, dbt = e(gamma), e(beta)
        check(L.hv_pixel_d_bwd_bf16(ptr(xd), ptr(w1), ptr(b1), ptr(w2), ptr(b2), ptr(gamma), ptr(beta), ptr(w3), ptr(b3), ptr(mean),
                                    ptr(invstd), ptr(out.grad.contiguous()), ptr(dx), ptr(dw1), ptr(db1), ptr(dw2), ptr(db2), ptr(dg),
                                    ptr(dbt), ptr(dw3), ptr(db3), n, 1, 64, h, w, kind, 0.2, ptr(ws), _lib.stream()))
        if param_grads:
            for mod, dw, db in ((c1, dw1, db1), (c2, dw2, db2), (c3, dw3, db3)):
                accumulate_param(mod.weight, dw)
                if db is not None:
                    accumulate_param(mod.bias, db)
            if bn is not None:
                accumulate_param(bn.weight, dg)
                accumulate_param(bn.bias, dbt)
        if need_dx:
            accumulate(x, dx)

    tape.keep.append(ws)
    tape.record(bwd)
    return out


def lrelu(tape, x):
    """LeakyReLU(0.2) as its own pass (after a tensor-core convolution, which has no activation epilogue)."""
    y = torch.empty_like(x.data)
    check(_L().hv_act_fwd(ptr(x.data), ptr(y), HV_ACT["lrelu"], y.numel(), _lib.stream()))
    out = Var(y)
    if tape is None:
        return out

    def bwd():
        if out.grad is None:
            return
        dx = torch.empty_like(y)
        check(_L().hv_act_bwd(ptr(y), ptr(out.grad.contiguous()), ptr(dx), HV_ACT["lrelu"], y.numel(), _lib.stream()))
        accumulate(x, dx)

    tape.record(bwd)
    return out


# ------------------------------------------------------------------------------------------- scalar losses
class Scratch:
    """Per-device reduction scratch (1024 floats) and 0-dim outputs."""
    _bufs = {}

    @classmethod
    def get(cls, dev):
        key = (dev.type, dev.index)
        if key not in cls._bufs:
            cls._bufs[key] = torch.empty(1024, device=dev, dtype=torch.float32)
        return cls._bufs[key]


def reduce_scalar(a, b, kind, scale, t=0.0):
    out = torch.empty(1, device=a.device, dtype=torch.float32)
    check(_L().hv_reduce_scalar(ptr(a), ptr(b), float(t), int(kind), a.numel(), float(scale), ptr(out), ptr(Scratch.get(a.device)),
                                _lib.stream()))
    return out


def l1_mean(a, b):
    """nn.L1Loss()(a, b) as a device scalar."""
    return reduce_scalar(a.contiguous(), b.contiguous(), 0, 1.0 / a.numel())


# GANLoss objectives (reference networks.py:212-278) -> (hv_reduce_scalar kind, hv_loss_grad kind)
GAN_KINDS = {"vanilla": (1, 1), "lsgan": (5, 2), "wgangp": (3, 3)}


def gan_loss(logits, mode, t, sign=1.0):
    """sign * mean over the logits of BCE-with-logits vs the constant t ('vanilla'), (x - t)^2 ('lsgan') or x ('wgangp', t unused),
    as a device scalar."""
    return reduce_scalar(logits.contiguous(), None, GAN_KINDS[mode][0], sign / logits.numel(), t)


def gan_loss_grad(logits, mode, t, g, sign=1.0):
    """d(g * gan_loss(logits, mode, t, sign))/d logits."""
    da = torch.empty_like(logits)
    check(_L().hv_loss_grad(ptr(logits), None, float(t), GAN_KINDS[mode][1], float(g) * sign / logits.numel(), None, 0, ptr(da), 0,
                            logits.numel(), _lib.stream()))
    return da


def l1_grad(a, b, g, scale=None, reciprocal=False):
    """d(g * S * mean|a-b|)/da with the optional device scalar S (or 1/S)."""
    da = torch.empty_like(a)
    check(_L().hv_loss_grad(ptr(a), ptr(b), 0.0, 0, float(g) / a.numel(), ptr(scale), int(reciprocal), ptr(da), 0, a.numel(),
                            _lib.stream()))
    return da


def dice(pred, gt, eps=1e-5):
    """diceCoeff(pred, gt, activation='none') (pix2pix_model.py:13-39): (mean dice as device scalar, sums for the backward)."""
    n = pred.shape[0]
    per = pred.numel() // n
    sums = torch.empty(n, 3, device=pred.device, dtype=torch.float32)
    dn = torch.empty(n, device=pred.device, dtype=torch.float32)
    check(_L().hv_dice_fwd(ptr(pred), ptr(gt), ptr(sums), ptr(dn), n, per, float(eps), _lib.stream()))
    mean = reduce_scalar(dn, None, 3, 1.0 / n)
    return mean, sums


def dice_grad(gt, sums, g_out, eps=1e-5):
    n = gt.shape[0]
    per = gt.numel() // n
    d = torch.empty_like(gt)
    check(_L().hv_dice_bwd(ptr(gt), ptr(sums), float(g_out), float(eps), ptr(d), n, per, 0, _lib.stream()))
    return d


class TensorTable:
    """Device table of the multi-tensor kernels (hv_adam_step_multi / hv_bucket_copy): n rows of six int64
    {p, g, m, v, count, first_chunk}.  The table is re-uploaded only when a pointer changed (gradient tensors are re-allocated every
    step, but the caching allocator hands the same blocks back once the step's allocation pattern has settled)."""

    def __init__(self):
        self.rows = None
        self.dev = None
        self.host = None
        self.chunks = 0

    def update(self, cols, counts, device):
        import numpy as np
        chunk = _L().hv_multi_tensor_chunk()
        first, c = [], 0
        for k in counts:
            first.append(c)
            c += (k + chunk - 1) // chunk
        rows = [tuple(col[i] for col in cols) + (counts[i], first[i]) for i in range(len(counts))]
        if rows != self.rows:
            arr = np.array(rows, dtype=np.int64)
            if self.host is None or self.host.shape != arr.shape:
                self.host = torch.empty(arr.shape, dtype=torch.int64).pin_memory()
                self.dev = torch.empty(arr.shape, dtype=torch.int64, device=device)
            else:
                torch.cuda.current_stream(device).synchronize()   # a previous async upload may still read the pinned staging
            self.host.copy_(torch.from_numpy(arr))
            self.dev.copy_(self.host, non_blocking=True)
            self.rows = rows
            self.chunks = c
        return self.dev, len(rows), self.chunks


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam(lr, betas) semantics (pix2pix_model.py:127-130); state keys mirror torch's.  ONE kernel launch per step for
    all parameters of the optimiser (hv_adam_step_multi); parameters with different step counts take one launch per tensor.  A
    torch.optim.Optimizer, so that torch's learning-rate schedulers drive param_groups[0]["lr"] (networks.get_scheduler)."""

    def __init__(self, params, lr=2e-4, betas=(0.5, 0.999), eps=1e-8):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps))
        self.params = self.param_groups[0]["params"]
        self._table = TensorTable()
        self._step = 0

    def zero_grad(self, set_to_none=True):
        for p in self.params:
            p.grad = None

    @torch.no_grad()
    def step(self):
        g = self.param_groups[0]
        live = [p for p in self.params if p.grad is not None]
        if not live:
            return
        for p in live:
            if p not in self.state:
                self.state[p] = {"step": 0, "exp_avg": torch.zeros_like(p), "exp_avg_sq": torch.zeros_like(p)}
        steps = {self.state[p]["step"] for p in live}
        if len(steps) != 1:   # parameters with different step counts (some had no gradient earlier): per tensor
            for p in live:
                st = self.state[p]
                st["step"] += 1
                grad = p.grad.contiguous()
                check(_L().hv_adam_step(ptr(p.data), ptr(grad), ptr(st["exp_avg"]), ptr(st["exp_avg_sq"]), p.numel(), float(g["lr"]),
                                        float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]), int(st["step"]), _lib.stream()))
                torch.autograd.graph.increment_version(p)
            return
        grads = [p.grad if p.grad.is_contiguous() else p.grad.contiguous() for p in live]
        cols = ([ptr(p.data) for p in live], [ptr(t) for t in grads], [ptr(self.state[p]["exp_avg"]) for p in live],
                [ptr(self.state[p]["exp_avg_sq"]) for p in live])
        table, n, chunks = self._table.update(cols, [p.numel() for p in live], live[0].device)
        step = steps.pop() + 1
        check(_L().hv_adam_step_multi(ptr(table), n, chunks, float(g["lr"]), float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]),
                                      int(step), _lib.stream()))
        for p in live:
            self.state[p]["step"] = step
            # the kernel wrote through raw pointers: tell torch (and the Generator's cached-plan signature, which compares
            # tensor._version) that the parameter changed in place, exactly as an eager optimizer step would
            torch.autograd.graph.increment_version(p)


class GradientBucket:
    """One flat fp32 buffer per net for the data-parallel gradient exchange (SURVEY 8e: 4 all-reduces per step, not one per tensor):
    gather (1 launch) -> all_reduce(SUM) on the flat buffer (NCCL over NVLink) -> scatter scaled by 1 / world (1 launch)."""

    def __init__(self):
        self._table = TensorTable()
        self.flat = None

    @torch.no_grad()
    def allreduce_mean_(self, grads, world, all_reduce):
        if world <= 1 or not grads:
            return
        grads = [t if t.is_contiguous() else t.contiguous() for t in grads]
        zero = [0] * len(grads)
        table, n, chunks = self._table.update(([ptr(t) for t in grads], zero, zero, zero), [t.numel() for t in grads], grads[0].device)
        size = chunks * _L().hv_multi_tensor_chunk()
        if self.flat is None or self.flat.numel() != size:
            self.flat = torch.empty(size, device=grads[0].device, dtype=torch.float32)
        check(_L().hv_bucket_copy(ptr(table), n, chunks, ptr(self.flat), 1.0, 1, _lib.stream()))
        all_reduce(self.flat)
        check(_L().hv_bucket_copy(ptr(table), n, chunks, ptr(self.flat), 1.0 / world, 0, _lib.stream()))
