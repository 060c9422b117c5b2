"""Op-level parity of the tcgen05 bf16 convolution kernel (csrc/conv_tc.cu) against fp32 torch convolutions on
bf16-ROUNDED operands (reference op: Conv2dBlock.forward, models/inpaint_networks.py:494-503).

Two angles:
* `hv_conv2d_bf16` (the stand-alone C-ABI op) over geometries the plan does not use (ragged extents and channel counts,
  N != 16), once through the geometry-specialised kernel instance (where one matches) and once through the generic
  FIXED = 0 instance (flags bit 1);
* every kernel instance of the generator plan (kx-packed inputs, space-to-depth, x-phase tail, tile pairs, two sources,
  fused upsample stores, dual heads): the output tap of each layer is recomputed from the plan's OWN bf16 input taps, so
  the tolerance is one bf16 rounding of the result, not the accumulated drift of a 30-layer network.

Tolerance: the kernel accumulates bf16 x bf16 products in fp32 and rounds the activated result to bf16; the expected value is
rounded the same way, so the two may differ by ONE bf16 ulp (2^-7 relative at worst) where fp32 summation-order noise straddles
a rounding boundary; heads stay fp32:  |got - want| <= 2^-7 |want| + 3e-5 * max|want|.
"""
import zlib

import pytest
import torch
import torch.nn.functional as F

import healthivert_gan_b200 as hv
from healthivert_gan_b200 import _lib
from healthivert_gan_b200._lib import HV_ACT, HV_SRC_DIRECT, check, ptr
from oracle import generator_ref as gr
from oracle import synth

pytestmark = pytest.mark.gpu


def _bf(t):
    return t.to(torch.bfloat16).to(torch.float32)


def _act(y, act):
    return {"elu": F.elu, "relu": F.relu, "sigmoid": torch.sigmoid, "none": lambda t: t,
            "clamp1": lambda t: t.clamp(-1, 1)}[act](y)


def _close(got, want, what, rounded=True):
    scale = float(want.abs().max())
    tol = (2.0 ** -7 * 1.001 if rounded else 1e-5) * want.abs() + 3e-5 * max(scale, 1e-3)
    bad = (got - want).abs() > tol
    assert not bool(bad.any()), (what, int(bad.sum()), float((got - want).abs().max()), scale)


def _conv_bf16(srcs, w, b, k, stride, dil, act, flags=0, heads=False):
    """hv_conv2d_bf16 on a channel concatenation of fp32 NCHW CUDA tensors."""
    d = _lib.hv_conv_desc()
    n, _, h, wd = srcs[0].shape
    cin = 0
    for i, t in enumerate(srcs):
        d.src[i].ptr, d.src[i].channels, d.src[i].mode = ptr(t), t.shape[1], HV_SRC_DIRECT
        cin += t.shape[1]
    cout = w.shape[0]
    d.n, d.cin, d.cout, d.hin, d.win = n, cin, cout, h, wd
    d.k, d.stride, d.pad, d.dil, d.nsrc = k, stride, (k - 1) // 2 * dil, dil, len(srcs)
    d.act = HV_ACT["heads"] if heads else HV_ACT[act]
    ho, wo = h // stride, wd // stride
    sc = 2 if flags & 1 else 1
    if heads:
        y = torch.empty(n, 1, ho, wo, device="cuda")
        y2 = torch.empty_like(y)
    else:
        y, y2 = torch.empty(n, cout, ho * sc, wo * sc, device="cuda"), None
    check(_lib.lib().hv_conv2d_bf16(d, ptr(w), ptr(b), ptr(y), ptr(y2), flags, _lib.stream()))
    torch.cuda.synchronize()
    return (y, y2) if heads else y


# (n, [source channels], cout, k, stride, dil, h, w, act, up2)
CASES = [
    (3, [64], 64, 3, 1, 1, 64, 64, "elu", False),       # the trunk geometry (specialised instance 0x11334)
    (2, [64], 64, 3, 1, 2, 64, 64, "elu", False),
    (1, [64], 64, 3, 1, 4, 64, 64, "elu", False),
    (2, [64], 64, 3, 1, 8, 64, 64, "relu", False),
    (17, [64], 64, 3, 1, 16, 64, 64, "elu", False),     # N != 16, more images than one wave
    (2, [32], 32, 3, 1, 1, 48, 80, "elu", False),
    (3, [16], 32, 3, 2, 1, 64, 96, "elu", False),       # stride 2 = space-to-depth source
    (2, [32], 64, 3, 2, 1, 40, 56, "elu", False),
    (2, [24], 40, 3, 1, 1, 40, 56, "elu", False),       # ragged channel counts (padding channels / filters)
    (2, [16], 16, 5, 1, 1, 37, 53, "elu", False),       # 5x5, odd extents
    (1, [8], 8, 3, 1, 1, 33, 130, "none", False),
    (2, [64, 64], 64, 3, 1, 1, 64, 64, "elu", False),   # two sources (allconv11)
    (2, [32, 1], 32, 3, 1, 1, 48, 48, "elu", False),    # 33 -> 32 (conv19 without the kx packing)
    (2, [64], 64, 3, 1, 1, 32, 32, "elu", True),        # fused nearest x2 upsample on the store
    (2, [32], 16, 3, 1, 1, 64, 64, "sigmoid", False),
]


@pytest.mark.parametrize("generic", [0, 2])
@pytest.mark.parametrize("case", CASES, ids=lambda c: "n{}_c{}_o{}_k{}s{}d{}_{}x{}_{}{}".format(
    c[0], "+".join(map(str, c[1])), c[2], c[3], c[4], c[5], c[6], c[7], c[8], "_up2" if c[9] else ""))
def test_standalone_bf16_conv_against_bf16_rounded_torch(case, generic):
    n, chans, cout, k, stride, dil, h, w, act, up2 = case
    g = torch.Generator().manual_seed(zlib.crc32(repr(case).encode()) & 0xFFFF)
    srcs = [torch.randn(n, c, h, w, generator=g).cuda() for c in chans]
    cin = sum(chans)
    wt = (torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5).cuda()
    b = (torch.randn(cout, generator=g) * 0.1).cuda()
    got = _conv_bf16(srcs, wt, b, k, stride, dil, act, flags=(1 if up2 else 0) | generic)
    x = torch.cat([_bf(s) for s in srcs], 1).double().cpu()
    want = F.conv2d(x, _bf(wt).double().cpu(), b.double().cpu(), stride=stride, padding=(k - 1) // 2 * dil, dilation=dil)
    want = _bf(_act(want, act).float())
    if up2:
        want = want.repeat_interleave(2, 2).repeat_interleave(2, 3)
    _close(got.cpu(), want, case)


@pytest.mark.parametrize("generic", [0, 2])
def test_standalone_bf16_dual_heads(generic):
    g = torch.Generator().manual_seed(11)
    for chans in ([8], [8, 1]):
        srcs = [torch.randn(2, c, 48, 64, generator=g).cuda() for c in chans]
        cin = sum(chans)
        wt = (torch.randn(2, cin, 3, 3, generator=g) * 0.3).cuda()
        b = (torch.randn(2, generator=g) * 0.1).cuda()
        y, y2 = _conv_bf16(srcs, wt, b, 3, 1, 1, "none", flags=generic, heads=True)
        x = torch.cat([_bf(s) for s in srcs], 1).double().cpu()
        want = F.conv2d(x, _bf(wt).double().cpu(), b.double().cpu(), padding=1)
        _close(y.cpu(), want[:, 0:1].clamp(-1, 1).float(), ("clamp head", chans), rounded=False)
        # the sigmoid head uses the fast exponential (__expf): a few 1e-6 absolute
        assert float((y2.cpu() - torch.sigmoid(want[:, 1:2]).float()).abs().max()) <= 2e-5


# ------------------------------------------------------------------------------------------------ plan instances
@pytest.fixture(scope="module")
def gen_bf16(synthetic_sd):
    g = hv.Generator({"input_dim": 1, "ngf": 16}, True)
    g.load_state_dict(synthetic_sd)
    g = g.cuda().eval()
    g.precision = "bf16"
    return g


def _subpixel_expected(lo, cam_hi, w, b):
    """conv3x3(cat[nearest_x2(lo), cam_hi]) exactly as the sub-pixel upsample mode of the kernel computes it (tc_conv_setup `ups`):
    output parity (py, px) is a 3x3 conv over the LOW-res map whose tap (dy, dx) carries the fp32 SUM (in kernel order, then rounded to
    bf16) of the original taps landing on that low-res pixel; the full-resolution plane keeps its original (rounded) taps."""
    n, cin, h, wd = lo.shape
    cout = w.shape[0]
    out = torch.zeros(n, cout, 2 * h, 2 * wd, dtype=torch.float64)
    for py in range(2):
        for px in range(2):
            wl = torch.zeros(cout, cin, 3, 3, dtype=torch.float32)
            for ky in range(3):
                for kx in range(3):
                    dy, dx = (py + ky - 1) // 2, (px + kx - 1) // 2
                    wl[:, :, dy + 1, dx + 1] = wl[:, :, dy + 1, dx + 1] + w[:, :cin, ky, kx]
            y = F.conv2d(lo.double(), _bf(wl).double(), None, padding=1)
            if cam_hi is not None:
                y = y + F.conv2d(cam_hi.double(), _bf(w[:, cin:]).double(), None, padding=1)[:, :, py::2, px::2]
            out[:, :, py::2, px::2] = y
    return out + b.double().view(1, -1, 1, 1)


def _w_eff(sd, net, name):
    p = f"{net}.{name}.conv."
    w = sd[p + "weight_orig"]
    return (w / gr.sn_sigma(w, sd[p + "weight_u"], sd[p + "weight_v"])), sd[p + "bias"]


@pytest.mark.parametrize("n", [16, 3])
def test_every_plan_instance_against_bf16_rounded_torch(gen_bf16, synthetic_sd, n):
    """Each conv launch of the bf16 plan, checked in isolation: expected = act(conv(bf16 inputs the plan itself produced,
    bf16-rounded W/sigma) + bias) rounded to bf16.  n = 3 leaves partial waves and an odd tile count for the tile-pair instance."""
    x, mask, cam, ratio = synth.synthetic_slices(n, seed=300 + n)
    with torch.no_grad():
        out = gen_bf16(x.cuda(), mask.cuda(), cam.cuda(), ratio.cuda())
    torch.cuda.synchronize()
    layers = gr.all_layers()
    idx = {f"{l[0]}.{l[1]}": i for i, l in enumerate(layers)}
    tap = {}

    def T(name):
        if name not in tap:
            l = layers[idx[name]]
            t = gen_bf16.read_tap(idx[name]).cpu()
            tap[name] = t.reshape(n, l[3], int(round((t.numel() / n / l[3]) ** 0.5)), -1)
        return tap[name]

    up = lambda t: t.repeat_interleave(2, 2).repeat_interleave(2, 3)
    plane = lambda v: _bf(v.reshape(n, 1, 1, 1).expand(n, 1, 256, 256))
    xb, mb, camb, rb = _bf(x), _bf(mask), _bf(cam), plane(ratio)
    C, Fi = "coarse_generator.", "fine_generator."
    fine_in = lambda: torch.cat([xb, _bf(out[0].cpu()), mb, rb], 1)
    heads_in = lambda: torch.cat([T(Fi + "allconv16"), _bf(out[2].cpu())], 1)
    inputs = {   # every layer whose input is not simply the previous layer of the state_dict order
        C + "conv1": lambda: torch.cat([xb, rb, mb], 1),
        C + "conv20": lambda: torch.cat([up(T(C + "conv12")), camb[:, :, ::2, ::2]], 1),
        C + "conv19": lambda: torch.cat([up(T(C + "conv14")), camb], 1),
        C + "conv18": lambda: T(C + "conv16"),
        Fi + "conv1": fine_in,
        Fi + "pmconv1": fine_in,
        Fi + "pmconv9": lambda: gen_bf16.read_tap(47).cpu().reshape(n, 64, 64, 64),
        Fi + "allconv11": lambda: torch.cat([T(Fi + "conv10_atrous"), T(Fi + "pmconv10")], 1),
        Fi + "allconv12": lambda: T(Fi + "allconv11"),
        Fi + "allconv19": lambda: T(Fi + "allconv12"),
        Fi + "allconv13": lambda: up(T(Fi + "allconv19")),
        Fi + "allconv15": lambda: up(T(Fi + "allconv14")),
        Fi + "allconv17": heads_in,
        Fi + "allconv18": heads_in,
    }
    prev = None
    for net, name, cin, cout, k, stride, pad, dil, act in layers:
        full = f"{net}.{name}"
        src = inputs[full]() if full in inputs else T(prev)
        assert src.shape[1] == cin, (full, src.shape)
        w, b = _w_eff(synthetic_sd, net, name)
        if full == C + "conv19":      # sub-pixel upsample mode: per-parity summed taps over the low-res map of conv14 + the CAM plane
            want = _subpixel_expected(T(C + "conv14"), camb, w, b)
        elif full == Fi + "allconv15":
            want = _subpixel_expected(T(Fi + "allconv14"), None, w, b)
        elif full == Fi + "allconv13":
            want = _subpixel_expected(T(Fi + "allconv19"), None, w, b)
        else:
            want = F.conv2d(src.double(), _bf(w).double(), b.double(), stride=stride, padding=pad, dilation=dil)
        head = act in ("none", "sigmoid")
        # conv17 / allconv17 ('none') are followed by torch.clamp(-1, 1) (:115, :230), fused into the head epilogue
        want = want.clamp(-1, 1) if act == "none" else _act(want, act)
        want = want.float() if head else _bf(want.float())
        got = T(full)
        if act == "sigmoid":   # fast exponential (__expf) in the epilogue: a few 1e-6 absolute
            assert float((got - want).abs().max()) <= 2e-5, full
        else:
            _close(got, want, full, rounded=not head)
        prev = full

