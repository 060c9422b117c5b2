"""The contextual attention's tensor-core paths against float64 restatements of their own bf16 roundings.

(a) hv_ctx_attn_fwd_bf16 on features on a 2^-6 grid: the restatement (oracle/ctx_attn_rounded.py) reproduces the fp32
    logits bit for bit, so the offsets must be equal (ties included) and y within about two bf16 ulps (the bound of
    ctx_attn_rounded.y_bound); every negative control of the restatement must be rejected by the same check.
(b) the same op on the bf16 plan's own pmconv6 activations, with a stated model of the fp32 accumulation error.
(c) the plan's attention (tap 47, offsets, flow) equals the stand-alone op bit for bit; the same with one stream, and
    the paste GEMM at BN = 128 still passes (a).
(d) the flow image equals gr.flow_image of the kernel's offsets, with the reference's running maxrad across the batch.
(e) the training mode (hv_ctx_attn_fwd_tc / _bwd_tc) against float64 autograd whose dense contractions round their
    operands where tc_contract rounds them.
The references are computed on the GPU in float64.  Each test prints its largest error / bound (run with -s to see it).
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import healthivert_gan_b200 as hv
from healthivert_gan_b200 import train_ops as T
from oracle import ctx_attn_rounded as car
from oracle import generator_ref as gr
from oracle import synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda"
NAMES = [f"{l[0]}.{l[1]}" for l in gr.all_layers()]
TAP_PM6 = NAMES.index("fine_generator.pmconv6")
TAP_CA = len(NAMES)                     # 47: the attention output


def standalone(f, mask, scale=10.0, fuse=True, per_sample=False):
    """hv_ctx_attn_fwd_bf16 through the drop-in module: (y, offsets, flow)."""
    ca = hv.ContextualAttention(True, ksize=3, stride=1, rate=2, fuse_k=3, softmax_scale=scale, fuse=fuse)
    ca.precision = "bf16"
    ca.per_sample_mask = per_sample
    f = f.to(DEV).float().contiguous()
    y, flow = ca(f, f, mask.to(DEV))
    torch.cuda.synchronize()
    return y, ca.last_offsets.clone(), flow


def _report(tag, res):
    print(f"[ctx_attn] {tag}: error/bound {res['ratio']:.3f}, bad y {res['bad_y']}, bad offsets {res['bad_off']}, "
          f"near-ties exempt {res['ties_exempt']}")


# ----------------------------------------------------------------------------------------------------- (a) grid features
SCALES = (10.0, 1.0, 0.1)
BATCHES = (1, 3, 16, 17)   # 17 is beyond the plan's batch


@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("scale", SCALES)
@pytest.mark.parametrize("kind", car.MASKS)
def test_grid_features_pinned_to_rounded_restatement(kind, scale, fuse):
    """Masks differ per sample (sample i rolled by 24 i rows); both mask modes, batches cycling through BATCHES."""
    k = car.MASKS.index(kind) + SCALES.index(scale)
    for per_sample, n in ((False, BATCHES[k % 4]), (True, BATCHES[(k + 1) % 4])):
        f = car.grid_features(n, seed=n, device=DEV)
        mask = car.make_mask(kind, n, mixed=True).to(DEV)
        y, off, _ = standalone(f, mask, scale, fuse, per_sample)
        ref = car.restate(f, mask, scale, fuse, per_sample)
        res = car.check(y, off, ref)
        _report(f"grid {kind} scale={scale} fuse={fuse} per_sample={per_sample} n={n}", res)
        assert res["ok"], res
        if kind == "full":   # no valid background: every weight is 0
            assert float(y.abs().max()) == 0.0 and int(car.offsets_to_argmax(off).abs().max()) == 0


@pytest.mark.parametrize("variant,kind,scale,fuse,per_sample,n", car.CONTROL_CASES)
def test_negative_controls_are_rejected(variant, kind, scale, fuse, per_sample, n):
    f = car.grid_features(n, seed=n, device=DEV)
    mask = car.make_mask(kind, n, mixed=True).to(DEV)
    y, off, _ = standalone(f, mask, scale, fuse, per_sample)
    assert car.check(y, off, car.restate(f, mask, scale, fuse, per_sample))["ok"]
    res = car.check(y, off, car.restate(f, mask, scale, fuse, per_sample, variant=variant))
    _report(f"control {variant} on {kind}", res)
    assert not res["ok"], res


# ----------------------------------------------------------------------------------------------------- (b) realistic features
@pytest.fixture(scope="module")
def gen_bf16():
    g = hv.Generator({"input_dim": 1, "ngf": 16}, True)
    g.load_state_dict(synth.synthetic_generator_state_dict())
    g = g.cuda().eval()
    g.precision = "bf16"
    return g


def _plan_forward(g, n, seed, per_sample, return_flow=True):
    x, mask, cam, ratio = synth.synthetic_slices(n, seed=seed, per_sample_masks=True)
    g.per_sample_mask, g.return_flow = per_sample, return_flow
    with torch.no_grad():
        out = g(x.cuda(), mask.cuda(), cam.cuda(), ratio.cuda())
    torch.cuda.synchronize()
    return out, mask


def logit_error(ref, scale, fuse):
    """Per foreground row j, a bound on |z_kernel - z_restated| over all background columns, from this model:

    T[f][b] = fl32(sum_k P_fk P_bk) * inv[b] with K = 576.  The fp32 accumulator takes one rounding of at most 2^-23
    relative per K = 16 MMA step (truncating alignment allowed), each against a partial sum bounded by
    sum_k |P_fk P_bk| <= |P_f| |P_b| (Cauchy-Schwarz): 36 * 2^-23 = 72 u |P_f| |P_b|, u = 2^-24.  The kernel's
    sum of squares runs <= 24 sequential fmaf per lane and 5 shuffle levels (29 u), halved by the sqrt, plus the sqrt and
    the division: 17 u on inv[b].  The column scale adds 1 u.  Since |P_b| inv[b] <= 1, |dT[f][b]| <= 90 u |P_f|.
    The fuse sums up to 9 such terms in fp32 (8 u more, as |T| <= |P_f|):
        dz_j = scale * 98 u * sum_{s in fuse sources of j} |P_s|
    (without the fuse, s = j only).  The restatement's own fp32 T rounds at the same places, so the model bounds the
    kernel's deviation from it."""
    u = 2.0 ** -24
    pn = ref.P.norm(dim=-1)                                         # [n, L]
    if fuse:
        acc = torch.zeros_like(pn)
        for src, valid in car.fuse_sources(None, pn.device):
            acc = acc + torch.where(valid, pn[:, src], torch.zeros_like(acc))
    else:
        acc = pn
    return scale * 98 * u * acc


@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("per_sample", [False, True])
def test_plan_features_within_accumulation_model(gen_bf16, per_sample, fuse):
    """Input: the bf16 plan's pmconv6 activations on synthetic slices.  The argmax must equal the restatement's wherever the
    fp64 gap between the two largest fused logits exceeds 4 dz_j, and be within 4 dz_j of the maximum elsewhere; y within
    the bound of (a) plus the first-order weight error 0.25 fold(2 dz_j |R| @ A^T)."""
    n = 16
    _, mask = _plan_forward(gen_bf16, n, seed=81, per_sample=per_sample)
    f = gen_bf16.read_tap(TAP_PM6).reshape(n, 64, 64, 64)
    y, off, _ = standalone(f, mask, 10.0, fuse, per_sample)
    ref = car.restate(f, mask.to(DEV), 10.0, fuse, per_sample)
    dz = logit_error(ref, 10.0, fuse)
    bound = car.y_bound(ref, extra_dA=2 * dz[:, :, None] * ref.A64)
    res = car.check(y, off, ref, bound=bound, logit_tol=4 * dz)
    _report(f"plan features per_sample={per_sample} fuse={fuse} (max dz {float(dz.max()):.2e})", res)
    assert res["ok"], res


# ----------------------------------------------------------------------------------------------------- (c) plan == stand-alone
@pytest.mark.parametrize("return_flow", [True, False])
@pytest.mark.parametrize("per_sample", [False, True])
@pytest.mark.parametrize("n", [16, 3])
def test_plan_attention_equals_standalone_op(gen_bf16, n, per_sample, return_flow):
    """Tap 47 (the attention output inside the plan: two streams, PDL) == hv_ctx_attn_fwd_bf16 on the plan's own pmconv6
    output, byte for byte; offsets and flow equal as well."""
    out, mask = _plan_forward(gen_bf16, n, seed=90 + n, per_sample=per_sample, return_flow=return_flow)
    offsets = gen_bf16.last_offsets.clone()
    f = gen_bf16.read_tap(TAP_PM6).reshape(n, 64, 64, 64)
    y47 = gen_bf16.read_tap(TAP_CA).reshape(n, 64, 64, 64)
    y, off, flow = standalone(f, mask, 10.0, True, per_sample)
    assert y47.cpu().numpy().tobytes() == y.cpu().numpy().tobytes()
    assert torch.equal(offsets, off)
    if return_flow:
        assert torch.equal(out[4], flow)
    else:
        assert out[4] is None


_DUMP_PLAN = """
import sys, numpy as np, torch
sys.path.insert(0, {root!r})
import healthivert_gan_b200 as hv
from oracle import synth
g = hv.Generator({{'input_dim': 1, 'ngf': 16}}, True); g.load_state_dict(synth.synthetic_generator_state_dict())
g = g.cuda().eval(); g.precision = 'bf16'; g.per_sample_mask = True
x, mask, cam, ratio = (t.cuda() for t in synth.synthetic_slices(16, seed=95, per_sample_masks=True))
with torch.no_grad():
    o = g(x, mask, cam, ratio)
torch.cuda.synchronize()
np.savez({out!r}, y=g.read_tap({tap}).cpu().numpy(), off=g.last_offsets.cpu().numpy(), flow=o[4].cpu().numpy())
"""

_DUMP_GRID = """
import sys, numpy as np, torch
sys.path.insert(0, {root!r})
import healthivert_gan_b200 as hv
from oracle import ctx_attn_rounded as car
f = car.grid_features(3, seed=3, device='cuda')
mask = car.make_mask('band', 3, mixed=True).cuda()
ca = hv.ContextualAttention(True, ksize=3, stride=1, rate=2, fuse_k=3, softmax_scale=1.0, fuse=True)
ca.precision = 'bf16'; ca.per_sample_mask = True
y, _ = ca(f, f, mask)
torch.cuda.synchronize()
np.savez({out!r}, y=y.cpu().numpy(), off=ca.last_offsets.cpu().numpy())
"""


def _subprocess(script, path, **env_set):
    env = {k: v for k, v in os.environ.items() if k not in ("HV_NO_AUX_STREAM", "HV_GEMM_BN128")}
    env.update(env_set)
    r = subprocess.run([sys.executable, "-c", script.format(root=ROOT, out=str(path), tap=TAP_CA)], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return dict(np.load(path))


def test_plan_attention_without_aux_stream_is_bit_identical(tmp_path):
    """HV_NO_AUX_STREAM=1 runs the raw-patch / mask / offsets-flow launches on the attention's own stream."""
    two = _subprocess(_DUMP_PLAN, tmp_path / "two.npz")
    one = _subprocess(_DUMP_PLAN, tmp_path / "one.npz", HV_NO_AUX_STREAM="1")
    for k in two:
        assert two[k].tobytes() == one[k].tobytes(), k


def test_paste_gemm_bn128_passes_the_grid_pin(tmp_path):
    """HV_GEMM_BN128=1 tiles the paste GEMM 128 wide instead of 256: same bound as (a); also reports bit identity."""
    wide = _subprocess(_DUMP_GRID, tmp_path / "wide.npz")
    narrow = _subprocess(_DUMP_GRID, tmp_path / "narrow.npz", HV_GEMM_BN128="1")
    f = car.grid_features(3, seed=3, device=DEV)
    mask = car.make_mask("band", 3, mixed=True).to(DEV)
    ref = car.restate(f, mask, 1.0, True, True)
    for name, d in (("BN=256", wide), ("BN=128", narrow)):
        res = car.check(torch.from_numpy(d["y"]), torch.from_numpy(d["off"]), ref)
        _report(f"paste GEMM {name}", res)
        assert res["ok"], (name, res)
    print("[ctx_attn] paste GEMM BN=128 bit-identical to BN=256:",
          wide["y"].tobytes() == narrow["y"].tobytes() and np.array_equal(wide["off"], narrow["off"]))


# ----------------------------------------------------------------------------------------------------- (d) flow image
def test_flow_image_carries_maxrad_across_the_batch():
    """Sample 0 has no mask (self matches: offsets 0), sample 1 a wide band (long offsets), samples 2 and 3 narrow bands:
    their own largest offsets are below the running maximum, so the colour scale comes from sample 1.  At most 0.1 % of the
    pixels may differ from gr.flow_image of the kernel's offsets (atan2 rounding at floor boundaries), by one grey level."""
    g = torch.Generator().manual_seed(11)
    f = torch.relu(torch.randn(4, 64, 64, 64, generator=g)).to(torch.bfloat16).float()
    mask = torch.zeros(4, 1, 256, 256)
    mask[1, :, 60:200] = 1
    mask[2, :, 120:130] = 1
    mask[3, :, :, 100:112] = 1
    _, off, flow = standalone(f, mask, 10.0, True, True)
    off = off.cpu().long()
    rad = off.double().pow(2).sum(1).sqrt().flatten(1).amax(1)
    assert float(rad[0]) < float(rad[1]) and float(rad[2:].max()) < float(rad[:2].max()), rad
    want = gr.flow_image(off)
    diff = (flow.cpu() - want).abs()
    assert float(diff.max()) <= 1.0 / 255 + 1e-6
    assert float((diff > 1e-6).float().mean()) <= 1e-3


# ----------------------------------------------------------------------------------------------------- (e) training mode
class _RoundedMM(torch.autograd.Function):
    """C = bf16(X) @ bf16(Y); the backward rounds dC and the other operand (tc_contract's casts)."""

    @staticmethod
    def forward(ctx, X, Y):
        ctx.save_for_backward(X, Y)
        return car.bf16(X) @ car.bf16(Y)

    @staticmethod
    def backward(ctx, dC):
        X, Y = ctx.saved_tensors
        dCr = car.bf16(dC)
        return dCr @ car.bf16(Y).transpose(1, 2), car.bf16(X).transpose(1, 2) @ dCr


class _Similarity(torch.autograd.Function):
    """S[b][f] = sum_k bf16(P_bk inv_b) bf16(P_fk) (the row scale is applied before the cast, ca_cast_kernel).  Backward as
    ctx_attn_bwd_fp32: dG = dS inv; C1 = bf16(dG) @ bf16(P); C2 = bf16(dG)^T @ bf16(P); dinv[b] = sum_f dS S / inv.
    ``variant``: "no_c2" drops C2; "inv_fg" scales the foreground side instead."""

    @staticmethod
    def forward(ctx, P, inv, variant):
        ctx.variant = variant
        if variant == "inv_fg":
            S = car.bf16(P) @ car.bf16(P * inv[..., None]).transpose(1, 2)
        else:
            S = car.bf16(P * inv[..., None]) @ car.bf16(P).transpose(1, 2)
        ctx.save_for_backward(P, inv, S)
        return S

    @staticmethod
    def backward(ctx, dS):
        P, inv, S = ctx.saved_tensors
        Pr = car.bf16(P)
        if ctx.variant == "inv_fg":
            dG = car.bf16(dS * inv[:, None, :])
            dP = dG.transpose(1, 2) @ Pr + dG @ Pr
            return dP, (dS * S).sum(1) / inv, None
        dG = car.bf16(dS * inv[..., None])
        dP = dG @ Pr
        if ctx.variant != "no_c2":
            dP = dP + dG.transpose(1, 2) @ Pr
        return dP, (dS * S).sum(-1) / inv, None


def train_reference(f, mask, scale, variant=None):
    """float64 autograd of the training forward (fuse on, mask of sample 0) with the kernels' bf16 operand roundings."""
    P, R = car.patches(f)
    ss = (P * P).sum(-1)
    live = ss > 1e-8                                                 # |P| > 1e-4; elsewhere the clamp holds (and sqrt'(0) = inf)
    nrm = torch.where(live, torch.sqrt(torch.where(live, ss, torch.ones_like(ss))), torch.full_like(ss, 1e-4))
    S = _Similarity.apply(P, 1.0 / nrm, variant)                     # [n, L_b, L_f]
    U = car.fuse(S.transpose(1, 2))                                  # [n, L_f, L_b]
    mm = car.mask_valid(mask, False)[:, None, :]
    A = torch.softmax(U * mm * scale, dim=-1) * mm
    cols = _RoundedMM.apply(R, A.transpose(1, 2))                    # [n, C*16, L_f]
    return car.fold4(cols)


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp(min=1e-300))


# observed on one B200 (1000 W limit): y 2.4e-5 / df 1.1e-4 (relu features, scale 10), y <= 1.0e-6 / df <= 9.3e-6 on the grid cases; the
# controls land at y 0.25 (inv_norm on the foreground side) and df 0.73 (C2 dropped).  Tolerances: about 4x the worst observed.
TRAIN_TOL_Y, TRAIN_TOL_DF = 1e-4, 5e-4


def _train_case(case):
    g = torch.Generator().manual_seed(6)
    if case == "relu":
        f = torch.relu(torch.randn(2, 64, 64, 64, generator=g))
        scale = 10.0
    else:
        f = car.grid_features(2, seed=6)
        scale = 10.0 if case == "grid10" else 1.0
    mask = torch.zeros(2, 1, 256, 256)
    mask[:, :, 100:141] = 1
    dy = torch.randn(2, 64, 64, 64, generator=g)
    return f, mask, scale, dy


def _train_kernel(f, mask, scale, dy, bf16_backward):
    tape = T.Tape()
    fv = T.Var(f.cuda())
    y, _, _ = T.ctx_attention(tape, fv, mask.cuda(), scale, True, False)
    y.grad = dy.cuda()
    tape.backward()
    torch.cuda.synchronize()
    return y.data, fv.grad


def _train_ref(f, mask, scale, dy, variant=None):
    fd = f.double().to(DEV).requires_grad_()
    y = train_reference(fd, mask.to(DEV), scale, variant)
    y.backward(dy.double().to(DEV))
    return y.detach(), fd.grad


@pytest.fixture
def bf16_backward():
    prev = (T.BACKWARD_PRECISION, T.FORWARD_PRECISION)
    T.BACKWARD_PRECISION = T.FORWARD_PRECISION = "bf16"
    yield
    T.BACKWARD_PRECISION, T.FORWARD_PRECISION = prev


@pytest.mark.parametrize("case", ["relu", "grid10", "grid1"])
def test_training_tensor_core_mode_against_rounded_autograd(case, bf16_backward):
    f, mask, scale, dy = _train_case(case)
    y, df = _train_kernel(f, mask, scale, dy, bf16_backward)
    y_ref, df_ref = _train_ref(f, mask, scale, dy)
    ry, rdf = _rel(y, y_ref), _rel(df, df_ref)
    print(f"[ctx_attn] training {case}: rel L2 y {ry:.2e} (tol {TRAIN_TOL_Y:.0e}), df {rdf:.2e} (tol {TRAIN_TOL_DF:.0e})")
    assert torch.isfinite(y).all() and torch.isfinite(df).all()
    assert 0 < ry <= TRAIN_TOL_Y and rdf <= TRAIN_TOL_DF


@pytest.mark.parametrize("variant", ["no_c2", "inv_fg"])
def test_training_negative_controls_are_rejected(variant, bf16_backward):
    f, mask, scale, dy = _train_case("relu")
    y, df = _train_kernel(f, mask, scale, dy, bf16_backward)
    y_ref, df_ref = _train_ref(f, mask, scale, dy, variant)
    ry, rdf = _rel(y, y_ref), _rel(df, df_ref)
    print(f"[ctx_attn] training control {variant}: rel L2 y {ry:.2e}, df {rdf:.2e}")
    assert ry > TRAIN_TOL_Y or rdf > TRAIN_TOL_DF
