"""Contextual attention restated in float64, rounding where the bf16 tensor-core chain rounds.

TEST INFRASTRUCTURE — never imported by the product package.

``restate`` mirrors ``csrc/ctx_attn_tc.cu`` (the chain behind ``hv_ctx_attn_fwd_bf16`` and the generator plan's
attention) stage by stage, on any torch device:

* P (3x3 patches of the ::2 feature) and R (4x4 stride-2 patches) come from the bf16 features;
* ``inv_norm = 1 / max(sqrt(sum P^2), 1e-4)`` in fp32 (IEEE sqrtf and division: the library is built without fast-math);
* ``T[f][b] = fl32(fl32(sum_k P_f P_b) * inv_norm[b])`` (the GEMM's fp32 accumulator times its column scale);
* the fuse sums T in the kernel's order, ``cc`` outer, ``a`` inner, in fp32; flat indices outside [0, L) contribute 0;
* ``z = fl32(fl32(U * mm) * scale)``; softmax in float64 from the fp32 logits; ``A = softmax * mm``, rounded to bf16;
* ``cols = R @ bf16(A)^T`` in float64, rounded to bf16; ``y = bf16(0.25 * fold(cols))``;
* the argmax is taken over the unrounded A, ties going to the smallest index.

With ``rounded=False`` and float64 inputs every stage is exact float64 and the result is the plain closed form of
``oracle.generator_ref.contextual_attention`` (which ``tests/test_ctx_attn_ref_cpu.py`` checks).

``variant`` selects a deliberately wrong restatement (a negative control the tests must reject):
``"fuse2d"`` 2-D shifts instead of flat-index shifts; ``"fuse_a_only"`` only the ``a`` pass of the fuse; ``"no_trailing_mm"``
no ``* mm`` after the softmax; ``"mask_max8"`` an 8x8-max mask sampler instead of ``[::8, ::8]``; ``"mask_sample0"`` the
mask of sample 0 although ``per_sample_mask`` is set; ``"fold_count"`` fold divided by the real overlap count instead of 4;
``"tie_last"`` the last maximal index instead of the first.
"""
from __future__ import annotations

from types import SimpleNamespace

import torch
import torch.nn.functional as F

SIDE, L = 32, 1024
VARIANTS = ("fuse2d", "fuse_a_only", "no_trailing_mm", "mask_max8", "mask_sample0", "fold_count", "tie_last")
# the case on which each wrong variant must be rejected: (variant, mask kind, softmax_scale, fuse, per_sample_mask, n)
CONTROL_CASES = [
    ("fuse2d", "band_top", 10.0, True, False, 1),
    ("fuse2d", "band_bottom", 1.0, True, False, 3),
    ("fuse_a_only", "band", 10.0, True, False, 1),
    ("no_trailing_mm", "band", 0.1, True, False, 1),
    # not the [3, 44) band: the 3x3 dilation of the sampled mask already covers the block row an 8x8 max adds at the border
    ("mask_max8", "band_105_140", 10.0, True, False, 1),
    ("mask_max8", "row100", 10.0, True, False, 1),
    ("mask_sample0", "band", 10.0, True, True, 3),
    ("fold_count", "band", 1.0, True, False, 1),
    ("tie_last", "band", 10.0, True, False, 1),          # the zero and copied blocks of grid_features
]


def bf16(x):
    """Round to the nearest bf16 (ties to even), returned in x's dtype.  float64 goes through fp32 first, as the kernels
    round fp32 values."""
    return x.to(torch.float32).to(torch.bfloat16).to(x.dtype)


def _cm(i):
    return (i % SIDE) * SIDE + i // SIDE


def fuse_sources(variant=None, device="cpu"):
    """[(src, valid)] per fuse term in the kernel's summation order (cc outer, a inner): U[j][i] = sum T[src[j]][src[i]]
    over the terms where valid[j] and valid[i]."""
    idx = torch.arange(L, device=device)
    out = []
    for cc in (-1, 0, 1):
        if variant == "fuse_a_only" and cc != 0:
            continue
        for a in (-1, 0, 1):
            if variant == "fuse2d":
                h, w = idx // SIDE + cc, idx % SIDE + a
                valid = (h >= 0) & (h < SIDE) & (w >= 0) & (w < SIDE)
                src = h * SIDE + w
            else:
                p = _cm(idx) + cc
                v1 = (p >= 0) & (p < L)
                s = _cm(p.clamp(0, L - 1)) + a
                valid = v1 & (s >= 0) & (s < L)
                src = s
            out.append((src.clamp(0, L - 1), valid))
    return out


def fuse(T, variant=None):
    """The two identity-3x3 fuse convolutions on T [n, L_f, L_b], summed term by term in T's dtype."""
    U = torch.zeros_like(T)
    for src, valid in fuse_sources(variant, T.device):
        term = T[:, src][:, :, src]
        U = U + torch.where(valid[:, None] & valid[None, :], term, torch.zeros((), dtype=T.dtype, device=T.device))
    return U


def mask_valid(mask, per_sample_mask, variant=None):
    """mm [n, L] = 1 where the zero-padded 3x3 neighbourhood of the 1/8 mask is all zero (float64)."""
    n = mask.shape[0]
    m = mask.to(torch.float64)
    if not per_sample_mask or variant == "mask_sample0":
        m = m[:1].expand(n, -1, -1, -1)
    md = F.max_pool2d(m, 8) if variant == "mask_max8" else m[:, :, ::8, ::8]
    u = F.unfold(F.pad(md, (1, 1, 1, 1)), kernel_size=3)          # [n, 9, L]
    return (u.mean(dim=1) == 0.0).to(torch.float64)


def patches(f):
    """P [n, L, C*9] (rows = positions) and R [n, C*16, L] of features f [n, C, 64, 64]."""
    P = F.unfold(F.pad(f[:, :, ::2, ::2], (1, 1, 1, 1)), kernel_size=3).transpose(1, 2)
    R = F.unfold(F.pad(f, (1, 1, 1, 1)), kernel_size=4, stride=2)
    return P, R


def inv_norm(P, rounded=True):
    """1 / max(|P_l|, 1e-4) per row; in fp32 (correctly rounded, as sqrtf and 1.f / x are) when ``rounded``."""
    ss = (P * P).sum(dim=-1)
    if not rounded:
        return 1.0 / torch.clamp(torch.sqrt(ss), min=1e-4)
    nrm = torch.sqrt(ss).to(torch.float32)                       # sqrt of an fp32-exact sum: one rounding to fp32
    nrm = torch.maximum(nrm, torch.tensor(1e-4, dtype=torch.float32, device=P.device))
    return (1.0 / nrm.to(torch.float64)).to(torch.float32)       # 53 >= 2 * 24 + 2: the double rounding is innocuous


def logits(f, mask, softmax_scale=10.0, fuse_on=True, per_sample_mask=False, rounded=True, variant=None):
    """Fused, masked, scaled logits z [n, L_f, L_b] (fp32 values in float64 when ``rounded``), mm [n, L_b], P, R, inv."""
    f = f.to(torch.float64)
    if rounded:
        f = bf16(f)
    P, R = patches(f)
    inv = inv_norm(P, rounded)
    S = P @ P.transpose(1, 2)                                    # exact for features on a 2^-6 grid
    mm = mask_valid(mask.to(f.device), per_sample_mask, variant)
    if rounded:
        T = S.to(torch.float32) * inv[:, None, :]
        U = fuse(T, variant) if fuse_on else T
        z = (U * mm[:, None, :].to(torch.float32)) * torch.tensor(softmax_scale, dtype=torch.float32)
        z = z.to(torch.float64)
    else:
        T = S * inv[:, None, :]
        U = fuse(T, variant) if fuse_on else T
        z = U * mm[:, None, :] * softmax_scale
    return SimpleNamespace(z=z, mm=mm, P=P, R=R, inv=inv)


def restate(f, mask, softmax_scale=10.0, fuse_on=True, per_sample_mask=False, rounded=True, variant=None):
    """The whole chain.  Returns y [n, C, 64, 64], offsets [n, 2, 32, 32] (int64), argmax [n, L] and the float64
    intermediates the error bounds need: A64 (unrounded weights), A (as pasted), cols (as folded), R, z."""
    assert variant is None or variant in VARIANTS, variant
    lg = logits(f, mask, softmax_scale, fuse_on, per_sample_mask, rounded, variant)
    z, mm = lg.z, lg.mm
    e = torch.exp(z - z.amax(dim=-1, keepdim=True))
    A64 = e / e.sum(dim=-1, keepdim=True)
    if variant != "no_trailing_mm":
        A64 = A64 * mm[:, None, :]
    if variant == "tie_last":
        am = L - 1 - torch.argmax(A64.flip(-1), dim=-1)
    else:
        am = torch.argmax(A64, dim=-1)                           # first maximal index
    A = bf16(A64) if rounded else A64
    cols64 = lg.R @ A.transpose(1, 2)                            # [n, C*16, L_f]
    cols = bf16(cols64) if rounded else cols64
    y = F.fold(cols, output_size=(64, 64), kernel_size=4, stride=2, padding=1)
    if variant == "fold_count":
        ones = torch.ones_like(cols[:1])
        y = y / F.fold(ones, output_size=(64, 64), kernel_size=4, stride=2, padding=1)
    else:
        y = y * 0.25
    y64 = y
    if rounded:
        y = bf16(y)
    ar = torch.arange(L, device=am.device)
    off = torch.stack([am // SIDE - ar // SIDE, am % SIDE - ar % SIDE], dim=1).reshape(-1, 2, SIDE, SIDE)
    return SimpleNamespace(y=y, y64=y64, offsets=off, argmax=am, A64=A64, A=A, cols=cols, cols64=cols64, R=lg.R, z=z,
                           mm=mm, P=lg.P, inv=lg.inv)


# ----------------------------------------------------------------------------- error bounds and the check
EPS_A = 2.0 ** -13        # relative freedom of the kernel's fp32 weights: __expf, the order of the 1024-term sum, 1 / sum
GAMMA_PASTE = 2.0 ** -13  # fp32 accumulation of the paste GEMM over K = 1024: K * 2^-23 (truncating alignment allowed)
TIE_EPS = 2.0 ** -20      # top-two weights closer than this (but not equal) may swap under __expf


def bf16_spacing(x):
    """Distance between adjacent bf16 numbers at |x| (2^-133, the subnormal step, at zero)."""
    _, e = torch.frexp(x.abs())
    sp = torch.ldexp(torch.ones_like(x), e - 8)
    return torch.where(x == 0, torch.zeros_like(x), sp).clamp(min=2.0 ** -133)


def fold4(cols):
    return 0.25 * F.fold(cols, output_size=(64, 64), kernel_size=4, stride=2, padding=1)


def weight_freedom(A64, eps=EPS_A):
    """How far the bf16 weight the kernel pastes may lie from bf16(A64): the width of the bf16 rounding step when A64 is
    within eps (relative) of a rounding boundary, else 0; weights in fp32's subnormal range may also flush to 0."""
    dA = bf16(A64 * (1 + eps)) - bf16(A64 * (1 - eps))
    return torch.where(A64 < 2.0 ** -125, torch.maximum(dA, bf16(A64)), dA)


def y_bound(ref, extra_dA=None):
    """Per-element bound on |y - ref.y|:  spacing(y) + 0.25 fold(spacing(cols) + |R| @ dA^T + gamma |R| @ A^T).
    ``extra_dA`` [n, L_f, L_b] adds a first-order weight error (the realistic-feature case)."""
    Rabs = ref.R.abs()
    dA = weight_freedom(ref.A64)
    if extra_dA is not None:
        dA = dA + extra_dA
    dcols = Rabs @ dA.transpose(1, 2) + GAMMA_PASTE * (Rabs @ ref.A64.transpose(1, 2))
    bc = dcols + bf16_spacing(ref.cols.abs() + dcols)
    by = fold4(bc)
    return by + bf16_spacing(ref.y.abs() + by)


def check(y, offsets, ref, bound=None, logit_tol=None):
    """Compare a kernel's (y, offsets) with a restatement.  Returns a dict: ``ok``, ``ratio`` (max |y - y_ref| / bound),
    ``bad_y`` (elements over the bound), ``bad_off`` (rows whose argmax is not allowed), ``finite``.

    Argmax rule: equal to the restatement's, except (a) rows whose two largest weights differ by less than TIE_EPS relative
    without being equal, where any index within TIE_EPS of the maximum is allowed, or (b) with ``logit_tol`` [n, L_f] (the
    realistic case): rows where the fp64 gap between the two largest fused logits is at most logit_tol, where any index whose
    logit is within logit_tol of the maximum is allowed."""
    y = y.to(ref.y.device, torch.float64)
    am = offsets_to_argmax(offsets.to(ref.y.device))
    bound = y_bound(ref) if bound is None else bound
    err = (y - ref.y).abs()
    finite = bool(torch.isfinite(y).all())
    bad_y = int((err > bound).sum()) if finite else y.numel()
    ratio = float((err / bound).max()) if finite else float("inf")
    same = am == ref.argmax
    A64 = ref.A64
    got = torch.gather(A64, -1, am[..., None])[..., 0]
    if logit_tol is None:
        top = A64.topk(2, dim=-1).values
        t0, t1 = top[..., 0], top[..., 1]
        near = (t1 < t0) & (t0 - t1 <= TIE_EPS * t0)
        allowed = same | (near & (got >= t0 * (1 - TIE_EPS)))
    else:
        z = torch.where(ref.mm[:, None, :] > 0, ref.z, torch.full_like(ref.z, -float("inf")))   # background candidates only
        top = z.topk(2, dim=-1).values
        zgot = torch.gather(z, -1, am[..., None])[..., 0]
        near = top[..., 0] - top[..., 1] <= logit_tol
        allowed = same | (near & (zgot >= top[..., 0] - logit_tol))
    bad_off = int((~allowed).sum())
    return dict(ok=finite and bad_y == 0 and bad_off == 0, ratio=ratio, bad_y=bad_y, bad_off=bad_off, finite=finite,
                ties_exempt=int((near & ~same).sum()))


def offsets_to_argmax(off):
    """offsets [n, 2, 32, 32] (row, col of the argmax minus own position) -> flat argmax [n, L]."""
    off = off.reshape(off.shape[0], 2, L).to(torch.int64)
    ar = torch.arange(L, device=off.device)
    return (off[:, 0] + ar // SIDE) * SIDE + off[:, 1] + ar % SIDE


# ----------------------------------------------------------------------------- inputs
MASKS = ("empty", "full", "band", "band_top", "band_bottom", "band_3_44", "band_105_140", "row100", "row104", "columns", "blob")


def grid_features(n, seed=0, device="cpu"):
    """Features on the 2^-6 grid, integers in [-8, 15] (exact in bf16; every product and partial sum of the similarity
    GEMM is then an integer times 2^-12 below 2^17, exact in fp32), with a zero block (zero patches, the 1e-4 clamp, exact
    ties) and a block copied from elsewhere (exact ties between distinct non-zero patches).  Offsets are even, so both
    blocks sit on the ::2 grid of the similarity patches.  [n, 64, 64, 64] float32."""
    g = torch.Generator().manual_seed(seed)
    f = torch.randint(-8, 16, (n, 64, 64, 64), generator=g).to(torch.float32) * 2.0 ** -6
    f[:, :, 4:20, 4:28] = 0
    f[:, :, 44:60, 40:60] = f[:, :, 44:60, 4:24]
    return f.to(device)


def make_mask(kind, n, mixed=False, seed=0):
    """[n, 1, 256, 256] attention masks.  ``mixed``: sample i is the kind's mask rolled down by 24 i rows, so that
    masks differ per sample (empty and full stay as they are)."""
    m = torch.zeros(1, 1, 256, 256)
    if kind == "empty":
        pass
    elif kind == "full":
        m[:] = 1
    elif kind == "band":
        m[..., 100:141, :] = 1                 # the eval band
    elif kind == "band_top":
        m[..., 0:41, :] = 1
    elif kind == "band_bottom":
        m[..., 215:256, :] = 1
    elif kind == "band_3_44":
        m[..., 3:44, :] = 1                    # not aligned to the ::8 sampling
    elif kind == "band_105_140":
        m[..., 105:140, :] = 1                 # unaligned at both ends, away from the border
    elif kind == "row100":
        m[..., 100, :] = 1                     # invisible to [::8, ::8]
    elif kind == "row104":
        m[..., 104, :] = 1                     # visible
    elif kind == "columns":
        m[..., :, 60:101] = 1
    elif kind == "blob":
        g = torch.Generator().manual_seed(1000 + seed)
        yy, xx = torch.meshgrid(torch.arange(256.0), torch.arange(256.0), indexing="ij")
        cy, cx = (torch.rand(2, generator=g) * 128 + 64).tolist()
        ry, rx = (torch.rand(2, generator=g) * 40 + 20).tolist()
        m[0, 0] = (((yy - cy) / ry) ** 2 + ((xx - cx) / rx) ** 2 <= 1).float()
        m[0, 0] = torch.maximum(m[0, 0], (torch.rand(256, 256, generator=g) < 0.002).float())
    else:
        raise ValueError(kind)
    m = m.expand(n, -1, -1, -1).clone()
    if mixed:
        for i in range(1, n):
            m[i] = torch.roll(m[0], 24 * i, dims=1)
    return m
