"""The float64 restatement of the bf16 contextual-attention chain (oracle/ctx_attn_rounded.py), on the CPU.

* With every rounding switched off it is the plain closed form of oracle.generator_ref.contextual_attention.
* With the roundings on, each deliberately wrong variant is rejected by the same check the GPU tests apply to the kernels,
  on the case listed for it: every negative control of tests/test_gpu_ctx_attn.py can expose its bug.
"""
import pytest
import torch

from oracle import ctx_attn_rounded as car
from oracle import generator_ref as gr


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-300))


@pytest.fixture(scope="module")
def feats():
    g = torch.Generator().manual_seed(3)
    return torch.relu(torch.randn(3, 64, 64, 64, generator=g, dtype=torch.float64))


@pytest.mark.parametrize("fuse", [True, False])
@pytest.mark.parametrize("per_sample", [False, True])
def test_unrounded_restatement_is_the_closed_form(feats, fuse, per_sample):
    mask = car.make_mask("band", 3, mixed=True)
    got = car.restate(feats, mask, 10.0, fuse, per_sample, rounded=False)
    if per_sample:
        refs = [gr.contextual_attention(feats[i:i + 1], mask[i:i + 1], fuse=fuse) for i in range(3)]
        y_ref = torch.cat([r[0] for r in refs])
        off_ref = torch.cat([r[1] for r in refs])
    else:
        y_ref, off_ref = gr.contextual_attention(feats, mask, fuse=fuse)
    assert y_ref.dtype == torch.float64
    assert _rel(got.y, y_ref) <= 1e-10
    assert torch.equal(got.offsets, off_ref)


@pytest.mark.parametrize("scale", [10.0, 0.1])
def test_unrounded_restatement_matches_on_grid_features_and_edge_masks(scale):
    f = car.grid_features(3, seed=1).double()
    for kind in ("empty", "band_top", "row104", "blob"):
        mask = car.make_mask(kind, 3)
        got = car.restate(f, mask, scale, True, False, rounded=False)
        y_ref, off_ref = gr.contextual_attention(f, mask, softmax_scale=scale)
        assert _rel(got.y, y_ref) <= 1e-10, kind
        assert torch.equal(got.offsets, off_ref), kind


def test_rounded_restatement_passes_its_own_check_and_rounds_y_to_bf16():
    f = car.grid_features(3, seed=2)
    ref = car.restate(f, car.make_mask("band", 3, mixed=True), 1.0, True, True)
    assert torch.equal(ref.y, car.bf16(ref.y))
    assert car.check(ref.y, ref.offsets, ref)["ok"]
    full = car.restate(f, car.make_mask("full", 3), 10.0, True, False)
    assert float(full.y.abs().max()) == 0.0 and int(full.argmax.abs().max()) == 0


@pytest.mark.parametrize("variant,kind,scale,fuse,per_sample,n", car.CONTROL_CASES)
def test_each_negative_control_is_rejected_on_its_case(variant, kind, scale, fuse, per_sample, n):
    f = car.grid_features(n, seed=4)
    mask = car.make_mask(kind, n, mixed=per_sample)
    good = car.restate(f, mask, scale, fuse, per_sample)
    bad = car.restate(f, mask, scale, fuse, per_sample, variant=variant)
    res = car.check(good.y, good.offsets, bad)
    assert not res["ok"], (variant, res)
