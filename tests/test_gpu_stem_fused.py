"""The fused input stem (csrc/stem_tc.cu: conv1 -> conv2_downsample and conv1 | pmconv1 -> conv2_downsample, pmconv2_downsample, one
launch per stage) must reproduce the per-layer launches (HV_NO_STEM_FUSE=1) bit for bit: the seven outputs of the forward and the taps
of every layer of the two stems (conv1 / fine conv1 / pmconv1 are recomputed on demand after a fused forward).  The switch is read once
per process, so each mode runs in its own subprocess."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

TAPS = ("coarse_generator.conv1", "coarse_generator.conv2_downsample", "fine_generator.conv1", "fine_generator.pmconv1",
        "fine_generator.conv2_downsample", "fine_generator.pmconv2_downsample")

_DUMP = """
import sys, numpy as np, torch
sys.path.insert(0, {root!r})
import healthivert_gan_b200 as hv
from oracle import synth, generator_ref as gr
n = {n}
g = hv.Generator({{'input_dim': 1, 'ngf': 16}}, True); g.load_state_dict(synth.synthetic_generator_state_dict())
g = g.cuda().eval(); g.precision = 'bf16'
x, mask, cam, ratio = (t.cuda() for t in synth.synthetic_slices(n, seed=60 + n))
with torch.no_grad():
    o = g(x, mask, cam, ratio)
torch.cuda.synchronize()
idx = {{f"{{l[0]}}.{{l[1]}}": i for i, l in enumerate(gr.all_layers())}}
names = ("coarse_seg", "fine_seg", "x_stage1", "x_stage2", "flow", "pred1_h", "pred2_h")
arrs = {{k: o[i].cpu().numpy() for i, k in enumerate(names)}}
for name in {taps!r}:
    arrs[name] = g.read_tap(idx[name]).cpu().numpy()
np.savez({out!r}, **arrs)
"""


def _run(n, fuse, path, tail_fuse=True):
    env = dict(os.environ, HV_NO_STEM_FUSE="0" if fuse else "1", HV_NO_TAIL_FUSE="0" if tail_fuse else "1")
    r = subprocess.run([sys.executable, "-c", _DUMP.format(root=ROOT, n=n, taps=TAPS, out=str(path))], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return dict(np.load(path))


def _assert_bitwise_equal(fused, plain):
    assert fused.keys() == plain.keys()
    for k in fused:
        a, b = fused[k], plain[k]
        assert a.shape == b.shape, k
        assert np.isfinite(a).all(), k
        diff = 0.0 if np.array_equal(a, b) else float(np.abs(a.astype(np.float64) - b).max())
        assert a.tobytes() == b.tobytes(), f"{k}: max |diff| {diff}"


@pytest.mark.parametrize("n", [16, 3, 1])
def test_fused_stem_equals_per_layer_launches(tmp_path, n):
    """n = 16: one strip of 15 output rows per CTA; n = 3 and n = 1: other strip heights, a grid that does not fill the GPU."""
    _assert_bitwise_equal(_run(n, True, tmp_path / "fused.npz"), _run(n, False, tmp_path / "plain.npz"))


def test_fused_stem_without_fused_tail(tmp_path):
    """With the per-layer tails, the coarse mask of the fine input is packed by its own launch, not by the coarse tail."""
    _assert_bitwise_equal(_run(16, True, tmp_path / "fused.npz", tail_fuse=False),
                          _run(16, False, tmp_path / "plain.npz", tail_fuse=False))
