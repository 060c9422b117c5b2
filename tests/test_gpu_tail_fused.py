"""The fused thin tail (csrc/tail_tc.cu: conv16 -> conv17 | conv18 and allconv16 -> allconv17 | allconv18, one launch per stage) must
reproduce the per-layer launches (HV_NO_TAIL_FUSE=1) bit for bit: the four image / mask outputs of the forward and the conv15,
conv16 and allconv16 taps (conv16 / allconv16 are recomputed on demand after a fused forward).  The switch is read once per process,
so each mode runs in its own subprocess."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import healthivert_gan_b200 as hv
from oracle import generator_ref as gr

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_DUMP = """
import sys, numpy as np, torch
sys.path.insert(0, {root!r})
import healthivert_gan_b200 as hv
from oracle import synth, generator_ref as gr
n = {n}
g = hv.Generator({{'input_dim': 1, 'ngf': 16}}, True); g.load_state_dict(synth.synthetic_generator_state_dict())
g = g.cuda().eval(); g.precision = 'bf16'
x, mask, cam, ratio = (t.cuda() for t in synth.synthetic_slices(n, seed=40 + n))
with torch.no_grad():
    o = g(x, mask, cam, ratio)
torch.cuda.synchronize()
idx = {{f"{{l[0]}}.{{l[1]}}": i for i, l in enumerate(gr.all_layers())}}
arrs = {{k: o[i].cpu().numpy() for k, i in (("coarse_seg", 0), ("fine_seg", 1), ("x_stage1", 2), ("x_stage2", 3))}}
for name in ("coarse_generator.conv15", "coarse_generator.conv16", "fine_generator.allconv16"):
    arrs[name] = g.read_tap(idx[name]).cpu().numpy()
np.savez({out!r}, **arrs)
"""


def _run(n, fuse, path):
    env = dict(os.environ, HV_NO_TAIL_FUSE="0" if fuse else "1")
    r = subprocess.run([sys.executable, "-c", _DUMP.format(root=ROOT, n=n, out=str(path))], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return dict(np.load(path))


@pytest.mark.parametrize("n", [16, 3])
def test_fused_tail_equals_per_layer_launches(tmp_path, n):
    """n = 3: an odd image count (the second image of the last pair does not exist) and a different strip height."""
    fused = _run(n, True, tmp_path / "fused.npz")
    plain = _run(n, False, tmp_path / "plain.npz")
    assert fused.keys() == plain.keys()
    for k in fused:
        a, b = fused[k], plain[k]
        assert a.shape == b.shape, k
        assert np.isfinite(a).all(), k
        diff = 0.0 if np.array_equal(a, b) else float(np.abs(a.astype(np.float64) - b).max())
        assert a.tobytes() == b.tobytes(), f"{k}: max |diff| {diff}"


def test_slice_pipeline_with_fused_tail_equals_tensor_api(synthetic_sd):
    """The uint8 pipeline captures the forward (fused tails included) into a CUDA graph; per-sample masks as in the eval driver."""
    g = hv.Generator({"input_dim": 1, "ngf": 16}, True)
    g.load_state_dict(synthetic_sd)
    g = g.cuda().eval()
    g.precision = "bf16"
    g.per_sample_mask = True
    g.return_flow = False
    pipe = hv.SlicePipeline(g, batch=16, depth=2, use_graph=True)
    rng = np.random.Generator(np.random.PCG64(77))
    for k, n in enumerate((16, 5)):
        ct = rng.integers(0, 256, size=(n, 256, 256), dtype=np.uint8)
        cam = rng.integers(0, 256, size=(n, 256, 256), dtype=np.uint8)
        r0 = rng.integers(60, 150, size=n).astype(np.int32)
        rows = np.stack([r0, r0 + 41], axis=1).astype(np.int32)
        ratio = rng.random(n).astype(np.float32)
        x = (torch.from_numpy(ct).float().div(255) - 0.5) / 0.5
        c = 1 - torch.from_numpy(cam).float().div(255)
        m = torch.zeros(ct.shape, dtype=torch.float32)
        for i, (a, b) in enumerate(rows):
            m[i, a:b] = 1
        with torch.no_grad():
            out = g(x[:, None].cuda(), m[:, None].cuda(), c[:, None].cuda(), torch.from_numpy(ratio).cuda())
        torch.cuda.synchronize()
        s = pipe.slot(k)
        s.ct[:n], s.cam[:n], s.rows[:n], s.ratio[:n] = ct, cam, rows, ratio
        pipe.submit(k, n)
        pipe.wait(k)
        assert np.array_equal(s.ct_out[:n], ((out[3] + 1) * 127.5).to(torch.int32).to(torch.uint8).cpu().numpy()[:, 0])
        assert np.array_equal(s.fine_mask[:n].astype(bool), (out[1] > 0.5).cpu().numpy()[:, 0])
        assert np.array_equal(s.coarse_mask[:n].astype(bool), (out[0] > 0.5).cpu().numpy()[:, 0])
    pipe.close()
