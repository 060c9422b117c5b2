#!/usr/bin/env python
"""Smallest run that touches every new round-2 kernel family once (for `compute-sanitizer --tool memcheck`): bf16 forward (sub-pixel
upsample instances, split input packing), the uint8 pipeline with its CUDA graph, the fused post-forward kernel and one training
step in the tensor-core mode (dconv / gconv GEMM paths, multi-tensor Adam)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import healthivert_gan_b200 as hv
from healthivert_gan_b200.pix2pix_model import Pix2PixModel
from oracle import synth

torch.cuda.set_device(0)
g = hv.Generator({"input_dim": 1, "ngf": 16}, True)
g.load_state_dict(synth.synthetic_generator_state_dict())
g = g.cuda().eval()
g.precision = "bf16"
x, mask, cam, ratio = (t.cuda() for t in synth.synthetic_slices(2, seed=1))
with torch.no_grad():
    out = g(x, mask, cam, ratio)
torch.cuda.synchronize()
print("bf16 forward ok", float(out[3].abs().mean()))
rng = np.random.Generator(np.random.PCG64(0))
ct = rng.integers(0, 256, size=(2, 256, 256), dtype=np.uint8)
r = g.forward_u8(ct, ct[::-1].copy(), np.array([[100, 141], [90, 131]], np.int32), np.array([0.1, 0.7], np.float32))
print("uint8 pipeline ok", int(r[0].sum()), r[3], r[4])
if "--no-train" not in sys.argv:
    opt = synth.train_options(gpu_ids=[0], precision="bf16")
    m = Pix2PixModel(opt)
    m.setup(opt)
    m.netG.load_state_dict(synth.synthetic_generator_state_dict())
    m.train()
    m.set_input(synth.synthetic_train_batch(n=1, seed=7))
    m.optimize_parameters()
    torch.cuda.synchronize()
    print("bf16 training step ok", {k: round(v, 4) for k, v in m.get_current_losses().items()})
