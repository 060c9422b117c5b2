#!/usr/bin/env python
"""One golden training step (n = 2) in the tensor-core mode: gradient-norm deviations and gradient direction against the golden
vectors of the unmodified reference.  --g-forward selects the precision of the generator's forward."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from healthivert_gan_b200.pix2pix_model import Pix2PixModel
from oracle import synth

ap = argparse.ArgumentParser()
ap.add_argument("--g-forward", default="bf16")
ap.add_argument("--precision", default="bf16")
args = ap.parse_args()
gold = np.load(os.path.join(os.path.dirname(__file__), "..", "tests", "golden", "train_step_n2.npz"))
PROBES = np.array([0.0, 0.113, 0.271, 0.5, 0.733, 0.999])
if "probes" in gold:
    PROBES = gold["probes"]


def probe(t):
    t = t.detach().double().reshape(-1).cpu()
    return t[torch.from_numpy((PROBES * t.numel()).astype(np.int64))].numpy()


opt = synth.train_options(gpu_ids=[0], precision=args.precision, g_forward_precision=args.g_forward)
m = Pix2PixModel(opt)
m.setup(opt)
m.netG.load_state_dict(synth.synthetic_generator_state_dict())
for k, net in enumerate((m.netD_1, m.netD_2, m.netD_3), start=1):
    net.load_state_dict(synth.synthetic_discriminator_state_dict(seed=k))
m.train()
m.set_input(synth.synthetic_train_batch(n=2, seed=7))
m.optimize_parameters()
torch.cuda.synchronize()
dev = []
for tag, net in (("D_1", m.netD_1), ("G", m.netG)):
    params = dict(net.named_parameters())
    for i, name in enumerate(str(s) for s in gold[f"{tag}_names"]):
        gn, rn = float(params[name].grad.double().norm()), float(gold[f"{tag}_grad_norm"][i])
        dev.append((abs(gn - rn) / (rn + 1e-12), tag, name))
w = sorted([d for d in dev if not d[2].endswith("bias")], reverse=True)
b = sorted([d for d in dev if d[2].endswith("bias")], reverse=True)
print(args, {k: os.environ[k] for k in os.environ if k.startswith("HV_")})
print("  weights worst", [(round(d, 3), n.replace("_generator", "").replace(".conv.weight_orig", "")) for d, _, n in w[:8]], "mean", round(float(np.mean([d[0] for d in w])), 4))
print("  biases  worst", [(round(d, 3), n.replace("_generator", "").replace(".conv.bias", "")) for d, _, n in b[:8]], "mean", round(float(np.mean([d[0] for d in b])), 4))
