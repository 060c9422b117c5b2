#!/usr/bin/env python
"""Gradient agreement of the tensor-core training modes with the fp32 parity mode (same weights, same batch, one step each):
per-tensor cosine and norm ratio.  usage: python tools/dbg_train_cos.py [n]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from healthivert_gan_b200.pix2pix_model import Pix2PixModel
from oracle import synth

n = int(sys.argv[1]) if len(sys.argv) > 1 else 2


def grads(precision, g_forward):
    opt = synth.train_options(gpu_ids=[0], precision=precision, g_forward_precision=g_forward)
    m = Pix2PixModel(opt)
    m.setup(opt)
    m.netG.load_state_dict(synth.synthetic_generator_state_dict())
    for k, net in enumerate((m.netD_1, m.netD_2, m.netD_3), start=1):
        net.load_state_dict(synth.synthetic_discriminator_state_dict(seed=k))
    m.train()
    m.set_input(synth.synthetic_train_batch(n=n, seed=7))
    m.optimize_parameters()
    torch.cuda.synchronize()
    return {k: p.grad.double().flatten().clone() for k, p in m.netG.named_parameters()}


ref = grads("fp32", "fp32")
for label, args in (("bf16 backward (fp32 forward)", ("bf16", "fp32")), ("bf16 forward + backward", ("bf16", "bf16"))):
    g = grads(*args)
    rows = []
    for k in ref:
        a, b = g[k], ref[k]
        cos = float(a @ b / (a.norm() * b.norm() + 1e-300))
        rows.append((cos, float(a.norm() / (b.norm() + 1e-300)), k))
    rows.sort()
    allg, allr = torch.cat([g[k] for k in ref]), torch.cat([ref[k] for k in ref])
    print(label, ": whole-G cosine", round(float(allg @ allr / (allg.norm() * allr.norm())), 5), "norm ratio", round(float(allg.norm() / allr.norm()), 4))
    print("   lowest cosines:", [(round(c, 3), round(r, 3), k.replace("_generator", "").replace(".conv", "")) for c, r, k in rows[:8]])
