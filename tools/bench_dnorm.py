"""Fused InstanceNorm + LeakyReLU (hv_in_lrelu_fwd / hv_in_lrelu_bwd) at the batch-16 PatchGAN shapes, against torch's
F.instance_norm + F.leaky_relu (forward + autograd backward) on the same GPU.

CUDA events around each kernel call; a 256 MB buffer is overwritten before every timed call, because the three shapes together (82 MB)
would otherwise be read from the 126 MB L2.  GB/s counts 8 B per element forward (read x, write y) and 12 B per element backward
(read x and dy, write dx), for both implementations.
usage: python tools/bench_dnorm.py [--reps 30]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

from healthivert_gan_b200 import train_ops as T

SHAPES = [(16, 128, 64, 64), (16, 256, 32, 32), (16, 512, 31, 31)]


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True).stdout
        return dict(zip(q.split(","), [s.strip() for s in out.splitlines()[0].split(",")]))
    except (OSError, IndexError):
        return {"name": torch.cuda.get_device_name()}


def timed(fn, flush, reps):
    """median milliseconds of fn() over reps calls, L2 overwritten before each"""
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dnorm needs a GPU")
    flush = torch.empty(64 << 20, device="cuda", dtype=torch.float32)
    res = {"gpu": gpu_info(), "shapes": []}
    for shape in SHAPES:
        n, c, h, w = shape
        numel = n * c * h * w
        g = torch.Generator(device="cuda").manual_seed(c)
        x = torch.randn(shape, device="cuda", generator=g)
        dy = torch.randn(shape, device="cuda", generator=g)
        xv = T.Var(x)
        state = {}

        def hv_fwd():
            state["tape"] = T.Tape()
            state["out"] = T.in_lrelu(state["tape"], xv, None, 0.2, 1e-5)

        def hv_bwd():
            xv.grad = None
            state["out"].grad = dy
            state["tape"].backward()

        def torch_fwd():
            xt = x.detach().requires_grad_()
            state["xt"], state["yt"] = xt, F.leaky_relu(F.instance_norm(xt, eps=1e-5), 0.2)

        def torch_bwd():
            state["yt"].backward(dy)

        row = {"shape": list(shape)}
        for name, fwd, bwd in (("hv", hv_fwd, hv_bwd), ("torch", torch_fwd, torch_bwd)):
            for _ in range(3):                       # warm-up (module load, cudnn algorithm choice)
                fwd(); bwd()
            tf = timed(fwd, flush, args.reps)
            tb = []
            for _ in range(args.reps):
                fwd()
                tb.append(timed(bwd, flush, 1))
            tb = sorted(tb)[len(tb) // 2]
            row[name] = {"fwd_us": tf * 1e3, "bwd_us": tb * 1e3, "fwd_GBps": 8 * numel / tf / 1e6, "bwd_GBps": 12 * numel / tb / 1e6}
        hv_fwd(); hv_bwd(); torch_fwd(); torch_bwd()
        torch.cuda.synchronize()
        ref = state["yt"].detach()
        row["max_abs_y_vs_torch"] = float((state["out"].data - ref).abs().max())
        row["rel_dx_vs_torch"] = float((xv.grad - state["xt"].grad).norm() / state["xt"].grad.norm())
        res["shapes"].append(row)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
