"""PixelDiscriminator (netD='pixel', ndf = 64, batch 16 x 256^2) forward and backward: the fused tensor-core kernels
(train_ops.pixel_d), the layer path (run_blocks: SIMT 1x1 convs + norm kernels) and torch's own module under bf16 autocast, on the same
GPU, for each norm.

CUDA events around each call; a 256 MB buffer is overwritten before every timed call (the input plane and the fused kernels' working set
fit the 126 MB L2).  Medians of --reps calls.  The backward of each implementation is timed after a fresh forward.
GFLOP/s counts the 64 -> 128 product only (2 * 64 * 128 flops per pixel per GEMM: one GEMM per forward pass, three in the backward's
recompute + dh1 + dW2); the layer path and torch are given the same work count.
usage: python tools/bench_pixel_d.py [--reps 30] [--batch 16] [--size 256]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from healthivert_gan_b200 import networks, train_ops as T


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True).stdout
        return dict(zip(q.split(","), [s.strip() for s in out.splitlines()[0].split(",")]))
    except (OSError, IndexError):
        return {"name": torch.cuda.get_device_name()}


def timed(fn, flush, reps, before=None):
    """median milliseconds of fn() over reps calls, L2 overwritten (and before() run, untimed) ahead of each"""
    ts = []
    for _ in range(reps):
        if before is not None:
            before()
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
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=256)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_pixel_d needs a GPU")
    flush = torch.empty(64 << 20, device="cuda", dtype=torch.float32)
    n, s = args.batch, args.size
    pixels = n * s * s
    res = {"gpu": gpu_info(), "batch": n, "size": s, "reps": args.reps, "norms": []}
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(n, 1, s, s, device="cuda", generator=g)
    dy = torch.randn(n, 1, s, s, device="cuda", generator=g) / pixels ** 0.5
    for norm in ("batch", "instance", "none"):
        torch.manual_seed(0)
        net = networks.define_D(1, 64, "pixel", 3, norm, "normal", 0.02, []).cuda().train()
        row = {"norm": norm}
        state = {}

        def hv_fwd(prec):
            def f():
                net.precision = prec
                state["tape"] = T.Tape()
                state["x"] = T.Var(x, requires_grad=True)
                state["out"] = net.run(state["x"], state["tape"])
            return f

        def hv_bwd():
            for p in net.parameters():
                p.grad = None
            state["out"].grad = dy
            state["tape"].backward()

        def torch_fwd():
            xt = x.detach().requires_grad_()
            with torch.autocast("cuda", dtype=torch.bfloat16):
                state["yt"] = net.net(xt)

        def torch_bwd():
            state["yt"].float().backward(dy)

        for name, fwd, bwd in (("fused_bf16", hv_fwd("bf16"), hv_bwd), ("layers_fp32", hv_fwd("fp32"), hv_bwd),
                               ("torch_autocast_bf16", torch_fwd, torch_bwd)):
            for _ in range(3):                       # warm-up (module load, allocator, cudnn algorithm choice)
                fwd(); bwd()
            torch.cuda.synchronize()
            tf = timed(fwd, flush, args.reps)
            tb = timed(bwd, flush, args.reps, before=fwd)
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            fwd(); bwd()
            torch.cuda.synchronize()
            peak = torch.cuda.max_memory_allocated() - base
            row[name] = {"fwd_us": tf * 1e3, "bwd_us": tb * 1e3, "fwd_GFLOPs_64x128": 2 * 64 * 128 * pixels / tf / 1e6,
                         "bwd_GFLOPs_64x128": 3 * 2 * 64 * 128 * pixels / tb / 1e6, "input_GBps_fwd": 8 * pixels / tf / 1e6,
                         "peak_extra_MiB": peak / 2 ** 20}
        res["norms"].append(row)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
