"""Config-4 measurement: pix2pix training step, batch 16 (2 samples per rank under torchrun), fp32 kernels.
usage: python tools/bench_train.py [--batch 16] [--steps 5] [--norm batch|instance|none] [--gan-mode vanilla|lsgan|wgangp]
                                   [--netD basic|n_layers|pixel] [--n-layers-d 3]
       |   torchrun --nproc-per-node N tools/bench_train.py"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist

from healthivert_gan_b200 import _lib, sharding
from healthivert_gan_b200.pix2pix_model import Pix2PixModel
from oracle import synth


def discriminator_state_dict(seed, norm):
    """synthetic_discriminator_state_dict in the layout of define_D(norm=...): 'instance' drops the BatchNorm entries and gives convs
    2-4 a zero bias, 'none' drops the BatchNorm entries."""
    sd = synth.synthetic_discriminator_state_dict(seed=seed)
    if norm == "batch":
        return sd
    out = {k: v for k, v in sd.items() if k.split(".")[1] in ("0", "2", "5", "8", "11")}
    if norm == "instance":
        for i in (2, 5, 8):
            out[f"model.{i}.bias"] = torch.zeros(out[f"model.{i}.weight"].shape[0])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16, help="global batch")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16"], help="bf16: tensor-core training mode (D convs + G conv backward)")
    ap.add_argument("--d-precision", default=None, choices=["fp32", "bf16"], help="override for the PatchGAN convolutions alone")
    ap.add_argument("--device-batch", action="store_true", help="keep the batch on the device (no per-step H2D copy, no host sync): shows whether the host or the device bounds a step")
    ap.add_argument("--norm", default="batch", choices=["batch", "instance", "none"], help="the discriminators' normalisation (opt.norm)")
    ap.add_argument("--g-forward", default=None, choices=["fp32", "bf16"], help="override for the generator's conv forward alone")
    ap.add_argument("--gan-mode", default="vanilla", choices=["vanilla", "lsgan", "wgangp"], help="the GAN objective (opt.gan_mode)")
    ap.add_argument("--netD", default="basic", choices=["basic", "n_layers", "pixel"], help="the discriminator (opt.netD)")
    ap.add_argument("--n-layers-d", type=int, default=3, help="PatchGAN depth of --netD n_layers (opt.n_layers_D)")
    args = ap.parse_args()
    rank, world, local = sharding.world_from_env()
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    opt = synth.train_options(gpu_ids=[local], precision=args.precision, norm=args.norm, gan_mode=args.gan_mode, netD=args.netD,
                              n_layers_D=args.n_layers_d, **({'d_precision': args.d_precision} if args.d_precision else {}),
                              **({'g_forward_precision': args.g_forward} if args.g_forward else {}))
    m = Pix2PixModel(opt)
    m.setup(opt)
    m.netG.load_state_dict(synth.synthetic_generator_state_dict())
    if args.netD == "basic":       # the other discriminators keep define_D's seeded initialisation
        for k, net in enumerate((m.netD_1, m.netD_2, m.netD_3), start=1):
            net.load_state_dict(discriminator_state_dict(k, args.norm))
    m.train()
    m.world_size = world
    full = synth.synthetic_train_batch(n=args.batch, seed=7)
    idx = list(sharding.shard_contiguous(args.batch, rank, world))
    batch = {k: (v[idx[0]:idx[-1] + 1] if torch.is_tensor(v) else v[idx[0]:idx[-1] + 1]) for k, v in full.items()}
    if args.device_batch:
        batch = {k: (v.cuda() if torch.is_tensor(v) and k != "h2" else v) for k, v in batch.items()}
    for _ in range(args.warmup):
        m.set_input(batch)
        m.optimize_parameters()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        m.set_input(batch)
        m.optimize_parameters()
    e1.record()
    host = (time.perf_counter() - t0) / args.steps * 1e3     # time to ENQUEUE a step (the host runs ahead of the device unless it is the bound)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    wall = (time.perf_counter() - t0) / args.steps * 1e3
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    if rank == 0:
        print(json.dumps({"workload": "pix2pix optimize_parameters (BASELINE.json configs[3])", "global_batch": args.batch, "n_gpus": world,
                          "ms_per_step_device": ms, "ms_per_step_wall": wall, "ms_per_step_host_enqueue": host, "samples_per_s": args.batch / ms * 1e3,
                          "launches_per_step": (_lib.launch_count() - l0) / args.steps, "precision": args.precision, "d_precision": args.d_precision or args.precision, "norm": args.norm,
                          "gan_mode": args.gan_mode, "netD": args.netD, "n_layers_D": args.n_layers_d,
                          "losses": {k: round(v, 4) for k, v in m.get_current_losses().items()}}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
