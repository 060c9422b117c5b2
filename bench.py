#!/usr/bin/env python
"""bench.py — slices/sec of the two-stage generator forward (256x256), BASELINE.json's metric.

Workload (config.workload): BASELINE.json configs[1] = batch-16 256x256 two-stage generator
inference on one B200 (weights: oracle.synth random-init, spectral norm converged; inputs:
oracle.synth.synthetic_slices).  One "step" = one generator forward over one batch of 16 slices.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--precision fp32|bf16] [--impl reference] [--no-extras]
                  [--dump-outputs DIR]

* value      : slices/s with inputs resident in HBM; every step is timed with its own CUDA-event pair
               on the launching stream and L2 is flushed (256 MiB write) between steps.
* e2e        : the same metric through the public HOST interface (healthivert_gan_b200.SlicePipeline =
               hv_pipeline_* of the C ABI): uint8 CT / CAM planes + mask rows in pinned host memory in,
               uint8 CT / masks + heights out - what the reference's eval driver hands over and keeps
               (eval_3d_sagittal_twostage.py:84-121).  Per step inside the timed region: one H2D copy,
               one CUDA-graph launch of the whole forward, one D2H copy, a ring of 4 slots in flight.
* roofline   : the dominant kernel (the 64->64 3x3 conv family) timed live with CUDA events;
               achieved = algorithmic FLOPs per layer / mean time per layer.
* cpu_baseline : the reference forward on the host cores (rank 0, N=1 only): the UNMODIFIED reference modules
               staged under oracle/_ref by oracle/stage_ref.py (kind "reference"), else the oracle port ("port").
* extra      : (N=1) fp32-mode slices/s, the stock-PyTorch-on-this-GPU baselines (reference modules on cuda,
               TF32 off / on), config 3 (one 256^3 volume, sagittal + coronal + RHLV); (every N) config 4
               (pix2pix training step, global batch 16 sharded over the ranks, NCCL gradient all-reduce) and
               config 5 (volumes sharded over the ranks, no collective).
* --impl reference : the reference's CPU implementation on all host threads, same config / metric.
* --dump-outputs DIR : after the run, the seven outputs Generator.forward returned in the last timed step, as
               DIR/<name>.npy (float32, full size).  Weights and inputs are seeded, so the files of two builds compare
               output for output; with --impl reference they are the reference forward's outputs for rank 0's batch.
Multi-GPU (torchrun): weak scaling, every rank runs its own batch-16 stream of slices, no collective
on the data path; barrier + synchronize around the timed region, max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH = 16
FLOP_PER_SLICE = 17.54e9          # SURVEY.md §8(d): 14.187 (47 convs) + 1.208 + 2.147 (attention) GFLOP
METRIC = "slices/sec two-stage gen fwd (256x256)"
OUTPUT_NAMES = ("coarse_seg", "fine_seg", "x_stage1", "x_stage2", "flow", "pred1_h", "pred2_h")   # Generator.forward's tuple
WORKLOAD = f"batch-{BATCH} 256x256 two-stage generator inference (BASELINE.json configs[1])"


def _config(precision, world):
    """The `config` object both arms print (same keys, same values: the driver compares them)."""
    return {"workload": WORKLOAD, "batch": BATCH, "precision": precision,
            "l2": "flushed (256 MiB write) between steps",
            "timing": "per-step CUDA-event pairs on the launch stream, summed; max over ranks",
            "e2e_timing": "one CUDA-event pair around all steps; uint8 host interface, H2D / graph launch / D2H per step, 4 slots in flight",
            "parallelism": f"slice-sharded x{world}, no collective"}


def _traffic(precision):
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel per launch, from the committed ncu capture."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        with open(path) as fh:
            return json.load(fh).get(precision)
    except (OSError, ValueError):
        return None


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p["bf16_tflops_sustained"], "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (every 100 ms: measured on B200, polling every 20 ms
    takes driver locks often enough to slow the launch thread)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", os.environ.get("HV_CLOCK_MS", "100")], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference legs
def _reference_forward(device):
    """(callable forward(x, mask, cam, ratio), kind): the UNMODIFIED reference Generator staged under oracle/_ref when present
    (oracle/stage_ref.py), else the oracle port.  Inputs / weights are moved to `device`."""
    import torch
    from oracle import stage_ref, synth
    sd = synth.synthetic_generator_state_dict()
    if stage_ref.staged():
        stage_ref.import_reference()
        from models.inpaint_networks import Generator   # the staged reference module
        g = Generator({"input_dim": 1, "ngf": 16}, device.type == "cuda")
        g.load_state_dict(sd)
        g = g.to(device).eval()
        return (lambda *a: g(*a)), "reference"
    from oracle import generator_ref as gr
    sd = {k: v.to(device) for k, v in sd.items()}
    return (lambda *a: gr.generator_forward(sd, *a)), "port"


def _cpu_forward_rate(steps, warmup, batch=BATCH):
    """The reference forward on all host threads: slices/s over `steps` batches."""
    import torch
    from oracle import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    fwd, kind = _reference_forward(torch.device("cpu"))
    x, mask, cam, ratio = synth.synthetic_slices(batch, seed=123)
    with torch.no_grad():
        for _ in range(warmup):
            fwd(x, mask, cam, ratio)
        t0 = time.perf_counter()
        for _ in range(steps):
            out = fwd(x, mask, cam, ratio)
        dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps * 1e3, torch.get_num_threads(), kind, out


def run_reference(args, rank, world):
    if rank != 0:
        return
    # the CPU arm needs ~0.4 s per batch-16 step (each step = the full batch): the requested step count is kept up to 200 (80 s)
    steps = max(1, min(args.steps, 200))
    rate, ms, threads, kind, out = _cpu_forward_rate(steps, args.warmup)
    what = "the unmodified reference modules (oracle/_ref)" if kind == "reference" else "oracle port of the reference"
    sample = f"{steps} steps x batch {BATCH} (each step = one full batch-{BATCH} forward), {what}"
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": "slices/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(args.precision, world),
        "device": "host CPU, fp32",
        "cpu_baseline": {"value": rate, "unit": "slices/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": "slices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, host_outputs(out))


# ------------------------------------------------------------------------------------------------ extras
def _torch_gpu_baselines(dev, steps=10):
    """Stock PyTorch on this GPU: the reference modules (cuDNN / cuBLAS through ATen) on the same batch, TF32 off and on."""
    import torch
    from oracle import synth
    out = {}
    fwd, kind = _reference_forward(dev)
    x, mask, cam, ratio = (t.to(dev) for t in synth.synthetic_slices(BATCH, seed=123))
    for name, tf32 in (("fp32", False), ("tf32_cudnn_benchmark", True)):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.benchmark = tf32       # the reference sets cudnn.benchmark = True (models/base_model.py:37-38)
        with torch.no_grad():
            for _ in range(3):
                fwd(x, mask, cam, ratio)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fwd(x, mask, cam, ratio)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"slices_per_s": BATCH / ms * 1e3, "ms_per_step": ms}
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = False
    out["kind"] = kind
    out["what"] = ("Generator.forward of the unmodified reference modules" if kind == "reference" else "oracle port of the reference forward") + \
        f" on cuda, batch {BATCH}, eager PyTorch (cuDNN / cuBLAS), CUDA events around {steps} forwards"
    return out


def _torch_gpu_train_baseline(dev, steps=3):
    """optimize_parameters of the UNMODIFIED reference Pix2PixModel on this GPU (needs oracle/_ref), batch 16."""
    import contextlib
    import io
    import torch
    from oracle import stage_ref, synth
    if not stage_ref.staged():
        return {"unavailable": "oracle/_ref is not staged"}
    stage_ref.import_reference()
    with contextlib.redirect_stdout(io.StringIO()):
        from models.pix2pix_model import Pix2PixModel as RefModel
        opt = synth.train_options(gpu_ids=[dev.index])
        m = RefModel(opt)
        m.setup(opt)
    m.netG.load_state_dict(synth.synthetic_generator_state_dict())
    batch = synth.synthetic_train_batch(n=BATCH, seed=7)
    out = {}
    for name, tf32 in (("fp32", False), ("tf32_cudnn_benchmark", True)):
        torch.backends.cudnn.allow_tf32 = tf32
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.benchmark = tf32       # the reference sets cudnn.benchmark = True (models/base_model.py:37-38)
        for _ in range(3 if tf32 else 2):
            m.set_input(batch)
            m.optimize_parameters()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            m.set_input(batch)
            m.optimize_parameters()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"ms_per_step": ms, "samples_per_s": BATCH / ms * 1e3}
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = False
    out["ms_per_step"] = out["fp32"]["ms_per_step"]
    out["samples_per_s"] = out["fp32"]["samples_per_s"]
    out["kind"] = "reference"
    out["what"] = (f"unmodified reference Pix2PixModel.optimize_parameters on cuda, batch {BATCH}, eager PyTorch: fp32 (TF32 off; the top-level keys) and "
                   "TF32 + cudnn.benchmark")
    return out


def _train_step_rate(rank, world, local, steps=5, warmup=2, precision="bf16"):
    """BASELINE.json config 4: pix2pix training step, GLOBAL batch 16 sharded over the ranks (2 samples per rank at 8 GPUs),
    gradient all-reduce(mean) over NCCL; device time per step, max over ranks."""
    import torch
    import torch.distributed as dist
    from healthivert_gan_b200 import _lib, sharding
    from healthivert_gan_b200.pix2pix_model import Pix2PixModel
    from oracle import synth
    opt = synth.train_options(gpu_ids=[local], precision=precision)
    m = Pix2PixModel(opt)
    m.setup(opt)
    m.netG.load_state_dict(synth.synthetic_generator_state_dict())
    for k, net in enumerate((m.netD_1, m.netD_2, m.netD_3), start=1):
        net.load_state_dict(synth.synthetic_discriminator_state_dict(seed=k))
    m.train()
    m.world_size = world
    full = synth.synthetic_train_batch(n=BATCH, seed=7)
    idx = sharding.shard_contiguous(BATCH, rank, world)
    batch = {k: v[idx.start:idx.stop] for k, v in full.items()}
    for _ in range(warmup):
        m.set_input(batch)
        m.optimize_parameters()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        m.set_input(batch)
        m.optimize_parameters()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    launches = (_lib.launch_count() - l0) / steps
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    losses = {k: round(v, 4) for k, v in m.get_current_losses().items()}
    del m
    torch.cuda.empty_cache()
    return {"workload": "pix2pix optimize_parameters, global batch 16 (BASELINE.json configs[3])", "n_gpus": world,
            "samples_per_rank": len(idx), "ms_per_step": ms, "steps_per_s": 1e3 / ms, "samples_per_s": BATCH / ms * 1e3,
            "launches_per_step_rank0": launches,
            "dtype": ("tensor-core mode: generator conv forward / data / weight gradients, PatchGAN convs and the attention contractions with bf16 operands on "
                      "tcgen05, fp32 accumulate; output heads, losses, BatchNorm, spectral norm and Adam in fp32"
                      if precision == "bf16" else "fp32 SIMT kernels everywhere (parity mode)"),
            "collective": "4 NCCL all-reduces per step on flat gradient buckets (D_1, D_2, D_3, G)" if world > 1 else "none",
            "losses_rank0": losses}


def _volume_rate(g, rank, world, n_volumes, depth, batch=64):
    """Configs 3 / 5: whole synthetic straightened volumes through the batched three-stage synthesis (sagittal, and coronal when
    the volume is 256 deep), then the RHLV features; volumes sharded round-robin over the ranks, no collective."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from healthivert_gan_b200 import mask_ops, sharding
    from healthivert_gan_b200.volume import VolumeSynthesizer
    from oracle import synth

    def feats(label, fake, axis):
        lab, fk = (label == 20), (fake == 20)      # calculate_heights only asks `!= 0`: no float64 copies of the volumes
        loc = np.where(lab)[axis]
        return mask_ops.calculate_rhlv(fk, lab, int(np.mean(loc)), int((loc.max() - loc.min()) // 5), None, 0.7, axis=axis)

    vs = VolumeSynthesizer(g, batch=batch)
    mine = sharding.shard_round_robin(n_volumes, rank, world)
    vols = {v: synth.synthetic_volume(seed=v, depth=depth) for v in mine}
    coronal = depth == 256          # the generator is a 256x256 network: coronal planes are 256 x depth
    lab, ct, cam = synth.synthetic_volume(seed=999, depth=depth)
    vs.synthesize(ct, lab, cam, 20)
    if coronal:
        vs.synthesize(ct, lab, cam, 20, axis=1)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    dt = t_rhlv = 0.0
    slices = 0
    f0 = None
    for v in mine:
        label, ct, cam = vols[v]
        t0 = time.perf_counter()
        lab_dev = torch.as_tensor(label).cuda() if coronal else label      # two orientations: the label volume crosses PCIe once
        _, lab_s = vs.synthesize(ct, lab_dev, cam, 20, axis=2)
        lab_c = vs.synthesize(ct, lab_dev, cam, 20, axis=1)[1] if coronal else lab_s
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        slices += int(lab_s.any(axis=(0, 1)).sum()) + (int(lab_c.any(axis=(0, 2)).sum()) if coronal else 0)
        f = list(feats(label, lab_s, 2)[:3]) + list(feats(label, lab_c, 1)[:3])
        f0 = f0 or f
        dt += t1 - t0
        t_rhlv += time.perf_counter() - t1
    if world > 1:
        t = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        s = torch.tensor([float(slices)], device="cuda", dtype=torch.float64)
        dist.all_reduce(s)
        dt, slices = float(t), int(s)
    return {"volumes": n_volumes, "shape": [256, 256, depth], "n_gpus": world, "precision": g.precision, "seconds": dt,
            "volumes_per_s": n_volumes / dt, "output_slices": slices, "output_slices_per_s": slices / dt,
            "orientations": "sagittal + coronal" if coronal else "sagittal", "rhlv_tail_seconds_rank0": t_rhlv,
            "timing": "host clock around synthesize() with device synchronisation, incl. H2D of the float64 volumes and D2H of the results; max over ranks",
            "rhlv_2p5d_features_volume0": [round(float(x), 6) for x in (f0 or [])]}


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    import healthivert_gan_b200 as hv
    from healthivert_gan_b200 import _lib
    from healthivert_gan_b200.inpaint_networks import conv2d_fused
    from oracle import synth

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sd = synth.synthetic_generator_state_dict()
    g = hv.Generator({"input_dim": 1, "ngf": 16}, True)
    g.load_state_dict(sd)
    g = g.to(dev).eval()
    g.precision = args.precision
    g.return_flow = True
    x, mask, cam, ratio = (t.to(dev) for t in synth.synthetic_slices(BATCH, seed=123 + rank))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream()
    warm = max(args.warmup, 3)

    def step():
        with torch.no_grad():
            return g(x, mask, cam, ratio)

    for _ in range(warm):
        step()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident throughput
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    wall0 = time.perf_counter()
    launches0 = _lib.launch_count()
    evs = []
    for _ in range(args.steps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = step()
        e1.record(stream)
        evs.append((e0, e1))
    barrier()
    wall = time.perf_counter() - wall0
    launches = _lib.launch_count() - launches0
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    # host copies of the last timed step's outputs, taken before anything else runs on the generator; written at the end
    dumped = host_outputs(out) if args.dump_outputs and rank == 0 else None

    # ---------------- end to end through the public uint8 HOST interface (hv_pipeline_*), 4 slots in flight
    rng = np.random.Generator(np.random.PCG64(1000 + rank))
    depth = 4
    g.per_sample_mask, g.return_flow = True, False        # the eval driver's semantics: every slice has its own mask
    pipe = hv.SlicePipeline(g, batch=BATCH, depth=depth)
    for k in range(depth):                                 # every slot holds its own batch of synthetic uint8 planes
        s = pipe.slot(k)
        s.ct[:] = rng.integers(0, 256, size=s.ct.shape, dtype=np.uint8)
        s.cam[:] = rng.integers(0, 256, size=s.cam.shape, dtype=np.uint8)
        s.rows[:, 0] = 108
        s.rows[:, 1] = 149
        s.ct[:, 108:149] = 0
        s.ratio[:] = rng.random(BATCH).astype(np.float32)
    s_in, s_main, s_out = pipe.stream(0), pipe.stream(1), pipe.stream(2)

    def e2e_loop(nsteps):
        barrier()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(s_main)
        s_in.wait_event(t0)                 # no input copy starts before the clock does
        checksum = 0
        for i in range(nsteps):
            k = i % depth
            if i >= depth:
                pipe.wait(k)                # step i - depth has landed in host memory: the host reads its result ...
                checksum += int(pipe.slot(k).heights[1, 0] > 0)
            pipe.submit(k)                  # ... and the slot's (pinned) inputs go out again
        for k in range(depth):
            pipe.wait(k)
        t1.record(s_out)                    # after the last D2H copy
        t1.synchronize()
        barrier()
        return t0.elapsed_time(t1)

    e2e_loop(warm + depth)
    e2e_launch0 = _lib.launch_count()
    e2e_ms = e2e_loop(args.steps)
    e2e_launches = _lib.launch_count() - e2e_launch0
    clocks = sampler.stop() if rank == 0 else None
    h2d, d2h = pipe.h2d_bytes, pipe.d2h_bytes
    pipe.close()
    g.per_sample_mask, g.return_flow = False, True

    # ---------------- dominant kernel alone (roofline): the 64->64 3x3 conv family on the batch's 64x64 maps
    reps = 20
    kev = []
    if args.precision == "bf16":
        # layers 4..10 = coarse conv5, conv6, conv7..10_atrous, conv11: seven consecutive 64->64 3x3 layers of the plan, each
        # reading its predecessor's output exactly as in the forward (L2 flushed before the chain, not inside it)
        chain = list(range(4, 11))
        launch_k = lambda: g.run_chain(chain[0], len(chain), BATCH)
    else:
        a = torch.randn(BATCH, 64, 64, 64, device=dev)
        w = torch.randn(64, 64, 3, 3, device=dev) * 0.05
        b = torch.zeros(64, device=dev)
        chain = [0]
        launch_k = lambda: conv2d_fused([(a, 0)], w, b, 3, 1, 1, 1, "elu", 64, 64)
    step()
    for _ in range(3):
        launch_k()
    for _ in range(reps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        launch_k()
        e1.record(stream)
        kev.append((e0, e1))
    torch.cuda.synchronize()
    k_ms = sum(x0.elapsed_time(x1) for x0, x1 in kev) / (reps * len(chain))
    k_flop = 2.0 * BATCH * 64 * 64 * 64 * 576

    if world > 1:
        t = torch.tensor([dev_ms, e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, e2e_ms = t.tolist()
        lt = torch.tensor([launches, e2e_launches], device=dev, dtype=torch.int64)
        dist.all_reduce(lt)
        launches, e2e_launches = (int(v) for v in lt.tolist())

    # ---------------- extras: the other BASELINE configs and the honest baselines (same JSON line, `extra`)
    extra = {}
    if not args.no_extras:
        def guarded(name, fn):
            try:
                extra[name] = fn()
            except Exception as e:  # an extra must never cost the headline line
                extra[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
        if world == 1:
            def fp32_mode():
                g.precision = "fp32"
                try:
                    for _ in range(2):
                        step()
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    for _ in range(5):
                        step()
                    e1.record(stream)
                    torch.cuda.synchronize()
                    ms = e0.elapsed_time(e1) / 5
                    return {"slices_per_s": BATCH / ms * 1e3, "ms_per_step": ms, "what": "same workload, --precision fp32 (parity mode, max-abs <= 1e-3)"}
                finally:
                    g.precision = args.precision
            guarded("fp32_mode", fp32_mode)
            guarded("torch_gpu_baseline", lambda: _torch_gpu_baselines(dev))
            guarded("torch_gpu_train_baseline", lambda: _torch_gpu_train_baseline(dev))
            guarded("config3_volume", lambda: _volume_rate(g, rank, world, 1, 256))
        guarded("config4_train", lambda: _train_step_rate(rank, world, local_rank, precision="bf16"))
        guarded("config4_train_fp32_parity_mode", lambda: _train_step_rate(rank, world, local_rank, steps=3, precision="fp32"))
        guarded("config5_volumes", lambda: _volume_rate(g, rank, world, 2 * world, 64))

    if rank == 0:
        peaks = _peaks()
        value = world * BATCH * args.steps / (dev_ms * 1e-3)
        e2e = world * BATCH * args.steps / (e2e_ms * 1e-3)
        achieved = k_flop / (k_ms * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": value, "unit": "slices/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic",
            "config": _config(args.precision, world),
            "e2e": {"value": e2e, "unit": "slices/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / args.steps, "api": "healthivert_gan_b200.SlicePipeline (hv_pipeline_submit / hv_pipeline_wait)",
                    "kernels_per_step": e2e_launches / max(1, args.steps * world)},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "conv 64->64 3x3 (fp32 SIMT parity kernel)"
                         if args.precision == "fp32" else "conv 64->64 3x3 (tcgen05 bf16)",
                         "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                         "frac": achieved / peaks["bf16_tflops"], "traffic": _traffic(args.precision),
                         "algorithmic_flop_per_launch": k_flop, "launch_us": k_ms * 1e3,
                         "launches_timed": f"{reps} x {len(chain)} layers (CUDA events around each chain of consecutive 64->64 layers, L2 flushed before each chain)",
                         "peak_source": peaks["source"] + " burst bf16 (kernel timed alone)",
                         "whole_forward_tensor_frac_sustained": value / world * FLOP_PER_SLICE / (peaks["bf16_tflops_sustained"] * 1e12)},
            "wall_s_timed_region": wall,
            "extra": extra,
        }
        if world == 1 and not args.no_cpu_baseline:
            rate, ms, threads, kind, _ = _cpu_forward_rate(10, 1)
            what = "the unmodified reference modules (oracle/_ref)" if kind == "reference" else "oracle port of the reference forward"
            line["cpu_baseline"] = {"value": rate, "unit": "slices/s", "cores": threads, "kind": kind,
                                    "sample": f"10 steps x batch {BATCH} of the same workload ({ms:.0f} ms/step), {what}"}
        print(json.dumps(line), flush=True)
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


def host_outputs(out):
    """Generator.forward's 7-tuple as named float32 host arrays."""
    return {name: t.float().cpu().numpy() for name, t in zip(OUTPUT_NAMES, out)}


def dump_outputs(directory, arrays):
    """One float32 .npy per output of Generator.forward, full size (about 28 MB for batch 16)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("HV_PRECISION", "bf16"), choices=["fp32", "bf16"],
                    help="bf16 = tcgen05 tensor-core mode (headline); fp32 = SIMT parity mode")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the `extra` sub-records (configs 3/4/5, fp32 mode, torch baselines)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0's batch; with --impl reference, the reference "
                         "forward's) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
