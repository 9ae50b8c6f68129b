#!/usr/bin/env python
"""Headline benchmark: LaVie base T2V denoise steps/s at 320x512x16 with classifier-free guidance (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # this repo's B200 path (one process per GPU; N > 1 under
                                                             # torch.distributed.run: CFG halves x frame shards)
    python bench.py --impl reference --steps K --warmup W    # the UNMODIFIED reference forward on the host CPU cores
    python bench.py --workload interp|vsr|encoders           # BASELINE configs 4 / 5 and the once-per-video stages
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/*.npy

A "step" is one CFG denoising step of VideoGenPipeline's loop (pipeline_videogen.py:664-689): the UNet forward on
[2,4,16,40,64] (uncond + cond), the guidance combine and the DDIM update.  Weights are deterministic random-init of
the architecture (no checkpoint offline), inputs synthetic.

Prints ONE JSON line (rank 0).  `value` = steps/s with the latents resident in HBM; `e2e` = the same step driven
through the public module API from pinned HOST buffers (H2D of latents + text, D2H of the new latents, every step);
`roofline` = the dominant kernel (tcgen05 implicit-GEMM conv / GEMM) timed per launch with CUDA events;
`cpu_baseline` = the unmodified reference model (baseline/_ref, copied there by __graft_entry__.build(); the CPU oracle
port when it is absent) timed on this box's cores; `parity` = the product's forward at the headline shape against that
CPU forward (N = 1), or every rank's partitioned forward against the un-sharded one on its own GPU (N > 1).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOAD = "base T2V 320x512x16 (latent 4x16x40x64), CFG batch 2, 77 text tokens, DDIM"
FRAMES, LAT_H, LAT_W = 16, 40, 64
# SURVEY.md 8d: algorithmic FLOPs of one CFG step (conv 8006.5 + linears/1x1 6595.6 + attention cores 1617.2 GFLOP)
STEP_GFLOP = 16219.4


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"bf16_tflops": p.get("bf16_tflops_sustained", p.get("bf16_tflops")), "hbm_gbs": p.get("hbm_gbs"),
                "source": "MEASURED_PEAKS.json (sustained bf16; kernel timed inside a long step)"}
    return {"bf16_tflops": 1590.0, "hbm_gbs": 6650.0, "source": "fallback of B200_PROFILING.md"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.lines, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        return False

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm)}


DUMP_BYTES = 64_000_000


def dump_outputs(directory, arrays):
    """--dump-outputs: write what the timed path returned in its last step, one float32 DIR/<name>.npy per array.  The
    inputs are seeded, so two builds run with the same arguments can be compared output for output.  The dump stays
    within 64 MB: an array larger than its share is written as <name>_sample.npy, a fixed seeded choice of its elements
    (the same positions for the same shape)."""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    share = (DUMP_BYTES // len(arrays) - 256) // 4          # elements per array; 256 bytes for the .npy header
    for name, t in arrays.items():
        a = t.detach().cpu().float()
        if a.numel() > share:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:share].sort().values
            a, name = a.reshape(-1)[idx], f"{name}_sample"
        np.save(os.path.join(directory, f"{name}.npy"), a.numpy())


# ----------------------------------------------------------------------------------------------- CPU legs
CONFIG = {"workload": WORKLOAD, "weights": "random-init (seeded), 909.1 M params", "timesteps": "DDIM, 50 steps"}


def reference_forward():
    """The reference's own forward on the host CPU: the UNMODIFIED reference model from baseline/_ref (copied there by
    __graft_entry__.build(), kind "reference"), else the CPU oracle port (kind "port").  Returns (fn, kind)."""
    from lavie_b200.synthetic import synthetic_state_dict
    from oracle import reference_loader as R
    sd = synthetic_state_dict(seed=0)
    if R.available("base"):
        ref = R.load_reference_unet("base", sd)

        def fwd(sample, t, text):
            with torch.no_grad():
                return ref(sample, t, encoder_hidden_states=text).sample
        return fwd, "reference"
    from oracle import unet3d_oracle as O
    return (lambda sample, t, text: O.unet_forward(sd, sample, t, text)), "port"


def timed_forward(fwd, frames: int):
    """One CPU forward on the bench inputs restricted to the first `frames` frames (all other dimensions full size)."""
    from lavie_b200.synthetic import synthetic_inputs
    sample, t, text = synthetic_inputs(2, FRAMES, LAT_H, LAT_W, seed=0)
    sample = sample[:, :, :frames].contiguous()
    t0 = time.time()
    out = fwd(sample, t, text)
    return time.time() - t0, out


def cpu_baseline():
    """N=1 line: ONE full-size forward ([2,4,16,40,64], fp32) of the reference on all host cores.  Its output is kept:
    it is the parity reference of the product's forward on the same inputs (`parity` key of the line)."""
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    fwd, kind = reference_forward()
    timed_forward(fwd, 1)                                  # warm-up (allocator, oneDNN primitive caches)
    dt, out = timed_forward(fwd, FRAMES)
    what = "unmodified reference UNet3DConditionModel (baseline/_ref)" if kind == "reference" else "CPU oracle port"
    return {"value": 1.0 / dt, "unit": "steps/s", "cores": threads, "kind": kind,
            "sample": f"1 full forward of the {what}, fp32, [2,4,{FRAMES},{LAT_H},{LAT_W}] = {dt:.2f} s "
                      f"(guidance combine + DDIM update are negligible on CPU)", "seconds_per_step": dt}, out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation on all host cores.  Every bench step is a BOUNDED SAMPLE
    of the workload: the reference forward on the first f of the 16 frames (everything else at full size; conv / spatial
    attention / FF work is per frame), f chosen so that the K + W steps finish in ~2.5 minutes.  `ms_per_step` is the
    measured wall time of one such bench step; `value` = (f / 16 of a denoise step) / that time."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    fwd, kind = reference_forward()
    total = max(1, args.steps + args.warmup)
    timed_forward(fwd, 1)
    t1, _ = timed_forward(fwd, 1)
    frames = 1
    for f in (2, 4, 8, 16):
        if t1 * f * total <= 150.0:
            frames = f
    for _ in range(args.warmup):
        timed_forward(fwd, frames)
    times = []
    for _ in range(args.steps):
        dt, out = timed_forward(fwd, frames)
        times.append(dt)
    step_s = sum(times) / len(times)
    frac = frames / FRAMES
    value = frac / step_s
    sample = (f"per bench step: one forward of the {'unmodified reference (baseline/_ref)' if kind == 'reference' else 'CPU oracle port'}"
              f" on {frames} of {FRAMES} frames = {frac:g} of a denoise step, measured {step_s:.2f} s")
    line = {"impl": "reference", "metric": "denoise steps/s (320x512x16, CFG)", "value": value, "unit": "steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": CONFIG, "setup": {"device": "host CPU", "threads": threads, "sample_fraction": frac},
            "cpu_baseline": {"value": value, "unit": "steps/s", "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"noise_pred": out})
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- B200 path
def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def run_b200(args):
    import torch.distributed as dist
    from lavie_b200 import UNet3DConditionModel, ops
    from lavie_b200.pipeline import CFGDenoiser, DDIMSchedule
    from lavie_b200.synthetic import synthetic_inputs, synthetic_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with torch.distributed.run (one process per GPU), see module docstring")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    unet = UNet3DConditionModel()
    unet.load_state_dict(synthetic_state_dict(seed=0), strict=True)
    unet = unet.to(dev).eval()
    sample, t_check, text = synthetic_inputs(2, FRAMES, LAT_H, LAT_W, seed=0)
    latents0 = sample[:1].contiguous()                 # [1,4,16,40,64]
    sched = DDIMSchedule(50)
    timesteps = sched.timesteps

    # ---- parity reference of this run: the un-sharded forward of the bench inputs on THIS GPU (outside any timing) ----
    full_out = unet(sample.to(dev), t_check, encoder_hidden_states=text.to(dev)).sample
    torch.cuda.synchronize()

    # ---- partitioning (SURVEY.md 8e): ONE video, strong scaling ----
    # N = 1: both CFG halves on one GPU.  N >= 2: rank = half * P + shard.  The uncond / cond halves never interact
    # inside the UNet, so they go to the two halves of the ranks; each half shards the 16 frames over P = N/2 GPUs
    # (all-to-all around every temporal attention, all-reduce of the 5-D GroupNorm sums).  The latents stay
    # frame-sharded across steps: after the forward the two ranks holding the same frames exchange their noise
    # predictions (all_gather of 2 x 655/P KB) and each applies the fused guidance + DDIM update to its frames.
    jobs, scaling = 1, "strong"
    parity = None
    if world == 1:
        parallelism = "single"
        pair_group, half, P, shard_idx = None, None, 1, 0
    else:
        if world % 2 or FRAMES % (world // 2):
            raise SystemExit("--gpus must be 1, 2, 4 or 8")
        P = world // 2
        half, shard_idx = rank // P, rank % P
        parallelism = "cfg2" if P == 1 else f"cfg2 x frames{P}"
        frame_group = None
        for hh in range(2):
            g = dist.new_group(list(range(hh * P, hh * P + P)))
            if hh == half:
                frame_group = g
        pair_group = None
        for ss in range(P):
            g = dist.new_group([ss, P + ss])
            if ss == shard_idx:
                pair_group = g
        unet.set_frame_sharding(frame_group)
        fl = FRAMES // P
        latents0 = latents0[:, :, shard_idx * fl:(shard_idx + 1) * fl].contiguous()
        # every rank: its shard of the SAME inputs through the sharded path (CUDA graph + peer-memory exchanges, exactly
        # what is timed below) against the slice of the un-sharded forward computed above
        shard_in = sample[half:half + 1, :, shard_idx * fl:(shard_idx + 1) * fl].contiguous().to(dev)
        shard_out = None
        for _ in range(2):                              # second call = graph replay
            shard_out = unet(shard_in, t_check, encoder_hidden_states=text[half:half + 1].to(dev)).sample
        err = rel_l2(shard_out, full_out[half:half + 1, :, shard_idx * fl:(shard_idx + 1) * fl])
        errs = [None] * world
        dist.all_gather_object(errs, err)
        parity = {"rel_l2": max(errs), "per_rank": [round(e, 6) for e in errs], "tolerance": 2e-2,
                  "vs": "un-sharded forward of the same inputs on the rank's own GPU",
                  "shape": [2, 4, FRAMES, LAT_H, LAT_W]}
        if max(errs) > 2e-2:
            raise SystemExit(f"sharded forward differs from the un-sharded one: worst rel-L2 {max(errs):.3e} > 2e-2")

    lat = latents0.to(dev)
    txt = text.to(dev)
    den = CFGDenoiser(unet, 7.5, sched)
    gather = [torch.empty((1,) + tuple(lat.shape[1:]), dtype=torch.float32, device=dev) for _ in range(2)]

    def one_step(latents, t, text_in=None):
        if world == 1:
            return den.step(latents, t, txt if text_in is None else text_in)
        noise = unet(latents, t, encoder_hidden_states=txt[half:half + 1] if text_in is None else text_in).sample
        dist.all_gather(gather, noise.contiguous(), group=pair_group)
        a_t, a_prev = sched.alphas(t)
        return ops.cfg_ddim_step(gather[0], gather[1], 7.5, a_t, a_prev, latents)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    x = lat
    for i in range(max(args.warmup, 3)):
        x = one_step(x, timesteps[i % len(timesteps)])
    barrier()
    launches0 = ops.LAUNCHES
    graph_launches = unet.launches_per_step() if hasattr(unet, "launches_per_step") else None

    # ---- timed region: K steps, latents resident in HBM ----
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        ev0.record()
        for i in range(args.steps):
            x = one_step(x, timesteps[i % len(timesteps)])
        ev1.record()
        barrier()
    dump = {"latents": x.cpu()} if args.dump_outputs else None
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        tmax = torch.tensor([ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax)
    ms_per_step = ms / args.steps
    value = jobs * 1e3 / ms_per_step
    eager_launches = ops.LAUNCHES - launches0
    per_step = graph_launches if graph_launches is not None else 0
    gpu_launches = eager_launches + (per_step * args.steps if unet.use_cuda_graph else 0)

    # ---- e2e: the same step through the public module API from pinned HOST buffers.  Every step: H2D of the latents
    # and the text embedding, the step, D2H of the new latents; the next step's input IS that host copy, so the host
    # waits for the copy's event (not a device-wide synchronize) before it enqueues the next step. ----
    lat_host = [latents0.clone().pin_memory(), torch.empty_like(latents0).pin_memory()]
    txt_host = (text if world == 1 else text[half:half + 1]).contiguous().pin_memory()
    done = torch.cuda.Event()
    for i in range(2):                                   # warm the pinned-buffer path
        new = one_step(lat_host[0].to(dev, non_blocking=True), timesteps[i], txt_host.to(dev, non_blocking=True))
        lat_host[1].copy_(new, non_blocking=True)
    barrier()
    lat_host[0].copy_(latents0)
    t0 = time.perf_counter()
    for i in range(args.steps):
        src, dst = lat_host[i & 1], lat_host[(i + 1) & 1]
        new = one_step(src.to(dev, non_blocking=True), timesteps[i % len(timesteps)],
                       txt_host.to(dev, non_blocking=True))
        dst.copy_(new, non_blocking=True)
        done.record()
        done.synchronize()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        tmax = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e_s = float(tmax)
    e2e_value = jobs * args.steps / e2e_s
    h2d = lat_host[0].numel() * 4 + txt_host.numel() * 4
    d2h = lat_host[0].numel() * 4

    # ---- roofline of the dominant kernel: per-launch CUDA events over one eager (un-graphed) step ----
    # (every rank runs the eager pass: with frame sharding its collectives need the whole group; rank 0 reports)
    roofline, kernels = None, None
    was = unet.use_cuda_graph
    unet.use_cuda_graph = False
    model_in = torch.cat([lat, lat]) if world == 1 else lat
    text_in = txt if world == 1 else txt[half:half + 1]
    unet(model_in, 500, encoder_hidden_states=text_in)                # eager warm-up
    ops.PROFILE = []
    if world == 1:
        # keep the GPU busy while the host enqueues the eager step, so that the event pairs bracket back-to-back kernel
        # execution and not the ~20 us the host needs per ctypes launch (which would be charged to the small kernels)
        torch.cuda._sleep(150_000_000)
    unet(model_in, 500, encoder_hidden_states=text_in)
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    unet.use_cuda_graph = was
    weight_bytes = sum(v.numel() * v.element_size() for v in unet.packed_tensors())
    if rank == 0:
        peaks = measured_peaks()
        agg = {}
        for name, flops, nbytes, e0, e1, _tag in prof:
            a = agg.setdefault(name, [0, 0.0, 0.0, 0.0])
            a[0] += 1
            a[1] += e0.elapsed_time(e1)
            a[2] += flops
            a[3] += nbytes
        total_ms = sum(a[1] for a in agg.values())
        kernels = {k: {"launches": a[0], "ms": round(a[1], 3), "share": round(a[1] / total_ms, 4),
                       "gflop": round(a[2] / 1e9, 1), "gbytes": round(a[3] / 1e9, 3),
                       "tflops": round(a[2] / (a[1] * 1e-3) / 1e12, 1) if a[2] else None,
                       "gbs": round(a[3] / (a[1] * 1e-3) / 1e9, 1) if a[3] else None}
                   for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1])}
        dom = "gemm_bf16_tcgen05"
        d = agg[dom]
        achieved = d[2] / (d[1] * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            traffic = tj.get("dram_bytes_per_launch")
            traffic_src = "STATIC: " + tj.get("source", "ncu --set full capture committed under profiles/")
        roofline = {"kernel": dom, "bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"],
                    "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"], "traffic": traffic,
                    "traffic_source": traffic_src,
                    "launches_per_step": d[0], "avg_launch_ms": d[1] / d[0],
                    "algorithmic_gflop_per_launch": d[2] / d[0] / 1e9, "share_of_step": d[1] / total_ms,
                    "peak_source": peaks["source"]}

    cpu = None
    used_graph = bool(unet.use_cuda_graph)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu, ref_out = cpu_baseline()
        err = rel_l2(full_out.cpu(), ref_out)
        parity = {"rel_l2": err, "tolerance": 2e-2, "shape": [2, 4, FRAMES, LAT_H, LAT_W],
                  "vs": ("unmodified reference forward, fp32 CPU (baseline/_ref)" if cpu["kind"] == "reference"
                         else "CPU oracle port, fp32")}
        if not err <= 2e-2:
            raise SystemExit(f"parity FAILED at the headline shape: rel-L2 {err:.3e} > 2e-2")
        # the fp32-accumulate check mode (north star: <= 1e-3) on the same inputs, same launch sequence
        del unet
        torch.cuda.empty_cache()
        chk = UNet3DConditionModel(check_mode=True)
        chk.load_state_dict(synthetic_state_dict(seed=0), strict=True)
        chk = chk.to(dev).eval()
        out_chk = chk(sample.to(dev), t_check, encoder_hidden_states=text.to(dev)).sample.cpu()
        err_chk = rel_l2(out_chk, ref_out)
        parity["check_mode"] = {"rel_l2": err_chk, "tolerance": 1e-3,
                                "what": "split-bf16 operands through the same tcgen05 GEMM/conv mainloops, fp32 "
                                        "epilogues / norms / attention (UNet3DConditionModel(check_mode=True))"}
        if not err_chk <= 1e-3:
            raise SystemExit(f"check-mode parity FAILED at the headline shape: rel-L2 {err_chk:.3e} > 1e-3")

    if rank == 0:
        line = {"metric": "denoise steps/s (320x512x16, CFG)", "value": value, "unit": "steps/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic", "config": CONFIG,
                "setup": {"parallelism": parallelism, "independent_videos": jobs, "cuda_graph": used_graph,
                          "l2": "no flush: one step streams 1.8 GB of weights and several GB of activations, "
                                ">> 126 MB L2",
                          "launches_per_step_per_rank": per_step, "weight_bytes_per_rank": weight_bytes},
                "parity": parity,
                "step_tflops": STEP_GFLOP / ms_per_step / 1e3,
                "clocks": clocks.summary(),
                "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "gpu_launches": gpu_launches, "roofline": roofline, "cpu_baseline": cpu, "kernels": kernels}
        if dump is not None:
            dump_outputs(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)        # captured NCCL graphs make process-group teardown hang; nothing left to clean up


# ----------------------------------------------------------------------------------------------- config 4 (N1)
INTERP_WORKLOAD = "interpolation UNet 320x512, 16 -> 61 frames (latent 8x61x40x64), CFG batch 2 (scale 4.0), respaced DDIM"
INTERP_FRAMES = 61


def run_interp(args):
    """BASELINE config 4 (python bench.py --workload interp [--gpus N under torchrun]): a step = forward_with_cfg of the
    interpolation UNet on cat([x_t, key-frame latents], 1) = [2,8,61,40,64] + the DDIM update
    (interpolation/sample.py:138-166).  N >= 2: the cond / uncond halves go to the two halves of the ranks and each half
    shards its 61 frames over P = N/2 GPUs (16/15/15/15 at N = 8): SparseCausal halo exchange, all-to-all around the
    temporal attention and GroupNorm sum exchange over NVLink peer memory; the sharded forward of every rank is checked
    against the un-sharded one on its own GPU.  N = 1 parity: a bounded sample (the first 5 frames at full spatial size)
    against the unmodified reference model, whose full-size CPU forward needs a 51 GB score tensor (SURVEY 6)."""
    import torch.distributed as dist
    from lavie_b200 import UNet3DConditionModel, ops
    from lavie_b200.config import INTERP_CONFIG
    from lavie_b200.pipeline import InterpolationSampler
    from lavie_b200.synthetic import synthetic_state_dict
    from oracle import reference_loader as R
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sd = synthetic_state_dict(INTERP_CONFIG, seed=0)
    unet = UNet3DConditionModel(INTERP_CONFIG)
    unet.load_state_dict(sd, strict=True)
    unet = unet.to(dev).eval()
    g = torch.Generator().manual_seed(4)
    z = torch.randn(1, 4, INTERP_FRAMES, LAT_H, LAT_W, generator=g)
    cond = torch.randn(1, 4, INTERP_FRAMES, LAT_H, LAT_W, generator=g)
    text = torch.randn(2, 77, 768, generator=g)                    # [prompt, negative prompt]
    sampler = InterpolationSampler(unet, 4.0, 50)
    ts = sampler.timesteps[::-1]
    parity = None

    if world == 1:
        parallelism = "single"
        z2, c2 = torch.cat([z, z]), torch.cat([cond, cond])
        x, cnd, txt = z2.to(dev), c2.to(dev), text.to(dev)

        def one_step(x, cnd, txt, i):
            gd = unet.forward_with_cfg(torch.cat([x, cnd], dim=1), ts[i % 50], encoder_hidden_states=txt, cfg_scale=4.0)
            a, b = sampler.coefficients(49 - (i % 50))
            return ops.cfg_linear_step(gd, gd, 0.0, a, b, x)
        host_in = [z2, c2, text]
    else:
        if world % 2 or (LAT_H * LAT_W) % (world // 2):
            raise SystemExit("--gpus must be 1, 2, 4 or 8")
        P = world // 2
        half, shard_idx = rank // P, rank % P
        counts = [INTERP_FRAMES // P + (1 if r < INTERP_FRAMES % P else 0) for r in range(P)]
        off = sum(counts[:shard_idx])
        parallelism = "cfg2" if P == 1 else f"cfg2 x frames{P} ({'/'.join(map(str, counts))})"
        frame_group = pair_group = None
        for hh in range(2):
            gg = dist.new_group(list(range(hh * P, hh * P + P)))
            if hh == half:
                frame_group = gg
        for ss in range(P):
            gg = dist.new_group([ss, P + ss])
            if ss == shard_idx:
                pair_group = gg
        my_text = text[half:half + 1].to(dev)                       # half 0 = cond prompt, half 1 = negative prompt
        full_in = torch.cat([z, cond], dim=1).to(dev)
        full_out = unet(full_in, 500, encoder_hidden_states=my_text).sample
        unet.set_frame_sharding(frame_group, frame_counts=counts if P > 1 else None)
        sl = slice(off, off + counts[shard_idx])
        shard_out = None
        for _ in range(2):
            shard_out = unet(full_in[:, :, sl].contiguous(), 500, encoder_hidden_states=my_text).sample
        err = rel_l2(shard_out, full_out[:, :, sl])
        errs = [None] * world
        dist.all_gather_object(errs, err)
        parity = {"rel_l2": max(errs), "per_rank": [round(e, 6) for e in errs], "tolerance": 2e-2,
                  "vs": "un-sharded forward of the same inputs on the rank's own GPU",
                  "shape": [1, 8, INTERP_FRAMES, LAT_H, LAT_W]}
        if max(errs) > 2e-2:
            raise SystemExit(f"sharded interpolation forward differs from the un-sharded one: {max(errs):.3e}")
        del full_out, full_in
        x, cnd, txt = z[:, :, sl].contiguous().to(dev), cond[:, :, sl].contiguous().to(dev), my_text
        gather = [torch.empty_like(x) for _ in range(2)]

        def one_step(x, cnd, txt, i):
            eps = unet(torch.cat([x, cnd], dim=1), ts[i % 50], encoder_hidden_states=txt).sample
            dist.all_gather(gather, eps.contiguous(), group=pair_group)      # [cond eps, uncond eps] of my frames
            a, b = sampler.coefficients(49 - (i % 50))
            return ops.cfg_linear_step(gather[1], gather[0], 4.0, a, b, x)
        host_in = [z[:, :, sl].contiguous(), cond[:, :, sl].contiguous(), text[half:half + 1].contiguous()]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        x = one_step(x, cnd, txt, i)
    barrier()
    per_step = unet.launches_per_step() + 2
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        ev0.record()
        for i in range(args.steps):
            x = one_step(x, cnd, txt, i)
        ev1.record()
        barrier()
    dump = {"latents": x.cpu()} if args.dump_outputs else None
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        tmax = torch.tensor([ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax)
    ms_per_step = ms / args.steps
    # e2e: host buffers in, new latents out, every step
    xh = [host_in[0].clone().pin_memory(), torch.empty_like(host_in[0]).pin_memory()]
    ch, th = host_in[1].clone().pin_memory(), host_in[2].clone().pin_memory()
    done = torch.cuda.Event()
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        new = one_step(xh[i & 1].to(dev, non_blocking=True), ch.to(dev, non_blocking=True),
                       th.to(dev, non_blocking=True), i)
        xh[(i + 1) & 1].copy_(new, non_blocking=True)
        done.record()
        done.synchronize()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        tmax = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e_s = float(tmax)
    # per-kernel profile of one eager forward (every rank runs it: the sharded exchanges need the whole group)
    unet.use_cuda_graph = False
    m_in = (torch.cat([torch.cat([z, z]), torch.cat([cond, cond])], dim=1) if world == 1 else
            torch.cat([host_in[0], host_in[1]], dim=1)).to(dev)
    unet(m_in, 500, encoder_hidden_states=txt)
    ops.PROFILE = []
    if world == 1:
        torch.cuda._sleep(300_000_000)
    unet(m_in, 500, encoder_hidden_states=txt)
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    unet.use_cuda_graph = True
    agg = {}
    for name, flops, nbytes, e0, e1, _tag in prof:
        a = agg.setdefault(name, [0, 0.0, 0.0, 0.0])
        a[0] += 1; a[1] += e0.elapsed_time(e1); a[2] += flops; a[3] += nbytes
    total_ms = sum(a[1] for a in agg.values())
    kernels = {k: {"launches": a[0], "ms": round(a[1], 3), "share": round(a[1] / total_ms, 4),
                   "gflop": round(a[2] / 1e9, 1), "tflops": round(a[2] / (a[1] * 1e-3) / 1e12, 1) if a[2] else None,
                   "gbs": round(a[3] / (a[1] * 1e-3) / 1e9, 1) if a[3] else None}
               for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1])}
    step_gflop = sum(a[2] for a in agg.values()) / 1e9 * world      # every rank does 1/world of the step
    peaks = measured_peaks()
    d = agg["gemm_bf16_tcgen05"]
    achieved = d[2] / (d[1] * 1e-3) / 1e12
    roofline = {"kernel": "gemm_bf16_tcgen05", "bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"],
                "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"], "traffic": None,
                "launches_per_step": d[0], "share_of_step": d[1] / total_ms, "peak_source": peaks["source"]}
    # N = 1: parity + CPU baseline on a bounded sample: 5 frames, full spatial size
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        f = 5
        threads = os.cpu_count() or 1
        torch.set_num_threads(threads)
        m5 = torch.cat([torch.cat([z, cond], dim=1)[:1, :, :f]] * 2).contiguous()
        if R.available("interpolation"):
            ref = R.load_reference_unet("interp", sd)
            kind = "reference"
            fwd = lambda: ref(m5, 500, encoder_hidden_states=text).sample
        else:
            from oracle import interp_oracle as IO
            kind = "port"
            fwd = lambda: IO.unet_forward(sd, m5, 500, text)
        with torch.no_grad():
            t0 = time.time()
            ref_out = fwd()
            dt = time.time() - t0
        out5 = unet(m5.to(dev), 500, encoder_hidden_states=txt).sample.cpu()
        err = rel_l2(out5, ref_out)
        parity = {"rel_l2": err, "tolerance": 2e-2, "shape": [2, 8, f, LAT_H, LAT_W],
                  "vs": f"{'unmodified reference interpolation UNet (baseline/_ref)' if kind == 'reference' else 'CPU oracle port'}, fp32"}
        frac = f / INTERP_FRAMES
        cpu = {"value": frac / dt, "unit": "steps/s", "cores": threads, "kind": kind,
               "sample": f"1 forward on {f} of {INTERP_FRAMES} frames ({frac:.3f} of a step; the full-size CPU forward "
                         f"needs a 51 GB score tensor) = {dt:.2f} s"}
        if not err <= 2e-2:
            raise SystemExit(f"interp parity FAILED: {err:.3e}")
    if rank == 0:
        line = {"metric": "denoise steps/s (interpolation 320x512, 61 frames, CFG)", "value": 1e3 / ms_per_step,
                "unit": "steps/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "bf16", "data": "synthetic",
                "config": {"workload": INTERP_WORKLOAD, "weights": "random-init (seeded), 909.1 M params"},
                "setup": {"parallelism": parallelism, "cuda_graph": True, "launches_per_step_per_rank": per_step},
                "parity": parity, "step_gflop": step_gflop, "step_tflops": step_gflop / ms_per_step,
                "clocks": clocks.summary(),
                "e2e": {"value": args.steps / e2e_s, "unit": "steps/s",
                        "h2d_bytes_per_step": (xh[0].numel() + ch.numel() + th.numel()) * 4,
                        "d2h_bytes_per_step": xh[0].numel() * 4},
                "gpu_launches": per_step * args.steps, "roofline": roofline, "cpu_baseline": cpu, "kernels": kernels}
        if dump is not None:
            dump_outputs(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


# ----------------------------------------------------------------------------------------------- config 5 (N2)
VSR_WORKLOAD = "VSR x4-upscaler UNet3D, 1280x2048x{f} output (latent 4+3 ch x {f} x {h} x {w}), CFG batch 2, 77 text tokens, DDIM"


def run_vsr(args):
    """BASELINE config 5 on ONE GPU (python bench.py --workload vsr): a step = the VSR UNet forward on the CFG batch
    ([2,4,F,320,512] latent + [2,3,F,320,512] noised low-res frames, noise level 50, the reference pipeline's call
    vsr/models/pipeline_stable_diffusion_upscale_video_3d.py:712-727) + guidance + DDIM update.  The reference's sample.py
    feeds 16 frames as two independent 8-frame chunks (vsr/sample.py:100-118); the default here runs the 16 frames as ONE
    video (same FLOPs, temporal attention / frame convs over 16 frames), --vsr-frames 8 runs one chunk.  Frame sharding of this
    model is not built (its frame convolutions need a halo exchange), so N > 1 is refused.  Parity + CPU baseline: a bounded
    sample (2 frames, 80x128 crop = 1/128 of the pixels; the model is convolutional apart from its 40x64-level
    self-attention) against the unmodified reference on the host cores."""
    from lavie_b200 import ops
    from lavie_b200.config import VSR_CONFIG
    from lavie_b200.pipeline import DDIMSchedule
    from lavie_b200.synthetic import synthetic_state_dict
    from lavie_b200.vsr import UNet3DVSRModel
    from oracle import reference_loader as R
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world not in (1, 2, 4, 8) or args.gpus != world or (world > 2 and args.vsr_frames % (world // 2)):
        raise SystemExit("--workload vsr runs on 1, 2, 4 or 8 GPUs (CFG halves x frame shards)")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world >= 2:
        dist.init_process_group("nccl", device_id=dev)
    Fr, H, W = args.vsr_frames, args.vsr_height, args.vsr_width
    # N >= 2: rank = half * P + shard; the CFG halves go to the two halves of the ranks, each half shards the frames over
    # P = N / 2 GPUs (halo exchange of the frame convs, all-reduced GroupNorm sums, all-to-all around temporal attention)
    P = max(world // 2, 1)
    half, shard_idx = (rank // P, rank % P) if world >= 2 else (0, 0)
    frame_group = pair_group = None
    if world >= 2:
        for hh in range(2):
            gg = dist.new_group(list(range(hh * P, hh * P + P)))
            if hh == half:
                frame_group = gg
        for ss in range(P):
            gg = dist.new_group([ss, P + ss])
            if ss == shard_idx:
                pair_group = gg
    fl = Fr // P
    fsl = slice(shard_idx * fl, (shard_idx + 1) * fl)
    sd = synthetic_state_dict(VSR_CONFIG, seed=0)
    unet = UNet3DVSRModel()
    unet.load_state_dict(sd, strict=True)
    unet = unet.to(dev).eval()
    g = torch.Generator().manual_seed(5)
    lat = torch.randn(1, 4, Fr, H, W, generator=g)
    low = torch.randn(2, 3, Fr, H, W, generator=g)
    low[1] = low[0]
    text = torch.randn(2, 77, 1024, generator=g)
    labels = torch.tensor([50, 50])
    sched = DDIMSchedule(50)
    ts = sched.timesteps
    x, lowd, txt = lat.to(dev), low.to(dev), text.to(dev)
    if world >= 2:
        x, lowd = x[:, :, fsl].contiguous(), lowd[:, :, fsl].contiguous()

    gather = [torch.empty((1, 4, fl, H, W), dtype=torch.float32, device=dev) for _ in range(2)]

    def one_step(x, lowd, txt, i):
        t = ts[i % len(ts)]
        a_t, a_prev = sched.alphas(t)
        if world == 1:
            eps = unet(torch.cat([x, x]), t, lowd, encoder_hidden_states=txt, class_labels=labels).sample
            return ops.cfg_ddim_step(eps[:1].contiguous(), eps[1:].contiguous(), 5.0, a_t, a_prev, x)
        # CFG split: the ranks of half h evaluate batch item h (its own prompt) on their frames; the two noise predictions
        # of the same frames are exchanged between the pair
        eps = unet(x, t, lowd[half:half + 1], encoder_hidden_states=txt[half:half + 1], class_labels=labels[half:half + 1]).sample
        dist.all_gather(gather, eps.contiguous(), group=pair_group)
        return ops.cfg_ddim_step(gather[0], gather[1], 5.0, a_t, a_prev, x)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    parity2 = None
    if world >= 2:
        # every rank: its (half, frame shard) through the partitioned path against the un-sharded batch-1 forward of the
        # same half on its own GPU (outside any timing)
        xf, lf = lat.to(dev), low.to(dev)
        full = unet(xf, 500, lf[half:half + 1], encoder_hidden_states=txt[half:half + 1], class_labels=labels[half:half + 1]).sample
        unet._graphs.clear()
        if P > 1:
            unet.set_frame_sharding(frame_group)
        mine = unet(x, 500, lowd[half:half + 1], encoder_hidden_states=txt[half:half + 1], class_labels=labels[half:half + 1]).sample
        err = rel_l2(mine, full[:, :, fsl])
        errs = [None] * world
        dist.all_gather_object(errs, err)
        parity2 = {"rel_l2": max(errs), "per_rank": [round(e, 6) for e in errs], "tolerance": 2e-2,
                   "vs": "un-sharded batch-1 forward of the same CFG half on the rank's own GPU", "shape": [1, 7, Fr, H, W]}
        del full, mine, xf, lf
        torch.cuda.empty_cache()
    for i in range(max(args.warmup, 3)):
        x = one_step(x, lowd, txt, i)
    barrier()
    if P > 1:                                    # sharded steps run eagerly: count the C-ABI calls of one step
        l0 = ops.LAUNCHES
        x = one_step(x, lowd, txt, 0)
        per_step = ops.LAUNCHES - l0
        barrier()
    else:
        per_step = unet.launches_per_step() + 1
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        ev0.record()
        for i in range(args.steps):
            x = one_step(x, lowd, txt, i)
        ev1.record()
        barrier()
    dump = {"latents": x.cpu()} if args.dump_outputs else None
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        tmax = torch.tensor([ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax)
    ms_per_step = ms / args.steps
    peak_mem = torch.cuda.max_memory_allocated() / 2 ** 30
    # e2e: latents + low-res frames + text from pinned host buffers every step, new latents back
    lat_s, low_s = (lat, low) if world == 1 else (lat[:, :, fsl].contiguous(), low[:, :, fsl].contiguous())
    xh = [lat_s.clone().pin_memory(), torch.empty_like(lat_s).pin_memory()]
    lh, th = low_s.clone().pin_memory(), text.clone().pin_memory()
    done = torch.cuda.Event()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(args.steps):
        new = one_step(xh[i & 1].to(dev, non_blocking=True), lh.to(dev, non_blocking=True),
                       th.to(dev, non_blocking=True), i)
        xh[(i + 1) & 1].copy_(new, non_blocking=True)
        done.record()
        done.synchronize()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        tmax = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e_s = float(tmax)
    # per-kernel CUDA-event profile of one eager forward
    unet.use_cuda_graph = False
    if world == 1:
        m_in, l_in, t_in, c_in = torch.cat([x, x]), lowd, txt, labels
    else:
        m_in, l_in, t_in, c_in = x, lowd[half:half + 1], txt[half:half + 1], labels[half:half + 1]
    unet(m_in, 500, l_in, encoder_hidden_states=t_in, class_labels=c_in)
    ops.PROFILE = []
    torch.cuda._sleep(300_000_000)
    unet(m_in, 500, l_in, encoder_hidden_states=t_in, class_labels=c_in)
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    unet.use_cuda_graph = True
    agg = {}
    for name, flops, nbytes, e0, e1, _tag in prof:
        a = agg.setdefault(name, [0, 0.0, 0.0, 0.0])
        a[0] += 1; a[1] += e0.elapsed_time(e1); a[2] += flops; a[3] += nbytes
    total_ms = sum(a[1] for a in agg.values())
    kernels = {k: {"launches": a[0], "ms": round(a[1], 3), "share": round(a[1] / total_ms, 4),
                   "gflop": round(a[2] / 1e9, 1), "tflops": round(a[2] / (a[1] * 1e-3) / 1e12, 1) if a[2] else None,
                   "gbs": round(a[3] / (a[1] * 1e-3) / 1e9, 1) if a[3] else None}
               for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1])}
    step_gflop = sum(a[2] for a in agg.values()) / 1e9 * world
    peaks = measured_peaks()
    d = agg["gemm_bf16_tcgen05"]
    achieved = d[2] / (d[1] * 1e-3) / 1e12
    roofline = {"kernel": "gemm_bf16_tcgen05", "bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"],
                "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"], "traffic": None,
                "launches_per_step": d[0], "avg_launch_ms": d[1] / d[0], "share_of_step": d[1] / total_ms,
                "algorithmic_gflop_per_launch": d[2] / d[0] / 1e9, "peak_source": peaks["source"]}
    parity, cpu = parity2, None
    if world > 1 and parity2["rel_l2"] > 2e-2:
        raise SystemExit(f"vsr CFG-split parity FAILED: {parity2['rel_l2']:.3e}")
    if rank != 0:
        torch.cuda.synchronize()
        dist.barrier()
        os._exit(0)
    if world == 1 and not args.no_cpu_baseline:
        f, hh, ww = min(2, Fr), min(80, H), min(128, W)
        threads = os.cpu_count() or 1
        torch.set_num_threads(threads)
        s_lat = torch.cat([lat, lat])[:, :, :f, :hh, :ww].contiguous()
        s_low = low[:, :, :f, :hh, :ww].contiguous()
        if R.available("vsr"):
            ref = R.load_reference_unet("vsr", sd)
            kind = "reference"
            fwd = lambda: ref(s_lat, 500, s_low, encoder_hidden_states=text, class_labels=labels).sample
        else:
            from oracle import vsr_oracle as V
            kind = "port"
            fwd = lambda: V.unet_forward(sd, s_lat, 500, s_low, text, labels)
        with torch.no_grad():
            t0 = time.time()
            ref_out = fwd()
            dt = time.time() - t0
        out_s = unet(s_lat.to(dev), 500, s_low.to(dev), encoder_hidden_states=txt, class_labels=labels).sample.cpu()
        err = rel_l2(out_s, ref_out)
        frac = (f * hh * ww) / (Fr * H * W)
        parity = {"rel_l2": err, "tolerance": 2e-2, "shape": [2, 7, f, hh, ww],
                  "vs": f"{'unmodified reference UNet3DVSRModel (baseline/_ref)' if kind == 'reference' else 'CPU oracle port'}, fp32"}
        cpu = {"value": frac / dt, "unit": "steps/s", "cores": threads, "kind": kind,
               "sample": f"1 forward on {f} frames x {hh}x{ww} of {Fr} x {H}x{W} ({frac:.5f} of a step's pixels) = {dt:.2f} s"}
        if not err <= 2e-2:
            raise SystemExit(f"vsr parity FAILED: {err:.3e}")
    line = {"metric": "denoise steps/s (VSR 320x512 latent, CFG)", "value": 1e3 / ms_per_step, "unit": "steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": VSR_WORKLOAD.format(f=Fr, h=H, w=W), "weights": "random-init (seeded), 691.0 M params"},
            "setup": {"parallelism": "single" if world == 1 else ("cfg2" if P == 1 else f"cfg2 x frames{P}"),
                      "cuda_graph": P == 1,
                      "launches_per_step_per_rank": per_step,
                      "peak_mem_gb": round(peak_mem, 1)},
            "parity": parity, "step_gflop": step_gflop, "step_tflops": step_gflop / ms_per_step,
            "clocks": clocks.summary(),
            "e2e": {"value": args.steps / e2e_s, "unit": "steps/s",
                    "h2d_bytes_per_step": (xh[0].numel() + lh.numel() + th.numel()) * 4,
                    "d2h_bytes_per_step": xh[0].numel() * 4},
            "gpu_launches": per_step * args.steps, "roofline": roofline, "cpu_baseline": cpu, "kernels": kernels}
    if dump is not None:
        dump_outputs(args.dump_outputs, dump)
    print(json.dumps(line), flush=True)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


# ----------------------------------------------------------------------------------------------- N4: encoders
def run_encoders(args):
    """SURVEY 8f row N4 (python bench.py --workload encoders): the two once-per-video stages around the denoiser on ONE
    GPU.  A step = decode_latents of one 16-frame video (latents [1,4,16,40,64] -> uint8 [1,16,320,512,3],
    pipeline_videogen.py:422-429) + the text encoding of its [negative, positive] prompt pair (CLIP ViT-L/14 text tower,
    [2,77] ids, pipeline_videogen.py:337-348, 395-406).  value = videos/s with the latents resident; e2e = latents and ids
    from pinned host buffers, uint8 frames and embeddings back on the host.  CPU baseline: the oracle ports on a bounded
    sample (2 frames for the VAE).  The VAE oracle is parity-unpinned (no diffusers offline), the CLIP oracle is pinned to
    transformers."""
    from lavie_b200 import ops
    from lavie_b200.clip import SD14_TEXT, CLIPTextEncoder, clip_synthetic_state_dict
    from lavie_b200.vae import VAEDecoder, vae_synthetic_state_dict
    if int(os.environ.get("WORLD_SIZE", "1")) != 1 or args.gpus != 1:
        raise SystemExit("--workload encoders runs on one GPU (replicas only: nothing to shard in a once-per-video stage)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    vsd, csd = vae_synthetic_state_dict(0), clip_synthetic_state_dict(SD14_TEXT, 0)
    vae = VAEDecoder(); vae.load_state_dict(vsd, strict=True); vae = vae.to(dev).eval()
    clip = CLIPTextEncoder(); clip.load_state_dict(csd, strict=True); clip = clip.to(dev).eval()
    g = torch.Generator().manual_seed(6)
    lat = 0.18215 * torch.randn(1, 4, FRAMES, LAT_H, LAT_W, generator=g)
    ids = torch.randint(0, 49408, (2, 77), generator=g)
    latd, idsd = lat.to(dev), ids.to(dev)

    def one_step(l, i):
        z = l.permute(0, 2, 1, 3, 4).reshape(FRAMES, 4, LAT_H, LAT_W)
        return vae.decode(z, scale=1.0 / 0.18215, as_uint8=True), clip(i)[0]

    for _ in range(max(args.warmup, 3)):
        one_step(latd, idsd)
    torch.cuda.synchronize()
    l0 = ops.LAUNCHES
    one_step(latd, idsd)
    per_step = ops.LAUNCHES - l0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(0) as clocks:
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.steps):
            video, emb = one_step(latd, idsd)
        ev1.record()
        torch.cuda.synchronize()
    dump = {"video": video.cpu(), "text_embedding": emb.cpu()} if args.dump_outputs else None
    ms_per_step = ev0.elapsed_time(ev1) / args.steps
    lh, ih = lat.clone().pin_memory(), ids.clone().pin_memory()
    vid_h = torch.empty((FRAMES, 8 * LAT_H, 8 * LAT_W, 3), dtype=torch.uint8).pin_memory()
    emb_h = torch.empty((2, 77, 768), dtype=torch.float32).pin_memory()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, e = one_step(lh.to(dev, non_blocking=True), ih.to(dev, non_blocking=True))
        vid_h.copy_(v, non_blocking=True)
        emb_h.copy_(e, non_blocking=True)
        torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    ops.PROFILE = []
    torch.cuda._sleep(100_000_000)
    one_step(latd, idsd)
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    agg = {}
    for name, flops, nbytes, e0, e1, _tag in prof:
        a = agg.setdefault(name, [0, 0.0, 0.0, 0.0])
        a[0] += 1; a[1] += e0.elapsed_time(e1); a[2] += flops; a[3] += nbytes
    total_ms = sum(a[1] for a in agg.values())
    kernels = {k: {"launches": a[0], "ms": round(a[1], 3), "share": round(a[1] / total_ms, 4),
                   "gflop": round(a[2] / 1e9, 1), "tflops": round(a[2] / (a[1] * 1e-3) / 1e12, 1) if a[2] else None,
                   "gbs": round(a[3] / (a[1] * 1e-3) / 1e9, 1) if a[3] else None}
               for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1])}
    peaks = measured_peaks()
    d = agg["gemm_bf16_tcgen05"]
    achieved = d[2] / (d[1] * 1e-3) / 1e12
    roofline = {"kernel": "gemm_bf16_tcgen05", "bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"],
                "unit": "TFLOP/s", "frac": achieved / peaks["bf16_tflops"], "traffic": None, "launches_per_step": d[0],
                "avg_launch_ms": d[1] / d[0], "share_of_step": d[1] / total_ms,
                "algorithmic_gflop_per_launch": d[2] / d[0] / 1e9, "peak_source": peaks["source"]}
    parity, cpu = None, None
    if not args.no_cpu_baseline:
        from oracle import clip_oracle as CO, vae_oracle as VO
        threads = os.cpu_count() or 1
        torch.set_num_threads(threads)
        f = 2
        t0 = time.time()
        ref_img = VO.decode(vsd, (lat / 0.18215)[0, :, :f].permute(1, 0, 2, 3).contiguous())
        ref_emb = CO.clip_text_forward(csd, ids, 12)
        dt = time.time() - t0
        z = (latd / 0.18215)[0, :, :f].permute(1, 0, 2, 3).contiguous()
        err_v = rel_l2(vae.decode(z).sample.cpu(), ref_img)
        err_c = rel_l2(clip(idsd)[0].cpu(), ref_emb)
        parity = {"vae_rel_l2": err_v, "vae_tolerance": 4e-2, "clip_rel_l2": err_c, "clip_tolerance": 2e-2,
                  "vs": "CPU oracle ports, fp32 (VAE: restatement of the diffusers decoder, parity unpinned; CLIP: pinned "
                        "to transformers.CLIPTextModel)", "shape": [f, 4, LAT_H, LAT_W]}
        cpu = {"value": (f / FRAMES) / dt, "unit": "videos/s", "cores": threads, "kind": "port",
               "sample": f"VAE decode of {f} of {FRAMES} frames + the full 2-prompt text encoding = {dt:.2f} s"}
        if not (err_v <= 4e-2 and err_c <= 2e-2):
            raise SystemExit(f"encoder parity FAILED: vae {err_v:.3e}, clip {err_c:.3e}")
    line = {"metric": "videos/s (VAE decode 16 x 320x512 + CLIP encode of the prompt pair)", "value": 1e3 / ms_per_step,
            "unit": "videos/s", "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "decode_latents [1,4,16,40,64] -> uint8 [1,16,320,512,3] + CLIP ViT-L/14 text tower on "
                                   "[2,77] ids", "weights": "random-init (seeded), 49.5 M + 123.1 M params"},
            "setup": {"parallelism": "single", "cuda_graph": False, "launches_per_step_per_rank": per_step},
            "parity": parity, "clocks": clocks.summary(),
            "e2e": {"value": args.steps / e2e_s, "unit": "videos/s", "h2d_bytes_per_step": lh.numel() * 4 + ih.numel() * 8,
                    "d2h_bytes_per_step": vid_h.numel() + emb_h.numel() * 4},
            "gpu_launches": per_step * args.steps, "roofline": roofline, "cpu_baseline": cpu, "kernels": kernels}
    if dump is not None:
        dump_outputs(args.dump_outputs, dump)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="base", choices=["base", "interp", "vsr", "encoders"],
                    help="base = BASELINE config 1-3 (the headline); interp = config 4; vsr = config 5 on one GPU")
    ap.add_argument("--vsr-frames", type=int, default=16)
    ap.add_argument("--vsr-height", type=int, default=320)
    ap.add_argument("--vsr-width", type=int, default=512)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs runs in one process (each rank of a sharded run holds only its frames)")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "interp":
        run_interp(args)
    elif args.workload == "vsr":
        run_vsr(args)
    elif args.workload == "encoders":
        run_encoders(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
