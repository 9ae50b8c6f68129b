"""Times the whole VSR stage: VSRSampler.upscale of a 320x512 video to 1280x2048 (8-frame chunks, 50 v-prediction DDIM
steps per chunk, CFG guidance 5, noise level 50, text [2, 77, 1024]) with synthetic VSR-UNet and x4-VAE weights.

    python tools/bench_vsr_stage.py --frames 16 [--steps 50]
    torchrun --nproc_per_node 8 tools/bench_vsr_stage.py --frames 61 --gpus 8      # chunk-parallel over 8 GPUs

A warm-up call with one step per chunk captures the step graph of every chunk length and warms the decode (and, under
torchrun, the gather); then one timed call.  Reported: ms per CFG step for each chunk length (CUDA events around every
chunk's loop, divided by its steps; the once-per-chunk noising of the low-resolution frames is inside), the loop and x4
decode totals (sums of CUDA events, summed over this rank's chunks), the stage wall time (host clock around the call,
which ends with the frames on the host, after a synchronise; the slowest rank under torchrun), peak device memory, the
sha256 of the returned frames (equal across GPU counts for the same seed), and the GPU's name and power limit.
"""
import argparse
import hashlib
import json
import os
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from bench_vae_x4 import gpu_identity  # noqa: E402
from lavie_b200.config import VSR_CONFIG  # noqa: E402
from lavie_b200.pipeline import VSRSampler  # noqa: E402
from lavie_b200.synthetic import synthetic_state_dict  # noqa: E402
from lavie_b200.vae import X4_BLOCK_OUT, VAEDecoder, vae_synthetic_state_dict  # noqa: E402
from lavie_b200.vsr import UNet3DVSRModel  # noqa: E402

H, W = 320, 512
STAGE_STEPS = 50


class TimedSampler(VSRSampler):
    """VSRSampler with CUDA events around every chunk's loop."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.chunk_events = []

    def _chunk(self, lr, lr_noise, x, text):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = super()._chunk(lr, lr_noise, x, text)
        e1.record()
        self.chunk_events.append((lr.shape[2], e0, e1))
        return out


class TimedVAE:
    """The x4 decoder with CUDA events around every decode_latents call."""

    def __init__(self, vae):
        self.vae, self.upscale, self.events = vae, vae.upscale, []

    def decode_latents(self, latents):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = self.vae.decode_latents(latents)
        e1.record()
        self.events.append((e0, e1))
        return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=STAGE_STEPS)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--chunk-frames", type=int, default=8)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_vsr_stage needs a CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.gpus != world:
        raise SystemExit(f"--gpus {a.gpus} needs torchrun with {a.gpus} processes (WORLD_SIZE is {world})")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    group = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD
    if rank == 0:
        print(gpu_identity())
        if a.steps != STAGE_STEPS:
            print(f"NOTE: {a.steps} steps per chunk, SHORTER than the stage's {STAGE_STEPS}: loop and wall times are "
                  f"those of the shorter run")

    unet = UNet3DVSRModel()
    unet.load_state_dict(synthetic_state_dict(VSR_CONFIG, seed=0), strict=True)
    unet = unet.to(dev).eval()
    vae = VAEDecoder.x4_upscaler()
    vae.load_state_dict(vae_synthetic_state_dict(seed=0, block_out_channels=X4_BLOCK_OUT), strict=True)
    vae = TimedVAE(vae.to(dev).eval())
    g = torch.Generator().manual_seed(0)
    frames = torch.randint(0, 256, (1, a.frames, H, W, 3), generator=g, dtype=torch.uint8)
    text = torch.randn(2, 77, 1024, generator=g).to(dev)

    # warm-up: one step per chunk captures each chunk length's step graph and warms the decode
    TimedSampler(unet, 5.0, 50, num_inference_steps=1, chunk_frames=a.chunk_frames).upscale(
        frames, text, vae, generator=torch.Generator().manual_seed(1), group=group)
    vae.events = []
    sampler = TimedSampler(unet, 5.0, 50, num_inference_steps=a.steps, chunk_frames=a.chunk_frames)
    torch.cuda.synchronize()
    if group is not None:
        dist.barrier()
    torch.cuda.reset_peak_memory_stats(dev)
    t0 = time.perf_counter()
    video = sampler.upscale(frames, text, vae, generator=torch.Generator().manual_seed(2), group=group)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    peak = torch.cuda.max_memory_allocated(dev) / 2 ** 30

    per_len = {}
    for n, e0, e1 in sampler.chunk_events:
        per_len.setdefault(n, []).append(e0.elapsed_time(e1))
    loop_ms = sum(sum(v) for v in per_len.values())
    decode_ms = sum(e0.elapsed_time(e1) for e0, e1 in vae.events)
    mine = {"rank": rank, "wall_s": wall, "loop_ms": loop_ms, "decode_ms": decode_ms, "peak_gib": peak,
            "ms_per_step": {n: sum(v) / len(v) / a.steps for n, v in per_len.items()},
            "chunks": {n: len(v) for n, v in per_len.items()}}
    every = [mine]
    if group is not None:
        every = [None] * world
        dist.all_gather_object(every, mine)
    if rank == 0:
        assert video.shape == (1, a.frames, 4 * H, 4 * W, 3) and video.dtype == torch.uint8
        steps_ms = {}
        for r in every:
            for n, ms in r["ms_per_step"].items():
                steps_ms.setdefault(n, []).append(ms)
        result = {
            "stage": f"VSR x4 {H}x{W} -> {4 * H}x{4 * W}, {a.frames} frames, chunks of {a.chunk_frames}",
            "gpus": world, "steps_per_chunk": a.steps, "shorter_than_stage": a.steps != STAGE_STEPS,
            "ms_per_cfg_step": {f"{n}-frame chunk": round(max(v), 2) for n, v in sorted(steps_ms.items())},
            "loop_ms_per_rank_max": round(max(r["loop_ms"] for r in every), 1),
            "decode_ms_per_rank_max": round(max(r["decode_ms"] for r in every), 1),
            "loop_ms_all_ranks": round(sum(r["loop_ms"] for r in every), 1),
            "decode_ms_all_ranks": round(sum(r["decode_ms"] for r in every), 1),
            "stage_wall_s": round(max(r["wall_s"] for r in every), 2),
            "peak_mem_gib_max_rank": round(max(r["peak_gib"] for r in every), 1),
            "chunks_per_rank": [sum(r["chunks"].values()) for r in every],
            "video_sha256": hashlib.sha256(video.numpy().tobytes()).hexdigest()[:16],
            "gpu": gpu_identity(),
        }
        print(json.dumps(result))
    if group is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
