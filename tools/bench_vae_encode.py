"""Times the VAE encoder on one GPU: ``VAEEncoder.encode_video`` of uint8 videos [1, F, 320, 512, 3] (the interpolation
stage's conditioning frames) and the Downsample2D conv with its one-sided (0, 1) padding against the pad-1 stride-2 conv.

    python tools/bench_vae_encode.py [--reps 5] [--frames 16 61] [--log profiles/r3_bench_vae_encode.log]

1. encode_video (sampled posterior) of F frames at 320x512 -> fp32 latents [1, 4, F, 40, 64], timed end to end with CUDA
   events around the device work (frames already on the device), then once more with per-launch CUDA events to split
   the time into convolutions, norms, attention and input / posterior launches.  Conv TFLOP/s = the convs' algorithmic
   FLOPs (2 M N K per launch, from the shapes) over their summed launch times.
2. The three Downsample2D convs of a 16-frame encode (128, 256 and 512 channels) as pad (0, 1) and as pad (1, 1), the same
   kernel with different im2col bounding-box corners, alternating in this process.
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from lavie_b200 import ops  # noqa: E402
from lavie_b200.vae import VAEEncoder, vae_encoder_synthetic_state_dict  # noqa: E402

DEV = "cuda"
H, W = 320, 512
LINES = []


def say(s=""):
    print(s, flush=True)
    LINES.append(s)


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"power limit unknown ({e})"
    return f"{name}; power limit, max SM clock: {q}"


def timed(fn, reps):
    """Per-call milliseconds of fn() from CUDA events, one measurement per repetition."""
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def med(t):
    return sorted(t)[len(t) // 2]


def phase_of(kernel, tag):
    if kernel in ("lavie_im2col_frames_bf16", "lavie_posterior_sample_f32"):
        return "input / posterior"
    if "groupnorm" in kernel:
        return "norms"
    if kernel == "lavie_softmax_rows_bf16" or (tag.startswith("gemm") and "K=512" in tag and " N=512 " in tag) or \
            (tag.startswith("gemm M=") and ("N=2560 " in tag or "K=2560" in tag)):
        return "attention"
    return "convs"


def bench_encode(frames_list, reps):
    m = VAEEncoder()
    m.load_state_dict(vae_encoder_synthetic_state_dict(seed=0), strict=True)
    m = m.to(DEV).eval()
    say(f"\n== encode_video, uint8 [1,F,{H},{W},3] -> latents [1,4,F,{H // 8},{W // 8}], "
        f"{m.frames_per_group(H, W)} frames per group ==")
    for F in frames_list:
        frames = torch.randint(0, 256, (1, F, H, W, 3), dtype=torch.uint8,
                               generator=torch.Generator().manual_seed(F)).to(DEV)
        gen = torch.Generator(device=DEV)
        run = lambda: m.encode_video(frames, generator=gen.manual_seed(0))   # noqa: E731
        run()
        torch.cuda.synchronize()
        t = timed(run, reps)
        say(f"  F={F:2d}: encode_video median {med(t):8.1f} ms ({med(t) / F:6.2f} ms/frame; all: "
            + ", ".join(f"{x:.1f}" for x in t) + ")")
        ops.PROFILE = []
        run()
        torch.cuda.synchronize()
        phases, conv_flops = {}, 0.0
        for kernel, fl, _nb, e0, e1, tag in ops.PROFILE:
            ph = phase_of(kernel, tag)
            phases[ph] = phases.get(ph, 0.0) + e0.elapsed_time(e1)
            if ph == "convs":
                conv_flops += fl
        n = len(ops.PROFILE)
        ops.PROFILE = None
        total = sum(phases.values())
        say(f"        per-phase split ({n} launches, per-launch events, sum {total:.1f} ms): " + ", ".join(
            f"{k} {v:.1f} ms ({100 * v / total:.0f} %)" for k, v in sorted(phases.items(), key=lambda kv: -kv[1])))
        say(f"        convs: {conv_flops / F / 1e12:.3f} TFLOP per frame (algorithmic, from shapes), "
            f"{conv_flops / phases['convs'] / 1e9:.1f} TFLOP/s over their launch times")
        del frames
        torch.cuda.empty_cache()


def bench_downsample(reps, F=16):
    say(f"\n== Downsample2D conv, {F} frames of a {H}x{W} encode: pad (0,1) vs pad (1,1), stride 2, alternating ==")
    g = torch.Generator(device=DEV).manual_seed(0)
    h, w = H, W
    for C in (128, 256, 512):
        x = torch.randn(F * h * w, C, generator=g, device=DEV).to(torch.bfloat16)
        wt = (torch.randn(C, 9 * C, generator=g, device=DEV) / (3 * C ** 0.5)).to(torch.bfloat16)
        b = torch.zeros(C, device=DEV)
        runs = {p: (lambda p=p: ops.conv3x3(x, F, h, w, wt, stride=2, padding=p, bias=b, stats=True))
                for p in ((0, 1), (1, 1))}
        for f in runs.values():
            f()
        torch.cuda.synchronize()
        t = {p: [] for p in runs}
        for _ in range(reps):
            for p, f in runs.items():
                t[p] += timed(f, 1)
        ho, wo = ops.conv3x3_out_size(h, 2, (0, 1)), ops.conv3x3_out_size(w, 2, (0, 1))
        flops = 2.0 * F * ho * wo * C * 9 * C
        say(f"  C={C:3d} {h}x{w} -> {ho}x{wo}: " + "; ".join(
            f"pad {p} median {med(v):.3f} ms ({flops / med(v) / 1e9:.1f} TFLOP/s; all: " + ", ".join(
                f"{x:.3f}" for x in v) + ")" for p, v in t.items())
            + f"; (0,1)/(1,1) = {med(t[(0, 1)]) / med(t[(1, 1)]):.3f}")
        h, w = ho, wo
        del x, wt
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--frames", type=int, nargs="*", default=[16, 61])
    ap.add_argument("--log", default=os.path.join("profiles", "r3_bench_vae_encode.log"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_vae_encode needs a CUDA device")
    say(gpu_identity())
    bench_encode(a.frames, a.reps)
    bench_downsample(a.reps)
    os.makedirs(os.path.dirname(os.path.abspath(a.log)), exist_ok=True)
    with open(a.log, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
