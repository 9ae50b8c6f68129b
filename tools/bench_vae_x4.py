"""Times the x4-upscaler VAE decode on one GPU: the fused d = 512 mid-block attention against a yardstick built from the
GEMM kernels, and whole decodes of a [1,4,F,320,512] latent.

    python tools/bench_vae_x4.py [--reps 3] [--frames 8 16]

1. Attention at S = 320 * 512 = 163 840 tokens per frame, 1 and 8 frames: lavie_attention_wide_bf16.  The yardstick runs
   query blocks of 4096 rows as Q K^T (ops.gemm) -> row softmax -> P V (ops.gemm against V^T, as the SD VAE path does).
   ops.softmax_rows_ takes rows of at most 4096 keys, so at 163 840 keys the yardstick's softmax pass is torch.softmax
   (a memory-bound pass over the same 1.3 GB score block).  The kernel and the yardstick run alternately in this
   process; their full-size outputs are compared (rel-L2), and 1024 sampled query rows of the kernel are checked
   against float64 over all keys.  q, k, v are 168 MB each, larger than the 126 MB L2.
   Algorithmic FLOPs are 4 S^2 d per frame; the kernel executes 6 S^2 d (each of its two CTAs per query tile computes
   the full Q K^T for its half of the output columns), the yardstick 4 S^2 d.
2. decode_latents of F frames of a 320x512 latent -> uint8 [1,F,1280,2048,3], timed end to end, then once more with
   per-launch CUDA events to split the time into attention, convolutions and norms.
"""
import argparse
import math
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from lavie_b200 import ops  # noqa: E402
from lavie_b200.vae import X4_BLOCK_OUT, VAEDecoder, vae_synthetic_state_dict  # noqa: E402
from lavie_b200.vae_attention import attention_wide  # noqa: E402

DEV = "cuda"
D = 512
H_LAT, W_LAT = 320, 512
S = H_LAT * W_LAT
QBLOCK = 4096


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


def yardstick(q, k, v, frames, out):
    """Q K^T -> softmax -> P V per 4096-row query block, from the GEMM kernels."""
    for f in range(frames):
        rows = slice(f * S, (f + 1) * S)
        vt = v[rows].t().contiguous()                         # V^T [512, S]: P V = P (V^T)^T on ops.gemm
        for a in range(0, S, QBLOCK):
            b = min(a + QBLOCK, S)
            s = ops.gemm(q[rows][a:b], k[rows])               # [block, S] scores (scale folded into q)
            if S <= 4096:
                ops.softmax_rows_(s, 1.0)
            else:
                s = torch.softmax(s, dim=-1)
            ops.gemm(s, vt, out=out[rows][a:b])
    return out


def sampled_parity(q, k, v, o, nrows=1024):
    rows = torch.randperm(S, generator=torch.Generator().manual_seed(0))[:nrows].to(DEV)
    s = q[:S][rows].double() @ k[:S].double().T
    ref = torch.softmax(s, dim=-1) @ v[:S].double()
    err = (o[:S][rows].double() - ref)
    return float(err.norm() / ref.norm()), float(err.abs().max()), float(ref.abs().max())


def bench_attention(reps):
    g = torch.Generator(device=DEV).manual_seed(0)
    frames_max = 8
    q = (torch.randn(frames_max * S, D, generator=g, device=DEV) * (3.0 / math.sqrt(D))).to(torch.bfloat16)
    k = torch.randn(frames_max * S, D, generator=g, device=DEV).to(torch.bfloat16)
    v = torch.randn(frames_max * S, D, generator=g, device=DEV).to(torch.bfloat16)
    o_k = torch.empty(frames_max * S, D, dtype=torch.bfloat16, device=DEV)
    o_y = torch.empty(frames_max * S, D, dtype=torch.bfloat16, device=DEV)
    alg = 4.0 * S * S * D
    exe_k, exe_y = 6.0 * S * S * D, 4.0 * S * S * D

    def kern(n):
        return lambda: attention_wide(q[:n * S], k[:n * S], v[:n * S], n, S, out=o_k[:n * S])

    kern(1)()
    yardstick(q, k, v, 1, o_y)                                # warm-up of every shape
    torch.cuda.synchronize()
    tk, ty = [], []
    for _ in range(reps):                                     # alternate kernel and yardstick
        tk += timed(kern(1), 1)
        ty += timed(lambda: yardstick(q, k, v, 1, o_y), 1)
    rel = float((o_k[:S].double() - o_y[:S].double()).norm() / o_y[:S].double().norm())
    print(f"\n== mid-block attention, one head d=512, S={S} tokens per frame (inputs {3 * q.numel() * 2 / 1e9:.2f} GB) ==")
    for name, t, exe in (("fused kernel", tk, exe_k), ("yardstick (GEMM + softmax + GEMM)", ty, exe_y)):
        best, med = min(t), sorted(t)[len(t) // 2]
        print(f"  1 frame  {name:36s} median {med:8.2f} ms  best {best:8.2f} ms  "
              f"algorithmic {alg / med / 1e9:7.1f} TFLOP/s  executed {exe / med / 1e9:7.1f} TFLOP/s  (all: "
              + ", ".join(f"{x:.2f}" for x in t) + ")")
    print(f"  kernel / yardstick time: {sorted(tk)[len(tk) // 2] / sorted(ty)[len(ty) // 2]:.3f}")
    print(f"  full-size cross-check: rel-L2(kernel, yardstick) = {rel:.3e}")
    r, mx, ref_mx = sampled_parity(q, k, v, o_k)
    print(f"  production-size sampled parity: 1024 query rows vs float64 over all {S} keys: rel-L2 {r:.3e}, "
          f"max |err| {mx:.3e} (max |ref| {ref_mx:.3e})")
    n = frames_max
    kern(n)()
    torch.cuda.synchronize()
    t8 = timed(kern(n), max(2, reps - 1))
    med = sorted(t8)[len(t8) // 2]
    print(f"  {n} frames fused kernel: median {med:8.2f} ms = {med / n:7.2f} ms/frame  algorithmic "
          f"{n * alg / med / 1e9:7.1f} TFLOP/s  executed {n * exe_k / med / 1e9:7.1f} TFLOP/s  (all: "
          + ", ".join(f"{x:.2f}" for x in t8) + ")")
    del q, k, v, o_k, o_y
    torch.cuda.empty_cache()


def phase_of(kernel, tag):
    if kernel == "attn_wide_kernel":
        return "attention (fused kernel)"
    if tag.startswith("gemm") and tag.endswith("K=512") and (" N=1536 " in tag or " N=512 " in tag):
        return "attention (q/k/v + proj GEMMs)"
    if "groupnorm" in kernel:
        return "norms"
    if tag.startswith(("conv3x3", "upsample_conv3x3", "gemm")) or kernel in (
            "lavie_im2col3x3_bf16", "lavie_upsample_nearest2x", "lavie_conv_in", "lavie_pointwise_conv_nchw_f32"):
        return "convs"
    return "other (" + kernel + ")"


def bench_decode(frames_list, reps):
    sd = vae_synthetic_state_dict(seed=0, block_out_channels=X4_BLOCK_OUT)
    m = VAEDecoder.x4_upscaler()
    m.load_state_dict(sd, strict=True)
    m = m.to(DEV).eval()
    print(f"\n== x4 decode_latents, [1,4,F,{H_LAT},{W_LAT}] -> uint8 [1,F,{4 * H_LAT},{4 * W_LAT},3], "
          f"{m.frames_per_group(H_LAT, W_LAT)} frames per group ==")
    for F in frames_list:
        lat = 0.08333 * torch.randn(1, 4, F, H_LAT, W_LAT, generator=torch.Generator().manual_seed(F))
        z = lat.permute(0, 2, 1, 3, 4).reshape(F, 4, H_LAT, W_LAT).to(DEV)
        run = lambda: m.decode(z, scale=1 / 0.08333, as_uint8=True)   # noqa: E731  (device part of decode_latents)
        run()
        torch.cuda.synchronize()
        t = timed(run, reps)
        med = sorted(t)[len(t) // 2]
        t0 = time.perf_counter()
        video = m.decode_latents(lat.to(DEV))
        host = (time.perf_counter() - t0) * 1e3
        assert video.shape == (1, F, 4 * H_LAT, 4 * W_LAT, 3) and video.dtype == torch.uint8
        print(f"  F={F:2d}: device decode median {med:9.1f} ms ({med / F:7.1f} ms/frame; all: "
              + ", ".join(f"{x:.1f}" for x in t) + f"); decode_latents incl. copy to host {host:9.1f} ms")
        ops.PROFILE = []
        run()
        torch.cuda.synchronize()
        phases = {}
        for kernel, _fl, _nb, e0, e1, tag in ops.PROFILE:
            ph = phase_of(kernel, tag)
            phases[ph] = phases.get(ph, 0.0) + e0.elapsed_time(e1)
        n = len(ops.PROFILE)
        ops.PROFILE = None
        total = sum(phases.values())
        print(f"        per-phase split ({n} launches, per-launch events, sum {total:.1f} ms): " + ", ".join(
            f"{k} {v:.1f} ms ({100 * v / total:.0f} %)" for k, v in sorted(phases.items(), key=lambda kv: -kv[1])))
        del video, z
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--frames", type=int, nargs="*", default=[8, 16])
    ap.add_argument("--skip-attention", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_vae_x4 needs a CUDA device")
    print(gpu_identity())
    if not a.skip_attention:
        bench_attention(a.reps)
    if a.frames:
        bench_decode(a.frames, a.reps)


if __name__ == "__main__":
    main()
