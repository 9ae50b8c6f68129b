"""The x4-upscaler VAE decoder (lavie_b200.vae.VAEDecoder.x4_upscaler) and its fused single-head d = 512 mid-block
attention (lavie_b200.vae_attention.attention_wide -> lavie_attention_wide_bf16).

GPU tests check the kernel launch by launch against a float64 reference with an element-wise bound from the rounding
model, probe the key tails, check determinism and that nothing outside the output view is written, sample the kernel
at its production size (163 840 tokens), and compare the whole decoder with the oracle restatement
(oracle/vae_x4_oracle.py, parity unpinned).  CPU tests pin the parameter layouts and the frame grouping."""
import hashlib
import math
import os
import re

import pytest
import torch

from conftest import rel_l2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda"
D = 512
# The x4 decoder stacks 21 convolutions, 21 GroupNorms and the attention block.  With weights and every intermediate
# rounded to bf16 on the CPU, the oracle itself sits 2.0e-2 .. 2.1e-2 (rel-L2) from its fp32 run at the four decoder
# geometries below, so the tolerance is 4e-2, the same margin the SD VAE test keeps over its 2.3e-2.
X4_TOL = 4e-2


# ------------------------------------------------------------------------------------------------ kernel reference
def _qkv(frames, S, seed, score_std=3.0, device=DEV):
    """bf16 q, k, v [frames * S, 512]; q carries the scale, so the scores have about ``score_std`` spread."""
    g = torch.Generator(device=device).manual_seed(seed)
    q = (torch.randn(frames * S, D, generator=g, device=device) * (score_std / math.sqrt(D))).to(torch.bfloat16)
    k = torch.randn(frames * S, D, generator=g, device=device).to(torch.bfloat16)
    v = torch.randn(frames * S, D, generator=g, device=device).to(torch.bfloat16)
    return q, k, v


def _reference(q, k, v, frames, S, rows=None):
    """float64 softmax(q k^T) v per frame and the element-wise bound of the kernel's rounding, the one the per-launch
    audit holds the kernel to (tests/test_launch_audit.py, RHO_WIDE and c_attn_wide): bf16 output rounding, bf16
    probabilities in P V, the fp32 score error of the K = 512 tcgen05 product (c_gemm(512) of each key's sum |q| |k|) and
    the fp32 chains over the S keys.  ``rows``: only these query rows (indices within a frame) of every frame."""
    from test_launch_audit import wide_attention_ref
    o, bnd = wide_attention_ref(q, k, v, frames, S, rows)
    return o.reshape(-1, D), bnd.reshape(-1, D)


def _check(out, ref, bnd, what):
    err = (out.double() - ref).abs()
    worst = float((err / bnd).max())
    i = int((err / bnd).argmax())
    assert worst <= 1.0, (f"{what}: element {divmod(i, D)} off by {float(err.flatten()[i]):.3e}, bound "
                          f"{float(bnd.flatten()[i]):.3e}")
    r = rel_l2(out, ref)
    assert r < 5e-3, f"{what}: rel-L2 {r:.3e}"
    return worst, r


@pytest.mark.gpu
@pytest.mark.parametrize("frames,S", [(1, 1), (2, 7), (1, 127), (3, 128), (1, 129), (2, 1000), (1, 2560), (1, 4129)])
def test_wide_attention_vs_fp64(frames, S):
    from lavie_b200.vae_attention import attention_wide
    q, k, v = _qkv(frames, S, seed=frames * 10007 + S)
    out = attention_wide(q, k, v, frames, S)
    assert out.shape == (frames * S, D) and out.dtype == torch.bfloat16
    ref, bnd = _reference(q, k, v, frames, S)
    _check(out, ref, bnd, f"attention_wide frames={frames} S={S}")


@pytest.mark.gpu
@pytest.mark.parametrize("S", [127, 129, 1000, 4129])
def test_wide_attention_tail_probes(S):
    """A dropped or duplicated key shows up as V = 1 not giving 1, or as a key-index ramp not matching the reference.
    Peaky scores (spread 8) and a self-similar q ~ k make single keys, including the last partial tile's, dominate."""
    from lavie_b200.vae_attention import attention_wide
    q, k, _ = _qkv(1, S, seed=S, score_std=8.0)
    out = attention_wide(q, k, torch.ones(S, D, dtype=torch.bfloat16, device=DEV), 1, S)
    assert float((out.float() - 1).abs().max()) <= 2.0 ** -7, "V = 1 probe"
    j = torch.arange(S, device=DEV, dtype=torch.float64)
    ramp = torch.stack([j, j.remainder(64)], dim=1).repeat(1, D // 2).to(torch.bfloat16)   # even columns j, odd j mod 64
    x = torch.randn(S, D, generator=torch.Generator(device=DEV).manual_seed(S + 1), device=DEV)
    for qq, kk, what in ((q, k, "peaky"), ((0.1 * x).to(torch.bfloat16), x.to(torch.bfloat16), "self-similar")):
        out = attention_wide(qq, kk, ramp, 1, S)
        ref, bnd = _reference(qq, kk, ramp, 1, S)
        _check(out, ref, bnd, f"key ramp ({what}) S={S}")


@pytest.mark.gpu
def test_wide_attention_deterministic_and_writes_only_its_view():
    from lavie_b200.vae_attention import attention_wide
    frames, S = 2, 333
    q, k, v = _qkv(frames, S, seed=5)
    a = attention_wide(q, k, v, frames, S)
    b = attention_wide(q, k, v, frames, S)
    assert torch.equal(a, b)
    buf = torch.full((frames * S + 2, 640), 7.0, dtype=torch.bfloat16, device=DEV)
    view = buf[1:frames * S + 1, 64:64 + D]
    attention_wide(q, k, v, frames, S, out=view)
    assert torch.equal(view, a)
    mask = torch.ones_like(buf, dtype=torch.bool)
    mask[1:frames * S + 1, 64:64 + D] = False
    assert bool((buf[mask] == 7.0).all()), "wrote outside the output view"
    # strided inputs (q, k, v as column slices of one [rows, 1536] buffer, as the decoder passes them)
    qkv = torch.cat([q, k, v], dim=1)
    c = attention_wide(qkv[:, :D], qkv[:, D:2 * D], qkv[:, 2 * D:], frames, S)
    assert torch.equal(c, a)


@pytest.mark.gpu
def test_wide_attention_rejects_bad_arguments():
    from lavie_b200 import _lib
    from lavie_b200.ops import _stream
    lib = _lib.load()
    t = torch.zeros(64, D, dtype=torch.bfloat16, device=DEV)
    p = t.data_ptr()
    assert lib.lavie_attention_wide_bf16(p, D, p, D, p, D, p, D, 1, 0, _stream()) == -1
    assert lib.lavie_attention_wide_bf16(p, 500, p, D, p, D, p, D, 1, 64, _stream()) == -1
    assert lib.lavie_attention_wide_bf16(p, 516, p, 516, p, 516, p, 516, 1, 60, _stream()) == -2
    assert lib.lavie_attention_wide_bf16(p + 2, D, p, D, p, D, p, D, 1, 32, _stream()) == -2
    assert b"attention_wide" in lib.lavie_last_error()


@pytest.mark.gpu
def test_wide_attention_production_size_sampled():
    """One frame of a 320x512 latent: 163 840 tokens.  1024 random query rows against float64 over all keys."""
    from lavie_b200.vae_attention import attention_wide
    S = 320 * 512
    q, k, v = _qkv(1, S, seed=163840)
    out = attention_wide(q, k, v, 1, S)
    rows = torch.randperm(S, generator=torch.Generator().manual_seed(0))[:1024].to(DEV)
    ref, bnd = _reference(q, k, v, 1, S, rows=rows)
    worst, r = _check(out[rows], ref, bnd, "attention_wide S=163840 (sampled)")
    print(f"S=163840, 1024 sampled rows: worst error / bound = {worst:.3f}, rel-L2 = {r:.3e}")


# ------------------------------------------------------------------------------------------------ decoder
@pytest.fixture(scope="module")
def x4():
    from lavie_b200.vae import X4_BLOCK_OUT, VAEDecoder, vae_synthetic_state_dict
    sd = vae_synthetic_state_dict(seed=0, block_out_channels=X4_BLOCK_OUT)
    m = VAEDecoder.x4_upscaler()
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval(), sd


@pytest.mark.gpu
@pytest.mark.parametrize("N,h,w", [(3, 8, 8), (2, 16, 24), (1, 40, 64), (1, 12, 20)])
def test_x4_decode_vs_oracle(x4, N, h, w):
    """(1, 12, 20): 240 tokens, not a multiple of the 128-query or 64-key tile, and W = 20 / 40 has no fused
    upsample conv (nearest x2 + conv instead)."""
    from lavie_b200 import ops
    from oracle import vae_x4_oracle as V
    if (h, w) == (12, 20):
        assert not ops.upsample_conv3x3_supported(h, w, 512)
    m, sd = x4
    z = torch.randn(N, 4, h, w, generator=torch.Generator().manual_seed(h * w))
    ref = V.decode(sd, z)
    out = m.decode(z.to(DEV)).sample
    assert out.shape == ref.shape == (N, 3, 4 * h, 4 * w) and out.dtype == torch.float32
    assert rel_l2(out.cpu(), ref) < X4_TOL


@pytest.mark.gpu
def test_x4_decode_latents_uint8(x4):
    """The VSR pipeline's decode: [B,4,F,h,w] -> uint8 [B,F,4h,4w,3] on the host, 1/0.08333 folded into the kernels."""
    from oracle import vae_x4_oracle as V
    m, sd = x4
    lat = 0.08333 * torch.randn(1, 4, 3, 16, 16, generator=torch.Generator().manual_seed(9))
    ref = V.decode_latents(sd, lat)
    out = m.decode_latents(lat.to(DEV))
    assert out.shape == ref.shape == (1, 3, 64, 64, 3) and out.dtype == torch.uint8 and out.device.type == "cpu"
    diff = (out.int() - ref.int()).abs()
    assert float(diff.float().mean()) < 1.0 and int(diff.max()) <= 12


@pytest.mark.gpu
def test_x4_decode_grouping_matches_one_group(x4):
    """Five frames with the launch bound lowered to two frames' worth: groups of 2, 2, 1 against one group of 5."""
    m, _ = x4
    z = torch.randn(5, 4, 8, 8, generator=torch.Generator().manual_seed(4)).to(DEV)
    fe = m.frame_elements(8, 8)
    assert m.frames_per_group(8, 8, 2 * fe + 1) == 2
    one = m.decode(z).sample
    grouped = m.decode(z, max_launch_elements=2 * fe + 1).sample
    assert grouped.shape == one.shape
    for f in range(5):
        assert rel_l2(grouped[f].cpu(), one[f].cpu()) < 1e-2, f
    u1 = m.decode(z, as_uint8=True)
    u2 = m.decode(z, as_uint8=True, max_launch_elements=2 * fe + 1)
    assert u2.shape == u1.shape == (5, 32, 32, 3)
    assert float((u1.int() - u2.int()).abs().float().mean()) < 1.0


@pytest.mark.gpu
def test_x4_loads_a_full_autoencoder_checkpoint_layout(x4):
    """Encoder-side keys are dropped; post-0.16 attention names (and 1x1-conv shaped attention weights) are accepted."""
    from lavie_b200.vae import VAEDecoder, load_vae_state_dict
    m, sd = x4
    full = dict(sd)
    full["encoder.conv_in.weight"] = torch.zeros(128, 3, 3, 3)
    full["encoder.mid_block.attentions.0.to_q.weight"] = torch.zeros(512, 512)
    full["quant_conv.weight"] = torch.zeros(8, 8, 1, 1)
    a = "decoder.mid_block.attentions.0"
    for new, old in (("to_q", "query"), ("to_k", "key"), ("to_v", "value"), ("to_out.0", "proj_attn")):
        full[f"{a}.{new}.weight"] = full.pop(f"{a}.{old}.weight").reshape(512, 512, 1, 1)
        full[f"{a}.{new}.bias"] = full.pop(f"{a}.{old}.bias")
    m2 = VAEDecoder.x4_upscaler()
    load_vae_state_dict(m2, full, strict=True)
    m2 = m2.to(DEV).eval()
    z = torch.randn(1, 4, 8, 8, generator=torch.Generator().manual_seed(2)).to(DEV)
    assert torch.equal(m2.decode(z).sample, m.decode(z).sample)


# ------------------------------------------------------------------------------------------------ CPU
def test_x4_param_spec_matches_published_config():
    from lavie_b200.vae import X4_BLOCK_OUT, VAEDecoder, vae_decoder_param_spec
    spec = vae_decoder_param_spec(X4_BLOCK_OUT)
    assert len(spec) == 114
    d = "decoder."
    assert spec[d + "conv_in.weight"] == (512, 4, 3, 3)
    assert spec[d + "mid_block.attentions.0.query.weight"] == (512, 512)
    assert spec[d + "up_blocks.0.resnets.2.conv2.weight"] == (512, 512, 3, 3)
    assert spec[d + "up_blocks.0.upsamplers.0.conv.weight"] == (512, 512, 3, 3)
    assert spec[d + "up_blocks.1.resnets.0.conv1.weight"] == (256, 512, 3, 3)
    assert spec[d + "up_blocks.1.resnets.0.conv_shortcut.weight"] == (256, 512, 1, 1)
    assert spec[d + "up_blocks.1.upsamplers.0.conv.weight"] == (256, 256, 3, 3)
    assert spec[d + "up_blocks.2.resnets.0.conv_shortcut.weight"] == (128, 256, 1, 1)
    assert d + "up_blocks.2.upsamplers.0.conv.weight" not in spec
    assert not any(k.startswith(d + "up_blocks.3.") for k in spec)
    assert spec[d + "conv_norm_out.weight"] == (128,) and spec[d + "conv_out.weight"] == (3, 128, 3, 3)
    m = VAEDecoder.x4_upscaler()
    assert m.config.scaling_factor == 0.08333 and m.config.block_out_channels == (128, 256, 512) and m.upscale == 4
    assert set(m.state_dict()) == set(spec)
    from oracle import vae_x4_oracle as V
    assert V.BLOCK_OUT == X4_BLOCK_OUT and V.SCALING == m.config.scaling_factor


def test_sd_param_spec_unchanged():
    from lavie_b200.vae import VAEDecoder, vae_decoder_param_spec
    spec = vae_decoder_param_spec()
    assert len(spec) == 140
    assert hashlib.sha256(repr(list(spec.items())).encode()).hexdigest() == (
        "73ba096be8697419ba4108fae7ec096168bd87c9f4bfbe6d8031e87265766a05")
    m = VAEDecoder()
    assert m.config.scaling_factor == 0.18215 and m.upscale == 8 and not m.wide_attention


def test_x4_oracle_output_shape():
    from lavie_b200.vae import X4_BLOCK_OUT, vae_synthetic_state_dict
    from oracle import vae_x4_oracle as V
    sd = vae_synthetic_state_dict(seed=1, block_out_channels=X4_BLOCK_OUT)
    z = torch.randn(2, 4, 4, 6, generator=torch.Generator().manual_seed(0))
    assert V.decode(sd, z).shape == (2, 3, 16, 24)
    lat = torch.randn(1, 4, 2, 4, 6, generator=torch.Generator().manual_seed(1))
    out = V.decode_latents(sd, lat)
    assert out.shape == (1, 2, 16, 24, 3) and out.dtype == torch.uint8


def test_x4_frame_grouping_from_geometry():
    """At a 320x512 latent the largest map is the 256-channel upsampled 1280x2048 one: 6.7e8 elements per frame, so three
    frames per group keep every launch under 2^31 elements."""
    from lavie_b200.vae import VAEDecoder
    m = VAEDecoder.x4_upscaler()
    assert m.frame_elements(320, 512) == 256 * 1280 * 2048
    assert m.frames_per_group(320, 512) == 3
    assert m.frames_per_group(8, 8) * m.frame_elements(8, 8) <= 2 ** 31 - 1
    assert VAEDecoder().frames_per_group(40, 64) >= 16        # the SD video of the benchmark stays one group
    with pytest.raises(ValueError):
        m.frames_per_group(320, 512, max_launch_elements=10 ** 8)


def test_wide_attention_symbol_declared():
    from lavie_b200 import _lib
    text = open(os.path.join(ROOT, "include", "lavie_b200.h")).read()
    assert re.search(r"\bint lavie_attention_wide_bf16\s*\(", text)
    assert "lavie_attention_wide_bf16" in _lib.SIGNATURES
