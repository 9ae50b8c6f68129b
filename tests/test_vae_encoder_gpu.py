"""The VAE encoder (lavie_b200.vae.VAEEncoder) and the kernels only it needs: the 3x3 conv with Downsample2D's
one-sided (0, 1) padding (ops.conv3x3(padding=(0, 1)) -> lavie_conv3x3_pad_bf16), conv_in patch rows from uint8 frames
(lavie_im2col_frames_bf16) and the posterior sample (lavie_posterior_sample_f32).

GPU tests check each kernel against float64 with element-wise bounds from the rounding model of tests/test_launch_audit.py,
and the whole encoder against the oracle restatement (oracle/vae_encoder_oracle.py, parity unpinned).  CPU tests pin the
parameter layout, the output-size formula, the argument checks and the ABI declarations."""
import ctypes
import os
import re

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2
from test_launch_audit import U, c_gemm, check_colsums, gn_scale_shift64

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda"
F64 = torch.float64
# The encoder stacks 21 convolutions, 20 GroupNorms and the mid-block attention.  With weights and every intermediate
# rounded to bf16 on the CPU, the oracle itself sits 1.1e-2 .. 1.3e-2 (mean) and 1.4e-2 .. 1.5e-2 (logvar) rel-L2 from
# its fp32 run at the four geometries below (a sample with unit noise: 4.6e-3 .. 4.8e-3), so the tolerance is 3e-2.
ENC_TOL = 3e-2


def _splits(M, N, K):
    """split-K factor the planner picks for this conv (its fp32 reduction adds to the accumulation bound)."""
    from lavie_b200 import _lib, ops
    bn, s, tail, ts = (ctypes.c_int() for _ in range(4))
    assert _lib.load().lavie_gemm_plan(M, N, K, 1, 0, ops.WORKSPACE_BYTES, bn, s, tail, ts) == 0
    return max(s.value, ts.value, 1)


def _down_ref(x, NF, H, W, w, bias):
    """float64 F.conv2d(F.pad(x, (0, 1, 0, 1)), w, stride=2) + bias, and the element-wise bound of the kernel: bf16 output
    rounding plus the fp32 accumulation over |x| |w| (c_gemm)."""
    C, N = x.shape[1], w.shape[0]
    xi = x.to(F64).reshape(NF, H, W, C).permute(0, 3, 1, 2)
    wi = w.to(F64).reshape(N, 3, 3, C).permute(0, 3, 1, 2)
    ref = F.conv2d(F.pad(xi, (0, 1, 0, 1)), wi, stride=2) + bias.to(F64)[None, :, None, None]
    s = F.conv2d(F.pad(xi.abs(), (0, 1, 0, 1)), wi.abs(), stride=2) + bias.to(F64).abs()[None, :, None, None]
    Ho, Wo = ref.shape[2], ref.shape[3]
    ref = ref.permute(0, 2, 3, 1).reshape(NF * Ho * Wo, N)
    s = s.permute(0, 2, 3, 1).reshape(NF * Ho * Wo, N)
    c = c_gemm(9 * C, _splits(NF * Ho * Wo, N, 9 * C)) * (1 + U)
    return ref, U * ref.abs() + c * s, Ho, Wo


def _conv_inputs(NF, H, W, C, N, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(NF * H * W, C, generator=g, device=DEV).to(torch.bfloat16)
    w = (torch.randn(N, 9 * C, generator=g, device=DEV) / (3 * C ** 0.5)).to(torch.bfloat16)
    b = torch.randn(N, generator=g, device=DEV) * 0.1
    return x, w, b


# ------------------------------------------------------------------------------------------------ padded conv
@pytest.mark.gpu
@pytest.mark.parametrize("NF,H,W,C", [(2, 64, 64, 128), (3, 33, 47, 256), (1, 50, 80, 512), (4, 10, 6, 128),
                                      (2, 25, 41, 512), (5, 16, 24, 256)])
def test_downsample_conv_vs_fp64(NF, H, W, C):
    """Odd and ragged H / W (33 x 47, 25 x 41, 10 x 6), output rows per launch that are not a multiple of 128 (3 x 16 x 23
    = 1104, 2 x 12 x 20 = 480), several frames.  The fused column statistics must match the output, and the GroupNorm
    (scale, shift) folded from them a float64 GroupNorm of the output."""
    from lavie_b200 import ops
    x, w, b = _conv_inputs(NF, H, W, C, C, seed=NF * H * W + C)
    out = ops.conv3x3(x, NF, H, W, w, stride=2, padding=(0, 1), bias=b, stats=True)
    ref, bnd, Ho, Wo = _down_ref(x, NF, H, W, w, b)
    assert (Ho, Wo) == (ops.conv3x3_out_size(H, 2, (0, 1)), ops.conv3x3_out_size(W, 2, (0, 1)))
    assert out.shape == (NF * Ho * Wo, C)
    err = (out.to(F64) - ref).abs()
    worst = float((err / bnd).max())
    at = divmod(int((err / bnd).argmax()), C)
    assert worst <= 1.0, f"element (row, channel) {at}: err {float(err[at]):.3e} bound {float(bnd[at]):.3e}"
    assert rel_l2(out, ref) < 2.5e-3
    cmp = check_colsums(out._gn_colsums, out)
    assert cmp.ok, str(cmp)
    g = torch.Generator(device=DEV).manual_seed(C)
    gamma = 1 + 0.1 * torch.randn(C, generator=g, device=DEV)
    beta = 0.1 * torch.randn(C, generator=g, device=DEV)
    if C >= 256 and (Ho * Wo) % 32 == 0:
        assert ops.colsums(out, Ho * Wo) is not None          # the statistics below come from the conv's epilogue
    ss = ops.groupnorm_scale_shift(out, NF, Ho * Wo, gamma, beta, 1e-6)
    scale, shift, b_scale, b_shift = gn_scale_shift64(out, NF, gamma, beta, 1e-6)
    assert bool(((ss[..., 0].to(F64) - scale).abs() <= b_scale).all())
    assert bool(((ss[..., 1].to(F64) - shift).abs() <= b_shift).all())


@pytest.mark.gpu
def test_downsample_conv_deterministic_writes_only_its_view_and_pad11_is_unchanged():
    from lavie_b200 import _lib, ops
    NF, H, W, C = 2, 30, 42, 256
    x, w, b = _conv_inputs(NF, H, W, C, C, seed=7)
    a = ops.conv3x3(x, NF, H, W, w, stride=2, padding=(0, 1), bias=b)
    assert torch.equal(a, ops.conv3x3(x, NF, H, W, w, stride=2, padding=(0, 1), bias=b))
    M = a.shape[0]
    buf = torch.full((M + 2, C + 128), 7.0, dtype=torch.bfloat16, device=DEV)
    view = buf[1:M + 1, 64:64 + C]
    ops.conv3x3(x, NF, H, W, w, stride=2, padding=(0, 1), bias=b, out=view)
    assert torch.equal(view, a)
    mask = torch.ones_like(buf, dtype=torch.bool)
    mask[1:M + 1, 64:64 + C] = False
    assert bool((buf[mask] == 7.0).all()), "wrote outside the output view"
    # pad (1, 1) through the padded entry point is the existing conv, bit for bit
    for stride in (1, 2):
        new = ops.conv3x3(x, NF, H, W, w, stride=stride, bias=b)
        old = torch.empty_like(new)
        ep = ops._epilogue(b)
        ws = ops._workspace(x.device)
        assert _lib.load().lavie_conv3x3_bf16(x.data_ptr(), NF, H, W, C, stride, w.data_ptr(), old.data_ptr(), C, C,
                                              ctypes.byref(ep), 0, ws.data_ptr(), ws.numel(), ops._stream()) == 0
        assert torch.equal(new, old)


@pytest.mark.gpu
def test_downsample_conv_rejects_the_im2col_fallback_and_bad_padding():
    from lavie_b200 import _lib, ops
    x, w, _ = _conv_inputs(1, 8, 8, 128, 128, seed=1)
    with pytest.raises(ValueError, match="im2col"):
        ops.conv3x3(x, 1, 8, 8, w, stride=2, padding=(0, 1), force_im2col=True)
    x32 = torch.zeros(64, 32, dtype=torch.bfloat16, device=DEV)
    w32 = torch.zeros(32, 9 * 32, dtype=torch.bfloat16, device=DEV)
    with pytest.raises(ValueError, match="im2col"):
        ops.conv3x3(x32, 1, 8, 8, w32, stride=2, padding=(0, 1))
    out = torch.empty(64, 128, dtype=torch.bfloat16, device=DEV)
    lib = _lib.load()
    for pb, pa in ((2, 1), (1, -1)):
        assert lib.lavie_conv3x3_pad_bf16(x.data_ptr(), 1, 8, 8, 128, 1, pb, pa, w.data_ptr(), out.data_ptr(), 128, 128,
                                          None, 0, None, 0, ops._stream()) == -1
    assert b"padding" in lib.lavie_last_error()


# ------------------------------------------------------------------------------------------------ uint8 frames
def _frames(N, H, W, seed):
    f = torch.randint(0, 256, (N, H, W, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(seed))
    f[0, 0, 0] = 0
    f[-1, -1, -1] = 255
    return f


def _normalize_cpu(frames):
    """The reference's normalisation on the CPU, where torch divides with IEEE rounding: [N, 3, H, W] fp32."""
    return (frames.permute(0, 3, 1, 2).float() / 255 - 0.5) / 0.5


@pytest.mark.gpu
@pytest.mark.parametrize("N,H,W", [(2, 8, 8), (3, 17, 30), (1, 64, 96)])
def test_im2col_frames_matches_im2col_input_and_zero_borders(N, H, W):
    from lavie_b200 import _lib, ops
    from lavie_b200.vae_encode_ops import im2col_frames
    frames = _frames(N, H, W, seed=H * W)
    kpad = ops.conv_in_kpad(3)
    col = im2col_frames(frames.to(DEV), kpad)
    x = _normalize_cpu(frames)
    ref = torch.empty_like(col)
    xd = x.reshape(N, 3, 1, H, W).contiguous().to(DEV)
    assert _lib.load().lavie_im2col_input_bf16(xd.data_ptr(), None, N, 3, 1, H, W, kpad, ref.data_ptr(),
                                               ops._stream()) == 0
    assert torch.equal(col, ref)
    want = torch.zeros(N * H * W, kpad, dtype=torch.bfloat16)
    want[:, :27] = F.unfold(x, 3, padding=1).transpose(1, 2).reshape(N * H * W, 27).to(torch.bfloat16)
    assert torch.equal(col.cpu(), want)                 # K = c*9 + kh*3 + kw, zeros outside the image and beyond 27
    c = col.cpu().reshape(N, H, W, kpad)[..., :27].reshape(N, H, W, 3, 3, 3)
    assert c[:, 0, :, :, 0].abs().max() == 0 and c[:, -1, :, :, 2].abs().max() == 0
    assert c[:, :, 0, :, :, 0].abs().max() == 0 and c[:, :, -1, :, :, 2].abs().max() == 0


# ------------------------------------------------------------------------------------------------ posterior
def _moments(N, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    m = torch.randn(N, 8, h, w, generator=g)
    m[:, 4:] *= 12.0                                     # logvar spread wide enough to cross both clamp limits
    m[0, 4, 0, :4] = torch.tensor([-50.0, -30.0, 20.0, 45.0])
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("with_noise", [False, True])
def test_posterior_sample_vs_fp64(with_noise):
    from lavie_b200.vae_encode_ops import posterior_sample
    B, Fr, h, w = 2, 3, 5, 7
    m = _moments(B * Fr, h, w, seed=3)
    noise = torch.randn(B * Fr, 4, h, w, generator=torch.Generator().manual_seed(4)) if with_noise else None
    scale = 0.18215
    out = posterior_sample(m.to(DEV), B, Fr, scale, None if noise is None else noise.to(DEV)).cpu()
    mean, lv = m[:, :4].to(F64), m[:, 4:].to(F64)
    assert float(lv.min()) < -30 and float(lv.max()) > 20
    if noise is None:
        want = (m[:, :4] * scale).reshape(B, Fr, 4, h, w).permute(0, 2, 1, 3, 4)
        assert torch.equal(out, want)                    # the mode: one fp32 product per element
        return
    std = torch.exp(0.5 * lv.clamp(-30, 20))
    ref = scale * (mean + std * noise.to(F64))
    bnd = 2.0 ** -20 * scale * (mean.abs() + std * noise.abs().to(F64)) + 1e-30
    ref, bnd = (t.reshape(B, Fr, 4, h, w).permute(0, 2, 1, 3, 4) for t in (ref, bnd))
    assert bool(((out.to(F64) - ref).abs() <= bnd).all())


@pytest.mark.gpu
def test_posterior_layout_with_frame_ramps():
    """mean[n, c, p] = n + c / 8 + p / 2^14 (exact in fp32): out[b, c, f, p] must hold frame n = b * F + f."""
    from lavie_b200.vae_encode_ops import posterior_sample
    B, Fr, h, w = 3, 5, 4, 6
    n = torch.arange(B * Fr, dtype=torch.float32)[:, None, None]
    c = torch.arange(4, dtype=torch.float32)[None, :, None] / 8
    p = torch.arange(h * w, dtype=torch.float32)[None, None, :] / 2 ** 14
    m = torch.zeros(B * Fr, 8, h * w)
    m[:, :4] = n + c + p
    out = posterior_sample(m.reshape(B * Fr, 8, h, w).to(DEV), B, Fr, 1.0).cpu()
    assert out.shape == (B, 4, Fr, h, w)
    bi = torch.arange(B)[:, None, None, None, None]
    fi = torch.arange(Fr)[None, None, :, None, None]
    ci = torch.arange(4)[None, :, None, None, None]
    pi = torch.arange(h * w).reshape(1, 1, 1, h, w)
    assert torch.equal(out, (bi * Fr + fi).float() + ci.float() / 8 + pi.float() / 2 ** 14)


# ------------------------------------------------------------------------------------------------ encoder
@pytest.fixture(scope="module")
def enc():
    from lavie_b200.vae import VAEEncoder, vae_encoder_synthetic_state_dict
    sd = vae_encoder_synthetic_state_dict(seed=0)
    m = VAEEncoder()
    m.load_state_dict(sd, strict=True)
    return m.to(DEV).eval(), sd


@pytest.mark.gpu
@pytest.mark.parametrize("N,H,W", [(2, 64, 64), (3, 128, 192), (1, 320, 512), (2, 200, 320)])
def test_encode_vs_oracle(enc, N, H, W):
    """(2, 200, 320): a 25 x 40 latent, odd latent height, so the last downsample reads the one-sided pad row."""
    from oracle import vae_encoder_oracle as E
    m, sd = enc
    g = torch.Generator().manual_seed(H * W + N)
    x = torch.rand(N, 3, H, W, generator=g) * 2 - 1
    noise = torch.randn(N, 4, H // 8, W // 8, generator=g)
    mom = E.moments(sd, x)
    mean, logvar, _ = E.posterior(mom)
    dist = m.encode(x.to(DEV)).latent_dist
    assert dist.mean.shape == (N, 4, H // 8, W // 8) and dist.mean.dtype == torch.float32
    errs = {"mean": rel_l2(dist.mean.cpu(), mean), "logvar": rel_l2(dist.logvar.cpu(), logvar),
            "sample": rel_l2(dist.sample(noise=noise.to(DEV)).cpu(), E.sample(mom, noise))}
    print(f"encode {N}x{H}x{W}: " + ", ".join(f"{k} rel-L2 {v:.3e}" for k, v in errs.items()))
    assert all(v < ENC_TOL for v in errs.values()), errs
    assert torch.equal(dist.mode(), dist.mean)


@pytest.mark.gpu
def test_encode_video_is_encode_of_the_normalised_frames(enc):
    """Bit for bit: the uint8 path (normalisation inside the patch-row kernel, posterior into [B, 4, F, h, w]) equals
    encode() of the frames normalised on the CPU, sampled, scaled and rearranged; and it matches the oracle."""
    from oracle import vae_encoder_oracle as E
    m, sd = enc
    B, Fr, H, W = 2, 3, 64, 96
    frames = _frames(B * Fr, H, W, seed=11).reshape(B, Fr, H, W, 3)
    noise = torch.randn(B * Fr, 4, H // 8, W // 8, generator=torch.Generator().manual_seed(12))
    lat = m.encode_video(frames, noise=noise)
    assert lat.shape == (B, 4, Fr, H // 8, W // 8) and lat.is_cuda and lat.dtype == torch.float32
    x = _normalize_cpu(frames.reshape(B * Fr, H, W, 3))
    dist = m.encode(x.to(DEV)).latent_dist
    want = (dist.sample(noise=noise.to(DEV)) * 0.18215).reshape(B, Fr, 4, H // 8, W // 8).permute(0, 2, 1, 3, 4)
    assert torch.equal(lat, want)
    mode = m.encode_video(frames, sample=False)
    assert torch.equal(mode, (dist.mode() * 0.18215).reshape(B, Fr, 4, H // 8, W // 8).permute(0, 2, 1, 3, 4))
    ref = E.encode_video(sd, frames, noise)
    assert rel_l2(lat.cpu(), ref) < ENC_TOL
    assert rel_l2(mode.cpu(), E.encode_video(sd, frames)) < ENC_TOL


@pytest.mark.gpu
def test_encode_video_generator_draws(enc):
    m, _ = enc
    frames = _frames(2, 64, 64, seed=5).reshape(1, 2, 64, 64, 3)
    a = m.encode_video(frames, generator=torch.Generator().manual_seed(7))
    b = m.encode_video(frames, generator=torch.Generator().manual_seed(7))
    assert torch.equal(a, b)
    noise = torch.randn((2, 4, 8, 8), generator=torch.Generator().manual_seed(7))
    assert torch.equal(a, m.encode_video(frames, noise=noise))          # diffusers' randn_tensor on a CPU generator
    c = m.encode_video(frames, generator=torch.Generator(device=DEV).manual_seed(7))
    assert torch.equal(c, m.encode_video(frames, noise=torch.randn((2, 4, 8, 8), generator=torch.Generator(
        device=DEV).manual_seed(7), device=DEV)))
    assert not torch.equal(a, m.encode_video(frames, generator=torch.Generator().manual_seed(8)))


@pytest.mark.gpu
def test_encode_regrouping(enc):
    """Five frames with the launch bound lowered to two frames' worth: groups of 2, 2, 1 against one group of 5.  The
    per-frame work is the same, but the GroupNorm statistics chunking and the GEMM plans (split-K) follow the rows of each
    launch, so the fp32 summation order changes; a flipped bf16 rounding then propagates through 21 convolutions.  On a
    B200 the two runs differ by 8.6e-3 rel-L2 (not bit-identical), inside the bf16 spread ENC_TOL is set from."""
    m, _ = enc
    frames = _frames(5, 64, 64, seed=9).reshape(1, 5, 64, 64, 3)
    fe = m.frame_elements(64, 64)
    assert m.frames_per_group(64, 64, 2 * fe + 1) == 2
    one = m.encode_video(frames, sample=False)
    grouped = m.encode_video(frames, sample=False, max_launch_elements=2 * fe + 1)
    assert grouped.shape == one.shape == (1, 4, 5, 8, 8)
    for f in range(5):
        assert rel_l2(grouped[:, :, f].cpu(), one[:, :, f].cpu()) < ENC_TOL, f
    print(f"regrouped encode: bit-identical = {torch.equal(grouped, one)}, "
          f"rel-L2 = {rel_l2(grouped.cpu(), one.cpu()):.3e}")


@pytest.mark.gpu
def test_full_autoencoder_checkpoint_loads_into_encoder_and_decoder(enc):
    """One AutoencoderKL dict (encoder, decoder, quant_conv, post_quant_conv; post-0.16 attention names, 1x1-conv shaped
    attention weights) loads strictly into both modules."""
    from lavie_b200.vae import VAEDecoder, VAEEncoder, load_vae_state_dict, vae_synthetic_state_dict
    m, sd = enc
    dsd = vae_synthetic_state_dict(seed=0)
    full = dict(sd)
    full.update(dsd)
    for side in ("encoder", "decoder"):
        a = f"{side}.mid_block.attentions.0"
        for new, old in (("to_q", "query"), ("to_k", "key"), ("to_v", "value"), ("to_out.0", "proj_attn")):
            full[f"{a}.{new}.weight"] = full.pop(f"{a}.{old}.weight").reshape(512, 512, 1, 1)
            full[f"{a}.{new}.bias"] = full.pop(f"{a}.{old}.bias")
    e2, d2 = VAEEncoder(), VAEDecoder()
    load_vae_state_dict(e2, full, strict=True)
    load_vae_state_dict(d2, full, strict=True)
    e2, d2 = e2.to(DEV).eval(), d2.to(DEV).eval()
    x = torch.rand(1, 3, 64, 64, generator=torch.Generator().manual_seed(2)) * 2 - 1
    assert torch.equal(e2.encode(x.to(DEV)).latent_dist.parameters, m.encode(x.to(DEV)).latent_dist.parameters)
    d1 = VAEDecoder()
    d1.load_state_dict(dsd, strict=True)
    z = torch.randn(1, 4, 8, 8, generator=torch.Generator().manual_seed(3)).to(DEV)
    assert torch.equal(d2.decode(z).sample, d1.to(DEV).eval().decode(z).sample)


# ------------------------------------------------------------------------------------------------ CPU
def test_encoder_param_spec_and_oracle_keys():
    from lavie_b200.vae import VAEEncoder, vae_encoder_param_spec, vae_encoder_synthetic_state_dict
    from oracle import vae_encoder_oracle as E
    spec = vae_encoder_param_spec()
    assert len(spec) == 108
    e = "encoder."
    assert spec[e + "conv_in.weight"] == (128, 3, 3, 3)
    assert spec[e + "down_blocks.0.resnets.1.conv2.weight"] == (128, 128, 3, 3)
    assert spec[e + "down_blocks.0.downsamplers.0.conv.weight"] == (128, 128, 3, 3)
    assert spec[e + "down_blocks.1.resnets.0.conv_shortcut.weight"] == (256, 128, 1, 1)
    assert spec[e + "down_blocks.2.resnets.0.conv1.weight"] == (512, 256, 3, 3)
    assert spec[e + "down_blocks.2.downsamplers.0.conv.weight"] == (512, 512, 3, 3)
    assert e + "down_blocks.3.downsamplers.0.conv.weight" not in spec
    assert e + "down_blocks.3.resnets.0.conv_shortcut.weight" not in spec
    assert spec[e + "mid_block.attentions.0.query.weight"] == (512, 512)
    assert spec[e + "conv_norm_out.weight"] == (512,) and spec[e + "conv_out.weight"] == (8, 512, 3, 3)
    assert spec["quant_conv.weight"] == (8, 8, 1, 1)
    assert all(k.startswith((e, "quant_conv.")) for k in spec)
    m = VAEEncoder()
    assert set(m.state_dict()) == set(spec) and m.config.scaling_factor == 0.18215
    assert E.BLOCK_OUT == m.config.block_out_channels and E.SCALING == m.config.scaling_factor
    # the oracle reads exactly the spec's keys: it runs on them alone, and fails without any one of them
    sd = vae_encoder_synthetic_state_dict(seed=1)
    assert list(sd) == list(spec)
    x = torch.rand(1, 3, 8, 8, generator=torch.Generator().manual_seed(0)) * 2 - 1
    assert E.moments(sd, x).shape == (1, 8, 1, 1)
    for k in spec:
        part = {kk: v for kk, v in sd.items() if kk != k}
        with pytest.raises((KeyError, RuntimeError)):             # a missing conv_shortcut shows as a shape mismatch
            E.moments(part, x)


def test_oracle_encode_video_shape():
    from lavie_b200.vae import vae_encoder_synthetic_state_dict
    from oracle import vae_encoder_oracle as E
    sd = vae_encoder_synthetic_state_dict(seed=2)
    frames = _frames(2 * 3, 16, 24, seed=1).reshape(2, 3, 16, 24, 3)
    assert E.encode_video(sd, frames).shape == (2, 4, 3, 2, 3)
    assert E.encode_video(sd, frames, torch.randn(6, 4, 2, 3)).shape == (2, 4, 3, 2, 3)


def test_conv_output_size_formula():
    from lavie_b200 import ops
    for n in range(1, 41):
        for stride in (1, 2):
            assert ops.conv3x3_out_size(n, stride) == (n - 1) // stride + 1          # pad (1, 1): the existing formula
            for pad in ((0, 1), (1, 0), (0, 0), (1, 1)):
                got = ops.conv3x3_out_size(n, stride, pad)
                if n + pad[0] + pad[1] < 3:
                    assert got == 0
                    continue
                y = F.conv2d(F.pad(torch.zeros(1, 1, n, 1), (0, 0) + pad), torch.zeros(1, 1, 3, 1), stride=(stride, 1))
                assert got == y.shape[2] == (n + pad[0] + pad[1] - 3) // stride + 1, (n, stride, pad)


def test_encoder_rejects_bad_arguments():
    """Rejected before any launch; a valid request on a CPU module fails loudly instead of falling back."""
    from lavie_b200.vae import VAEEncoder
    m = VAEEncoder()
    u8 = lambda *s: torch.zeros(*s, dtype=torch.uint8)
    for bad in (torch.zeros(1, 3, 60, 64), torch.zeros(1, 3, 64, 68), torch.zeros(1, 4, 64, 64), torch.zeros(3, 64, 64),
                torch.zeros(1, 3, 24, 24),                     # 3 x 3 latent: 9 tokens, not a multiple of 8
                torch.zeros(1, 3, 512, 576),                   # 64 x 72 latent: 4608 tokens > 4096
                u8(1, 3, 64, 64)):
        with pytest.raises(ValueError):
            m.encode(bad)
    for bad in (u8(1, 2, 64, 64, 4), u8(1, 2, 60, 64, 3), torch.zeros(1, 2, 64, 64, 3), u8(2, 64, 64, 3)):
        with pytest.raises(ValueError):
            m.encode_video(bad)
    with pytest.raises(ValueError):
        m.encode_video(u8(1, 2, 64, 64, 3), noise=torch.zeros(2, 4, 8, 7))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA"):
            m.encode(torch.zeros(1, 3, 64, 64))
        with pytest.raises(RuntimeError, match="CUDA"):
            m.encode_video(u8(1, 2, 64, 64, 3))


def test_encoder_frame_grouping_from_geometry():
    """At 320 x 512 the largest map is conv_in's 128-channel output: 2.1e7 elements per frame, 102 frames per group, so a
    61-frame video is one group."""
    from lavie_b200.vae import VAEEncoder
    m = VAEEncoder()
    assert m.frame_elements(320, 512) == 128 * 320 * 512
    assert m.frames_per_group(320, 512) == 102
    with pytest.raises(ValueError):
        m.frames_per_group(320, 512, max_launch_elements=10 ** 7)


def test_encoder_abi_declared():
    from lavie_b200 import _lib
    text = open(os.path.join(ROOT, "include", "lavie_b200.h")).read()
    for name in ("lavie_conv3x3_pad_bf16", "lavie_conv3x3_out_size", "lavie_im2col_frames_bf16",
                 "lavie_posterior_sample_f32"):
        assert re.search(rf"\bint {name}\s*\(", text), name
        assert name in _lib.SIGNATURES, name
    assert _lib.load().lavie_abi_version() == 1
