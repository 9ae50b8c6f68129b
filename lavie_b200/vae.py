"""VAE decoder on the B200 path (SURVEY.md 8f row N4): ``vae.decode(latents).sample`` as the pipelines call it once per
video (base/pipelines/pipeline_videogen.py:422-429), frame by frame in one batch.

The reference takes ``AutoencoderKL`` from diffusers 0.16 (un-vendored third party; in-tree mirror of the wrapper at
vsr/models/autoencoder_kl.py:179-192).  This module keeps the decode-side ``state_dict`` layout of that class
(``post_quant_conv.*``, ``decoder.*``; encoder-side keys of a full checkpoint are ignored by ``load_vae_state_dict``) and
runs the published Stable-Diffusion VAE decoder as C-ABI launches that reuse the denoiser's kernels: implicit-GEMM 3x3
convs on tcgen05, per-frame GroupNorm + SiLU, nearest-x2 upsample; the single-head 2560-token mid-block attention is two
GEMMs around a row-softmax kernel (Q K^T per frame, P V against V^T produced directly by a GEMM).  bf16 activations, fp32
accumulation.  No CPU fallback.

The same class runs the x4-upscaler VAE that the VSR pipeline decodes with (``VAEDecoder.x4_upscaler()``, published
``vae/config.json`` of the x4 upscaler: block_out_channels (128, 256, 512), layers_per_block 2, 32 groups, scaling
factor 0.08333, two upsamplers, so the output is x4).  Its mid-block attention sees h * w tokens per frame at the
latent resolution (163 840 at 320x512), far beyond a materialised score matrix: it runs the fused single-head d = 512
kernel of ``vae_attention`` instead.  Frames are decoded in groups sized from the geometry so that no tensor of any
launch passes 2^31 elements.

``VAEEncoder`` runs the encode side of the same Stable-Diffusion VAE (``encoder.*``, ``quant_conv.*``): the video
frames the interpolation stage conditions on become latents (interpolation/sample.py, ``auto_inpainting_copy_no_mask``:
``vae.encode(frames).latent_dist.sample().mul_(0.18215)``).  It shares the decoder's ResnetBlock2D, mid-block attention
and their weight packing; Downsample2D is the implicit-GEMM conv with one-sided (0, 1) padding, conv_in reads uint8
frames directly, and the diagonal-Gaussian posterior is sampled straight into the [B, 4, F, h, w] latent layout."""
from __future__ import annotations

import math
from collections import OrderedDict
from types import SimpleNamespace
from typing import Dict, Optional, Tuple

import torch
from torch import nn

from . import ops
from .packing import pack_conv1x1, pack_conv3x3, pack_upsample_conv3x3
from .synthetic import _gen
from .vae_attention import attention_wide
from .vae_encode_ops import im2col_frames, posterior_sample

BF16 = torch.bfloat16
F32 = torch.float32
UP_CHANNELS = (512, 512, 256, 128)          # reversed block_out_channels of the SD VAE
SCALING = 0.18215                            # pipeline_videogen.py:424
SD_BLOCK_OUT = (128, 256, 512, 512)
# stabilityai/stable-diffusion-x4-upscaler vae/config.json
X4_BLOCK_OUT = (128, 256, 512)
X4_SCALING = 0.08333
MAX_LAUNCH_ELEMENTS = 2 ** 31 - 1           # largest tensor one launch may address with 32-bit element indices


def _conv_spec(spec, p, co, ci, k):
    spec[f"{p}.weight"] = (co, ci, k, k)
    spec[f"{p}.bias"] = (co,)


def _norm_spec(spec, p, c):
    spec[f"{p}.weight"] = (c,)
    spec[f"{p}.bias"] = (c,)


def _resnet_spec(spec, p, ci, co):
    _norm_spec(spec, f"{p}.norm1", ci)
    _conv_spec(spec, f"{p}.conv1", co, ci, 3)
    _norm_spec(spec, f"{p}.norm2", co)
    _conv_spec(spec, f"{p}.conv2", co, co, 3)
    if ci != co:
        _conv_spec(spec, f"{p}.conv_shortcut", co, ci, 1)


def _mid_block_spec(spec, m, c):
    """UNetMidBlock2D: ResnetBlock2D, single-head AttentionBlock (0.16 names), ResnetBlock2D."""
    _resnet_spec(spec, f"{m}.resnets.0", c, c)
    a = f"{m}.attentions.0"
    _norm_spec(spec, f"{a}.group_norm", c)
    for n in ("query", "key", "value", "proj_attn"):
        spec[f"{a}.{n}.weight"] = (c, c)
        spec[f"{a}.{n}.bias"] = (c,)
    _resnet_spec(spec, f"{m}.resnets.1", c, c)


def vae_decoder_param_spec(block_out_channels=SD_BLOCK_OUT, layers_per_block: int = 2
                           ) -> "OrderedDict[str, Tuple[int, ...]]":
    """Decode-side parameters of diffusers' AutoencoderKL (0.16 names).  Default: the Stable Diffusion VAE."""
    up_channels = tuple(reversed(block_out_channels))
    top = up_channels[0]
    spec: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
    _conv_spec(spec, "post_quant_conv", 4, 4, 1)
    _conv_spec(spec, "decoder.conv_in", top, 4, 3)
    _mid_block_spec(spec, "decoder.mid_block", top)
    prev = top
    for i, c in enumerate(up_channels):
        for j in range(layers_per_block + 1):
            _resnet_spec(spec, f"decoder.up_blocks.{i}.resnets.{j}", prev if j == 0 else c, c)
        if i != len(up_channels) - 1:
            _conv_spec(spec, f"decoder.up_blocks.{i}.upsamplers.0.conv", c, c, 3)
        prev = c
    _norm_spec(spec, "decoder.conv_norm_out", up_channels[-1])
    _conv_spec(spec, "decoder.conv_out", 3, up_channels[-1], 3)
    return spec


def vae_encoder_param_spec(block_out_channels=SD_BLOCK_OUT, layers_per_block: int = 2
                           ) -> "OrderedDict[str, Tuple[int, ...]]":
    """Encode-side parameters of diffusers' AutoencoderKL (0.16 names): Encoder (conv_in, DownEncoderBlock2D with a
    Downsample2D conv on every block but the last, mid block, conv_norm_out, conv_out to 2 x 4 moment channels) and
    quant_conv.  Default: the Stable Diffusion VAE (108 keys)."""
    spec: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
    _conv_spec(spec, "encoder.conv_in", block_out_channels[0], 3, 3)
    prev = block_out_channels[0]
    for i, c in enumerate(block_out_channels):
        for j in range(layers_per_block):
            _resnet_spec(spec, f"encoder.down_blocks.{i}.resnets.{j}", prev if j == 0 else c, c)
        if i != len(block_out_channels) - 1:
            _conv_spec(spec, f"encoder.down_blocks.{i}.downsamplers.0.conv", c, c, 3)
        prev = c
    top = block_out_channels[-1]
    _mid_block_spec(spec, "encoder.mid_block", top)
    _norm_spec(spec, "encoder.conv_norm_out", top)
    _conv_spec(spec, "encoder.conv_out", 8, top, 3)
    _conv_spec(spec, "quant_conv", 8, 8, 1)
    return spec


def _synthetic(spec, seed: int, tag: str):
    sd = OrderedDict()
    for key, shape in spec.items():
        g = _gen(seed, tag + key)
        if ".norm" in key or "group_norm" in key or "conv_norm_out" in key:
            t = 0.1 * torch.randn(shape, generator=g) + (1.0 if key.endswith("weight") else 0.0)
        else:
            wshape = spec[key[: -len("bias")] + "weight"] if key.endswith("bias") else shape
            t = (torch.rand(shape, generator=g) * 2.0 - 1.0) / math.sqrt(math.prod(wshape[1:]))
        sd[key] = t
    return sd


def vae_synthetic_state_dict(seed: int = 0, block_out_channels=SD_BLOCK_OUT):
    """Seeded decoder weights; ``block_out_channels=X4_BLOCK_OUT`` draws the x4-upscaler layout."""
    tag = "vae:" if tuple(block_out_channels) == SD_BLOCK_OUT else f"vae{tuple(block_out_channels)}:"
    return _synthetic(vae_decoder_param_spec(block_out_channels), seed, tag)


def vae_encoder_synthetic_state_dict(seed: int = 0):
    """Seeded weights of the Stable Diffusion VAE's encoder side (``VAEEncoder``); together with
    ``vae_synthetic_state_dict`` a full AutoencoderKL state dict."""
    return _synthetic(vae_encoder_param_spec(), seed, "vae-encoder:")


# diffusers renamed the attention block's parameters after 0.16; accept both spellings
_ATTN_ALIASES = {"to_q": "query", "to_k": "key", "to_v": "value", "to_out.0": "proj_attn"}


def load_vae_state_dict(module: "_VAEModule", sd, strict: bool = True):
    """Load the side of an ``AutoencoderKL`` checkpoint that ``module`` runs: a ``VAEDecoder`` takes the decoder and
    post_quant_conv keys, a ``VAEEncoder`` the encoder and quant_conv keys; the other side's keys are dropped, newer
    attention parameter names are mapped to the 0.16 ones."""
    out = {}
    for k, v in sd.items():
        if not k.startswith(module.STATE_PREFIXES):
            continue
        for new, old in _ATTN_ALIASES.items():
            k = k.replace(f"attentions.0.{new}.", f"attentions.0.{old}.")
        if k.endswith("weight") and v.dim() == 4 and ".attentions." in k:
            v = v.reshape(v.shape[0], v.shape[1])
        out[k] = v
    return module.load_state_dict(out, strict=strict)


def _pack_resnet(sd, p, f32, b16):
    r = {"g1": f32(f"{p}.norm1.weight"), "b1": f32(f"{p}.norm1.bias"),
         "w1": b16(pack_conv3x3(sd[f"{p}.conv1.weight"], dtype=None)), "cb1": f32(f"{p}.conv1.bias"),
         "g2": f32(f"{p}.norm2.weight"), "b2": f32(f"{p}.norm2.bias"),
         "w2": b16(pack_conv3x3(sd[f"{p}.conv2.weight"], dtype=None)), "cb2": f32(f"{p}.conv2.bias")}
    if f"{p}.conv_shortcut.weight" in sd:
        r["wsc"] = b16(pack_conv1x1(sd[f"{p}.conv_shortcut.weight"], dtype=None))
        r["bsc"] = f32(f"{p}.conv_shortcut.bias")
    return r


def _pack_attention(sd, a, C, wide, f32, b16, dev):
    s = C ** -0.5                                   # folded into the query projection: scores leave the GEMM scaled
    t = {"g": f32(f"{a}.group_norm.weight"), "b": f32(f"{a}.group_norm.bias"),
         "w_q": b16(sd[f"{a}.query.weight"].float() * s),
         "b_q": (sd[f"{a}.query.bias"].float() * s).to(dev).contiguous(),
         "w_k": b16(sd[f"{a}.key.weight"]), "b_k": f32(f"{a}.key.bias"),
         "w_v": b16(sd[f"{a}.value.weight"]), "b_v": f32(f"{a}.value.bias"),
         "w_o": b16(sd[f"{a}.proj_attn.weight"]), "b_o": f32(f"{a}.proj_attn.bias")}
    if wide:                                        # q, k, v from one GEMM: [rows, 3C], read as strided views
        t["w_qkv"] = torch.cat([t.pop("w_q"), t.pop("w_k"), t.pop("w_v")]).contiguous()
        t["b_qkv"] = torch.cat([t.pop("b_q"), t.pop("b_k"), t.pop("b_v")]).contiguous()
    return t


def _pack_conv_out(w, b, dev):
    """conv_out's few filters zero-padded to the CONV_OUT_PAD rows of ops.conv_out_tc."""
    wp = torch.zeros((ops.CONV_OUT_PAD, 9 * w.shape[1]), dtype=F32)
    wp[:w.shape[0]] = pack_conv3x3(w.float().cpu(), dtype=None)
    bp = torch.zeros(ops.CONV_OUT_PAD, dtype=F32)
    bp[:w.shape[0]] = b.float().cpu()
    return wp.to(device=dev, dtype=BF16).contiguous(), bp.to(dev)


class _VAEModule(nn.Module):
    """What the VAE decoder and encoder share: parameters registered from a spec (``state_dict`` = diffusers'
    AutoencoderKL names), lazy packing on CUDA, the ResnetBlock2D and single-head mid-block attention launches, and the
    frame grouping that keeps every launch under ``max_launch_elements``."""

    STATE_PREFIXES: Tuple[str, ...] = ()
    _ANCHOR = ""                                    # module whose weight tells the device / dtype
    _GEOMETRY = ""                                  # what the h x w of frames_per_group measures

    def __init__(self, spec):
        super().__init__()
        for key, shape in spec.items():
            prefix, leaf = key.rsplit(".", 1)
            cur = self
            for p in prefix.split("."):
                nxt = cur._modules.get(p)
                if nxt is None:
                    nxt = nn.Module()
                    cur.add_module(p, nxt)
                cur = nxt
            cur.register_parameter(leaf, nn.Parameter(torch.empty(shape), requires_grad=False))
        self._packed = None
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._invalidate())

    def _invalidate(self):
        self._packed = None

    def _apply(self, fn, *a, **kw):
        out = super()._apply(fn, *a, **kw)
        self._invalidate()
        return out

    @property
    def device(self):
        return getattr(self, self._ANCHOR).weight.device

    @property
    def dtype(self):
        return getattr(self, self._ANCHOR).weight.dtype

    def _state_for_packing(self):
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError(f"lavie_b200.{type(self).__name__} runs on CUDA (sm_100a) only; move it with .to('cuda')")
        sd = {k: v.detach() for k, v in self.state_dict().items()}
        f32 = lambda k: sd[k].to(device=dev, dtype=F32).contiguous()
        b16 = lambda t: t.to(device=dev, dtype=BF16).contiguous()
        return dev, sd, f32, b16

    # ------------------------------------------------------------------ blocks
    def _resnet(self, p, x, N, H, W):
        r = self._packed[p]
        h = ops.groupnorm(x, N, H * W, r["g1"], r["b1"], 1e-6, silu=True)
        h = ops.conv3x3(h, N, H, W, r["w1"], bias=r["cb1"], stats=True)
        h = ops.groupnorm(h, N, H * W, r["g2"], r["b2"], 1e-6, silu=True)
        sc = ops.gemm(x, r["wsc"], bias=r["bsc"]) if "wsc" in r else x
        return ops.conv3x3(h, N, H, W, r["w2"], bias=r["cb2"], residual=sc, stats=True)

    def _attention(self, a, x, N, HW, wide):
        """diffusers 0.16 AttentionBlock (one head of C channels) per frame."""
        t = self._packed[a]
        C = x.shape[1]
        n = ops.groupnorm(x, N, HW, t["g"], t["b"], 1e-6, silu=False)
        if wide:
            qkv = ops.gemm(n, t["w_qkv"], bias=t["b_qkv"])                # [rows, 3C]; q already scaled by C^-1/2
            o = attention_wide(qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:], N, HW)
            return ops.gemm(o, t["w_o"], bias=t["b_o"], residual=x, stats=True)
        if HW % 8:
            raise ValueError("the VAE mid-block attention needs h * w to be a multiple of 8")
        q = ops.gemm(n, t["w_q"], bias=t["b_q"])                          # already scaled by C^-1/2
        k = ops.gemm(n, t["w_k"], bias=t["b_k"])
        o = torch.empty((N * HW, C), dtype=BF16, device=x.device)
        for f in range(N):
            rows = slice(f * HW, (f + 1) * HW)
            s = ops.gemm(q[rows], k[rows])                                # scores [HW, HW] = q k^T (k rows are the "weights")
            ops.softmax_rows_(s, 1.0)
            vt = ops.gemm(t["w_v"], n[rows])                              # V^T [C, HW] = Wv n^T, no transpose pass
            # P V + b_v: rows of P sum to one, so the value bias moves behind the product
            ops.gemm(s, vt, bias=t["b_v"], out=o[rows])
        return ops.gemm(o, t["w_o"], bias=t["b_o"], residual=x, stats=True)

    def frame_elements(self, h: int, w: int) -> int:
        raise NotImplementedError

    def frames_per_group(self, h: int, w: int, max_launch_elements: int = MAX_LAUNCH_ELEMENTS) -> int:
        per_frame = self.frame_elements(h, w)
        if per_frame > max_launch_elements:
            raise ValueError(f"one frame of a {h}x{w} {self._GEOMETRY} needs {per_frame} elements in one launch "
                             f"(limit {max_launch_elements}); {self._VERB} it in tiles")
        return max_launch_elements // per_frame


class VAEDecoder(_VAEModule):
    """``decode(z).sample`` of an AutoencoderKL decoder + the pipelines' ``decode_latents``.  No arguments: the Stable
    Diffusion VAE (x8); ``VAEDecoder.x4_upscaler()``: the x4-upscaler VAE of the VSR pipeline."""

    STATE_PREFIXES = ("decoder.", "post_quant_conv.")
    _ANCHOR = "post_quant_conv"
    _GEOMETRY, _VERB = "latent", "decode"

    def __init__(self, block_out_channels=SD_BLOCK_OUT, scaling_factor: float = SCALING, layers_per_block: int = 2):
        block_out_channels = tuple(int(c) for c in block_out_channels)
        # the SD VAE keeps its GEMM + row-softmax attention (2560 tokens at its 40x64 latent); every other configuration
        # runs the fused wide kernel, which has no token limit
        wide_attention = block_out_channels != SD_BLOCK_OUT
        if wide_attention and block_out_channels[-1] != 512:
            raise ValueError("the fused mid-block attention needs block_out_channels[-1] == 512")
        super().__init__(vae_decoder_param_spec(block_out_channels, layers_per_block))
        self.config = SimpleNamespace(scaling_factor=scaling_factor, latent_channels=4,
                                      block_out_channels=block_out_channels, layers_per_block=layers_per_block,
                                      norm_num_groups=32)
        self.up_channels = tuple(reversed(block_out_channels))
        self.upscale = 2 ** (len(block_out_channels) - 1)
        self.wide_attention = wide_attention

    @classmethod
    def x4_upscaler(cls) -> "VAEDecoder":
        """The VAE of the x4 upscaler (the VSR pipeline's decoder): [N,4,h,w] -> [N,3,4h,4w]."""
        return cls(X4_BLOCK_OUT, X4_SCALING)

    def _pack(self):
        dev, sd, f32, b16 = self._state_for_packing()
        P: Dict[str, object] = {}
        for key in sd:
            if key.endswith(".conv1.weight"):
                p = key[: -len(".conv1.weight")]
                P[p] = _pack_resnet(sd, p, f32, b16)
            if key.endswith(".upsamplers.0.conv.weight"):
                p = key[: -len(".weight")]
                P[p] = (b16(pack_conv3x3(sd[key], dtype=None)), f32(f"{p}.bias"), pack_upsample_conv3x3(sd[key]).to(dev))
        a = "decoder.mid_block.attentions.0"
        P[a] = _pack_attention(sd, a, self.up_channels[0], self.wide_attention, f32, b16, dev)
        P["pq"] = (f32("post_quant_conv.weight").reshape(4, 4).contiguous(), f32("post_quant_conv.bias"))
        P["conv_in"] = (f32("decoder.conv_in.weight"), f32("decoder.conv_in.bias"))
        P["conv_out"] = _pack_conv_out(sd["decoder.conv_out.weight"], sd["decoder.conv_out.bias"], dev)
        P["norm_out"] = (f32("decoder.conv_norm_out.weight"), f32("decoder.conv_norm_out.bias"))
        self._packed = P
        return P

    def frame_elements(self, h: int, w: int) -> int:
        """Largest tensor, in elements per frame, that any launch of a decode at an h x w latent touches: the mid-block
        q/k/v rows at the latent resolution, and every level's maps at the channel count they enter and leave with
        (an upsampled map keeps the channels of the level below it)."""
        top = self.up_channels[0]
        most = 3 * top * h * w
        prev, H, W = top, h, w
        for i, c in enumerate(self.up_channels):
            most = max(most, max(prev, c) * H * W)
            if i != len(self.up_channels) - 1:
                H, W = 2 * H, 2 * W
                most = max(most, c * H * W)
            prev = c
        return max(most, ops.CONV_OUT_PAD * H * W)

    def _decode_group(self, zin, scale, as_uint8):
        P = self._packed
        N, _, h, w = zin.shape
        zq = ops.pointwise_conv_nchw(zin, P["pq"][0], P["pq"][1], scale)
        x = ops.conv_in(zq.reshape(N, 4, 1, h, w), P["conv_in"][0], P["conv_in"][1])
        H, W = h, w
        x = self._resnet("decoder.mid_block.resnets.0", x, N, H, W)
        x = self._attention("decoder.mid_block.attentions.0", x, N, H * W, self.wide_attention)
        x = self._resnet("decoder.mid_block.resnets.1", x, N, H, W)
        levels = len(self.up_channels)
        for i in range(levels):
            for j in range(self.config.layers_per_block + 1):
                x = self._resnet(f"decoder.up_blocks.{i}.resnets.{j}", x, N, H, W)
            if i != levels - 1:
                wu, bu, w4 = P[f"decoder.up_blocks.{i}.upsamplers.0.conv"]
                if ops.upsample_conv3x3_supported(H, W, x.shape[1]):          # Upsample2D without the 4x copy
                    x = ops.upsample_conv3x3(x, N, H, W, w4, bias=bu, stats=True)
                    H, W = 2 * H, 2 * W
                else:
                    x = ops.upsample_nearest2x(x, N, H, W)
                    H, W = 2 * H, 2 * W
                    x = ops.conv3x3(x, N, H, W, wu, bias=bu, stats=True)
        ss = ops.groupnorm_scale_shift(x, N, H * W, P["norm_out"][0], P["norm_out"][1], 1e-6)
        if as_uint8:
            hact = ops.groupnorm_apply(x, ss, N, H * W, True)
            y = ops.conv3x3(hact, N, H, W, P["conv_out"][0], bias=P["conv_out"][1], block_n=64, algo_n=3)
            return ops.image_to_uint8(y).reshape(N, H, W, 3)
        return ops.conv_out_tc(x, ss, N, 1, H, W, P["conv_out"][0], P["conv_out"][1], 3).reshape(N, 3, H, W)

    @torch.no_grad()
    def decode(self, z: torch.Tensor, return_dict: bool = True, scale: float = 1.0, as_uint8: bool = False,
               max_launch_elements: int = MAX_LAUNCH_ELEMENTS):
        """AutoencoderKL.decode (mirror vsr/models/autoencoder_kl.py:179-198): z [N,4,h,w] -> ``.sample`` [N,3,sh,sw] in
        z's dtype, s = 8 (SD VAE) or 4 (x4 upscaler).  ``scale`` multiplies z first (decode_latents' 1/scaling_factor);
        ``as_uint8`` returns the pipelines' uint8 frames [N, sh, sw, 3] instead.  Frames run in groups of at most
        ``frames_per_group(h, w, max_launch_elements)``; lowering the bound only regroups the same per-frame work."""
        if z.dim() != 4 or z.shape[1] != 4:
            raise ValueError(f"z must be [N,4,h,w], got {tuple(z.shape)}")
        if self._packed is None:
            self._pack()
        dev = self.device
        N, _, h, w = z.shape
        zin = z.to(device=dev, dtype=F32).contiguous()
        G = self.frames_per_group(h, w, max_launch_elements)
        if N <= G:
            out = self._decode_group(zin, scale, as_uint8)
        else:
            out = torch.cat([self._decode_group(zin[a:a + G], scale, as_uint8) for a in range(0, N, G)])
        if as_uint8:
            return out
        out = out.to(z.dtype) if z.dtype != F32 else out
        if not return_dict:
            return (out,)
        return SimpleNamespace(sample=out)

    @torch.no_grad()
    def decode_latents(self, latents: torch.Tensor) -> torch.Tensor:
        """The pipelines' decode_latents: [B,4,F,h,w] -> uint8 [B,F,sh,sw,3] on the host, with the 1/scaling_factor
        scaling and the uint8 conversion inside the kernels.  SD VAE: VideoGenPipeline.decode_latents
        (base/pipelines/pipeline_videogen.py:422-429); x4 upscaler: the VSR pipeline's decode
        (vsr/models/pipeline_stable_diffusion_upscale_video_3d.py:741-771)."""
        B, C, Fr, h, w = latents.shape
        z = latents.permute(0, 2, 1, 3, 4).reshape(B * Fr, C, h, w)
        video = self.decode(z, scale=1.0 / self.config.scaling_factor, as_uint8=True)
        s = self.upscale
        return video.reshape(B, Fr, s * h, s * w, 3).cpu().contiguous()


def _randn(shape, generator, device) -> torch.Tensor:
    """diffusers' randn_tensor for one generator: draw on the generator's device (a CPU generator draws on the CPU),
    then move to ``device``."""
    rand_device = device
    if generator is not None:
        if generator.device.type != device.type:
            if generator.device.type != "cpu":
                raise ValueError(f"cannot draw {device.type} noise from a {generator.device.type} generator")
            rand_device = torch.device("cpu")
    return torch.randn(shape, generator=generator, device=rand_device, dtype=F32).to(device)


def _noise_like(shape, generator, noise, device) -> torch.Tensor:
    if noise is None:
        return _randn(shape, generator, device)
    if tuple(noise.shape) != tuple(shape):
        raise ValueError(f"noise must be {tuple(shape)}, got {tuple(noise.shape)}")
    return noise.to(device=device, dtype=F32).contiguous()


class DiagonalGaussianDistribution:
    """The posterior ``AutoencoderKL.encode`` returns as ``.latent_dist``: ``parameters`` = the quant_conv moments fp32
    [N, 8, h, w] (mean | logvar) on the device.  ``sample`` runs the posterior kernel; ``logvar`` (clamped to [-30, 20]),
    ``std`` and ``var`` are derived on access for inspection."""

    def __init__(self, parameters: torch.Tensor):
        self.parameters = parameters
        self.mean = parameters[:, :4]

    @property
    def logvar(self) -> torch.Tensor:
        return torch.clamp(self.parameters[:, 4:], -30.0, 20.0)

    @property
    def std(self) -> torch.Tensor:
        return torch.exp(0.5 * self.logvar)

    @property
    def var(self) -> torch.Tensor:
        return torch.exp(self.logvar)

    def sample(self, generator: Optional[torch.Generator] = None, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        """mean + std * noise, fp32 [N, 4, h, w]; noise is drawn like diffusers' randn_tensor(mean.shape, generator)
        unless given."""
        N, _, h, w = self.parameters.shape
        eps = _noise_like((N, 4, h, w), generator, noise, self.parameters.device)
        return posterior_sample(self.parameters, N, 1, 1.0, eps).reshape(N, 4, h, w)

    def mode(self) -> torch.Tensor:
        return self.mean


class VAEEncoder(_VAEModule):
    """``encode(x).latent_dist`` of the Stable Diffusion AutoencoderKL's encoder, and ``encode_video``: uint8 frames
    [B, F, H, W, 3] (what ``VAEDecoder.decode_latents`` returns) -> scaled latents [B, 4, F, H/8, W/8], the
    interpolation stage's ``x_start`` (interpolation/sample.py: ``vae.encode(frames).latent_dist.sample().mul_(0.18215)``).

    Launches: conv_in on the tensor cores (the uint8 frames are normalised inside the patch-row kernel), four
    DownEncoderBlock2D (two ResnetBlock2D each; Downsample2D = F.pad(x, (0, 1, 0, 1)) + stride-2 conv as one
    implicit-GEMM conv with one-sided padding), the mid block (shared with ``VAEDecoder``), GroupNorm + SiLU + conv_out to
    8 moment channels on the tensor cores, quant_conv (1x1, fp32), and the posterior sample."""

    STATE_PREFIXES = ("encoder.", "quant_conv.")
    _ANCHOR = "quant_conv"
    _GEOMETRY, _VERB = "image", "encode"

    def __init__(self):
        super().__init__(vae_encoder_param_spec(SD_BLOCK_OUT, 2))
        self.config = SimpleNamespace(scaling_factor=SCALING, latent_channels=4, in_channels=3,
                                      block_out_channels=SD_BLOCK_OUT, layers_per_block=2, norm_num_groups=32)
        self.downscale = 2 ** (len(SD_BLOCK_OUT) - 1)

    def _pack(self):
        dev, sd, f32, b16 = self._state_for_packing()
        P: Dict[str, object] = {}
        for key in sd:
            if key.endswith(".conv1.weight"):
                p = key[: -len(".conv1.weight")]
                P[p] = _pack_resnet(sd, p, f32, b16)
            if key.endswith(".downsamplers.0.conv.weight"):
                p = key[: -len(".weight")]
                P[p] = (b16(pack_conv3x3(sd[key], dtype=None)), f32(f"{p}.bias"))
        a = "encoder.mid_block.attentions.0"
        P[a] = _pack_attention(sd, a, SD_BLOCK_OUT[-1], False, f32, b16, dev)
        P["conv_in"] = (ops.pack_conv_in(sd["encoder.conv_in.weight"], dev), f32("encoder.conv_in.bias"))
        P["norm_out"] = (f32("encoder.conv_norm_out.weight"), f32("encoder.conv_norm_out.bias"))
        P["conv_out"] = _pack_conv_out(sd["encoder.conv_out.weight"], sd["encoder.conv_out.bias"], dev)
        P["quant"] = (f32("quant_conv.weight").reshape(8, 8).contiguous(), f32("quant_conv.bias"))
        self._packed = P
        return P

    def _levels(self, H: int, W: int):
        """(channels, H, W) of each DownEncoderBlock2D's input map; the last entry is the mid block's."""
        out = []
        for i in range(len(SD_BLOCK_OUT)):
            out.append((SD_BLOCK_OUT[max(i - 1, 0)], H, W))
            if i != len(SD_BLOCK_OUT) - 1:
                H, W = ops.conv3x3_out_size(H, 2, (0, 1)), ops.conv3x3_out_size(W, 2, (0, 1))
        out.append((SD_BLOCK_OUT[-1], H, W))
        return out

    def check_geometry(self, H: int, W: int) -> None:
        """ValueError unless an H x W image can be encoded: H and W multiples of 8, and a mid block of h * w tokens that
        the single-head attention (GEMM + row softmax) takes: a multiple of 8, at most 4096."""
        if H <= 0 or W <= 0 or H % self.downscale or W % self.downscale:
            raise ValueError(f"image height and width must be positive multiples of {self.downscale}, got {H}x{W}")
        h, w = H // self.downscale, W // self.downscale
        if (h * w) % 8 or h * w > 4096:
            raise ValueError(f"the mid-block attention at a {h}x{w} latent needs h * w to be a multiple of 8 and at most "
                             f"4096 tokens, got {h * w}")

    def frame_elements(self, H: int, W: int) -> int:
        """Largest tensor, in elements per frame, that any launch of an encode of an H x W image touches: the conv_in
        patch rows, every level's maps at the channel counts they enter and leave with, the downsampled maps, and at the
        latent resolution the mid-block q/k/v rows and the padded conv_out rows."""
        levels = self._levels(H, W)
        most = max(3, ops.conv_in_kpad(3), SD_BLOCK_OUT[0]) * H * W
        for i, c in enumerate(SD_BLOCK_OUT):
            cin, h, w = levels[i]
            most = max(most, max(cin, c) * h * w)
            _, h2, w2 = levels[i + 1]
            most = max(most, c * h2 * w2)
        _, h, w = levels[-1]
        return max(most, 3 * SD_BLOCK_OUT[-1] * h * w, ops.CONV_OUT_PAD * h * w)

    def _encode_group(self, x, frames: bool):
        """One group of frames -> moments fp32 [N, 8, h, w].  x: fp32 [N, 3, H, W], or uint8 [N, H, W, 3] (frames)."""
        P = self._packed
        wi, bi = P["conv_in"]
        if frames:
            N, H, W, _ = x.shape
            h = ops.gemm(im2col_frames(x, wi.shape[1]), wi, bias=bi)
        else:
            N, _, H, W = x.shape
            h = ops.conv_in_tc(x.reshape(N, 3, 1, H, W), wi, bi)
        levels = len(SD_BLOCK_OUT)
        for i in range(levels):
            for j in range(self.config.layers_per_block):
                h = self._resnet(f"encoder.down_blocks.{i}.resnets.{j}", h, N, H, W)
            if i != levels - 1:
                wd, bd = P[f"encoder.down_blocks.{i}.downsamplers.0.conv"]
                h = ops.conv3x3(h, N, H, W, wd, stride=2, padding=(0, 1), bias=bd, stats=True)
                H, W = ops.conv3x3_out_size(H, 2, (0, 1)), ops.conv3x3_out_size(W, 2, (0, 1))
        h = self._resnet("encoder.mid_block.resnets.0", h, N, H, W)
        h = self._attention("encoder.mid_block.attentions.0", h, N, H * W, False)
        h = self._resnet("encoder.mid_block.resnets.1", h, N, H, W)
        ss = ops.groupnorm_scale_shift(h, N, H * W, P["norm_out"][0], P["norm_out"][1], 1e-6)
        y = ops.conv_out_tc(h, ss, N, 1, H, W, P["conv_out"][0], P["conv_out"][1], 8)
        return ops.pointwise_conv_nchw(y.reshape(N, 8, H, W), P["quant"][0], P["quant"][1])

    def _moments(self, x, frames: bool, max_launch_elements: int):
        H, W = (x.shape[1], x.shape[2]) if frames else (x.shape[2], x.shape[3])
        G = self.frames_per_group(H, W, max_launch_elements)
        N = x.shape[0]
        if N <= G:
            return self._encode_group(x, frames)
        return torch.cat([self._encode_group(x[a:a + G], frames) for a in range(0, N, G)])

    @torch.no_grad()
    def encode(self, x: torch.Tensor, return_dict: bool = True, max_launch_elements: int = MAX_LAUNCH_ELEMENTS):
        """AutoencoderKL.encode: x float [N, 3, H, W] in [-1, 1] -> ``.latent_dist`` (DiagonalGaussianDistribution over
        [N, 4, H/8, W/8]).  Frames run in groups of at most ``frames_per_group(H, W, max_launch_elements)``."""
        if x.dim() != 4 or x.shape[1] != 3 or not x.is_floating_point():
            raise ValueError(f"x must be a float [N,3,H,W] image batch, got {tuple(x.shape)} {x.dtype}")
        self.check_geometry(x.shape[2], x.shape[3])
        if self._packed is None:
            self._pack()
        xin = x.to(device=self.device, dtype=F32).contiguous()
        dist = DiagonalGaussianDistribution(self._moments(xin, False, max_launch_elements))
        if not return_dict:
            return (dist,)
        return SimpleNamespace(latent_dist=dist)

    @torch.no_grad()
    def encode_video(self, frames: torch.Tensor, generator: Optional[torch.Generator] = None,
                     noise: Optional[torch.Tensor] = None, sample: bool = True,
                     max_launch_elements: int = MAX_LAUNCH_ELEMENTS) -> torch.Tensor:
        """uint8 video [B, F, H, W, 3] -> fp32 latents [B, 4, F, H/8, W/8] * scaling_factor on the device: the frames are
        encoded as one batch of B*F images (frame n = b*F + f) normalised as (x / 255 - 0.5) / 0.5, the posterior is
        sampled (``sample=False``: its mode) and scaled.  noise: fp32 [B*F, 4, H/8, W/8], the shape the reference's
        ``latent_dist.sample()`` draws; by default drawn from ``generator`` like diffusers' randn_tensor."""
        if frames.dtype != torch.uint8 or frames.dim() != 5 or frames.shape[-1] != 3:
            raise ValueError(f"frames must be uint8 [B,F,H,W,3], got {tuple(frames.shape)} {frames.dtype}")
        B, Fr, H, W, _ = frames.shape
        self.check_geometry(H, W)
        dev = self.device
        lat = (B * Fr, 4, H // self.downscale, W // self.downscale)
        eps = _noise_like(lat, generator, noise, dev) if sample else None
        if self._packed is None:
            self._pack()
        fr = frames.to(dev).reshape(B * Fr, H, W, 3).contiguous()
        return posterior_sample(self._moments(fr, True, max_launch_elements), B, Fr, self.config.scaling_factor, eps)
