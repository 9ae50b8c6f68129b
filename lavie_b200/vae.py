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
launch passes 2^31 elements."""
from __future__ import annotations

import math
from collections import OrderedDict
from types import SimpleNamespace
from typing import Dict, Tuple

import torch
from torch import nn

from . import ops
from .packing import pack_conv1x1, pack_conv3x3, pack_upsample_conv3x3
from .synthetic import _gen
from .vae_attention import attention_wide

BF16 = torch.bfloat16
F32 = torch.float32
UP_CHANNELS = (512, 512, 256, 128)          # reversed block_out_channels of the SD VAE
SCALING = 0.18215                            # pipeline_videogen.py:424
SD_BLOCK_OUT = (128, 256, 512, 512)
# stabilityai/stable-diffusion-x4-upscaler vae/config.json
X4_BLOCK_OUT = (128, 256, 512)
X4_SCALING = 0.08333
MAX_LAUNCH_ELEMENTS = 2 ** 31 - 1           # largest tensor one launch may address with 32-bit element indices


def vae_decoder_param_spec(block_out_channels=SD_BLOCK_OUT, layers_per_block: int = 2
                           ) -> "OrderedDict[str, Tuple[int, ...]]":
    """Decode-side parameters of diffusers' AutoencoderKL (0.16 names).  Default: the Stable Diffusion VAE."""
    up_channels = tuple(reversed(block_out_channels))
    top = up_channels[0]
    spec: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()

    def conv(p, co, ci, k):
        spec[f"{p}.weight"] = (co, ci, k, k)
        spec[f"{p}.bias"] = (co,)

    def norm(p, c):
        spec[f"{p}.weight"] = (c,)
        spec[f"{p}.bias"] = (c,)

    def resnet(p, ci, co):
        norm(f"{p}.norm1", ci)
        conv(f"{p}.conv1", co, ci, 3)
        norm(f"{p}.norm2", co)
        conv(f"{p}.conv2", co, co, 3)
        if ci != co:
            conv(f"{p}.conv_shortcut", co, ci, 1)

    conv("post_quant_conv", 4, 4, 1)
    conv("decoder.conv_in", top, 4, 3)
    resnet("decoder.mid_block.resnets.0", top, top)
    a = "decoder.mid_block.attentions.0"
    norm(f"{a}.group_norm", top)
    for n in ("query", "key", "value", "proj_attn"):
        spec[f"{a}.{n}.weight"] = (top, top)
        spec[f"{a}.{n}.bias"] = (top,)
    resnet("decoder.mid_block.resnets.1", top, top)
    prev = top
    for i, c in enumerate(up_channels):
        for j in range(layers_per_block + 1):
            resnet(f"decoder.up_blocks.{i}.resnets.{j}", prev if j == 0 else c, c)
        if i != len(up_channels) - 1:
            conv(f"decoder.up_blocks.{i}.upsamplers.0.conv", c, c, 3)
        prev = c
    norm("decoder.conv_norm_out", up_channels[-1])
    conv("decoder.conv_out", 3, up_channels[-1], 3)
    return spec


def vae_synthetic_state_dict(seed: int = 0, block_out_channels=SD_BLOCK_OUT):
    """Seeded decoder weights; ``block_out_channels=X4_BLOCK_OUT`` draws the x4-upscaler layout."""
    sd = OrderedDict()
    spec = vae_decoder_param_spec(block_out_channels)
    tag = "vae:" if tuple(block_out_channels) == SD_BLOCK_OUT else f"vae{tuple(block_out_channels)}:"
    for key, shape in spec.items():
        g = _gen(seed, tag + key)
        if ".norm" in key or "group_norm" in key or "conv_norm_out" in key:
            t = 0.1 * torch.randn(shape, generator=g) + (1.0 if key.endswith("weight") else 0.0)
        else:
            wshape = spec[key[: -len("bias")] + "weight"] if key.endswith("bias") else shape
            t = (torch.rand(shape, generator=g) * 2.0 - 1.0) / math.sqrt(math.prod(wshape[1:]))
        sd[key] = t
    return sd


# diffusers renamed the attention block's parameters after 0.16; accept both spellings
_ATTN_ALIASES = {"to_q": "query", "to_k": "key", "to_v": "value", "to_out.0": "proj_attn"}


def load_vae_state_dict(module: "VAEDecoder", sd, strict: bool = True):
    """Load the decode side of an ``AutoencoderKL`` checkpoint: encoder / quant_conv keys are dropped, newer attention
    parameter names are mapped to the 0.16 ones."""
    out = {}
    for k, v in sd.items():
        if not (k.startswith("decoder.") or k.startswith("post_quant_conv.")):
            continue
        for new, old in _ATTN_ALIASES.items():
            k = k.replace(f"attentions.0.{new}.", f"attentions.0.{old}.")
        if k.endswith("weight") and v.dim() == 4 and ".attentions." in k:
            v = v.reshape(v.shape[0], v.shape[1])
        out[k] = v
    return module.load_state_dict(out, strict=strict)


class VAEDecoder(nn.Module):
    """``decode(z).sample`` of an AutoencoderKL decoder + the pipelines' ``decode_latents``.  No arguments: the Stable
    Diffusion VAE (x8); ``VAEDecoder.x4_upscaler()``: the x4-upscaler VAE of the VSR pipeline."""

    def __init__(self, block_out_channels=SD_BLOCK_OUT, scaling_factor: float = SCALING, layers_per_block: int = 2):
        super().__init__()
        block_out_channels = tuple(int(c) for c in block_out_channels)
        self.config = SimpleNamespace(scaling_factor=scaling_factor, latent_channels=4,
                                      block_out_channels=block_out_channels, layers_per_block=layers_per_block,
                                      norm_num_groups=32)
        self.up_channels = tuple(reversed(block_out_channels))
        self.upscale = 2 ** (len(block_out_channels) - 1)
        # the SD VAE keeps its GEMM + row-softmax attention (2560 tokens at its 40x64 latent); every other configuration
        # runs the fused wide kernel, which has no token limit
        self.wide_attention = block_out_channels != SD_BLOCK_OUT
        if self.wide_attention and self.up_channels[0] != 512:
            raise ValueError("the fused mid-block attention needs block_out_channels[-1] == 512")
        for key, shape in vae_decoder_param_spec(block_out_channels, layers_per_block).items():
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

    @classmethod
    def x4_upscaler(cls) -> "VAEDecoder":
        """The VAE of the x4 upscaler (the VSR pipeline's decoder): [N,4,h,w] -> [N,3,4h,4w]."""
        return cls(X4_BLOCK_OUT, X4_SCALING)

    def _invalidate(self):
        self._packed = None

    def _apply(self, fn, *a, **kw):
        out = super()._apply(fn, *a, **kw)
        self._invalidate()
        return out

    @property
    def device(self):
        return self.post_quant_conv.weight.device

    @property
    def dtype(self):
        return self.post_quant_conv.weight.dtype

    def _pack(self):
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError("lavie_b200.VAEDecoder runs on CUDA (sm_100a) only; move it with .to('cuda')")
        sd = {k: v.detach() for k, v in self.state_dict().items()}
        f32 = lambda k: sd[k].to(device=dev, dtype=F32).contiguous()
        b16 = lambda t: t.to(device=dev, dtype=BF16).contiguous()
        P: Dict[str, object] = {}
        for key in sd:
            if key.endswith(".conv1.weight"):
                p = key[: -len(".conv1.weight")]
                r = {"g1": f32(f"{p}.norm1.weight"), "b1": f32(f"{p}.norm1.bias"),
                     "w1": b16(pack_conv3x3(sd[f"{p}.conv1.weight"], dtype=None)), "cb1": f32(f"{p}.conv1.bias"),
                     "g2": f32(f"{p}.norm2.weight"), "b2": f32(f"{p}.norm2.bias"),
                     "w2": b16(pack_conv3x3(sd[f"{p}.conv2.weight"], dtype=None)), "cb2": f32(f"{p}.conv2.bias")}
                if f"{p}.conv_shortcut.weight" in sd:
                    r["wsc"] = b16(pack_conv1x1(sd[f"{p}.conv_shortcut.weight"], dtype=None))
                    r["bsc"] = f32(f"{p}.conv_shortcut.bias")
                P[p] = r
            if key.endswith(".upsamplers.0.conv.weight"):
                p = key[: -len(".weight")]
                P[p] = (b16(pack_conv3x3(sd[key], dtype=None)), f32(f"{p}.bias"), pack_upsample_conv3x3(sd[key]).to(dev))
        a = "decoder.mid_block.attentions.0"
        C = self.up_channels[0]
        s = C ** -0.5                                   # folded into the query projection: scores leave the GEMM scaled
        P[a] = {"g": f32(f"{a}.group_norm.weight"), "b": f32(f"{a}.group_norm.bias"),
                "w_q": b16(sd[f"{a}.query.weight"].float() * s),
                "b_q": (sd[f"{a}.query.bias"].float() * s).to(dev).contiguous(),
                "w_k": b16(sd[f"{a}.key.weight"]), "b_k": f32(f"{a}.key.bias"),
                "w_v": b16(sd[f"{a}.value.weight"]), "b_v": f32(f"{a}.value.bias"),
                "w_o": b16(sd[f"{a}.proj_attn.weight"]), "b_o": f32(f"{a}.proj_attn.bias")}
        if self.wide_attention:                         # q, k, v from one GEMM: [rows, 3C], read as strided views
            t = P[a]
            t["w_qkv"] = torch.cat([t.pop("w_q"), t.pop("w_k"), t.pop("w_v")]).contiguous()
            t["b_qkv"] = torch.cat([t.pop("b_q"), t.pop("b_k"), t.pop("b_v")]).contiguous()
        P["pq"] = (f32("post_quant_conv.weight").reshape(4, 4).contiguous(), f32("post_quant_conv.bias"))
        P["conv_in"] = (f32("decoder.conv_in.weight"), f32("decoder.conv_in.bias"))
        wp = torch.zeros((ops.CONV_OUT_PAD, 9 * self.up_channels[-1]), dtype=F32)
        wp[:3] = pack_conv3x3(sd["decoder.conv_out.weight"].float().cpu(), dtype=None)
        bp = torch.zeros(ops.CONV_OUT_PAD, dtype=F32)
        bp[:3] = sd["decoder.conv_out.bias"].float().cpu()
        P["conv_out"] = (wp.to(device=dev, dtype=BF16).contiguous(), bp.to(dev))
        P["norm_out"] = (f32("decoder.conv_norm_out.weight"), f32("decoder.conv_norm_out.bias"))
        self._packed = P
        return P

    # ------------------------------------------------------------------ blocks
    def _resnet(self, p, x, N, H, W):
        r = self._packed[p]
        h = ops.groupnorm(x, N, H * W, r["g1"], r["b1"], 1e-6, silu=True)
        h = ops.conv3x3(h, N, H, W, r["w1"], bias=r["cb1"], stats=True)
        h = ops.groupnorm(h, N, H * W, r["g2"], r["b2"], 1e-6, silu=True)
        sc = ops.gemm(x, r["wsc"], bias=r["bsc"]) if "wsc" in r else x
        return ops.conv3x3(h, N, H, W, r["w2"], bias=r["cb2"], residual=sc, stats=True)

    def _attention(self, x, N, HW):
        """diffusers 0.16 AttentionBlock (one head of 512 channels) per frame."""
        t = self._packed["decoder.mid_block.attentions.0"]
        C = 512
        n = ops.groupnorm(x, N, HW, t["g"], t["b"], 1e-6, silu=False)
        if self.wide_attention:
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

    def frames_per_group(self, h: int, w: int, max_launch_elements: int = MAX_LAUNCH_ELEMENTS) -> int:
        per_frame = self.frame_elements(h, w)
        if per_frame > max_launch_elements:
            raise ValueError(f"one frame of a {h}x{w} latent needs {per_frame} elements in one launch "
                             f"(limit {max_launch_elements}); decode it in tiles")
        return max_launch_elements // per_frame

    def _decode_group(self, zin, scale, as_uint8):
        P = self._packed
        N, _, h, w = zin.shape
        zq = ops.pointwise_conv_nchw(zin, P["pq"][0], P["pq"][1], scale)
        x = ops.conv_in(zq.reshape(N, 4, 1, h, w), P["conv_in"][0], P["conv_in"][1])
        H, W = h, w
        x = self._resnet("decoder.mid_block.resnets.0", x, N, H, W)
        x = self._attention(x, N, H * W)
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
