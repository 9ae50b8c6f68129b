"""CPU oracle for the x4-upscaler VAE decoder (SURVEY 8f row N4) -- TEST INFRASTRUCTURE, NOT PRODUCT.

**PARITY UNPINNED**, for the same reason as oracle/vae_oracle.py: the reference decodes with ``diffusers.AutoencoderKL``
(``diffusers==0.16.0``, third party, not vendored and not installable offline).  This file restates the published
decoder of the x4-upscaler VAE (stabilityai/stable-diffusion-x4-upscaler ``vae/config.json``: block_out_channels
(128, 256, 512), layers_per_block 2, 32 groups, eps 1e-6, latent channels 4, scaling factor 0.08333): conv_in ->
UNetMidBlock2D (ResnetBlock2D, single-head AttentionBlock of 512 channels, ResnetBlock2D) -> three UpDecoderBlock2D
(three ResnetBlock2D each, nearest-x2 Upsample2D + 3x3 conv on the first two) -> GroupNorm -> SiLU -> conv_out, so
[N,4,h,w] -> [N,3,4h,4w]; and the VSR pipeline's decode (vsr/models/pipeline_stable_diffusion_upscale_video_3d.py:741-771),
which is ``decode_latents`` of the SD pipelines with 1/0.08333 in place of 1/0.18215.  The ResnetBlock2D and
AttentionBlock restatements are the SD oracle's own (imported unchanged).  No reference run or golden vector of the real
class exists here; the GPU path is tested against THIS restatement only.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .vae_oracle import EPS, GROUPS, attention_block, resnet2d

BLOCK_OUT = (128, 256, 512)
UP_CHANNELS = tuple(reversed(BLOCK_OUT))
SCALING = 0.08333


@torch.no_grad()
def decode(sd, z: torch.Tensor) -> torch.Tensor:
    """AutoencoderKL._decode (mirror vsr/models/autoencoder_kl.py:179-192) of the x4 VAE: z [N,4,h,w] -> [N,3,4h,4w]."""
    sd = {k: v.float() for k, v in sd.items()}
    x = F.conv2d(z.float(), sd["post_quant_conv.weight"], sd["post_quant_conv.bias"])
    x = F.conv2d(x, sd["decoder.conv_in.weight"], sd["decoder.conv_in.bias"], padding=1)
    x = resnet2d(sd, "decoder.mid_block.resnets.0", x)
    x = attention_block(sd, "decoder.mid_block.attentions.0", x)
    x = resnet2d(sd, "decoder.mid_block.resnets.1", x)
    for i in range(len(UP_CHANNELS)):
        for j in range(3):
            x = resnet2d(sd, f"decoder.up_blocks.{i}.resnets.{j}", x)
        if i != len(UP_CHANNELS) - 1:
            x = F.interpolate(x, scale_factor=2.0, mode="nearest")
            x = F.conv2d(x, sd[f"decoder.up_blocks.{i}.upsamplers.0.conv.weight"],
                         sd[f"decoder.up_blocks.{i}.upsamplers.0.conv.bias"], padding=1)
    x = F.group_norm(x, GROUPS, sd["decoder.conv_norm_out.weight"], sd["decoder.conv_norm_out.bias"], EPS)
    return F.conv2d(F.silu(x), sd["decoder.conv_out.weight"], sd["decoder.conv_out.bias"], padding=1)


@torch.no_grad()
def decode_latents(sd, latents: torch.Tensor) -> torch.Tensor:
    """The VSR pipeline's decode (vsr/models/pipeline_stable_diffusion_upscale_video_3d.py:741-771):
    [B,4,F,h,w] -> uint8 [B,F,4h,4w,3]."""
    B, C, Fr, h, w = latents.shape
    z = (1 / SCALING * latents).permute(0, 2, 1, 3, 4).reshape(B * Fr, C, h, w)
    video = decode(sd, z)
    video = video.reshape(B, Fr, 3, video.shape[-2], video.shape[-1]).permute(0, 1, 3, 4, 2)
    return ((video / 2 + 0.5) * 255).add_(0.5).clamp_(0, 255).to(dtype=torch.uint8).contiguous()
