"""CPU oracle for the VAE encoder (SURVEY 8f row N4) -- TEST INFRASTRUCTURE, NOT PRODUCT.

**PARITY UNPINNED**, for the same reason as oracle/vae_oracle.py: the reference encodes with ``diffusers.AutoencoderKL``
(``diffusers==0.16.0``, third party, not vendored and not installable offline).  Its caller is the interpolation stage,
which encodes its conditioning frames before the DDIM loop (interpolation/sample.py, ``auto_inpainting_copy_no_mask``:
``vae.encode(frames).latent_dist.sample().mul_(0.18215)``); the in-tree mirror of the wrapper
(vsr/models/autoencoder_kl.py, ``AutoencoderKL.encode``) shows the call order ``encoder`` -> ``quant_conv`` ->
``DiagonalGaussianDistribution`` but imports the ``Encoder`` itself from diffusers.  The reference tree was not
available when this file was written, so neither the line numbers of those calls nor which frames the interpolation
stage encodes (its 16 key frames, or the copied-out video at the output frame count) could be checked here;
``encode_video`` takes whatever frames the caller passes.

This file restates the published diffusers-0.16 ``Encoder`` of the Stable Diffusion VAE (block_out_channels
(128, 256, 512, 512), layers_per_block 2, 32 groups, eps 1e-6, double_z): conv_in -> four DownEncoderBlock2D (two
ResnetBlock2D each, ``Downsample2D(padding=0)`` = ``F.pad(x, (0, 1, 0, 1))`` + stride-2 pad-0 3x3 conv on the first
three) -> UNetMidBlock2D (ResnetBlock2D, single-head AttentionBlock, ResnetBlock2D) -> GroupNorm -> SiLU -> conv_out
(512 -> 8), then ``quant_conv`` (1x1, 8 -> 8) and ``DiagonalGaussianDistribution`` (logvar clamped to [-30, 20],
std = exp(logvar / 2), sample = mean + std * noise).  The ResnetBlock2D and AttentionBlock restatements are the SD
decoder oracle's own (imported unchanged).  No reference run or golden vector of the real class exists here; the GPU
path is tested against THIS restatement only.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .vae_oracle import EPS, GROUPS, attention_block, resnet2d

BLOCK_OUT = (128, 256, 512, 512)
LAYERS_PER_BLOCK = 2
SCALING = 0.18215


def downsample2d(sd, p, x):
    """diffusers Downsample2D(use_conv=True, padding=0): pad right and bottom by one, then a stride-2 pad-0 conv."""
    x = F.pad(x, (0, 1, 0, 1), mode="constant", value=0)
    return F.conv2d(x, sd[f"{p}.conv.weight"], sd[f"{p}.conv.bias"], stride=2)


@torch.no_grad()
def moments(sd, x: torch.Tensor) -> torch.Tensor:
    """quant_conv(Encoder(x)): x [N,3,H,W] in [-1, 1] -> moments [N,8,H/8,W/8] (mean | logvar)."""
    sd = {k: v.float() for k, v in sd.items()}
    h = F.conv2d(x.float(), sd["encoder.conv_in.weight"], sd["encoder.conv_in.bias"], padding=1)
    for i in range(len(BLOCK_OUT)):
        for j in range(LAYERS_PER_BLOCK):
            h = resnet2d(sd, f"encoder.down_blocks.{i}.resnets.{j}", h)
        if i != len(BLOCK_OUT) - 1:
            h = downsample2d(sd, f"encoder.down_blocks.{i}.downsamplers.0", h)
    h = resnet2d(sd, "encoder.mid_block.resnets.0", h)
    h = attention_block(sd, "encoder.mid_block.attentions.0", h)
    h = resnet2d(sd, "encoder.mid_block.resnets.1", h)
    h = F.group_norm(h, GROUPS, sd["encoder.conv_norm_out.weight"], sd["encoder.conv_norm_out.bias"], EPS)
    h = F.conv2d(F.silu(h), sd["encoder.conv_out.weight"], sd["encoder.conv_out.bias"], padding=1)
    return F.conv2d(h, sd["quant_conv.weight"], sd["quant_conv.bias"])


def posterior(m: torch.Tensor):
    """DiagonalGaussianDistribution(moments): (mean, clamped logvar, std)."""
    mean, logvar = torch.chunk(m, 2, dim=1)
    logvar = torch.clamp(logvar, -30.0, 20.0)
    return mean, logvar, torch.exp(0.5 * logvar)


def sample(m: torch.Tensor, noise: torch.Tensor) -> torch.Tensor:
    mean, _, std = posterior(m)
    return mean + std * noise


def normalize_frames(frames: torch.Tensor) -> torch.Tensor:
    """uint8 [N,H,W,3] -> float [N,3,H,W]: (x / 255 - 0.5) / 0.5."""
    x = frames.permute(0, 3, 1, 2).float()
    return (x / 255 - 0.5) / 0.5


@torch.no_grad()
def encode_video(sd, frames: torch.Tensor, noise=None) -> torch.Tensor:
    """uint8 video [B,F,H,W,3] -> latents [B,4,F,H/8,W/8]: the frames as one (b f) batch,
    ``vae.encode(x).latent_dist.sample().mul_(0.18215)`` with ``noise`` [B*F,4,h,w] (None: the mode), rearranged
    "(b f) c h w -> b c f h w"."""
    B, Fr, H, W, _ = frames.shape
    m = moments(sd, normalize_frames(frames.reshape(B * Fr, H, W, 3)))
    z = posterior(m)[0] if noise is None else sample(m, noise.float())
    z = z * SCALING
    return z.reshape(B, Fr, 4, H // 8, W // 8).permute(0, 2, 1, 3, 4).contiguous()
