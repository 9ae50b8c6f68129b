"""Launches that only the VAE encoder needs: conv_in's patch rows straight from uint8 video frames
(``lavie_im2col_frames_bf16``) and the diagonal-Gaussian posterior, sampled and scaled into the interpolation model's
latent layout (``lavie_posterior_sample_f32``).  They live outside ``ops`` for the reason ``vae_attention`` does: ``ops``
holds the kernels shared by the denoisers and encoders, and these serve the VAE encoder alone."""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from ._lib import check
from .ops import BF16, F32, _Launch, _ptr, _stream


def im2col_frames(frames: torch.Tensor, kpad: int) -> torch.Tensor:
    """frames: uint8 [N, H, W, 3] channels-last on the device -> bf16 [N*H*W, kpad] conv_in patch rows of the image
    (frames / 255 - 0.5) / 0.5, K index c*9 + kh*3 + kw, zero outside the image and beyond 27."""
    lib = _lib.load()
    assert frames.dtype == torch.uint8 and frames.is_cuda and frames.is_contiguous() and frames.dim() == 4
    N, H, W, C = frames.shape
    assert C == 3, tuple(frames.shape)
    col = torch.empty((N * H * W, kpad), dtype=BF16, device=frames.device)
    with _Launch("lavie_im2col_frames_bf16", 0.0, 1.0 * frames.numel() + 2.0 * col.numel(), f"im2col_frames N={N}"):
        check(lib.lavie_im2col_frames_bf16(frames.data_ptr(), N, H, W, kpad, col.data_ptr(), _stream()),
              "lavie_im2col_frames_bf16")
    return col


def posterior_sample(moments: torch.Tensor, B: int, F: int, scale: float = 1.0,
                     noise: Optional[torch.Tensor] = None) -> torch.Tensor:
    """moments: fp32 [B*F, 8, h, w] (mean | logvar); noise: fp32 [B*F, 4, h, w] or None (the mode).  Returns fp32
    [B, 4, F, h, w] = scale * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise)."""
    lib = _lib.load()
    assert moments.dtype == F32 and moments.is_cuda and moments.is_contiguous() and moments.dim() == 4
    N, C8, h, w = moments.shape
    assert C8 == 8 and N == B * F, (tuple(moments.shape), B, F)
    if noise is not None:
        assert noise.dtype == F32 and noise.is_contiguous() and noise.device == moments.device
        assert tuple(noise.shape) == (N, 4, h, w), tuple(noise.shape)
    out = torch.empty((B, 4, F, h, w), dtype=F32, device=moments.device)
    with _Launch("lavie_posterior_sample_f32", 0.0, 4.0 * (moments.numel() + 2 * out.numel()),
                 f"posterior N={N} hw={h * w}"):
        check(lib.lavie_posterior_sample_f32(moments.data_ptr(), _ptr(noise), B, F, h * w, float(scale),
                                             out.data_ptr(), _stream()), "lavie_posterior_sample_f32")
    return out
