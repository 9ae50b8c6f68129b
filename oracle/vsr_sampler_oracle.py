"""CPU oracle of the VSR stage's sampling loop -- TEST INFRASTRUCTURE, NOT PRODUCT.

The x4-upscaler pipeline (vsr/models/pipeline_stable_diffusion_upscale_video_3d.py:709-738, diffusers 0.16
``StableDiffusionUpscalePipeline`` order) over the 8-frame chunks of vsr/sample.py:100-118, driving
``oracle.vsr_oracle.unet_forward``.  All scheduler arithmetic in float64; x0 and eps are formed explicitly, not through
the product's linear (A, B) form.

Unpinned (restated, not run against the reference here):

* the scheduler configs, from the published ``stabilityai/stable-diffusion-x4-upscaler`` ``scheduler`` (DDIMScheduler:
  scaled_linear 1e-4 .. 2e-2, 1000 steps, prediction_type v_prediction, steps_offset 1, set_alpha_to_one False,
  clip_sample False) and ``low_res_scheduler`` (DDPMScheduler: scaled_linear 1e-4 .. 2e-2, 1000 steps) configs;
* the timestep spacing: the reference's VSR scheduler is the vendored vsr/diffusion/scheduling_ddim.py, whose
  ``set_timesteps`` (:267-290) is a modified linspace variant; the stock 0.16 spacing ``(arange(n) * ratio)[::-1] +
  steps_offset`` is used here (callers may pass their own list);
* the draw order: per chunk, the low-resolution noise before the initial latents (diffusers 0.16 draws the image noise
  before ``prepare_latents``); the tests share explicit noise tensors instead of generator parity;
* the uint8 normalisation of low-resolution frames, (x / 255 - 0.5) / 0.5, as for the VAE encoder's input.
"""
from __future__ import annotations

from typing import Callable, List, Optional

import numpy as np
import torch

from . import vsr_oracle as V


def scaled_linear_alphas_cumprod(num_train: int = 1000, beta_start: float = 1e-4, beta_end: float = 2e-2) -> torch.Tensor:
    """diffusers' scaled_linear: linspace(sqrt(b0), sqrt(b1), n, float32) ** 2, cumprod of 1 - betas (float32)."""
    betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train, dtype=torch.float32) ** 2
    return torch.cumprod(1.0 - betas, dim=0)


def add_noise(x: torch.Tensor, noise: torch.Tensor, level: int) -> torch.Tensor:
    """DDPMScheduler.add_noise with the low_res_scheduler's alpha-bar (float32, as diffusers computes it)."""
    acp = scaled_linear_alphas_cumprod()
    return acp[level] ** 0.5 * x.float() + (1 - acp[level]) ** 0.5 * noise.float()


class DDIMV:
    """diffusers 0.16 DDIMScheduler.step, prediction_type v_prediction, eta 0, set_alpha_to_one False."""

    def __init__(self, steps: int = 50, num_train: int = 1000, steps_offset: int = 1,
                 timesteps: Optional[List[int]] = None):
        self.acp = scaled_linear_alphas_cumprod(num_train).double()
        n = steps if timesteps is None else len(timesteps)
        self.ratio = num_train // n
        self.timesteps = timesteps if timesteps is not None else \
            ((np.arange(n) * self.ratio).round()[::-1] + steps_offset).astype(np.int64).tolist()
        self.init_noise_sigma = 1.0

    def step(self, v, i, sample):
        t = self.timesteps[i]
        prev = t - self.ratio
        a_t = self.acp[t]
        a_p = self.acp[prev] if prev >= 0 else self.acp[0]
        x, v = sample.double(), v.double()
        x0 = a_t.sqrt() * x - (1 - a_t).sqrt() * v
        eps = a_t.sqrt() * v + (1 - a_t).sqrt() * x
        return a_p.sqrt() * x0 + (1 - a_p).sqrt() * eps


@torch.no_grad()
def vsr_loop(sd, low_res: torch.Tensor, text: torch.Tensor, latents: torch.Tensor, low_res_noise: torch.Tensor,
             scheduler: DDIMV, guidance: float = 5.0, noise_level: int = 50, chunk_frames: int = 8,
             forward: Optional[Callable] = None) -> torch.Tensor:
    """low_res float [1,3,F,h,w] in [-1, 1], text [2,L,1024] = cat([negative, positive]), latents [1,4,F,h,w] and
    low_res_noise [1,3,F,h,w] for the whole video -> final latents [1,4,F,h,w]; every chunk an independent pipeline call."""
    forward = forward or (lambda x, t, lr, e, c: V.unet_forward(sd, x, t, lr, e, c))
    labels = torch.tensor([noise_level, noise_level])
    out = []
    for s in range(0, low_res.shape[2], chunk_frames):
        sl = slice(s, s + chunk_frames)
        lr = add_noise(low_res[:, :, sl], low_res_noise[:, :, sl], noise_level)
        lr2 = torch.cat([lr, lr])
        x = latents[:, :, sl].float() * scheduler.init_noise_sigma
        for i, t in enumerate(scheduler.timesteps):
            pred = forward(torch.cat([x, x]), t, lr2, text, labels)
            u, c = pred.chunk(2)
            x = scheduler.step(u + guidance * (c - u), i, x).float()
        out.append(x)
    return torch.cat(out, dim=2)
