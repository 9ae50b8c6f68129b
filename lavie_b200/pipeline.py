"""The caller of the denoiser: the classifier-free-guidance loop of ``VideoGenPipeline.__call__``
(base/pipelines/pipeline_videogen.py:664-689) with the three schedulers the reference wires up (predict.py:74-96:
DDIM, DDPM, EulerDiscrete), restated over the B200 module.

Per step: ``cat([latents]*2)`` -> ``scheduler.scale_model_input`` -> ``unet(...)`` -> ``u + g (t - u)`` ->
``scheduler.step``.  Guidance combine + scheduler update run as ONE small kernel: every epsilon-prediction update is
``a * latents + b * eps (+ c * noise)`` (``lavie_cfg_linear_step``; DDIM keeps its dedicated ``lavie_cfg_ddim_step``), the
coefficients are computed here in float64 per step.  EulerDiscrete's ``scale_model_input`` (x / sqrt(sigma^2 + 1)) is
folded into conv_in through ``unet(..., input_scale=...)``.  Scheduler constants follow the reference's sampling config
(base/configs/sample.yaml:23-25: linear betas 1e-4..2e-2) and diffusers 0.16.0 (DDIM mirror in the reference:
vsr/diffusion/scheduling_ddim.py:259-265, 345-394; DDPM / EulerDiscrete from the published 0.16.0 sources).

``VSRSampler`` is the caller of the VSR denoiser: the x4-upscaler pipeline's loop (v-prediction DDIM, noise-augmented
low-resolution frames) over vsr/sample.py's chunks of 8 frames, optionally spread over the ranks of a process group.
"""
from __future__ import annotations

import math
from typing import Callable, Dict, List, Optional, Tuple

import numpy as np
import torch

from . import ops
from .config import VSR_CONFIG
from .vae import _noise_like

F32 = torch.float32


def _alphas_cumprod(num_train_timesteps: int, beta_start: float, beta_end: float,
                    beta_schedule: str = "linear") -> torch.Tensor:
    """diffusers' betas in float32: ``linear`` or ``scaled_linear`` (linspace of the square roots, squared)."""
    if beta_schedule == "linear":
        betas = torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=torch.float32)
    elif beta_schedule == "scaled_linear":
        betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
    else:
        raise ValueError(f"unknown beta_schedule {beta_schedule!r}; choose 'linear' or 'scaled_linear'")
    return torch.cumprod(1.0 - betas, dim=0)


class DDIMSchedule:
    """DDIMScheduler, eta = 0, steps_offset 1, set_alpha_to_one False, clip_sample False.

    ``prediction_type`` "epsilon" (the base pipeline's) or "v_prediction" (the x4 upscaler's); ``beta_schedule`` "linear"
    or "scaled_linear".  ``timesteps``: an explicit descending list replacing the stock diffusers 0.16 spacing
    ``(arange(n) * ratio)[::-1] + steps_offset``, e.g. the vendored VSR scheduler's own ``set_timesteps``; then n is its
    length and the previous timestep of every step is still ``t - num_train_timesteps // n``, as ``step()`` computes it."""
    name = "ddim"
    needs_noise = False

    def __init__(self, num_inference_steps: int = 50, num_train_timesteps: int = 1000, beta_start: float = 1e-4,
                 beta_end: float = 2e-2, steps_offset: int = 1, beta_schedule: str = "linear",
                 prediction_type: str = "epsilon", timesteps: Optional[List[int]] = None):
        if prediction_type not in ("epsilon", "v_prediction"):
            raise ValueError(f"unknown prediction_type {prediction_type!r}; choose 'epsilon' or 'v_prediction'")
        self.prediction_type = prediction_type
        self.alphas_cumprod = _alphas_cumprod(num_train_timesteps, beta_start, beta_end, beta_schedule)
        if timesteps is not None:
            timesteps = [int(t) for t in timesteps]
            if not timesteps or any(not 0 <= t < num_train_timesteps for t in timesteps):
                raise ValueError(f"timesteps must be a non-empty list in [0, {num_train_timesteps})")
            num_inference_steps = len(timesteps)
        self.ratio = num_train_timesteps // num_inference_steps
        if timesteps is None:
            timesteps = ((torch.arange(num_inference_steps) * self.ratio).flip(0) + steps_offset).tolist()
        self.timesteps: List[int] = timesteps
        self.init_noise_sigma = 1.0

    def alphas(self, t: int):
        prev = t - self.ratio
        a_t = float(self.alphas_cumprod[t])
        a_prev = float(self.alphas_cumprod[prev]) if prev >= 0 else float(self.alphas_cumprod[0])
        return a_t, a_prev

    def input_scale(self, i: int) -> float:
        return 1.0

    def coefficients(self, i: int):
        """(a, b, c_noise) of latents' = a latents + b out + c noise, out the model output.  epsilon:
        x0 = (x - sqrt(1-a_t) eps) / sqrt(a_t).  v_prediction: x0 = sqrt(a_t) x - sqrt(1-a_t) v and
        eps = sqrt(a_t) v + sqrt(1-a_t) x, so x' = sqrt(a_p) x0 + sqrt(1-a_p) eps is linear in (x, v) too."""
        a_t, a_p = self.alphas(self.timesteps[i])
        if self.prediction_type == "v_prediction":
            return (math.sqrt(a_p * a_t) + math.sqrt((1 - a_p) * (1 - a_t)),
                    math.sqrt(1 - a_p) * math.sqrt(a_t) - math.sqrt(a_p) * math.sqrt(1 - a_t), 0.0)
        return (math.sqrt(a_p / a_t), math.sqrt(1 - a_p) - math.sqrt(a_p) * math.sqrt(1 - a_t) / math.sqrt(a_t), 0.0)


class DDPMSchedule:
    """DDPMScheduler (diffusers 0.16.0): ancestral sampling, variance_type fixed_small, clip_sample False."""
    name = "ddpm"
    needs_noise = True

    def __init__(self, num_inference_steps: int = 50, num_train_timesteps: int = 1000, beta_start: float = 1e-4,
                 beta_end: float = 2e-2):
        self.alphas_cumprod = _alphas_cumprod(num_train_timesteps, beta_start, beta_end).double()
        self.ratio = num_train_timesteps // num_inference_steps
        self.timesteps: List[int] = (torch.arange(num_inference_steps) * self.ratio).flip(0).tolist()
        self.init_noise_sigma = 1.0

    def input_scale(self, i: int) -> float:
        return 1.0

    def coefficients(self, i: int):
        t = self.timesteps[i]
        prev = t - self.ratio
        a_t = float(self.alphas_cumprod[t])
        a_p = float(self.alphas_cumprod[prev]) if prev >= 0 else 1.0
        b_t, b_p = 1.0 - a_t, 1.0 - a_p
        cur_a = a_t / a_p
        cur_b = 1.0 - cur_a
        c_x0 = math.sqrt(a_p) * cur_b / b_t            # weight of the predicted x0
        c_x = math.sqrt(cur_a) * b_p / b_t             # weight of the current sample
        sigma = math.sqrt(max(b_p / b_t * cur_b, 1e-20)) if t > 0 else 0.0
        # x0 = (x - sqrt(b_t) eps) / sqrt(a_t)
        return (c_x0 / math.sqrt(a_t) + c_x, -c_x0 * math.sqrt(b_t) / math.sqrt(a_t), sigma)


class EulerDiscreteSchedule:
    """EulerDiscreteScheduler (diffusers 0.16.0), linear sigma interpolation, s_churn = 0 (deterministic)."""
    name = "eulerdiscrete"
    needs_noise = False

    def __init__(self, num_inference_steps: int = 50, num_train_timesteps: int = 1000, beta_start: float = 1e-4,
                 beta_end: float = 2e-2):
        acp = _alphas_cumprod(num_train_timesteps, beta_start, beta_end).double().numpy()
        ts = np.linspace(0, num_train_timesteps - 1, num_inference_steps, dtype=float)[::-1].copy()
        sig = ((1 - acp) / acp) ** 0.5
        sig = np.interp(ts, np.arange(0, len(sig)), sig)
        self.sigmas = np.concatenate([sig, [0.0]]).astype(np.float32).astype(np.float64)
        self.timesteps: List[float] = ts.tolist()        # fractional timesteps go to the time embedding as they are
        self.init_noise_sigma = float(self.sigmas.max())

    def input_scale(self, i: int) -> float:
        return float(1.0 / math.sqrt(self.sigmas[i] ** 2 + 1.0))

    def coefficients(self, i: int):
        # x0 = x - sigma eps; derivative = (x - x0) / sigma = eps; x' = x + eps (sigma_next - sigma)
        return (1.0, float(self.sigmas[i + 1] - self.sigmas[i]), 0.0)


def make_schedule(name: str, num_inference_steps: int = 50, **kw):
    """'ddim' | 'ddpm' | 'eulerdiscrete' -- the keys of predict.py:74-96's scheduler table."""
    table = {"ddim": DDIMSchedule, "ddpm": DDPMSchedule, "eulerdiscrete": EulerDiscreteSchedule}
    if name not in table:
        raise ValueError(f"unknown sample_method {name!r}; choose from {sorted(table)}")
    return table[name](num_inference_steps, **kw)


class CFGDenoiser:
    """One CFG denoising step on device-resident state.  ``text`` = cat([negative, positive]) [2, L, ctx] exactly as
    ``_encode_prompt`` returns it (pipeline_videogen.py:418)."""

    def __init__(self, unet, guidance_scale: float = 7.5, schedule=None):
        self.unet = unet
        self.guidance_scale = float(guidance_scale)
        self.schedule = schedule or DDIMSchedule()
        self._model_in = None
        self._index = {t: i for i, t in enumerate(self.schedule.timesteps)}

    def step(self, latents: torch.Tensor, t, text: torch.Tensor, noise: Optional[torch.Tensor] = None,
             generator: Optional[torch.Generator] = None) -> torch.Tensor:
        """latents fp32 [1,C,F,H,W] on the device -> next latents (new tensor).  ``noise``: the variance noise of a
        stochastic scheduler (DDPM); drawn from ``generator`` on the latents' device when omitted, like diffusers'
        ``randn_tensor``."""
        if self._model_in is None or self._model_in.shape[1:] != latents.shape[1:]:
            self._model_in = torch.empty((2,) + tuple(latents.shape[1:]), dtype=F32, device=latents.device)
        self._model_in[0].copy_(latents[0])          # torch.cat([latents] * 2), pipeline_videogen.py:666
        self._model_in[1].copy_(latents[0])
        sched = self.schedule
        i = self._index[t]
        noise_pred = self.unet(self._model_in, t, encoder_hidden_states=text, input_scale=sched.input_scale(i)).sample
        if isinstance(sched, DDIMSchedule) and sched.prediction_type == "epsilon":
            a_t, a_prev = sched.alphas(t)
            return ops.cfg_ddim_step(noise_pred[0:1], noise_pred[1:2], self.guidance_scale, a_t, a_prev, latents)
        a, b, c = sched.coefficients(i)
        if c != 0.0 and noise is None:
            noise = torch.randn(latents.shape, generator=generator, device=latents.device, dtype=F32)
        return ops.cfg_linear_step(noise_pred[0:1], noise_pred[1:2], self.guidance_scale, a, b, latents,
                                   noise=noise if c != 0.0 else None, c_noise=c)

    def loop(self, latents: torch.Tensor, text: torch.Tensor,
             callback: Optional[Callable[[int, int, torch.Tensor], None]] = None,
             noises: Optional[list] = None, generator: Optional[torch.Generator] = None) -> torch.Tensor:
        latents = latents.to(device=self.unet.device, dtype=F32).contiguous() * self.schedule.init_noise_sigma
        text = text.to(self.unet.device)
        for i, t in enumerate(self.schedule.timesteps):
            noise = None if noises is None else noises[i].to(device=latents.device, dtype=F32).contiguous()
            latents = self.step(latents, t, text, noise=noise, generator=generator)
            if callback is not None:
                callback(i, t, latents)
        return latents


class InterpolationSampler:
    """The caller of the frame-interpolation denoiser (interpolation/sample.py:138-166 ``auto_inpainting_copy_no_mask``
    -> interpolation/diffusion/gaussian_diffusion.py ``ddim_sample_loop`` with eta 0, clip_denoised False, use_concat):
    respaced DDIM (respace.py:9-63: ``count`` timesteps with a fractional stride) over cat([x_t, key-frame latents], 1)
    with ``forward_with_cfg`` (cfg_scale 4.0, text = [prompt, negative prompt]).  The reference's ``p_mean_variance``
    runs the UNet TWICE per step by accident (a failed ``.sample`` attribute access re-invokes the model,
    gaussian_diffusion.py:284-291); the result is identical, so one evaluation is made here."""

    def __init__(self, unet, cfg_scale: float = 4.0, num_steps: int = 50, num_train: int = 1000):
        self.unet = unet
        self.cfg_scale = float(cfg_scale)
        betas = torch.linspace(1e-4, 2e-2, num_train, dtype=torch.float64)
        acp = torch.cumprod(1.0 - betas, dim=0)
        stride = 1 if num_steps <= 1 else (num_train - 1) / (num_steps - 1)
        self.timesteps = [round(i * stride) for i in range(num_steps)]            # ascending; sampled in reverse
        self.ab = acp[self.timesteps]
        self.ab_prev = torch.cat([torch.ones(1, dtype=torch.float64), self.ab[:-1]])

    def coefficients(self, i: int):
        """x0 = x / sqrt(ab) - sqrt(1/ab - 1) eps;  x' = sqrt(ab_prev) x0 + sqrt(1 - ab_prev) eps."""
        ab, abp = float(self.ab[i]), float(self.ab_prev[i])
        return (math.sqrt(abp) / math.sqrt(ab), math.sqrt(1.0 - abp) - math.sqrt(abp) * math.sqrt(1.0 / ab - 1.0))

    @torch.no_grad()
    def loop(self, z: torch.Tensor, x_start: torch.Tensor, text: torch.Tensor) -> torch.Tensor:
        """z, x_start: [2, 4, F, H, W] (both CFG halves, as the reference passes them); text [2, L, ctx]."""
        dev = self.unet.device
        x = z.to(device=dev, dtype=F32).contiguous()
        cond = x_start.to(device=dev, dtype=F32).contiguous()
        text = text.to(dev)
        for i in reversed(range(len(self.timesteps))):
            # forward_with_cfg (text ordered [cond, uncond]) on cat([x_t, x_start], 1); the guided eps comes back for
            # both halves and the DDIM update (eta 0) is applied to the whole batch, as gaussian_diffusion.py:587-642 does
            g = self.unet.forward_with_cfg(torch.cat([x, cond], dim=1), self.timesteps[i], encoder_hidden_states=text,
                                           cfg_scale=self.cfg_scale).contiguous()
            a, b = self.coefficients(i)
            x = ops.cfg_linear_step(g, g, 0.0, a, b, x)
        return x


# ---------------------------------------------------------------------------------------------------- video super-resolution
# the x4 upscaler's low_res_scheduler: DDPMScheduler, scaled_linear betas 1e-4 .. 2e-2 over 1000 steps
LOW_RES_ALPHAS_CUMPROD = _alphas_cumprod(1000, 1e-4, 2e-2, "scaled_linear")


def add_low_res_noise(low_res: torch.Tensor, noise: torch.Tensor, noise_level: int) -> torch.Tensor:
    """``low_res_scheduler.add_noise(low_res, noise, noise_level)``: sqrt(ab) x + sqrt(1 - ab) n with ab the
    low_res_scheduler's alpha-bar at ``noise_level`` (both factors formed in float32, as diffusers does)."""
    level = int(noise_level)
    if not 0 <= level <= VSR_CONFIG.max_noise_level:
        raise ValueError(f"noise_level must be in [0, {VSR_CONFIG.max_noise_level}], got {noise_level}")
    ab = LOW_RES_ALPHAS_CUMPROD[level]
    return float(ab.sqrt()) * low_res + float((1 - ab).sqrt()) * noise


def chunk_plan(frames: int, chunk_frames: int) -> List[Tuple[int, int]]:
    """(first frame, frame count) of every chunk of vsr/sample.py: consecutive ``chunk_frames``, the last may be shorter."""
    return [(s, min(chunk_frames, frames - s)) for s in range(0, frames, chunk_frames)]


def rank_chunks(num_chunks: int, world: int, rank: int) -> List[int]:
    """The chunks rank ``rank`` of ``world`` runs: rank, rank + world, rank + 2 world, ..."""
    return list(range(rank, num_chunks, world))


def _gather_chunks(own: Dict[int, torch.Tensor], plan, group, tail, dtype, device) -> torch.Tensor:
    """Every rank's chunks ([frames, *tail] each, keyed by chunk index) -> the whole video [F, *tail] on every rank.  Each
    rank packs its chunks into ceil(K / P) zero-padded slots of the longest chunk, one all_gather moves the equal-size
    buffers, and chunk k is read back from rank k % P, slot k // P: a copy, so the gather is exact."""
    import torch.distributed as dist
    P = dist.get_world_size(group)
    slots = -(-len(plan) // P)
    buf = torch.zeros((slots, max(n for _, n in plan)) + tuple(tail), dtype=dtype, device=device)
    for k, t in own.items():
        buf[k // P, :t.shape[0]].copy_(t)
    every = [torch.empty_like(buf) for _ in range(P)]
    dist.all_gather(every, buf, group=group)
    return torch.cat([every[k % P][k // P, :n] for k, (_, n) in enumerate(plan)])


class VSRSampler:
    """The VSR stage: StableDiffusionUpscalePipeline's loop (diffusers 0.16 order, restated by the reference in
    vsr/models/pipeline_stable_diffusion_upscale_video_3d.py:709-738) over the chunks of vsr/sample.py:100-118.

    Every chunk of ``chunk_frames`` consecutive frames is an independent pipeline call: its low-resolution frames are
    noised once (``add_low_res_noise`` at ``noise_level``), then per step ``unet(cat([x, x]), t, cat([lr, lr]), text,
    class_labels=[level, level])``, guidance ``u + g (c - u)`` and the DDIM update run as one ``cfg_linear_step``.  Each
    chunk length captures its own step graph (a video has at most two).  The default schedule is the x4 upscaler's: DDIM,
    v-prediction, scaled_linear betas 1e-4 .. 2e-2, steps_offset 1, stock diffusers 0.16 timestep spacing; pass
    ``schedule=DDIMSchedule(..., timesteps=[...])`` for another spacing.

    Noise: per chunk in chunk order, first the low-resolution noise [1,3,f,h,w], then the initial latents [1,4,f,h,w]
    (diffusers draws the image noise before ``prepare_latents``), from ``generator`` on the generator's device.  Explicit
    ``low_res_noise`` [1,3,F,h,w] / ``latents`` [1,4,F,h,w] for the whole video replace the corresponding draws.

    ``group`` (torch.distributed, NCCL): rank r runs chunks r, r + P, ...  Every rank draws every chunk's noise, so with a
    generator seeded alike on every rank the result is the single-GPU result, returned whole on every rank."""

    def __init__(self, unet, guidance_scale: float = 5.0, noise_level: int = 50, num_inference_steps: int = 50,
                 chunk_frames: int = 8, schedule: Optional[DDIMSchedule] = None):
        if not 0 <= int(noise_level) <= VSR_CONFIG.max_noise_level:
            raise ValueError(f"noise_level must be in [0, {VSR_CONFIG.max_noise_level}], got {noise_level}")
        if int(chunk_frames) < 1:
            raise ValueError(f"chunk_frames must be >= 1, got {chunk_frames}")
        if schedule is None:
            schedule = DDIMSchedule(num_inference_steps, beta_schedule="scaled_linear", prediction_type="v_prediction")
        if not isinstance(schedule, DDIMSchedule):
            raise ValueError("VSRSampler steps a DDIMSchedule")
        self.unet = unet
        self.guidance_scale = float(guidance_scale)
        self.noise_level = int(noise_level)
        self.chunk_frames = int(chunk_frames)
        self.schedule = schedule

    def _low_res(self, low_res: torch.Tensor, dev) -> torch.Tensor:
        """float [1,3,F,h,w] in [-1, 1], or uint8 frames [1,F,h,w,3] normalised as (x / 255 - 0.5) / 0.5."""
        if low_res.dtype == torch.uint8:
            if low_res.dim() != 5 or low_res.shape[-1] != 3:
                raise ValueError(f"uint8 frames must be [1,F,h,w,3], got {tuple(low_res.shape)}")
            lr = (low_res.to(dev).permute(0, 4, 1, 2, 3).to(F32) / 255 - 0.5) / 0.5
        else:
            if low_res.dim() != 5 or low_res.shape[1] != 3:
                raise ValueError(f"low_res must be float [1,3,F,h,w], got {tuple(low_res.shape)}")
            lr = low_res.to(device=dev, dtype=F32)
        if lr.shape[0] != 1:
            raise ValueError(f"VSRSampler upscales one video (batch 1), got batch {lr.shape[0]}")
        mult = 1 << (len(self.unet.cfg.block_out_channels) - 1)
        if lr.shape[3] % mult or lr.shape[4] % mult:
            raise ValueError(f"frame height and width must be multiples of {mult}, got {tuple(lr.shape[3:])}")
        return lr.contiguous()

    def _run(self, low_res, text, generator, latents, low_res_noise, group):
        """This rank's chunks -> (chunk plan, {chunk index: final latents [1,4,f,h,w]}, (h, w))."""
        dev = self.unet.device
        lr = self._low_res(low_res, dev)
        if text.dim() != 3 or text.shape[0] != 2:
            raise ValueError(f"text must be cat([negative, positive]) [2, L, C], got {tuple(text.shape)}")
        _, _, Fr, h, w = lr.shape
        for name, t, c in (("low_res_noise", low_res_noise, 3), ("latents", latents, 4)):
            if t is not None and tuple(t.shape) != (1, c, Fr, h, w):
                raise ValueError(f"{name} must be {(1, c, Fr, h, w)}, got {tuple(t.shape)}")
        text = text.to(dev)
        plan = chunk_plan(Fr, self.chunk_frames)
        if group is None:
            mine = set(range(len(plan)))
        else:
            import torch.distributed as dist
            mine = set(rank_chunks(len(plan), dist.get_world_size(group), dist.get_rank(group)))
        out = {}
        for k, (s, n) in enumerate(plan):
            sl = slice(s, s + n)
            nz = _noise_like((1, 3, n, h, w), generator, None if low_res_noise is None else low_res_noise[:, :, sl], dev)
            x = _noise_like((1, 4, n, h, w), generator, None if latents is None else latents[:, :, sl], dev)
            if k in mine:
                out[k] = self._chunk(lr[:, :, sl], nz, x, text)
        return plan, out, (h, w)

    def _chunk(self, lr, lr_noise, x, text):
        sched = self.schedule
        lr = add_low_res_noise(lr, lr_noise, self.noise_level)
        lr2 = torch.cat([lr, lr])
        labels = torch.tensor([self.noise_level] * 2)
        x = x * sched.init_noise_sigma
        for i, t in enumerate(sched.timesteps):
            out = self.unet(torch.cat([x, x]), t, lr2, encoder_hidden_states=text, class_labels=labels).sample
            a, b, _ = sched.coefficients(i)
            x = ops.cfg_linear_step(out[0:1], out[1:2], self.guidance_scale, a, b, x)
        return x

    @torch.no_grad()
    def loop(self, low_res: torch.Tensor, text: torch.Tensor, generator: Optional[torch.Generator] = None,
             latents: Optional[torch.Tensor] = None, low_res_noise: Optional[torch.Tensor] = None,
             group=None) -> torch.Tensor:
        """low_res (float [1,3,F,h,w] or uint8 [1,F,h,w,3]), text [2, L, 1024] -> final latents fp32 [1,4,F,h,w] on the
        UNet's device (the whole video on every rank of ``group``)."""
        plan, out, (h, w) = self._run(low_res, text, generator, latents, low_res_noise, group)
        if group is None:
            return torch.cat([out[k] for k in range(len(plan))], dim=2)
        own = {k: v[0].transpose(0, 1) for k, v in out.items()}
        full = _gather_chunks(own, plan, group, (4, h, w), F32, self.unet.device)
        return full.transpose(0, 1).unsqueeze(0).contiguous()

    @torch.no_grad()
    def upscale(self, low_res: torch.Tensor, text: torch.Tensor, vae, generator: Optional[torch.Generator] = None,
                latents: Optional[torch.Tensor] = None, low_res_noise: Optional[torch.Tensor] = None,
                group=None) -> torch.Tensor:
        """``loop`` then ``vae.decode_latents`` (``VAEDecoder.x4_upscaler()``) chunk by chunk, as every pipeline call of
        the reference decodes its own chunk -> uint8 [1,F,4h,4w,3] on the host.  With ``group`` a rank decodes only its
        own chunks and the uint8 frames are gathered, so every rank returns the whole video."""
        plan, out, (h, w) = self._run(low_res, text, generator, latents, low_res_noise, group)
        frames = {k: vae.decode_latents(v)[0] for k, v in out.items()}
        if group is None:
            return torch.cat([frames[k] for k in range(len(plan))])[None]
        s = vae.upscale
        tail = (s * h, s * w, 3)
        return _gather_chunks(frames, plan, group, tail, torch.uint8, self.unet.device).cpu()[None]
