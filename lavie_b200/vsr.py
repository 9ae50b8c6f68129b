"""Drop-in replacement for the reference ``UNet3DVSRModel`` (vsr/models/unet.py:102-646), the x4 video
super-resolution denoiser (SURVEY.md 8f row N2, BASELINE config 5).

Same call signature ``forward(sample, timestep, low_res, encoder_hidden_states, class_labels) -> .sample`` and the same
1158-key ``state_dict`` as the reference built from ``vsr/configs/unet_3d_config.json``.  The weight packer, the
transformer block, the step walk, the forward body and the step graph are those of the base denoiser
(``UNet3DConditionModel`` in lavie_b200/unet.py), which follow the config's ``variant``, ``only_cross_attention``,
``num_class_embeds`` and ``temporal_modules`` there: the noise-level class embedding (``lavie_embedding_add``),
transformer blocks whose first attention reads the text on the three high-resolution levels (their K/V projections join
the one text GEMM of the step), Linear proj_in / proj_out.  This module adds what only the VSR UNet has:

* ``ResnetBlock3DCNN`` -- (k,1,1) convolutions over FRAMES -- as an implicit GEMM with K = k*C on a frame-padded map
  (``lavie_frame_conv_bf16``: the same TMA box shifted by whole frames; the GroupNorm-apply + SiLU pass writes straight
  into the padded buffer, whose pad frames stay zero), also the temporal ResNet in front of every transformer;
* a ``TemporalModule3D`` (frame ResNet (5,1,1) -> spatial ResNet -> 1x1 shift conv -> + input) behind every block;
* the forward signature with ``low_res`` and ``class_labels``, and frame sharding over the NCCL back end only.

There is no PyTorch compute fallback; the module raises on non-CUDA parameters like the base one.
"""
from __future__ import annotations

from typing import Dict, Optional, Union

import torch

from . import ops
from .config import VSR_CONFIG, UNetConfig
from .unet import BF16, F32, UNet3DConditionModel


def pack_frame_conv(w: torch.Tensor) -> torch.Tensor:
    """nn.Conv3d weight [Cout, Cin, k, 1, 1] -> [Cout, k*Cin] with K ordered (tap, cin) = the frame-conv GEMM's K order."""
    co, ci, k = w.shape[:3]
    return w.reshape(co, ci, k).permute(0, 2, 1).reshape(co, k * ci).contiguous()


class UNet3DVSRModel(UNet3DConditionModel):
    """B200-native LaVie VSR denoiser (bf16 activations, fp32 accumulation)."""
    _VARIANTS = ("vsr",)
    _TAPS = ("down0", "mid")            # behind the first and the mid TemporalModule3D (tests/golden/make_golden_vsr.py)

    def __init__(self, config: UNetConfig = VSR_CONFIG, use_cuda_graph: bool = True):
        super().__init__(config, use_cuda_graph=use_cuda_graph, check_mode=False)
        self._padbufs: Dict[tuple, torch.Tensor] = {}

    def set_frame_sharding(self, group=None, backend: str = "nccl", frame_counts=None):
        """Frame sharding of the VSR denoiser (BASELINE config 5): every rank of `group` holds F / P consecutive frames of
        one CFG half.  Per-frame work is shard-local; the 5-D GroupNorm sums are all-reduced, the tokens go all-to-all
        around every temporal attention (both as in the base model, NCCL back end), and every (k,1,1) frame convolution
        first receives k//2 halo frames of its (GroupNorm-applied) input from each neighbour (NCCL send / recv).  The
        peer-memory back end of the base model is not wired to this variant.  Sharded steps run eagerly (no step graph)."""
        if group is not None and (backend != "nccl" or frame_counts is not None):
            raise NotImplementedError("the VSR denoiser shards equal frame counts over the NCCL back end only")
        super().set_frame_sharding(group, backend="nccl" if group is not None else "p2p")
        self._padbufs = {}          # pad frames that held halos must not be mistaken for the zero padding of an un-sharded run

    def _invalidate(self):
        super()._invalidate()
        self._padbufs = {}

    def _only_cross_for(self, p: str) -> bool:
        """only_cross_attention of the level a transformer prefix belongs to (vsr/models/unet.py:134-139, 272)."""
        oca = self.cfg.only_cross_attention
        parts = p.split(".")
        if parts[0] == "mid_block":
            return bool(oca[-1])
        i = int(parts[1])
        return bool(oca[i] if parts[0] == "down_blocks" else oca[len(oca) - 1 - i])

    # ------------------------------------------------------------------ blocks
    def _padbuf(self, k: int, B: int, Fr: int, HW: int, C: int, dev) -> torch.Tensor:
        """[B, (F + k - 1) * HW, C] bf16 whose k//2 leading / trailing frames are zero and stay zero: every user writes the
        F interior frames only.  One buffer per shape: its producer (GroupNorm apply) and its only consumer (the frame
        conv) are adjacent on the stream."""
        key = (k, B, Fr, HW, C)
        buf = self._padbufs.get(key)
        if buf is None:
            buf = torch.zeros((B, (Fr + k - 1) * HW, C), dtype=BF16, device=dev)
            self._padbufs[key] = buf
        return buf

    def _frame_conv_block(self, x, ss, B, Fr, HW, k, w, bias, row_bias, residual):
        """GroupNorm apply + SiLU into the frame-padded buffer, then the (k,1,1) conv; one launch pair per batch item."""
        rps = Fr * HW
        C = x.shape[1]
        buf = self._padbuf(k, B, Fr, HW, C, x.device)
        lo = (k // 2) * HW
        out = torch.empty((B * rps, w.shape[0]), dtype=BF16, device=x.device)
        # the consumer's GroupNorm statistics come out of the conv's epilogue (one buffer, each item fills its slabs)
        cs = ops._new_colsums(B * rps, w.shape[0], x.device) if (ops.FUSE_GN_STATS and rps % 32 == 0) else None
        for b in range(B):
            rows = slice(b * rps, (b + 1) * rps)
            ops.groupnorm_apply(x[rows], ss[b:b + 1], 1, rps, True, out=buf[b, lo:lo + rps])
            if self._shard is not None:
                self._exchange_frame_halo(buf[b], k // 2, Fr, HW)
            ops.frame_conv(buf[b], k, HW, w, bias=bias, row_bias=None if row_bias is None else row_bias[b:b + 1],
                           rows_per_batch=rps, residual=None if residual is None else residual[rows], out=out[rows],
                           colsums_out=None if cs is None else cs[b * rps // 32:(b + 1) * rps // 32])
        if cs is not None:
            out._gn_colsums = cs
        return out

    def _exchange_frame_halo(self, buf, pad: int, Fr: int, HW: int):
        """Frame-sharded (k,1,1) conv: fill the pad frames from the neighbours (lavie_b200.sharding.exchange_frame_halo)."""
        from .sharding import exchange_frame_halo
        group, P, idx = self._shard
        exchange_frame_halo(buf, pad, Fr, HW, group, P, idx)

    def _resnet_cnn(self, p, x, temb_all, B, Fr, HW):
        """ResnetBlock3DCNN.forward (vsr/models/resnet.py:284-316): both GroupNorms see the 5-D tensor (eps 1e-6)."""
        r = self._packed[p]
        rps = Fr * HW
        ss = self._gn5_scale_shift(x, None, B, rps, r["g1"], r["b1"], 1e-6)
        rb = None
        if p in self._packed["temb_slices"]:
            off, cout = self._packed["temb_slices"][p]
            rb = temb_all[:, off:off + cout]
        h = self._frame_conv_block(x, ss, B, Fr, HW, r["k"], r["w1"], r["cb1"], rb, None)
        ss = self._gn5_scale_shift(h, None, B, rps, r["g2"], r["b2"], 1e-6)
        return self._frame_conv_block(h, ss, B, Fr, HW, 3, r["w2"], r["cb2"], None, x)

    def _temporal_module(self, p, x, temb_all, B, Fr, H, W):
        """TemporalModule3D.forward (vsr/models/temporal_module.py:151-178; no attention layers, no video condition)."""
        h = self._resnet_cnn(f"{p}.resblocks_3d_t", x, temb_all, B, Fr, H * W)
        h = self._resnet(f"{p}.resblocks_3d_s", h, None, temb_all, B, Fr, H, W)
        w, b = self._packed[f"{p}.shift_conv"]
        return ops.gemm(h, w, bias=b, residual=x, stats=True)

    # ------------------------------------------------------------------ public forward
    @torch.no_grad()
    def forward(self, sample: torch.Tensor, timestep: Union[torch.Tensor, float, int], low_res: torch.Tensor,
                encoder_hidden_states: torch.Tensor = None, class_labels=20, low_res_clean=None, attention_mask=None,
                return_dict: bool = True, taps: Optional[dict] = None):
        """Same contract as vsr/models/unet.py:408-590: ``sample`` [B,4,F,H,W] noisy latent, ``low_res`` [B,3,F,H,W] the
        (noised) low-resolution frames, ``class_labels`` the noise level (int or int64 [B], <= max_noise_level).
        ``attention_mask`` never reaches the blocks in the reference either (unet_blocks.py); ``low_res_clean`` is unused
        there too."""
        if encoder_hidden_states is None:
            raise ValueError("encoder_hidden_states is required")
        if sample.dim() != 5 or low_res.dim() != 5 or sample.shape[0] != low_res.shape[0] or \
                sample.shape[2:] != low_res.shape[2:]:
            raise ValueError(f"sample [B,4,F,H,W] and low_res [B,3,F,H,W] expected, got {tuple(sample.shape)}, "
                             f"{tuple(low_res.shape)}")
        B, C, Fr, H, W = sample.shape
        n_down = len(self.cfg.block_out_channels) - 1
        if C + low_res.shape[1] != self.cfg.in_channels or H % (1 << n_down) or W % (1 << n_down):
            raise ValueError(f"sample + low_res need {self.cfg.in_channels} channels and H, W multiples of {1 << n_down}")
        if encoder_hidden_states.shape[0] != B or encoder_hidden_states.shape[-1] != self.cfg.cross_attention_dim:
            raise ValueError(f"encoder_hidden_states must be [B, L, {self.cfg.cross_attention_dim}]")
        if class_labels is None:
            raise ValueError("class_labels should be provided when num_class_embeds > 0")        # unet.py:496
        dev = self.device
        labels = torch.as_tensor(class_labels, dtype=torch.int64).reshape(-1)
        if bool((labels > self.cfg.max_noise_level).any()):
            raise ValueError(f"`noise_level` has to be <= {self.cfg.max_noise_level} but is {class_labels}")   # :499
        labels = labels.expand(B).contiguous().to(dev, non_blocking=True)
        x = torch.cat([sample.to(device=dev, dtype=F32), low_res.to(device=dev, dtype=F32)], dim=1)     # unet.py:446
        if self.cfg.center_input_sample:
            x = 2 * x - 1.0
        return self._forward(x, sample.dtype, timestep, encoder_hidden_states, return_dict, taps, labels=labels)

    @torch.no_grad()
    def forward_with_cfg(self, x, t, low_res, encoder_hidden_states=None, class_labels=20, cfg_scale: float = 4.0,
                         use_fp16: bool = False) -> torch.Tensor:
        """vsr/models/unet.py:592-618: the first half of the batch runs against [cond, uncond] conditioning; the guided
        noise is returned for both halves."""
        n = len(x) // 2
        combined = torch.cat([x[:n], x[:n]], dim=0)
        return self._guided(self.forward(combined, t, low_res, encoder_hidden_states, class_labels).sample, cfg_scale)
