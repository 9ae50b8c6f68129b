"""Drop-in replacement for the reference ``UNet3DConditionModel`` (base/models/unet.py:98-512).

Same call signature ``forward(sample, timestep, encoder_hidden_states, ...) -> .sample``, same 830-key
``state_dict`` (so ``lavie_base.pt`` or random-init weights of the architecture load with
``load_state_dict(strict=True)``), same helper methods the pipelines call.  The module tree only HOLDS the
parameters under the reference's names; the forward pass is a flat sequence of C-ABI kernel launches
(``lavie_b200.ops``) over channels-last bf16 activations.  There is no PyTorch compute fallback.
"""
from __future__ import annotations

from dataclasses import dataclass
from types import SimpleNamespace
from typing import Dict, Optional, Tuple, Union

import torch
from torch import nn

from . import ops
from .config import BASE_CONFIG, UNetConfig, param_spec
from .packing import (head_pitch, interleave_geglu, pack_conv1x1, pack_conv3x3, pack_upsample_conv3x3, pad_heads,
                      rel_pos_bias_table, rope_table)

BF16 = torch.bfloat16
F32 = torch.float32


@dataclass
class UNet3DConditionOutput:
    """Mirror of base/models/unet.py:93-95."""
    sample: torch.Tensor

    def __getitem__(self, i):
        return (self.sample,)[i]

    def to_tuple(self):
        return (self.sample,)


class _Config(SimpleNamespace):
    """``unet.config`` as the pipelines read it (attribute and item access, pipeline_videogen.py:141-160,606)."""

    def __getitem__(self, k):
        return getattr(self, k)

    def __contains__(self, k):
        return hasattr(self, k)

    def get(self, k, default=None):
        return getattr(self, k, default)


class _RotaryFreqs(nn.Module):
    """Holds ``rotary_emb.freqs`` (rotary_embedding_torch keeps it as a frozen Parameter)."""

    def __init__(self, n):
        super().__init__()
        self.freqs = nn.Parameter(torch.empty(n), requires_grad=False)


def _leaf_for(key_prefix: str, names: Dict[str, Tuple[int, ...]]) -> nn.Module:
    """A real torch module (uninitialised storage) for one parameter group, so `.modules()` probing, `.to()` and
    `state_dict()` behave as usual.  The leaves only HOLD parameters: forward() runs from packed copies, which are
    refreshed whenever a parameter object or its version counter changes (in-place edits, LoRA merges).  Wrapping a leaf
    (PEFT's target_modules=["to_q","to_k","to_v","to_out.0"], fine_tuning.py:296-308) changes the key set and is rejected
    in `_pack` -- merge the adapter into the base weights first."""
    w = names.get("weight")
    has_bias = "bias" in names
    last = key_prefix.rsplit(".", 1)[-1]
    if "freqs" in names:
        return _RotaryFreqs(names["freqs"][0])
    if last in ("relative_attention_bias", "class_embedding"):
        return torch.nn.utils.skip_init(nn.Embedding, w[0], w[1])
    if len(w) == 5:                      # the VSR UNet's (k,1,1) frame convolutions (vsr/models/resnet.py:253-254,269)
        return torch.nn.utils.skip_init(nn.Conv3d, w[1], w[0], tuple(w[2:]), padding=(w[2] // 2, 0, 0), bias=has_bias)
    if len(w) == 4:
        k = w[2]
        return torch.nn.utils.skip_init(nn.Conv2d, w[1], w[0], k, padding=k // 2, bias=has_bias)
    if len(w) == 2:
        return torch.nn.utils.skip_init(nn.Linear, w[1], w[0], bias=has_bias)
    if last in ("norm1", "norm2", "norm3", "norm_temp", "norm_temporal") and ".transformer_blocks." in key_prefix:
        return nn.LayerNorm(w[0])
    return nn.GroupNorm(32, w[0])


def _install(root: nn.Module, path: str, leaf: nn.Module) -> None:
    parts = path.split(".")
    cur = root
    for p in parts[:-1]:
        nxt = cur._modules.get(p)
        if nxt is None:
            nxt = nn.Module()
            cur.add_module(p, nxt)
        cur = nxt
    cur.add_module(parts[-1], leaf)


class UNet3DConditionModel(nn.Module):
    """B200-native LaVie base denoiser (and, by ``config.variant``, the interpolation one; the VSR one is the subclass
    lavie_b200.vsr.UNet3DVSRModel).  ``use_cuda_graph`` replays the whole step from one captured CUDA graph per
    input geometry (the reference launches ~1.9k kernels per step from Python)."""
    _VARIANTS = ("base", "interp")
    _TAPS = ("emb", "conv_in", "down0_res0", "down0_attn0", "mid", "up_out")     # the oracle's tap points (forward(taps=))

    def __init__(self, config: UNetConfig = BASE_CONFIG, use_cuda_graph: bool = True, check_mode: bool = False):
        """``check_mode=True``: the fp32-accumulate check mode of BASELINE's north star (rel-L2 <= 1e-3 vs the reference
        fp32 forward): same launch sequence, activations as split-bf16 triples through the same tcgen05 GEMM / conv
        mainloops with fp32 epilogues, fp32 norms and attention (lavie_b200/check.py).  For parity attribution, not speed."""
        super().__init__()
        if getattr(config, "variant", "base") not in self._VARIANTS:
            raise NotImplementedError(f"UNet variant {config.variant!r} is not served by {type(self).__name__} "
                                      f"(variants: {self._VARIANTS}; the VSR denoiser is lavie_b200.vsr.UNet3DVSRModel)")
        if check_mode and config.variant == "vsr":
            raise NotImplementedError("check mode covers the base and interpolation denoisers")
        self.cfg = config
        self.config = _Config(**config.to_dict())
        self.sample_size = config.sample_size
        self.check_mode = bool(check_mode)
        if self.check_mode:
            from . import check as _check
            self._k = _check
        else:
            self._k = ops
        self.use_cuda_graph = use_cuda_graph and not self.check_mode
        groups: Dict[str, Dict[str, Tuple[int, ...]]] = {}
        for key, shape in param_spec(config).items():
            prefix, leaf = key.rsplit(".", 1)
            groups.setdefault(prefix, {})[leaf] = shape
        for prefix, names in groups.items():
            _install(self, prefix, _leaf_for(prefix, names))
        self._packed = None
        self._shard = None            # (process group, P, index) when the frames of one CFG half span P GPUs
        self._shard_backend = "p2p"
        self._peer = None
        self._frame_counts = None
        self._retired_peers: list = []
        self._param_versions = None
        self._param_list = None
        self._scale_one = None
        self._graphs: Dict[tuple, dict] = {}
        self._tables: Dict[tuple, tuple] = {}
        self._text_seen = None        # (tensor, version, graph key) whose K/V projections sit in that graph's buffer
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._invalidate())

    # ------------------------------------------------------------------ reference-compatible helpers
    @property
    def dtype(self):
        return self.conv_in.weight.dtype

    @property
    def device(self):
        return self.conv_in.weight.device

    def set_use_memory_efficient_attention_xformers(self, valid: bool = True, attention_op=None):
        """No-op: attention always runs in the fused tcgen05 kernel (reference hook: attention.py:482-509)."""

    enable_xformers_memory_efficient_attention = set_use_memory_efficient_attention_xformers

    def disable_xformers_memory_efficient_attention(self):
        pass

    def set_attention_slice(self, slice_size):
        """No-op: the flash kernel never materialises the score matrix (reference: unet.py:297-360)."""

    def _set_gradient_checkpointing(self, module, value=False):
        pass

    def _invalidate(self):
        """Drop the packed (kernel-layout) weight copies and every captured step graph.  Called automatically after
        ``load_state_dict`` / ``.to()`` and when a parameter's version counter moved (in-place edits such as
        ``param.data.copy_`` or a LoRA merge); replacing or wrapping a leaf module (PEFT) is detected in ``forward``."""
        self._packed = None
        self._param_versions = None
        self._param_list = None
        self._graphs.clear()
        self._tables.clear()
        self._text_seen = None

    def _weights_fingerprint(self):
        # version counters of the parameters seen at packing time (~0.1 ms for 830 tensors); module surgery after the
        # first forward (wrapping a leaf) is NOT seen here -- call _invalidate() after it
        if self._param_list is None:
            self._param_list = list(self.parameters())
        return tuple(p._version for p in self._param_list)

    def packed_tensors(self):
        """Every device tensor of the packed weights (bench.py reports the per-rank weight bytes)."""
        out = []

        def walk(v):
            if torch.is_tensor(v):
                out.append(v)
            elif isinstance(v, dict):
                for x in v.values():
                    walk(x)
            elif isinstance(v, (tuple, list)):
                for x in v:
                    walk(x)
        walk(self._packed or {})
        return out

    def _apply(self, fn, *a, **kw):
        out = super()._apply(fn, *a, **kw)
        self._invalidate()
        return out

    def set_frame_sharding(self, group=None, backend: str = "p2p", frame_counts=None):
        """Frame sharding (SURVEY.md 8e): this rank holds F/P consecutive frames of the video; `group` is the
        torch.distributed process group of the P ranks that share one CFG half (rank order = frame order).
        Per-frame work (convs, per-frame GroupNorm, LayerNorm, spatial / cross attention, FF) runs shard-local;
        5-D GroupNorm statistics are all-reduced and the tokens are exchanged all-to-all around every temporal
        attention.  backend "p2p" (default) runs those exchanges inside this library's kernels over NVLink peer memory
        (csrc/p2p.cu); "nccl" keeps the exchanges in torch.distributed collectives.  `None` switches sharding off.
        `frame_counts` (p2p only): frames held by each rank of the group when the shards are uneven, e.g. [16,15,15,15]
        for the 61-frame interpolation model (default: every rank holds as many frames as this one).  The interpolation
        variant additionally exchanges the SparseCausal halo (frame 0 of the video + the left neighbour's last frame)."""
        if backend not in ("p2p", "nccl"):
            raise ValueError("backend must be 'p2p' or 'nccl'")
        if group is not None and self.check_mode:
            raise NotImplementedError("frame sharding is not available in check mode")
        if group is None:
            self._shard = None
        else:
            import torch.distributed as dist
            P = dist.get_world_size(group)
            self._shard = None if P == 1 else (group, P, dist.get_rank(group))
            if frame_counts is not None:
                if backend != "p2p" or len(frame_counts) != P:
                    raise ValueError("frame_counts needs the p2p backend and one entry per rank of the group")
        self._frame_counts = list(frame_counts) if (frame_counts is not None and self._shard is not None) else None
        self._shard_backend = backend
        self._peer = None
        self._graphs.clear()

    def _frames(self, f_local: int):
        """(global frame count, global index of this rank's first frame) of the sharded video."""
        _, P, idx = self._shard
        if self._frame_counts is None:
            return f_local * P, idx * f_local
        assert self._frame_counts[idx] == f_local, (self._frame_counts, idx, f_local)
        return sum(self._frame_counts), sum(self._frame_counts[:idx])

    def _peer_ctx(self, token_bytes: int, halo_bytes: int = 0, frame_off: int = -1):
        """Symmetric buffers of the frame group, created at the first sharded forward (collective call)."""
        if (self._peer is None or self._peer.token_bytes < token_bytes or self._peer.halo_bytes < halo_bytes
                or self._peer.frame_off != frame_off):
            from .p2p import PeerContext
            # graphs captured against the previous context have its peer pointers and epoch counter baked in
            self._graphs.clear()
            self._retired_peers.append(self._peer)      # keep the old symmetric buffers mapped until the module dies
            self._peer = PeerContext(self._shard[0], token_bytes, self.device, frame_off, halo_bytes)
        return self._peer

    def _gn5(self, x, x2, B, rows_local, gamma, beta, eps, silu):
        """nn.GroupNorm on the 5-D tensor: statistics span ALL frames (resnet.py:180,191; unet.py:504)."""
        if self._shard is None:
            return self._k.groupnorm(x, B, rows_local, gamma, beta, eps, silu=silu, x2=x2)
        ss = self._gn5_scale_shift(x, x2, B, rows_local, gamma, beta, eps)
        return ops.groupnorm_apply(x, ss, B, rows_local, silu, x2=x2)

    def _gn5_scale_shift(self, x, x2, B, rows_local, gamma, beta, eps):
        if self._shard is None:
            return self._k.groupnorm_scale_shift(x, B, rows_local, gamma, beta, eps, x2=x2)
        if self._shard_backend == "p2p":
            f_loc, f_total = self._shard_frames        # rows of one sample over ALL frame shards (shards may be uneven)
            return self._peer.gn_scale_shift(x, x2, B, rows_local, gamma, beta, eps,
                                             rows_global=rows_local // f_loc * f_total)
        import torch.distributed as dist
        group, P, _ = self._shard
        C = x.shape[1] + (x2.shape[1] if x2 is not None else 0)
        sums = ops.groupnorm_sums(x, B, rows_local, x2=x2)                  # fp64 [B, 32, 2] (producers' column sums if any)
        dist.all_reduce(sums, group=group)                                   # 512 B per call
        return ops.groupnorm_finalize_sums(sums, C, rows_local * P * (C // 32), gamma, beta, eps)

    def init_synthetic(self, seed: int = 0):
        """Deterministic random-init weights (lavie_b200.synthetic), loaded through the normal state_dict path."""
        from .synthetic import synthetic_state_dict
        sd = synthetic_state_dict(self.cfg, seed)
        self.load_state_dict(sd, strict=True)
        return self

    # ------------------------------------------------------------------ weight packing (post-load)
    def _pack(self):
        sd = {k: v.detach() for k, v in self.state_dict().items()}
        spec = param_spec(self.cfg)
        missing = [k for k in spec if k not in sd]
        if missing:
            raise RuntimeError(f"state_dict no longer has the reference layout (first missing key: {missing[0]}); "
                               "wrapped / replaced leaf modules (e.g. un-merged LoRA adapters) are not executed by the "
                               "fused path -- merge them into the base weights first")
        dev = self.device
        if dev.type != "cuda":
            raise RuntimeError(f"lavie_b200.{type(self).__name__} runs on CUDA (sm_100a) only; move it with .to('cuda')")
        heads = self.cfg.heads
        P: Dict[str, object] = {}

        def f32(k):
            return sd[k].to(device=dev, dtype=F32).contiguous()

        K = self._k

        def pack_conv3x3_(w):            # layout only; precision is decided by K.weight
            return pack_conv3x3(w, dtype=None)

        def pack_conv1x1_(w):            # 1x1 conv or Linear (the VSR model's proj_in / proj_out)
            return pack_conv1x1(w, dtype=None)

        def b16(t):                      # kernel-side weight matrix: bf16 (check mode: an (hi, lo) bf16 pair)
            return K.weight(t, dev)

        # every time_emb_proj in one matrix and every text K/V projection in another, rows in param_spec order
        temb_w, temb_b, temb_slices = [], [], {}
        kv_w = []
        temb_off = 0
        kv_off = 0

        for key, shape in spec.items():
            if not key.endswith(".conv1.weight"):
                continue
            p = key[: -len(".conv1.weight")]
            r = {"g1": f32(f"{p}.norm1.weight"), "b1": f32(f"{p}.norm1.bias"), "cb1": f32(f"{p}.conv1.bias"),
                 "g2": f32(f"{p}.norm2.weight"), "b2": f32(f"{p}.norm2.bias"), "cb2": f32(f"{p}.conv2.bias")}
            if len(shape) == 5:                                   # ResnetBlock3DCNN (vsr/models/resnet.py:220-316)
                from .vsr import pack_frame_conv
                r["k"] = shape[2]
                r["w1"] = b16(pack_frame_conv(sd[f"{p}.conv1.weight"]))
                r["w2"] = b16(pack_frame_conv(sd[f"{p}.conv2.weight"]))
            else:                                                 # ResnetBlock3D
                r["w1"] = b16(pack_conv3x3_(sd[f"{p}.conv1.weight"]))
                r["w2"] = b16(pack_conv3x3_(sd[f"{p}.conv2.weight"]))
                if f"{p}.conv_shortcut.weight" in sd:
                    r["wsc"] = b16(pack_conv1x1_(sd[f"{p}.conv_shortcut.weight"]))
                    r["bsc"] = f32(f"{p}.conv_shortcut.bias")
                if "temporal_block" in p:                         # TemporalModule3D builds it with the default eps
                    r["eps"] = 1e-6
            if f"{p}.time_emb_proj.weight" in sd:
                temb_w.append(sd[f"{p}.time_emb_proj.weight"])
                temb_b.append(sd[f"{p}.time_emb_proj.bias"])
                temb_slices[p] = (temb_off, shape[0])
                temb_off += shape[0]
            P[p] = r

        # the VSR tree names the temporal attention and its LayerNorm attn_temporal / norm_temporal
        tmp = "temporal" if self.cfg.variant == "vsr" else "temp"
        for key in spec:
            if not key.endswith(".proj_in.weight"):
                continue
            p = key[: -len(".proj_in.weight")]
            b = f"{p}.transformer_blocks.0"
            C = sd[f"{p}.norm.weight"].shape[0]
            d = C // heads
            hp = heads * head_pitch(d)
            only_cross = any(self.cfg.only_cross_attention) and self._only_cross_for(p)

            def qkv(a):
                return b16(torch.cat([pad_heads(sd[f"{b}.{a}.to_{x}.weight"], heads) for x in "qkv"], 0))

            def text_kv(a):              # rows of the one text K/V GEMM; returns their first column
                nonlocal kv_off
                kv_w.append(pad_heads(sd[f"{b}.{a}.to_k.weight"], heads))
                kv_w.append(pad_heads(sd[f"{b}.{a}.to_v.weight"], heads))
                kv_off += 2 * hp
                return kv_off - 2 * hp

            t = {"C": C, "d": d, "pitch": head_pitch(d), "hp": hp, "only_cross": only_cross,
                 "gn_g": f32(f"{p}.norm.weight"), "gn_b": f32(f"{p}.norm.bias"),
                 "w_in": b16(pack_conv1x1_(sd[f"{p}.proj_in.weight"])), "b_in": f32(f"{p}.proj_in.bias"),
                 "w_out": b16(pack_conv1x1_(sd[f"{p}.proj_out.weight"])), "b_out": f32(f"{p}.proj_out.bias")}
            for n, src in (("norm1", "norm1"), ("norm2", "norm2"), ("norm_temp", f"norm_{tmp}"), ("norm3", "norm3")):
                t[f"{n}_g"] = f32(f"{b}.{src}.weight")
                t[f"{n}_b"] = f32(f"{b}.{src}.bias")
            if only_cross:               # attn1 reads the text (the VSR model's only_cross_attention levels)
                t["attn1_q"] = b16(pad_heads(sd[f"{b}.attn1.to_q.weight"], heads))
                t["attn1_kv_off"] = text_kv("attn1")
            else:
                t["attn1_qkv"] = qkv("attn1")
            t["attn_temp_qkv"] = qkv(f"attn_{tmp}")
            for a, src in (("attn1", "attn1"), ("attn2", "attn2"), ("attn_temp", f"attn_{tmp}")):
                t[f"{a}_wo"] = b16(sd[f"{b}.{src}.to_out.0.weight"])
                t[f"{a}_bo"] = f32(f"{b}.{src}.to_out.0.bias")
            t["attn2_q"] = b16(pad_heads(sd[f"{b}.attn2.to_q.weight"], heads))
            t["kv_off"] = text_kv("attn2")
            wi, bi = interleave_geglu(sd[f"{b}.ff.net.0.proj.weight"], sd[f"{b}.ff.net.0.proj.bias"])
            t["ff1_w"], t["ff1_b"] = b16(wi), bi.to(device=dev, dtype=F32).contiguous()
            t["ff2_w"], t["ff2_b"] = b16(sd[f"{b}.ff.net.2.weight"]), f32(f"{b}.ff.net.2.bias")
            if self.cfg.variant != "interp":    # the interpolation model's temporal attention has neither (SURVEY 2 #13)
                t["rel_emb"] = f32(f"{b}.attn_{tmp}.time_rel_pos_bias.relative_attention_bias.weight")
                t["freqs"] = f32(f"{b}.attn_{tmp}.rotary_emb.freqs")
            P[p] = t

        for key in spec:
            if key.endswith(".shift_conv.weight"):                # TemporalModule3D's 1x1 conv
                p = key[: -len(".shift_conv.weight")]
                P[f"{p}.shift_conv"] = (b16(pack_conv1x1_(sd[key])), f32(f"{p}.shift_conv.bias"))
        for i in range(len(self.cfg.block_out_channels) - 1):
            P[f"down_blocks.{i}.downsamplers.0.conv"] = (
                b16(pack_conv3x3_(sd[f"down_blocks.{i}.downsamplers.0.conv.weight"])),
                f32(f"down_blocks.{i}.downsamplers.0.conv.bias"))
            P[f"up_blocks.{i}.upsamplers.0.conv"] = (
                b16(pack_conv3x3_(sd[f"up_blocks.{i}.upsamplers.0.conv.weight"])),
                f32(f"up_blocks.{i}.upsamplers.0.conv.bias"))
            if not self.check_mode:      # the fused upsample + conv reads phase-summed 2x2 taps (packing.py)
                P[f"up_blocks.{i}.upsamplers.0.conv4"] = pack_upsample_conv3x3(
                    sd[f"up_blocks.{i}.upsamplers.0.conv.weight"]).to(dev)
        boc0 = self.cfg.block_out_channels[0]
        P["conv_in"] = (f32("conv_in.weight"), f32("conv_in.bias"))
        if not self.check_mode:          # bf16 path: explicit im2col of the few input channels + one GEMM
            P["conv_in_tc"] = (ops.pack_conv_in(sd["conv_in.weight"], dev), f32("conv_in.bias"))
        P["conv_out"] = (sd["conv_out.weight"].permute(0, 2, 3, 1).to(device=dev, dtype=F32).contiguous(),
                         f32("conv_out.bias"))
        if not self.check_mode and boc0 % 64 == 0:
            # bf16 path: conv_out runs on the tensor cores with its Cout filters zero-padded to one 32-column chunk
            co = sd["conv_out.weight"].shape[0]
            wp = torch.zeros((ops.CONV_OUT_PAD, 9 * boc0), dtype=F32)
            wp[:co] = pack_conv3x3(sd["conv_out.weight"].float().cpu(), dtype=None)
            bp = torch.zeros(ops.CONV_OUT_PAD, dtype=F32)
            bp[:co] = sd["conv_out.bias"].float().cpu()
            P["conv_out_tc"] = (wp.to(device=dev, dtype=BF16).contiguous(), bp.to(dev), co)
        P["norm_out"] = (f32("conv_norm_out.weight"), f32("conv_norm_out.bias"))
        P["time1"] = (K.weight_small(sd["time_embedding.linear_1.weight"], dev), f32("time_embedding.linear_1.bias"))
        P["time2"] = (K.weight_small(sd["time_embedding.linear_2.weight"], dev), f32("time_embedding.linear_2.bias"))
        if self.cfg.num_class_embeds:
            P["class_emb"] = f32("class_embedding.weight")
        P["temb_w"] = K.weight_small(torch.cat(temb_w, 0), dev)
        P["temb_b"] = torch.cat(temb_b, 0).to(device=dev, dtype=F32).contiguous()
        P["temb_slices"] = temb_slices
        P["kv_w"] = b16(torch.cat(kv_w, 0))
        self._packed = P
        return P

    def _frame_tables(self, prefix: str, frames: int):
        key = (prefix, frames)
        if key not in self._tables:
            t = self._packed[prefix]
            self._tables[key] = (rope_table(t["freqs"], frames),
                                 rel_pos_bias_table(t["rel_emb"], frames, self.cfg.rel_pos_buckets,
                                                    self.cfg.rel_pos_max_distance))
        return self._tables[key]

    # ------------------------------------------------------------------ blocks (kernel launch sequences)
    def _resnet(self, p, x, x2, temb_all, B, Fr, H, W):
        """ResnetBlock3D.forward (resnet.py:177-207); (x, x2) = folded channel concat of the up path."""
        K = self._k
        r = self._packed[p]
        NF, rps = B * Fr, Fr * H * W
        eps = r.get("eps", self.cfg.norm_eps)
        h = self._gn5(x, x2, B, rps, r["g1"], r["b1"], eps, True)
        off, cout = self._packed["temb_slices"][p]
        # stats=True: the conv's epilogue also emits the column sums the NEXT GroupNorm needs (no second read of h)
        h = K.conv3x3(h, NF, H, W, r["w1"], bias=r["cb1"], row_bias=temb_all[:, off:off + cout], rows_per_batch=rps,
                      stats=True)
        h = self._gn5(h, None, B, rps, r["g2"], r["b2"], eps, True)
        if "wsc" in r:
            sc = K.gemm(x, r["wsc"], a2=x2, bias=r["bsc"])
        else:
            assert x2 is None
            sc = x
        return K.conv3x3(h, NF, H, W, r["w2"], bias=r["cb2"], residual=sc, stats=True)

    def _transformer(self, p, x, kv_all, B, Fr, H, W, text_len):
        """Transformer3DModel.forward + BasicTransformerBlock.forward (attention.py:358-407, 511-560; VSR tree:
        vsr/models/attention.py:386-438, 556-593)."""
        K = self._k
        t = self._packed[p]
        heads, d, pitch, hp = self.cfg.heads, t["d"], t["pitch"], t["hp"]
        NF, HW = B * Fr, H * W
        interp = self.cfg.variant == "interp"
        if self.cfg.variant == "vsr":          # the VSR transformer runs a temporal (3,1,1) ResNet on its input first
            x = self._resnet_cnn(f"{p}.resblock_temporal", x, None, B, Fr, HW)
        h = K.groupnorm(x, NF, HW, t["gn_g"], t["gn_b"], 1e-6, silu=False)            # per-frame GN (4-D input)
        tok = K.gemm(h, t["w_in"], bias=t["b_in"])
        # spatial self-attention; interpolation model: SparseCausalAttention, the keys of frame f are those of frame 0
        # and of frame f-1 (interpolation/models/attention.py:611-664) -- two key segments, never concatenated
        n = K.layernorm(tok, t["norm1_g"], t["norm1_b"])
        if t["only_cross"]:                    # attn1 reads the text (the VSR model's only_cross_attention levels)
            q = K.gemm(n, t["attn1_q"])
            ko = t["attn1_kv_off"]
            a = K.attention(q, K.cols(kv_all, ko, ko + hp), K.cols(kv_all, ko + hp, ko + 2 * hp), NF, heads, HW, text_len,
                            d, pitch, kv_batch_div=Fr)
        elif interp and self._shard is not None:
            # frame-sharded SparseCausal attention: q|k|v of the local frames land behind two halo frames that the first
            # rank (frame 0 of the video) and the left neighbour (its last frame) fill over NVLink
            assert B == 1, "frame sharding runs one CFG half per rank"
            ctx = self._peer
            ext = ctx.local("kvx", (2 + Fr) * HW, 3 * hp)
            qkv = ops.gemm(n, t["attn1_qkv"], out=ext[2 * HW:])
            ctx.push_halo(ext, Fr, HW)
            a = ops.attention(qkv[:, :hp], ext[:, hp:2 * hp], ext[:, 2 * hp:], Fr, heads, HW, HW, d, pitch,
                              sparse_causal_frames=Fr, sc_halo=2 if self._frames(Fr)[1] == 0 else 1)
        else:
            qkv = K.gemm(n, t["attn1_qkv"])
            a = K.attention(K.cols(qkv, 0, hp), K.cols(qkv, hp, 2 * hp), K.cols(qkv, 2 * hp, 3 * hp), NF, heads, HW, HW,
                            d, pitch, sparse_causal_frames=Fr if interp else 0)
        tok = K.gemm(a, t["attn1_wo"], bias=t["attn1_bo"], residual=tok)
        # text cross-attention: keys/values projected once per batch item, shared by its frames
        n = K.layernorm(tok, t["norm2_g"], t["norm2_b"])
        q = K.gemm(n, t["attn2_q"])
        ko = t["kv_off"]
        a = K.attention(q, K.cols(kv_all, ko, ko + hp), K.cols(kv_all, ko + hp, ko + 2 * hp), NF, heads, HW, text_len, d,
                        pitch, kv_batch_div=Fr)
        tok = K.gemm(a, t["attn2_wo"], bias=t["attn2_bo"], residual=tok)
        if interp:
            # interpolation block order (interpolation/models/attention.py:566-608): feed-forward BEFORE the temporal
            # attention, which is a plain attention over the frames of a pixel (no rotary embedding, no bias)
            n = K.layernorm(tok, t["norm3_g"], t["norm3_b"])
            g = K.gemm(n, t["ff1_w"], bias=t["ff1_b"], geglu=True)
            tok = K.gemm(g, t["ff2_w"], bias=t["ff2_b"], residual=tok)
            if self._shard is None:
                n = K.layernorm(tok, t["norm_temp_g"], t["norm_temp_b"])
                qkv = K.gemm(n, t["attn_temp_qkv"])
                a = K.frame_attention(qkv, B, Fr, HW, heads, d, pitch)
                tok = K.gemm(a, t["attn_temp_wo"], bias=t["attn_temp_bo"], residual=tok)
            else:
                # all-to-all to pixel sharding around the plain temporal attention (peer-memory back end only)
                if self._shard_backend != "p2p":
                    raise NotImplementedError("the interpolation model shards frames over the p2p back end only")
                _, P, _ = self._shard
                assert HW % P == 0, "frame sharding needs H*W divisible by the number of frame shards"
                hwp = HW // P
                f_total = self._frames(Fr)[0]
                ctx = self._peer
                recv = ctx.layernorm_scatter(tok, t["norm_temp_g"], t["norm_temp_b"], HW, frames_total=f_total)
                qkv = ops.gemm(recv, t["attn_temp_qkv"])
                a = ops.frame_attention(qkv, 1, f_total, hwp, heads, d, pitch)
                ops.gemm(a, t["attn_temp_wo"], bias=t["attn_temp_bo"], out=ctx.local("y", f_total * hwp, t["C"]))
                tok = ctx.add_gathered(tok, HW)
            return K.gemm(tok, t["w_out"], bias=t["b_out"], residual=x, stats=True)
        # temporal attention: frames read in place with a row stride of HW (no (b f) d c <-> (b d) f c copies)
        if self._shard is None:
            n = K.layernorm(tok, t["norm_temp_g"], t["norm_temp_b"])
            qkv = K.gemm(n, t["attn_temp_qkv"])
            rope, bias = self._frame_tables(p, Fr)
            a = K.temporal_attention(qkv, B, Fr, HW, heads, d, pitch, rope, bias)
            tok = K.gemm(a, t["attn_temp_wo"], bias=t["attn_temp_bo"], residual=tok)
        else:
            # frame-sharded: all-to-all to pixel sharding (every rank gets ALL frames of HW/P pixels), attend, and back
            import torch.distributed as dist
            group, P, _ = self._shard
            assert B == 1 and HW % P == 0, "frame sharding runs one CFG half per rank and needs H*W divisible by P"
            hwp = HW // P
            f_total = self._frames(Fr)[0]
            rope, bias = self._frame_tables(p, f_total)
            if self._shard_backend == "p2p":
                # the all-to-alls are the store side of the LayerNorm and the load side of the residual add
                ctx = self._peer
                recv = ctx.layernorm_scatter(tok, t["norm_temp_g"], t["norm_temp_b"], HW, frames_total=f_total)
                qkv = ops.gemm(recv, t["attn_temp_qkv"])
                a = ops.temporal_attention(qkv, 1, f_total, hwp, heads, d, pitch, rope, bias)
                ops.gemm(a, t["attn_temp_wo"], bias=t["attn_temp_bo"], out=ctx.local("y", f_total * hwp, t["C"]))
                tok = ctx.add_gathered(tok, HW)
                return self._ff_and_out(t, tok, x)
            send = ops.layernorm_scatter(tok, t["norm_temp_g"], t["norm_temp_b"], HW, hwp)   # [P, F_loc, hwp, C]
            recv = torch.empty_like(send)                                                     # [F, hwp, C]
            dist.all_to_all_single(recv, send, group=group)
            qkv = ops.gemm(recv, t["attn_temp_qkv"])
            a = ops.temporal_attention(qkv, 1, Fr * P, hwp, heads, d, pitch, rope, bias)
            y = ops.gemm(a, t["attn_temp_wo"], bias=t["attn_temp_bo"])                        # [F, hwp, C] = P chunks
            back = torch.empty_like(y)                                                        # [P, F_loc, hwp, C]
            dist.all_to_all_single(back, y, group=group)
            tok = ops.add_gathered(tok, back, HW, hwp)
        return self._ff_and_out(t, tok, x)

    def _upsample(self, p, x, NF, h, w):
        """Upsample3D.forward (resnet.py:44-76): nearest x2 in H and W, then the 3x3 conv.  Product path: four 2x2 phase
        convs on the low-resolution map (no 4x copy, 2.25x fewer FLOPs); check mode and geometries the 5-D output box does
        not cover materialise the upsampled map."""
        K = self._k
        P = self._packed
        wu, bu = P[f"{p}.conv"]
        w4 = P.get(f"{p}.conv4")
        if w4 is not None and ops.upsample_conv3x3_supported(h, w, x.shape[1]):
            # sharded runs keep the stand-alone statistics exchange (the phase segments are a single-GPU layout)
            return ops.upsample_conv3x3(x, NF, h, w, w4, bias=bu, stats=self._shard is None)
        x = K.upsample_nearest2x(x, NF, h, w)
        return K.conv3x3(x, NF, 2 * h, 2 * w, wu, bias=bu, stats=True)

    def _ff_and_out(self, t, tok, x):
        # GEGLU feed-forward, then proj_out + the block's residual (attention.py:558, 394-401)
        K = self._k
        n = K.layernorm(tok, t["norm3_g"], t["norm3_b"])
        g = K.gemm(n, t["ff1_w"], bias=t["ff1_b"], geglu=True)
        tok = K.gemm(g, t["ff2_w"], bias=t["ff2_b"], residual=tok)
        return K.gemm(tok, t["w_out"], bias=t["b_out"], residual=x, stats=True)

    def _step(self, sample: torch.Tensor, t: torch.Tensor, text: torch.Tensor, taps: Optional[dict] = None,
              input_scale: Optional[torch.Tensor] = None, kv_all: Optional[torch.Tensor] = None,
              labels: Optional[torch.Tensor] = None):
        """One denoiser evaluation.  sample fp32 [B,C,F,H,W] (VSR: latent | low-res frames), t fp32 [B], text [B*L, ctx]
        (bf16; fp32 in check mode), labels int64 [B] (VSR noise level) -> fp32 [B,Co,F,H,W].  ``kv_all``: the text K/V
        projections when the caller already holds them (graph path: they are computed once per prompt, not once per
        step -- the reference re-projects them in every attn2 call, attention.py:364)."""
        K = self._k
        P = self._packed
        cfg = self.cfg
        B, _, Fr, H, W = sample.shape
        text_len = text.shape[0] // B
        text = K.text_input(text, cfg.cross_attention_dim)
        boc = cfg.block_out_channels
        if self._shard is not None and self._shard_backend == "p2p":
            f_total, f_off = self._frames(Fr)
            P_ = self._shard[1]
            self._shard_frames = (Fr, f_total)
            halo = 0
            if cfg.variant == "interp":                # [2 halo frames | local frames] x q|k|v of level 0
                halo = (2 + max(self._frame_counts or [Fr])) * H * W * 3 * cfg.heads * head_pitch(boc[0] // cfg.heads) * 2
            # largest all-to-all buffer = level 0: all frames x this rank's pixel slice
            self._peer_ctx(B * f_total * (H * W // P_) * boc[0] * 2, halo, f_off if self._frame_counts else -1)

        def tap(name, x, C, h, w):
            if taps is not None and name in self._TAPS:
                taps[name] = K.to_float(x).reshape(B, Fr, h, w, C).permute(0, 4, 1, 2, 3).contiguous()

        # time embedding (unet.py:428-434) and all 22 time_emb_proj (resnet.py:187) in three small launches
        temb = K.timestep_embedding(t, boc[0])
        h1 = K.linear_smallm(temb, P["time1"][0], P["time1"][1], silu_out=True)
        emb = K.linear_smallm(h1, P["time2"][0], P["time2"][1])
        if cfg.num_class_embeds:               # + the noise-level class embedding (vsr/models/unet.py:494-507)
            ops.embedding_add(emb, P["class_emb"], labels)
        temb_all = K.linear_smallm(emb, P["temb_w"], P["temb_b"], silu_in=True)
        if taps is not None and "emb" in self._TAPS:
            taps["emb"] = emb.clone()
        # every K/V projection of the text in one GEMM (the base model's 16 cross-attentions)
        if kv_all is None:
            kv_all = K.gemm(text, P["kv_w"])

        if "conv_in_tc" in P:
            x = ops.conv_in_tc(sample, P["conv_in_tc"][0], P["conv_in_tc"][1], input_scale)
        else:
            x = K.conv_in(sample, P["conv_in"][0], P["conv_in"][1], input_scale)
        tap("conv_in", x, boc[0], H, W)
        skips = [x]
        h, w = H, W
        for i, kind in enumerate(cfg.down_block_types):
            for j in range(cfg.layers_per_block):
                x = self._resnet(f"down_blocks.{i}.resnets.{j}", x, None, temb_all, B, Fr, h, w)
                if i == 0 and j == 0:
                    tap("down0_res0", x, boc[0], h, w)
                if kind == "CrossAttnDownBlock3D":
                    x = self._transformer(f"down_blocks.{i}.attentions.{j}", x, kv_all, B, Fr, h, w, text_len)
                    if i == 0 and j == 0:
                        tap("down0_attn0", x, boc[0], h, w)
                skips.append(x)
            if i != len(boc) - 1:
                wd, bd = P[f"down_blocks.{i}.downsamplers.0.conv"]
                x = K.conv3x3(x, B * Fr, h, w, wd, stride=2, bias=bd, stats=True)
                h, w = h // 2, w // 2
                skips.append(x)
            if cfg.temporal_modules:
                x = self._temporal_module(f"down_temporal_blocks.{i}", x, temb_all, B, Fr, h, w)
            if i == 0:
                tap("down0", x, boc[0], h, w)
        x = self._resnet("mid_block.resnets.0", x, None, temb_all, B, Fr, h, w)
        x = self._transformer("mid_block.attentions.0", x, kv_all, B, Fr, h, w, text_len)
        x = self._resnet("mid_block.resnets.1", x, None, temb_all, B, Fr, h, w)
        if cfg.temporal_modules:
            x = self._temporal_module("mid_temporal_block", x, temb_all, B, Fr, h, w)
        tap("mid", x, boc[-1], h, w)
        for i, kind in enumerate(cfg.up_block_types):
            for j in range(cfg.layers_per_block + 1):
                skip = skips.pop()
                x = self._resnet(f"up_blocks.{i}.resnets.{j}", x, skip, temb_all, B, Fr, h, w)
                if kind == "CrossAttnUpBlock3D":
                    x = self._transformer(f"up_blocks.{i}.attentions.{j}", x, kv_all, B, Fr, h, w, text_len)
            if i != len(boc) - 1:
                x = self._upsample(f"up_blocks.{i}.upsamplers.0", x, B * Fr, h, w)
                h, w = 2 * h, 2 * w
            if cfg.temporal_modules:
                x = self._temporal_module(f"up_temporal_blocks.{i}", x, temb_all, B, Fr, h, w)
        tap("up_out", x, boc[0], h, w)
        ss = self._gn5_scale_shift(x, None, B, Fr * h * w, P["norm_out"][0], P["norm_out"][1], cfg.norm_eps)
        if "conv_out_tc" in P:
            wp, bp, co = P["conv_out_tc"]
            return ops.conv_out_tc(x, ss, B, Fr, h, w, wp, bp, co)
        return K.conv_out(x, ss, B, Fr, h, w, P["conv_out"][0], P["conv_out"][1])

    # ------------------------------------------------------------------ public forward
    @torch.no_grad()
    def forward(self, sample: torch.Tensor, timestep: Union[torch.Tensor, float, int],
                encoder_hidden_states: torch.Tensor = None, class_labels=None, attention_mask=None,
                use_image_num: int = 0, return_dict: bool = True, taps: Optional[dict] = None,
                input_scale: float = 1.0):
        """Same contract as base/models/unet.py:366-512 (interpolation/models/unet.py:313-451 for the "interp" variant).
        ``attention_mask`` is accepted and ignored exactly like the reference (it never reaches the blocks,
        unet_blocks.py:352); ``class_labels``/``use_image_num`` must be unset (no class embedding in these configs; joint
        image-video training is out of scope).  Extension: ``input_scale`` multiplies ``sample`` inside conv_in, i.e.
        ``unet(x, t, e, input_scale=s) == unet(scheduler.scale_model_input(x, t), t, e)`` for EulerDiscrete's
        s = 1 / sqrt(sigma^2 + 1) without a pass over the latents."""
        if class_labels is not None or use_image_num:
            raise NotImplementedError("class_labels / use_image_num are not part of the base T2V inference path")
        if encoder_hidden_states is None:
            raise ValueError("encoder_hidden_states is required")
        if sample.dim() != 5:
            raise ValueError(f"sample must be [B,C,F,H,W], got {tuple(sample.shape)}")
        B, C, Fr, H, W = sample.shape
        n_down = len(self.cfg.block_out_channels) - 1
        if C != self.cfg.in_channels or H % (1 << n_down) or W % (1 << n_down):
            raise ValueError(f"sample needs {self.cfg.in_channels} channels and H, W multiples of {1 << n_down}")
        if encoder_hidden_states.shape[0] != B or encoder_hidden_states.shape[-1] != self.cfg.cross_attention_dim:
            raise ValueError(f"encoder_hidden_states must be [B, L, {self.cfg.cross_attention_dim}]")
        dev = self.device
        out_dtype = sample.dtype
        if self.cfg.center_input_sample:
            sample = 2 * sample - 1.0
        x = sample.to(device=dev, dtype=F32, non_blocking=True).contiguous()
        if float(input_scale) == 1.0:
            if self._scale_one is None or self._scale_one.device != dev:
                self._scale_one = torch.ones(1, dtype=F32, device=dev)
            scale = self._scale_one
        else:
            scale = torch.full((1,), float(input_scale), dtype=F32, device=dev)
        return self._forward(x, out_dtype, timestep, encoder_hidden_states, return_dict, taps, scale=scale)

    def _forward(self, x, out_dtype, timestep, encoder_hidden_states, return_dict, taps, scale=None, labels=None):
        """What follows the argument checks in every denoiser's forward: x is the fp32 model input on the device."""
        fp = self._weights_fingerprint()
        if self._packed is not None and fp != self._param_versions:
            self._invalidate()                  # a parameter was edited in place or replaced since the last packing
        if self._packed is None:
            self._pack()
            self._param_versions = fp
        dev = self.device
        B = x.shape[0]
        # timestep normalisation of unet.py:413-426
        if not torch.is_tensor(timestep):
            t = torch.full((B,), float(timestep), dtype=F32, device=dev)
        else:
            t = timestep.to(device=dev, dtype=F32).reshape(-1).expand(B).contiguous()
        txt = encoder_hidden_states.to(device=dev, dtype=F32 if self.check_mode else BF16, non_blocking=True).reshape(
            -1, self.cfg.cross_attention_dim).contiguous()
        vsr = self.cfg.variant == "vsr"
        if self.use_cuda_graph and taps is None and not (vsr and self._shard is not None):   # sharded VSR: eager steps
            # the VSR step keeps its text K/V GEMM inside the graph; the others project each prompt once (text_src)
            out = self._graph_step(x, t, txt, scale, labels, None if vsr else encoder_hidden_states)
        else:
            out = self._step(x, t, txt, taps, scale, labels=labels)
        out = out.to(out_dtype) if out_dtype != F32 else out.clone()   # never hand out the graph's static buffer
        if not return_dict:
            return (out,)
        return UNet3DConditionOutput(sample=out)

    def launches_per_step(self) -> int:
        """Kernel launches of this library inside the most recently replayed step graph."""
        return getattr(self, "_last_graph_launches", 0)

    @torch.no_grad()
    def forward_with_cfg(self, x: torch.Tensor, t, encoder_hidden_states: torch.Tensor = None, class_labels=None,
                         cfg_scale: float = 4.0, use_fp16: bool = False) -> torch.Tensor:
        """base/models/unet.py:514-538 and interpolation/models/unet.py:453-474: the FIRST half of the batch is run twice,
        against encoder_hidden_states = [cond prompt(s), uncond prompt(s)]; returns uncond + s (cond - uncond) for both
        halves (a plain Tensor, like the reference).  ``use_fp16`` only chose the reference's input dtype; compute here
        is bf16/fp32-accumulate either way."""
        n = len(x) // 2
        half = x[:n]
        combined = torch.cat([half, half], dim=0)
        return self._guided(self.forward(combined, t, encoder_hidden_states, class_labels).sample, cfg_scale)

    def _guided(self, out, cfg_scale):
        """uncond + s (cond - uncond) from the prediction of a [cond | uncond] batch (the CFG arithmetic of both
        forward_with_cfg); channels past out_channels pass through."""
        n = len(out) // 2
        co = self.cfg.out_channels
        eps = out[:, :co].float().contiguous()
        g = ops.cfg_combine(eps[:n], eps[n:], cfg_scale).to(out.dtype)
        return g if out.shape[1] == co else torch.cat([g, out[:, co:]], dim=1)

    def _graph_step(self, x, t, txt, scale, labels, text_src):
        """Replay of the step graph captured for this input geometry.  With ``text_src`` (the caller's prompt tensor)
        the text K/V projections run outside the graph; without it they are part of the captured step."""
        key = (tuple(x.shape), tuple(txt.shape))
        g = self._graphs.get(key)
        if g is None:
            g = {"x": x.clone(), "t": t.clone(), "txt": txt.clone(), "kv": None,
                 "scale": None if scale is None else scale.clone(), "labels": None if labels is None else labels.clone()}
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):          # warm-up run: kernel attributes, table caches, zeroed VSR pad buffers
                if text_src is not None:
                    g["kv"] = ops.gemm(g["txt"], self._packed["kv_w"])
                self._step(g["x"], g["t"], g["txt"], None, g["scale"], g["kv"], g["labels"])
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            before = ops.LAUNCHES
            # with frame sharding the NCCL collectives of the step are captured too (same sequence on every rank)
            with torch.cuda.graph(graph):
                g["out"] = self._step(g["x"], g["t"], g["txt"], None, g["scale"], g["kv"], g["labels"])
            g["launches"] = ops.LAUNCHES - before      # kernel nodes of ours in the captured step
            g["graph"] = graph
            self._graphs[key] = g
        g["x"].copy_(x, non_blocking=True)
        g["t"].copy_(t, non_blocking=True)
        if scale is not None:
            g["scale"].copy_(scale, non_blocking=True)
        if labels is not None:
            g["labels"].copy_(labels, non_blocking=True)
        extra = 0
        if text_src is None:
            g["txt"].copy_(txt, non_blocking=True)
        else:
            # text K/V projections: once per prompt tensor, outside the captured step.  A caller that passes the SAME
            # tensor object, unmodified (version counter), step after step -- every pipeline of the reference does --
            # pays for the projection GEMM only on the first step.
            seen = self._text_seen
            if not (seen is not None and seen[0] is text_src and seen[1] == text_src._version and seen[2] == key):
                g["txt"].copy_(txt, non_blocking=True)
                ops.gemm(g["txt"], self._packed["kv_w"], out=g["kv"])
                extra = 1
                self._text_seen = (text_src, text_src._version, key)
        self._last_graph_launches = g["launches"] + extra
        g["graph"].replay()
        return g["out"]
