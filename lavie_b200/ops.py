"""Thin operator layer: torch CUDA tensors in, C-ABI kernel launches out.

PyTorch is used only for device memory and the current stream.  Every function enqueues on
``torch.cuda.current_stream()`` and returns the output tensor; nothing here computes with torch ops.
Activations are bf16 channels-last ``[rows, C]`` (rows = (b, f, y, x)), see include/lavie_b200.h.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import Epilogue, check

BF16 = torch.bfloat16
F32 = torch.float32

# Launch accounting (bench.py's "gpu_launches") and an optional per-launch CUDA-event profiler: set
# ``ops.PROFILE = []`` to collect (kernel, algorithmic_flops, algorithmic_bytes, start_event, end_event) per launch.
LAUNCHES = 0
PROFILE = None


class _Launch:
    """Counts one kernel launch; with ops.PROFILE set, brackets it with CUDA events on the launching stream."""

    def __init__(self, kernel: str, flops: float = 0.0, nbytes: float = 0.0, tag: str = ""):
        self.kernel, self.flops, self.nbytes, self.tag = kernel, flops, nbytes, tag

    def __enter__(self):
        global LAUNCHES
        LAUNCHES += 1
        if PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None and exc[0] is None:
            self.e1.record()
            PROFILE.append((self.kernel, self.flops, self.nbytes, self.e0, self.e1, self.tag))
        return False


# GroupNorm statistics emitted by the producing GEMM / conv epilogue (lavie_epilogue.col_stats).  LAVIE_FUSE_GN_STATS=0
# switches back to the stand-alone statistics pass (A/B timing).
import os as _os
FUSE_GN_STATS = _os.environ.get("LAVIE_FUSE_GN_STATS", "1") != "0"

WORKSPACE_BYTES = 128 << 20
_workspaces = {}


_ticket_bufs = {}


def _tickets(device, n: int) -> torch.Tensor:
    """Zero-initialised int32 tickets for "last block finalizes" kernels; the kernels leave them zero."""
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    t = _ticket_bufs.get(key)
    if t is None or t.numel() < n:
        t = torch.zeros(max(n, 256), dtype=torch.int32, device=device)
        _ticket_bufs[key] = t
    return t


def _workspace(device) -> torch.Tensor:
    """Caller-owned split-K scratch (fp32 partials), one per device, reused by every GEMM on the stream."""
    key = (device.type, device.index if device.index is not None else torch.cuda.current_device())
    ws = _workspaces.get(key)
    if ws is None:
        # zero-initialised: the last 64 KiB are the tickets of the in-kernel split-K reduction (lavie_gemm_bf16 contract:
        # zero before the first call, the library leaves them zero)
        ws = torch.zeros(WORKSPACE_BYTES, dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _rows2d(t: torch.Tensor) -> Tuple[int, int, int]:
    """(rows, cols, ld) of a 2-D bf16 view whose last dim is contiguous."""
    assert t.dim() == 2 and t.stride(1) == 1 and t.dtype == BF16 and t.is_cuda, (t.shape, t.stride(), t.dtype)
    return t.shape[0], t.shape[1], t.stride(0)


def _epilogue(bias=None, row_bias=None, rows_per_batch=1, residual=None, geglu=False, col_stats=None):
    if bias is None and row_bias is None and residual is None and not geglu and col_stats is None:
        return None
    ep = Epilogue()
    ep.col_stats = _ptr(col_stats)
    ep.bias = _ptr(bias)
    ep.row_bias = _ptr(row_bias)
    ep.rows_per_batch = int(rows_per_batch)
    ep.ld_row_bias = row_bias.stride(0) if row_bias is not None else 0
    ep.residual = _ptr(residual)
    ep.ld_residual = residual.stride(0) if residual is not None else 0
    ep.geglu = 1 if geglu else 0
    if bias is not None:
        assert bias.dtype == F32 and bias.is_contiguous()
    if row_bias is not None:
        assert row_bias.dtype == F32 and row_bias.dim() == 2 and row_bias.stride(1) == 1
    if residual is not None:
        _rows2d(residual)
    return ep


# ---- layout helpers shared with the check-mode provider (lavie_b200/check.py implements the same names on triples) ----
def cols(x: torch.Tensor, a: int, b: int) -> torch.Tensor:
    return x[:, a:b]


def weight(w: torch.Tensor, device) -> torch.Tensor:
    """kernel-side copy of a weight matrix: bf16, contiguous."""
    return w.to(device=device, dtype=BF16).contiguous()


weight_small = weight          # the time-embedding linears read bf16 weights too


def to_float(x: torch.Tensor) -> torch.Tensor:
    return x.float()


def text_input(text: torch.Tensor, ctx: int) -> torch.Tensor:
    return text                # already bf16 [B*L, ctx] (cast by the caller outside the captured graph)


def gemm(a: torch.Tensor, w: torch.Tensor, *, a2: Optional[torch.Tensor] = None, bias=None, row_bias=None,
         rows_per_batch=1, residual=None, geglu=False, out: Optional[torch.Tensor] = None, block_n: int = 0,
         stats: bool = False):
    """out[M,N] = [a | a2] @ w^T (+ fused epilogue).  w: bf16 [N, K] contiguous.  stats=True: the epilogue also emits the
    per-slab column sums the consuming GroupNorm needs (attached to the result, see `colsums`)."""
    lib = _lib.load()
    M, k0, lda = _rows2d(a)
    k1, lda2 = 0, 0
    if a2 is not None:
        M2, k1, lda2 = _rows2d(a2)
        assert M2 == M
    assert w.dtype == BF16 and w.is_contiguous() and w.shape[1] == k0 + k1, (w.shape, k0, k1)
    N = w.shape[0]
    n_out = N // 2 if geglu else N
    if out is None:
        out = torch.empty((M, n_out), dtype=BF16, device=a.device)
    Mo, No, ldo = _rows2d(out)
    assert Mo == M and No == n_out
    cs = _new_colsums(M, n_out, a.device) if stats and not geglu and FUSE_GN_STATS else None
    ep = _epilogue(bias, row_bias, rows_per_batch, residual, geglu, cs)
    ws = _workspace(a.device)
    with _Launch("gemm_bf16_tcgen05", 2.0 * M * N * (k0 + k1), 2.0 * (M * (k0 + k1) + N * (k0 + k1) + M * n_out),
                 f"gemm M={M} N={N} K={k0 + k1}{' geglu' if geglu else ''}"):
        rc = lib.lavie_gemm_bf16(a.data_ptr(), lda, k0, _ptr(a2), lda2, k1, w.data_ptr(), out.data_ptr(), ldo, M, N,
                                 ctypes.byref(ep) if ep is not None else None, block_n, ws.data_ptr(), ws.numel(),
                                 _stream())
    check(rc, "lavie_gemm_bf16")
    if cs is not None:
        out._gn_colsums = cs
    return out


def conv3x3_supported(H: int, W: int, C: int) -> bool:
    return bool(_lib.load().lavie_conv3x3_supported(H, W, C))


def im2col3x3(x: torch.Tensor, NF: int, H: int, W: int, stride: int = 1) -> torch.Tensor:
    """x: contiguous [NF*H*W, C] -> [NF*Ho*Wo, 9*C], K ordered (kh, kw, c)."""
    lib = _lib.load()
    rows, C, ld = _rows2d(x)
    assert rows == NF * H * W and ld == C
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    col = torch.empty((NF * Ho * Wo, 9 * C), dtype=BF16, device=x.device)
    with _Launch("lavie_im2col3x3_bf16"):
        check(lib.lavie_im2col3x3_bf16(x.data_ptr(), NF, H, W, C, stride, col.data_ptr(), _stream()), "lavie_im2col3x3_bf16")
    return col


def conv3x3_out_size(n: int, stride: int = 1, padding: Tuple[int, int] = (1, 1)) -> int:
    """Output extent of a 3x3 conv along one axis of n pixels with ``padding`` = (before, after) zero pixels."""
    return int(_lib.load().lavie_conv3x3_out_size(n, stride, padding[0], padding[1]))


def conv3x3(x: torch.Tensor, NF: int, H: int, W: int, w: torch.Tensor, *, stride: int = 1, bias=None, row_bias=None,
            rows_per_batch=1, residual=None, out: Optional[torch.Tensor] = None, block_n: int = 0,
            force_im2col: bool = False, stats: bool = False, algo_n: int = 0, padding: Tuple[int, int] = (1, 1)):
    """3x3 InflatedConv3d on a contiguous channels-last map; w: bf16 [N, 9*C] in (kh, kw, c) order.  ``algo_n``:
    real output channels when the weight rows are zero-padded (launch accounting only).  ``padding`` = (before, after)
    zero pixels on both axes: (1, 1) is the usual pad-1 conv, (0, 1) with stride 2 diffusers' Downsample2D(padding=0)."""
    lib = _lib.load()
    rows, C, ld = _rows2d(x)
    assert rows == NF * H * W and ld == C, "conv3x3 needs a contiguous channels-last input"
    N = w.shape[0]
    assert w.dtype == BF16 and w.is_contiguous() and w.shape[1] == 9 * C
    pad_b, pad_a = (int(p) for p in padding)
    if force_im2col or not conv3x3_supported(H, W, C):
        if (pad_b, pad_a) != (1, 1):
            raise ValueError(f"conv3x3: the explicit im2col path only pads (1, 1), got padding={tuple(padding)} "
                             f"(C={C}, force_im2col={force_im2col})")
        col = im2col3x3(x, NF, H, W, stride)
        return gemm(col, w, bias=bias, row_bias=row_bias, rows_per_batch=rows_per_batch, residual=residual, out=out,
                    block_n=block_n, stats=stats)
    Ho, Wo = conv3x3_out_size(H, stride, (pad_b, pad_a)), conv3x3_out_size(W, stride, (pad_b, pad_a))
    m_out = NF * Ho * Wo
    if out is None:
        out = torch.empty((m_out, N), dtype=BF16, device=x.device)
    Mo, No, ldo = _rows2d(out)
    assert Mo == m_out and No == N
    cs = _new_colsums(m_out, N, x.device) if stats and FUSE_GN_STATS else None
    ep = _epilogue(bias, row_bias, rows_per_batch, residual, False, cs)
    ws = _workspace(x.device)
    n_alg = algo_n or N
    pad_tag = "" if (pad_b, pad_a) == (1, 1) else f" pad=({pad_b},{pad_a})"
    with _Launch("gemm_bf16_tcgen05", 2.0 * m_out * n_alg * 9 * C, 2.0 * (rows * C + n_alg * 9 * C + m_out * n_alg),
                 f"conv3x3 M={m_out} N={N} K={9 * C} W={W} s={stride}{pad_tag}"):
        rc = lib.lavie_conv3x3_pad_bf16(x.data_ptr(), NF, H, W, C, stride, pad_b, pad_a, w.data_ptr(), out.data_ptr(),
                                        ldo, N, ctypes.byref(ep) if ep is not None else None, block_n, ws.data_ptr(),
                                        ws.numel(), _stream())
    check(rc, "lavie_conv3x3_pad_bf16")
    if cs is not None:
        out._gn_colsums = cs
    return out


def frame_conv(xpad: torch.Tensor, taps: int, tap_rows: int, w: torch.Tensor, *, bias=None, row_bias=None,
               rows_per_batch=1, residual=None, out: Optional[torch.Tensor] = None, block_n: int = 0,
               stats: bool = False, colsums_out: Optional[torch.Tensor] = None):
    """nn.Conv3d (taps,1,1) over frames (vsr/models/resnet.py:253-254,269) for ONE batch item.  xpad: bf16
    [(F + taps - 1) * tap_rows, C], the item's channels-last map with taps//2 zero frames on both sides;
    w: bf16 [N, taps*C] in (tap, c) order.  Returns [F * tap_rows, N].  ``colsums_out``: this item's slab range of a
    column-statistics buffer that spans several items (see `_new_colsums`)."""
    lib = _lib.load()
    rows_in, C, ld = _rows2d(xpad)
    M = rows_in - (taps - 1) * tap_rows
    N = w.shape[0]
    assert M > 0 and w.dtype == BF16 and w.is_contiguous() and w.shape[1] == taps * C, (w.shape, taps, C)
    if out is None:
        out = torch.empty((M, N), dtype=BF16, device=xpad.device)
    Mo, No, ldo = _rows2d(out)
    assert Mo == M and No == N
    cs = colsums_out if colsums_out is not None else (_new_colsums(M, N, xpad.device) if stats and FUSE_GN_STATS else None)
    ep = _epilogue(bias, row_bias, rows_per_batch, residual, False, cs)
    ws = _workspace(xpad.device)
    with _Launch("gemm_bf16_tcgen05", 2.0 * M * N * taps * C, 2.0 * (rows_in * C + N * taps * C + M * N),
                 f"frame_conv M={M} N={N} K={taps * C} taps={taps}"):
        rc = lib.lavie_frame_conv_bf16(xpad.data_ptr(), ld, rows_in, C, taps, tap_rows, w.data_ptr(), out.data_ptr(), ldo,
                                       M, N, ctypes.byref(ep) if ep is not None else None, block_n, ws.data_ptr(),
                                       ws.numel(), _stream())
    check(rc, "lavie_frame_conv_bf16")
    if cs is not None:
        out._gn_colsums = cs
    return out


def embedding_add(emb: torch.Tensor, table: torch.Tensor, labels: torch.Tensor):
    """emb[b] += table[labels[b]] in place (vsr/models/unet.py:494-507); emb fp32 [B, dim], labels int64 [B]."""
    lib = _lib.load()
    B, dim = emb.shape
    assert emb.dtype == F32 and emb.is_contiguous() and table.dtype == F32 and table.is_contiguous()
    assert table.shape[1] == dim and labels.dtype == torch.int64 and labels.numel() == B and labels.is_cuda
    with _Launch("lavie_embedding_add"):
        check(lib.lavie_embedding_add(emb.data_ptr(), table.data_ptr(), labels.data_ptr(), B, dim, table.shape[0],
                                      _stream()), "lavie_embedding_add")
    return emb


def upsample_conv3x3_supported(H: int, W: int, C: int) -> bool:
    return bool(_lib.load().lavie_upsample_conv3x3_supported(H, W, C))


def upsample_conv3x3(x: torch.Tensor, NF: int, H: int, W: int, w_phases: torch.Tensor, *, bias=None,
                     stats: bool = False, block_n: int = 0):
    """Upsample3D (nearest x2 in H and W, then 3x3 conv; resnet.py:44-76) without the upsampled copy: four 2x2 phase
    convs on the low-resolution map x [NF*H*W, C]; w_phases from packing.pack_upsample_conv3x3.  Returns the
    high-resolution map [NF*2H*2W, N]."""
    lib = _lib.load()
    rows, C, ld = _rows2d(x)
    assert rows == NF * H * W and ld == C, "upsample_conv3x3 needs a contiguous channels-last input"
    N = w_phases.shape[0] // 4
    assert w_phases.dtype == BF16 and w_phases.is_contiguous() and tuple(w_phases.shape) == (4 * N, 4 * C)
    out = torch.empty((4 * rows, N), dtype=BF16, device=x.device)
    cs = None
    if stats and FUSE_GN_STATS and N % 32 == 0 and rows % 32 == 0:
        cs = torch.empty((4 * (rows // 32), N // 32, 4, 2), dtype=F32, device=x.device)     # 4 phase segments
    ep = _epilogue(bias, None, 1, None, False, cs)
    # algorithmic work = the reference's op: a 3x3 conv on the 4x map
    with _Launch("gemm_bf16_tcgen05", 2.0 * 4 * rows * N * 9 * C, 2.0 * (rows * C + N * 9 * C + 4 * rows * N),
                 f"upsample_conv3x3 M={4 * rows} N={N} K={9 * C} W={2 * W} (16 tap-GEMMs on the low-res map)"):
        rc = lib.lavie_upsample_conv3x3_bf16(x.data_ptr(), NF, H, W, C, w_phases.data_ptr(), out.data_ptr(), N,
                                             ctypes.byref(ep) if ep is not None else None, block_n, _stream())
    check(rc, "lavie_upsample_conv3x3_bf16")
    if cs is not None:
        out._gn_colsums = cs
        out._gn_segs = 4
    return out


def _new_colsums(M: int, N: int, device) -> Optional[torch.Tensor]:
    """[slabs of 32 rows, 32-column chunks, 4 decade pieces, (sum, sumsq)] -- see lavie_epilogue.col_stats."""
    if N % 32:
        return None
    return torch.empty(((M + 31) // 32, N // 32, 4, 2), dtype=F32, device=device)


def colsums(x: torch.Tensor, rows_per_sample: int, x2: Optional[torch.Tensor] = None, allow_segments: bool = False):
    """The producers' column statistics of (x, x2) when every source carries them and slabs do not straddle samples;
    else None (the caller runs the stand-alone statistics pass).  Statistics written by the fused upsample conv come in
    4 phase segments (`_gn_segs`); only callers that can fold those (allow_segments) get them."""
    if rows_per_sample % 32:
        return None
    cs0 = getattr(x, "_gn_colsums", None)
    cs1 = getattr(x2, "_gn_colsums", None) if x2 is not None else None
    if cs0 is None or (x2 is not None and cs1 is None):
        return None
    for t in (x, x2):
        segs = getattr(t, "_gn_segs", 1) if t is not None else 1
        if segs > 1 and (not allow_segments or (rows_per_sample // 32) % segs):
            return None
    # micro-group width the producers used: 10 channels when their N is a multiple of 10 (base / interpolation model),
    # else 8 (VSR model); all sources and the consumer's 32 groups must agree on it
    c0 = x.shape[1]
    c1 = x2.shape[1] if x2 is not None else 0
    mg = 10 if c0 % 10 == 0 else 8
    if (c1 and (c1 % 10 == 0) != (mg == 10)) or ((c0 + c1) // 32) % mg or c0 % mg:
        return None
    return cs0, cs1


def groupnorm_scale_shift(x: torch.Tensor, samples: int, rows_per_sample: int, gamma: torch.Tensor,
                          beta: torch.Tensor, eps: float, groups: int = 32, x2: Optional[torch.Tensor] = None,
                          fused: bool = True):
    """Statistics + affine folded into per-(sample, channel) (scale, shift): fp32 [samples, C, 2].
    fused=False runs the two-launch form (stats, then finalize) -- same arithmetic, kept for the sharded path and tests."""
    lib = _lib.load()
    rows, c0, ld0 = _rows2d(x)
    c1, ld1 = 0, 0
    if x2 is not None:
        rows2, c1, ld1 = _rows2d(x2)
        assert rows2 == rows
    assert rows == samples * rows_per_sample
    C = c0 + c1
    ss = torch.empty((samples, C, 2), dtype=F32, device=x.device)
    assert gamma.dtype == F32 and beta.dtype == F32 and gamma.numel() == C
    cs = colsums(x, rows_per_sample, x2, allow_segments=True) if fused else None
    if cs is not None:
        # the statistics pass already happened in the producers' epilogues: fold their column sums (one small launch)
        s0 = getattr(x, "_gn_segs", 1)
        s1 = getattr(x2, "_gn_segs", 1) if x2 is not None else 1
        with _Launch("lavie_groupnorm_finalize_colsums", 0.0, 1.0 * (rows // 32) * C,
                     f"gn_colsums rows={rows} C={C} samples={samples}"):
            check(lib.lavie_groupnorm_finalize_colsums_seg(cs[0].data_ptr(), c0, s0, _ptr(cs[1]), c1, s1, samples,
                                                           rows_per_sample, groups, gamma.data_ptr(), beta.data_ptr(), eps,
                                                           ss.data_ptr(), _stream()), "lavie_groupnorm_finalize_colsums_seg")
        return ss
    chunks = lib.lavie_groupnorm_chunks(samples, rows_per_sample)
    partial = torch.empty((samples, chunks, groups, 2), dtype=F32, device=x.device)
    if not fused:
        with _Launch("lavie_groupnorm_stats", 0.0, 2.0 * rows * C, f"gn_stats rows={rows} C={C} samples={samples}"):
            check(lib.lavie_groupnorm_stats(x.data_ptr(), ld0, c0, _ptr(x2), ld1, c1, samples, rows_per_sample, groups,
                                            partial.data_ptr(), _stream()), "lavie_groupnorm_stats")
        with _Launch("lavie_groupnorm_finalize"):
            check(lib.lavie_groupnorm_finalize(partial.data_ptr(), samples, chunks, groups, C,
                                               rows_per_sample * (C // groups), gamma.data_ptr(), beta.data_ptr(), eps,
                                               ss.data_ptr(), _stream()), "lavie_groupnorm_finalize")
        return ss
    # one launch: the last block of each sample folds the partials into (scale, shift)
    with _Launch("lavie_groupnorm_scale_shift", 0.0, 2.0 * rows * C, f"gn_stats rows={rows} C={C} samples={samples}"):
        check(lib.lavie_groupnorm_scale_shift(x.data_ptr(), ld0, c0, _ptr(x2), ld1, c1, samples, rows_per_sample,
                                              groups, gamma.data_ptr(), beta.data_ptr(), eps, partial.data_ptr(),
                                              _tickets(x.device, samples).data_ptr(), ss.data_ptr(), _stream()),
              "lavie_groupnorm_scale_shift")
    return ss


def groupnorm_sums(x: torch.Tensor, samples: int, rows_per_sample: int, groups: int = 32,
                   x2: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Local (sum, sum of squares) per (sample, group) as fp64 [samples, groups, 2]: the quantity frame shards all-reduce."""
    lib = _lib.load()
    rows, c0, ld0 = _rows2d(x)
    c1, ld1 = 0, 0
    if x2 is not None:
        _, c1, ld1 = _rows2d(x2)
    assert rows == samples * rows_per_sample
    cs = colsums(x, rows_per_sample, x2)
    if cs is not None:
        sums = torch.empty((samples, groups, 2), dtype=torch.float64, device=x.device)
        with _Launch("lavie_groupnorm_reduce_colsums"):
            check(lib.lavie_groupnorm_reduce_colsums(cs[0].data_ptr(), c0, _ptr(cs[1]), c1, samples, rows_per_sample,
                                                     groups, sums.data_ptr(), _stream()), "lavie_groupnorm_reduce_colsums")
        return sums
    chunks = lib.lavie_groupnorm_chunks(samples, rows_per_sample)
    partial = torch.empty((samples, chunks, groups, 2), dtype=F32, device=x.device)
    with _Launch("lavie_groupnorm_stats", 0.0, 2.0 * rows * (c0 + c1), f"gn_stats rows={rows} C={c0 + c1} samples={samples}"):
        check(lib.lavie_groupnorm_stats(x.data_ptr(), ld0, c0, _ptr(x2), ld1, c1, samples, rows_per_sample, groups,
                                        partial.data_ptr(), _stream()), "lavie_groupnorm_stats")
    sums = torch.empty((samples, groups, 2), dtype=torch.float64, device=x.device)
    with _Launch("lavie_groupnorm_reduce"):
        check(lib.lavie_groupnorm_reduce(partial.data_ptr(), samples, chunks, groups, sums.data_ptr(), _stream()),
              "lavie_groupnorm_reduce")
    return sums


def groupnorm_finalize_sums(sums: torch.Tensor, C: int, count_per_group: int, gamma: torch.Tensor, beta: torch.Tensor,
                            eps: float) -> torch.Tensor:
    lib = _lib.load()
    samples, groups, _ = sums.shape
    assert sums.dtype == torch.float64 and sums.is_contiguous()
    ss = torch.empty((samples, C, 2), dtype=F32, device=sums.device)
    with _Launch("lavie_groupnorm_finalize_sums"):
        check(lib.lavie_groupnorm_finalize_sums(sums.data_ptr(), samples, groups, C, count_per_group, gamma.data_ptr(),
                                                beta.data_ptr(), eps, ss.data_ptr(), _stream()),
              "lavie_groupnorm_finalize_sums")
    return ss


def layernorm_scatter(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, hw: int, hwp: int, eps: float = 1e-5):
    """LayerNorm + scatter rows (f, pixel) -> (pixel // hwp, f, pixel % hwp) (all-to-all send layout)."""
    lib = _lib.load()
    rows, C, ldx = _rows2d(x)
    out = torch.empty((rows, C), dtype=BF16, device=x.device)
    with _Launch("lavie_layernorm_bf16", 0.0, 4.0 * rows * C, f"ln_scatter rows={rows} C={C}"):
        check(lib.lavie_layernorm_scatter_bf16(x.data_ptr(), ldx, gamma.data_ptr(), beta.data_ptr(), eps, out.data_ptr(),
                                               C, rows, C, hw, hwp, _stream()), "lavie_layernorm_scatter_bf16")
    return out


def add_gathered(res: torch.Tensor, z: torch.Tensor, hw: int, hwp: int):
    """res[(f, pixel)] + z[(pixel // hwp, f, pixel % hwp)] (all-to-all receive layout) -> new tensor."""
    lib = _lib.load()
    rows, C, ldr = _rows2d(res)
    rz, Cz, ldz = _rows2d(z)
    assert rz == rows and Cz == C
    out = torch.empty((rows, C), dtype=BF16, device=res.device)
    with _Launch("lavie_add_gathered_bf16", 0.0, 6.0 * rows * C):
        check(lib.lavie_add_gathered_bf16(res.data_ptr(), ldr, z.data_ptr(), ldz, out.data_ptr(), C, rows, C, hw, hwp,
                                          _stream()), "lavie_add_gathered_bf16")
    return out


def groupnorm_apply(x: torch.Tensor, scale_shift: torch.Tensor, samples: int, rows_per_sample: int, silu: bool,
                    x2: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None):
    lib = _lib.load()
    rows, c0, ld0 = _rows2d(x)
    c1, ld1 = 0, 0
    if x2 is not None:
        _, c1, ld1 = _rows2d(x2)
    C = c0 + c1
    if out is None:
        out = torch.empty((rows, C), dtype=BF16, device=x.device)
    _, _, ldy = _rows2d(out)
    with _Launch("lavie_groupnorm_apply", 0.0, 4.0 * rows * C, f"gn_apply rows={rows} C={C}"):
        check(lib.lavie_groupnorm_apply(x.data_ptr(), ld0, c0, _ptr(x2), ld1, c1, samples, rows_per_sample,
                                        scale_shift.data_ptr(), 1 if silu else 0, out.data_ptr(), ldy, _stream()),
              "lavie_groupnorm_apply")
    return out


def groupnorm(x, samples, rows_per_sample, gamma, beta, eps, silu, groups=32, x2=None):
    ss = groupnorm_scale_shift(x, samples, rows_per_sample, gamma, beta, eps, groups, x2)
    return groupnorm_apply(x, ss, samples, rows_per_sample, silu, x2)


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-5,
              out: Optional[torch.Tensor] = None):
    lib = _lib.load()
    rows, C, ldx = _rows2d(x)
    if out is None:
        out = torch.empty((rows, C), dtype=BF16, device=x.device)
    _, _, ldy = _rows2d(out)
    assert gamma.dtype == F32 and beta.dtype == F32
    with _Launch("lavie_layernorm_bf16", 0.0, 4.0 * rows * C, f"ln rows={rows} C={C}"):
        check(lib.lavie_layernorm_bf16(x.data_ptr(), ldx, gamma.data_ptr(), beta.data_ptr(), eps, out.data_ptr(), ldy,
                                       rows, C, _stream()), "lavie_layernorm_bf16")
    return out


def attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, batch: int, heads: int, Sq: int, Sk: int, d: int,
              head_pitch: int, kv_batch_div: int = 1, scale: Optional[float] = None,
              out: Optional[torch.Tensor] = None, sparse_causal_frames: int = 0, sc_halo: int = 0):
    """q: [batch*Sq, >=heads*pitch] view, k/v: [(batch/kv_batch_div)*Sk, ...] views; returns [batch*Sq, heads*d].
    sparse_causal_frames = F: batch = (video, frame), keys of frame f = [frame 0 | frame max(f-1, 0)] (2*Sk keys).
    sc_halo (frame sharding): k/v carry two extra leading frames [frame 0 | previous rank's last frame]; 2 on rank 0."""
    lib = _lib.load()
    rq, _, ldq = _rows2d(q)
    rk, _, ldk = _rows2d(k)
    rv, _, ldv = _rows2d(v)
    assert rq == batch * Sq and rk == (batch // kv_batch_div + (2 if sc_halo else 0)) * Sk and rv == rk and ldk == ldv
    if out is None:
        out = torch.empty((rq, heads * d), dtype=BF16, device=q.device)
    _, _, ldo = _rows2d(out)
    if scale is None:
        scale = d ** -0.5
    keys = Sk * (2 if sparse_causal_frames else 1)
    with _Launch("lavie_attention_bf16", 4.0 * batch * heads * Sq * keys * d,
                 2.0 * (rq + 2 * rk) * heads * head_pitch + 2.0 * rq * heads * d,
                 f"attn B={batch} Sq={Sq} Sk={keys} d={d}"):
        check(lib.lavie_attention_strided_bf16(q.data_ptr(), ldq, Sq * ldq, k.data_ptr(), v.data_ptr(), ldk, Sk * ldk,
                                               out.data_ptr(), ldo, Sq * ldo, batch, heads, Sq, Sk, d, head_pitch,
                                               kv_batch_div, sparse_causal_frames, sc_halo, scale, _stream()),
              "lavie_attention_strided_bf16")
    return out


def frame_attention(qkv: torch.Tensor, B: int, F: int, HW: int, heads: int, d: int, head_pitch: int,
                    out: Optional[torch.Tensor] = None):
    """Plain attention over the F frames of every pixel (the interpolation UNet's attn_temp,
    interpolation/models/attention.py:598-606), read in place: qkv rows = (b, f, pixel), columns q | k | v; sequence
    stride = HW rows, batch (pixel) stride = one row.  Any F (one launch per video: the pixels are the batch)."""
    lib = _lib.load()
    rows, cols, ld = _rows2d(qkv)
    hp = heads * head_pitch
    assert rows == B * F * HW and cols == 3 * hp
    if out is None:
        out = torch.empty((rows, heads * d), dtype=BF16, device=qkv.device)
    _, _, ldo = _rows2d(out)
    for b in range(B):
        base = qkv[b * F * HW:]
        o_b = out[b * F * HW:]
        with _Launch("lavie_attention_bf16", 4.0 * HW * heads * F * F * d, 2.0 * F * HW * (cols + heads * d),
                     f"frame_attn F={F} HW={HW} d={d}"):
            check(lib.lavie_attention_strided_bf16(base.data_ptr(), HW * ld, ld, base[:, hp:].data_ptr(),
                                                   base[:, 2 * hp:].data_ptr(), HW * ld, ld, o_b.data_ptr(), HW * ldo,
                                                   ldo, HW, heads, F, F, d, head_pitch, 1, 0, 0, d ** -0.5, _stream()),
                  "lavie_attention_strided_bf16")
    return out


def temporal_attention(qkv: torch.Tensor, B: int, F: int, HW: int, heads: int, d: int, head_pitch: int,
                       rope: torch.Tensor, bias: torch.Tensor, out: Optional[torch.Tensor] = None):
    """qkv: [B*F*HW, 3*heads*pitch] (q | k | v); rope fp32 [F, rot_pairs, 2]; bias fp32 [heads, F, F]."""
    lib = _lib.load()
    rows, cols, ld = _rows2d(qkv)
    assert rows == B * F * HW and cols == 3 * heads * head_pitch
    if out is None:
        out = torch.empty((rows, heads * d), dtype=BF16, device=qkv.device)
    _, _, ldo = _rows2d(out)
    assert rope.dtype == F32 and rope.is_contiguous() and rope.shape[0] == F
    assert bias.dtype == F32 and bias.is_contiguous() and tuple(bias.shape) == (heads, F, F)
    with _Launch("lavie_temporal_attention_bf16", 4.0 * B * HW * heads * F * F * d, 2.0 * rows * (cols + heads * d),
                 f"tattn F={F} HW={HW} d={d}"):
        check(lib.lavie_temporal_attention_bf16(qkv.data_ptr(), ld, heads * head_pitch, 2 * heads * head_pitch,
                                                out.data_ptr(), ldo, B, F, HW, heads, d, head_pitch, d ** -0.5,
                                                rope.data_ptr(), rope.shape[1], bias.data_ptr(), _stream()),
              "lavie_temporal_attention_bf16")
    return out


def linear_smallm(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], silu_in=False, silu_out=False):
    lib = _lib.load()
    assert x.dtype == F32 and x.is_contiguous() and x.dim() == 2
    M, K = x.shape
    assert w.dtype == BF16 and w.is_contiguous() and w.shape[1] == K
    N = w.shape[0]
    out = torch.empty((M, N), dtype=F32, device=x.device)
    with _Launch("lavie_linear_smallm"):
        check(lib.lavie_linear_smallm(x.data_ptr(), M, K, w.data_ptr(), _ptr(bias), out.data_ptr(), N, int(silu_in),
                                      int(silu_out), _stream()), "lavie_linear_smallm")
    return out


def timestep_embedding(t: torch.Tensor, dim: int):
    lib = _lib.load()
    assert t.dtype == F32 and t.is_contiguous() and t.dim() == 1
    out = torch.empty((t.shape[0], dim), dtype=F32, device=t.device)
    with _Launch("lavie_timestep_embedding"):
        check(lib.lavie_timestep_embedding(t.data_ptr(), t.shape[0], dim, out.data_ptr(), _stream()),
              "lavie_timestep_embedding")
    return out


def conv_in(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, input_scale: Optional[torch.Tensor] = None):
    """x fp32 [B,Cin,F,H,W] -> bf16 [B*F*H*W, Cout]; w fp32 [Cout,Cin,3,3]; computes conv(input_scale * x) with
    input_scale a device fp32 scalar tensor (None = 1)."""
    lib = _lib.load()
    assert x.dtype == F32 and x.is_contiguous() and x.dim() == 5
    B, Cin, Fr, H, W = x.shape
    Cout = w.shape[0]
    assert w.dtype == F32 and w.is_contiguous() and bias.dtype == F32
    out = torch.empty((B * Fr * H * W, Cout), dtype=BF16, device=x.device)
    with _Launch("lavie_conv_in"):
        assert input_scale is None or (input_scale.dtype == F32 and input_scale.is_cuda and input_scale.numel() == 1)
        check(lib.lavie_conv_in_scaled(x.data_ptr(), _ptr(input_scale), B, Cin, Fr, H, W, w.data_ptr(), bias.data_ptr(),
                                       Cout, out.data_ptr(), Cout, _stream()), "lavie_conv_in_scaled")
    return out


def conv_in_kpad(cin: int) -> int:
    """K of the conv_in GEMM: 9 * Cin rounded up to the GEMM's 64-deep K block."""
    return (9 * cin + 63) // 64 * 64


def conv_in_tc(x: torch.Tensor, w_pad: torch.Tensor, bias: torch.Tensor, input_scale: Optional[torch.Tensor] = None):
    """conv_in on the tensor cores: x fp32 [B,Cin,F,H,W] -> im2col rows [B*F*H*W, kpad] (bf16, scaled by input_scale) ->
    one GEMM against w_pad bf16 [Cout, kpad] (filters in (c, kh, kw) order, zero-padded) + bias -> bf16 [rows, Cout]."""
    lib = _lib.load()
    assert x.dtype == F32 and x.is_contiguous() and x.dim() == 5
    B, Cin, Fr, H, W = x.shape
    kpad = w_pad.shape[1]
    assert kpad == conv_in_kpad(Cin) and w_pad.dtype == BF16 and w_pad.is_contiguous()
    col = torch.empty((B * Fr * H * W, kpad), dtype=BF16, device=x.device)
    with _Launch("lavie_im2col_input_bf16", 0.0, 4.0 * x.numel() + 2.0 * col.numel()):
        assert input_scale is None or (input_scale.dtype == F32 and input_scale.is_cuda and input_scale.numel() == 1)
        check(lib.lavie_im2col_input_bf16(x.data_ptr(), _ptr(input_scale), B, Cin, Fr, H, W, kpad, col.data_ptr(),
                                          _stream()), "lavie_im2col_input_bf16")
    return gemm(col, w_pad, bias=bias)


def pack_conv_in(w: torch.Tensor, device) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> bf16 [Cout, kpad] in (c, kh, kw) order, zero-padded (conv_in_tc)."""
    co, ci = w.shape[:2]
    out = torch.zeros((co, conv_in_kpad(ci)), dtype=F32)
    out[:, :9 * ci] = w.detach().float().cpu().reshape(co, 9 * ci)
    return out.to(device=device, dtype=BF16).contiguous()


def conv_out(x: torch.Tensor, scale_shift: torch.Tensor, B: int, Fr: int, H: int, W: int, w: torch.Tensor,
             bias: torch.Tensor):
    """x bf16 [B*F*H*W, C] raw; w fp32 [Cout, 3, 3, C]; returns fp32 [B, Cout, F, H, W]."""
    lib = _lib.load()
    rows, C, ldx = _rows2d(x)
    assert rows == B * Fr * H * W
    Cout = w.shape[0]
    assert w.dtype == F32 and w.is_contiguous() and tuple(w.shape) == (Cout, 3, 3, C)
    out = torch.empty((B, Cout, Fr, H, W), dtype=F32, device=x.device)
    with _Launch("lavie_conv_out"):
        check(lib.lavie_conv_out(x.data_ptr(), ldx, scale_shift.data_ptr(), B, Fr, H, W, C, w.data_ptr(), bias.data_ptr(),
                                 Cout, out.data_ptr(), _stream()), "lavie_conv_out")
    return out


CONV_OUT_PAD = 32      # conv_out's Cout = 4 filters are zero-padded to one 32-column chunk of the GEMM epilogue


def conv_out_tc(x: torch.Tensor, scale_shift: torch.Tensor, B: int, Fr: int, H: int, W: int, w_pad: torch.Tensor,
                bias_pad: torch.Tensor, Cout: int):
    """conv_norm_out -> SiLU -> conv_out (unet.py:504-506) with the conv on the tensor cores: GroupNorm apply + SiLU
    (one pass, bf16), implicit-GEMM 3x3 conv against the zero-padded filters w_pad bf16 [32, 9*C], then the 4 real
    channels are unpacked into fp32 [B, Cout, F, H, W].  Needs C % 64 == 0 (im2col-mode TMA)."""
    lib = _lib.load()
    rows, C, _ = _rows2d(x)
    assert rows == B * Fr * H * W and w_pad.shape == (CONV_OUT_PAD, 9 * C) and Cout <= CONV_OUT_PAD
    h = groupnorm_apply(x, scale_shift, B, Fr * H * W, True)
    y = conv3x3(h, B * Fr, H, W, w_pad, bias=bias_pad, block_n=64, algo_n=Cout)
    out = torch.empty((B, Cout, Fr, H, W), dtype=F32, device=x.device)
    with _Launch("lavie_unpack_nchw_f32", 0.0, rows * (2.0 * CONV_OUT_PAD + 4.0 * Cout)):
        check(lib.lavie_unpack_nchw_f32(y.data_ptr(), y.stride(0), B, Cout, Fr, H, W, out.data_ptr(), _stream()),
              "lavie_unpack_nchw_f32")
    return out


def upsample_nearest2x(x: torch.Tensor, NF: int, H: int, W: int):
    lib = _lib.load()
    rows, C, ld = _rows2d(x)
    assert rows == NF * H * W and ld == C
    y = torch.empty((NF * 4 * H * W, C), dtype=BF16, device=x.device)
    with _Launch("lavie_upsample_nearest2x"):
        check(lib.lavie_upsample_nearest2x(x.data_ptr(), NF, H, W, C, y.data_ptr(), _stream()), "lavie_upsample_nearest2x")
    return y


def cfg_ddim_step(noise_uncond, noise_text, guidance: float, alpha_t: float, alpha_prev: float, latents,
                  out: Optional[torch.Tensor] = None):
    lib = _lib.load()
    for t in (noise_uncond, noise_text, latents):
        assert t.dtype == F32 and t.is_contiguous()
    if out is None:
        out = torch.empty_like(latents)
    with _Launch("lavie_cfg_ddim_step"):
        check(lib.lavie_cfg_ddim_step(noise_uncond.data_ptr(), noise_text.data_ptr(), guidance, alpha_t, alpha_prev,
                                      latents.data_ptr(), out.data_ptr(), latents.numel(), _stream()),
              "lavie_cfg_ddim_step")
    return out


def cfg_linear_step(noise_uncond, noise_text, guidance: float, a: float, b: float, latents, noise=None,
                    c_noise: float = 0.0, out: Optional[torch.Tensor] = None):
    """eps = u + g (t - u); out = a * latents + b * eps (+ c_noise * noise)."""
    lib = _lib.load()
    for t in (noise_uncond, noise_text, latents) + ((noise,) if noise is not None else ()):
        assert t.dtype == F32 and t.is_contiguous() and t.numel() == latents.numel()
    if out is None:
        out = torch.empty_like(latents)
    with _Launch("lavie_cfg_linear_step"):
        check(lib.lavie_cfg_linear_step(noise_uncond.data_ptr(), noise_text.data_ptr(), guidance, a, b, c_noise,
                                        latents.data_ptr(), _ptr(noise), out.data_ptr(), latents.numel(), _stream()),
              "lavie_cfg_linear_step")
    return out


def cfg_combine(cond, uncond, scale: float, duplicate: bool = True):
    """uncond + scale * (cond - uncond), returned as cat([g, g]) when `duplicate` (forward_with_cfg's contract)."""
    lib = _lib.load()
    assert cond.dtype == F32 and uncond.dtype == F32 and cond.is_contiguous() and uncond.is_contiguous()
    assert cond.shape == uncond.shape
    n = cond.numel()
    out = torch.empty(((2 if duplicate else 1) * cond.shape[0],) + tuple(cond.shape[1:]), dtype=F32, device=cond.device)
    second = out[cond.shape[0]:] if duplicate else None
    with _Launch("lavie_cfg_combine"):
        check(lib.lavie_cfg_combine(cond.data_ptr(), uncond.data_ptr(), float(scale), out.data_ptr(), _ptr(second), n,
                                    _stream()), "lavie_cfg_combine")
    return out


# ---- once-per-video encoders / decoders (SURVEY 8f N4): CLIP text encoder and VAE decoder pieces ----
def clip_embed(ids: torch.Tensor, tok: torch.Tensor, pos: torch.Tensor, L: int) -> torch.Tensor:
    """ids int64 [rows]; tok fp32 [V, C]; pos fp32 [>= L, C] -> bf16 [rows, C] (token + position embedding)."""
    lib = _lib.load()
    assert ids.dtype == torch.int64 and ids.is_cuda and ids.is_contiguous() and tok.dtype == F32 and pos.dtype == F32
    rows, C = ids.numel(), tok.shape[1]
    out = torch.empty((rows, C), dtype=BF16, device=ids.device)
    with _Launch("lavie_clip_embed"):
        check(lib.lavie_clip_embed(ids.data_ptr(), tok.data_ptr(), pos.data_ptr(), rows, L, C, tok.shape[0], out.data_ptr(),
                                   _stream()), "lavie_clip_embed")
    return out


def causal_attention_small(qkv: torch.Tensor, B: int, L: int, heads: int, d: int) -> torch.Tensor:
    lib = _lib.load()
    rows, cols, ld = _rows2d(qkv)
    assert rows == B * L and cols == 3 * heads * d
    out = torch.empty((rows, heads * d), dtype=BF16, device=qkv.device)
    with _Launch("lavie_causal_attention_small", 4.0 * B * heads * L * L * d / 2):
        check(lib.lavie_causal_attention_small(qkv.data_ptr(), ld, B, L, heads, d, d ** -0.5, out.data_ptr(), heads * d,
                                               _stream()), "lavie_causal_attention_small")
    return out


def activation_(x: torch.Tensor, kind: str) -> torch.Tensor:
    lib = _lib.load()
    assert x.dtype == BF16 and x.is_contiguous() and x.is_cuda
    with _Launch("lavie_activation_bf16", 0.0, 4.0 * x.numel()):
        check(lib.lavie_activation_bf16(x.data_ptr(), x.numel(), {"quick_gelu": 0, "gelu": 1}[kind], _stream()),
              "lavie_activation_bf16")
    return x


def softmax_rows_(s: torch.Tensor, scale: float) -> torch.Tensor:
    lib = _lib.load()
    rows, n, ld = _rows2d(s)
    with _Launch("lavie_softmax_rows_bf16", 0.0, 4.0 * rows * n):
        check(lib.lavie_softmax_rows_bf16(s.data_ptr(), ld, rows, n, float(scale), _stream()), "lavie_softmax_rows_bf16")
    return s


def pointwise_conv_nchw(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
    """1x1 conv on an fp32 NCHW map: x [N, Cin, h, w], w fp32 [Cout, Cin], bias fp32 [Cout] -> fp32 [N, Cout, h, w]
    = bias + w @ (scale * x) per pixel (AutoencoderKL.post_quant_conv with decode_latents' scaling folded in)."""
    lib = _lib.load()
    assert x.dtype == F32 and x.is_contiguous() and x.dim() == 4
    N, Cin, h, wd = x.shape
    Cout = w.shape[0]
    assert w.dtype == F32 and w.is_contiguous() and tuple(w.shape) == (Cout, Cin)
    assert bias.dtype == F32 and bias.is_contiguous() and bias.numel() == Cout
    out = torch.empty((N, Cout, h, wd), dtype=F32, device=x.device)
    with _Launch("lavie_pointwise_conv_nchw_f32"):
        check(lib.lavie_pointwise_conv_nchw_f32(x.data_ptr(), w.data_ptr(), bias.data_ptr(), float(scale), N, Cin, Cout,
                                                h * wd, out.data_ptr(), _stream()), "lavie_pointwise_conv_nchw_f32")
    return out


def image_to_uint8(y: torch.Tensor) -> torch.Tensor:
    """y bf16 [pixels, >= 4] channels-last (columns 0..2 = RGB in [-1, 1]) -> uint8 [pixels, 3]."""
    lib = _lib.load()
    rows, _, ld = _rows2d(y)
    out = torch.empty((rows, 3), dtype=torch.uint8, device=y.device)
    with _Launch("lavie_image_to_uint8"):
        check(lib.lavie_image_to_uint8(y.data_ptr(), ld, rows, out.data_ptr(), _stream()), "lavie_image_to_uint8")
    return out
