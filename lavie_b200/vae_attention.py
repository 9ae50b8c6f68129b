"""Single-head d = 512 attention of the x4-upscaler VAE decoder's mid block (``lavie_attention_wide_bf16``).

The VAE decoder's AttentionBlock runs at the latent resolution, so the x4 decoder sees h * w tokens per frame (163 840
at a 320x512 latent): a materialised score matrix would be tens of GB per frame.  This launches the fused kernel of
csrc/attention_wide.cu instead.  It lives outside ``ops`` on purpose: ``ops`` holds the kernels shared by the denoisers
and encoders, and this one serves the VAE alone."""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from ._lib import check
from .ops import BF16, _Launch, _rows2d, _stream

WIDE_D = 512


def attention_wide(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, frames: int, S: int,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """o = softmax(q k^T) v per frame.  q, k, v: bf16 [frames * S, 512] row-major views (the 512^-1/2 scale already in
    q); returns (or fills ``out``) bf16 [frames * S, 512]."""
    lib = _lib.load()
    rows = frames * S
    lds = []
    for t in (q, k, v):
        r, c, ld = _rows2d(t)
        assert r == rows and c == WIDE_D, (tuple(t.shape), frames, S)
        lds.append(ld)
    if out is None:
        out = torch.empty((rows, WIDE_D), dtype=BF16, device=q.device)
    r, c, ldo = _rows2d(out)
    assert r == rows and c == WIDE_D, (tuple(out.shape), frames, S)
    flops = 4.0 * frames * S * S * WIDE_D
    with _Launch("attn_wide_kernel", flops, 2.0 * 4 * rows * WIDE_D, f"attention_wide frames={frames} S={S}"):
        rc = lib.lavie_attention_wide_bf16(q.data_ptr(), lds[0], k.data_ptr(), lds[1], v.data_ptr(), lds[2],
                                           out.data_ptr(), ldo, frames, S, _stream())
    check(rc, "lavie_attention_wide_bf16")
    return out
