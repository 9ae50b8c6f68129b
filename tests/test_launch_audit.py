"""Per-launch audit: every kernel launch the denoisers and encoders issue, checked against a high-precision reference of
that one launch.

A recorder wraps the launching functions of `lavie_b200.ops` (all model code calls through the module attribute), clones
each call's tensor arguments before the call (outputs alias inputs: `out=` views, residual/out pairs, in-place ops), runs
the real function on the original tensors and compares the result, right away, with a reference computed in fp64 from
the cloned inputs.  Only a summary row per launch is kept.

Every comparison is element-wise, against a bound derived from the kernel's rounding model and written next to the
reference; the whole-tensor rel-L2 is a second check.  Attention launches are also re-issued with probe values (all
ones, a key-index ramp) that a mask off by one key moves by more than the bound.  Producer column statistics and the
bytes around `out=` views are checked too.  The comparators are plain torch: the CPU tests at the end inject defects into
a correct bf16 result and show that each is flagged, and that an uninjected result passes.
"""
import collections
import inspect
import math
import os
import sys

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2

F64 = torch.float64
BF16 = torch.bfloat16

# ------------------------------------------------------------------------------------------------ rounding model
U = 2.0 ** -8          # unit roundoff of bf16: one rounding to bf16 moves a value by at most U * |value|
U32 = 2.0 ** -24       # unit roundoff of fp32
# fitted-exponent GELU of the GEGLU epilogue (gelu_fast_f, lavie_b200/csrc/common.cuh): max |gelu_fast - gelu_erf| over the
# real line; test_gelu_fast_error_bound measures it on a dense grid in emulated fp32
E_GELU = 2.5e-6
GELU_SLOPE = 1.13      # max |d gelu / dx| (1.1289 at x = 1.4142)
SILU_SLOPE = 1.1       # max |d silu / dx| (1.0998 at x = 2.3994)


def c_gemm(K, splits=1):
    """Accumulation bound of the tensor-core GEMM, as a multiple of S = |A| |W|^T: products of bf16 are exact in fp32, each
    16-deep MMA step and each fp32 accumulator update rounds once (<= 2^-23 of the partial sums' absolute values, which are
    <= S), the split-K reduction adds `splits` fp32 additions, the epilogue three more (bias, row bias, residual)."""
    return (math.ceil(K / 16) + splits + 8) * 2.0 ** -23


C_ATTN_P = 2.0 ** -7    # attention: P rounded to bf16 before P V (U) against a row sum of the unrounded P (U), per sum_j p |v|
C_ATTN_P_F32 = 2.0 ** -18   # causal_attention_small keeps P in fp32 (__expf: 2^-21 relative, fp32 sums of <= 128 terms)
RHO_F32 = 2.0 ** -20    # score error of fp32 q.k over d <= 160 bf16 products, relative to scale * sum |q| |k|
RHO_ROPE = 2.0 ** -7 + 2.0 ** -16   # temporal attention: scale * q and k are rotated in fp32 and rounded to bf16 (2 U)
NORM_REL = 1e-5         # GroupNorm scale / shift and LayerNorm statistics: fp32 partial sums, fp64 combination
COLSUM_REL = 1e-5       # producer column sums of <= 32 x 10 bf16 values, fp32, relative to the sums of |x| and x^2


def tf32_off():
    """Turn TF32 off for cuBLAS and cuDNN; returns the previous settings for tf32_restore."""
    saved = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    return saved


def tf32_restore(saved):
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved


# ------------------------------------------------------------------------------------------------ comparator
class Cmp:
    """Element-wise comparison of `out` with `ref` under `bound` (broadcast to out's shape).  Large results are compared in
    blocks along their first dimension (`add` with the block's offset, then `finish`), so no full-size fp64 temporaries
    beyond the caller's own are needed."""

    STEP = 1 << 24          # elements per comparison block

    def __init__(self, what, out=None, ref=None, bound=None, rel_max=None, dims=None):
        self.what, self.rel_max, self.dims = what, rel_max, dims
        self.n_over, self.worst, self.worst_at, self.worst_err, self.worst_ref = 0, -1.0, (), 0.0, 0.0
        self._d2 = self._r2 = self._emax = 0.0
        if out is not None:
            self.add(out, ref, bound)
            self.finish()

    def add(self, out, ref, bound, row0=0):
        ref = torch.as_tensor(ref)
        bound = torch.as_tensor(bound, dtype=F64, device=out.device)
        if out.dim() == 0:
            out, ref, bound = out.reshape(1), ref.reshape(1), bound.reshape(1)
        ref = ref.expand(out.shape)
        bound = bound.expand(out.shape)
        per = max(1, out[0].numel()) if out.numel() else 1
        step = max(1, self.STEP // per)
        for lo in range(0, out.shape[0], step):
            o = out[lo:lo + step].detach().to(F64)
            r = ref[lo:lo + step].to(device=o.device, dtype=F64)
            err = (o - r).abs()
            ratio = torch.nan_to_num(err / bound[lo:lo + step].clamp_min(1e-300), nan=math.inf)
            self.n_over += int((ratio > 1).sum())
            self._d2 += float(torch.nan_to_num((o - r).pow(2), nan=math.inf).sum())
            self._r2 += float(r.pow(2).sum())
            self._emax = max(self._emax, float(torch.nan_to_num(err, nan=math.inf).max()))
            flat = int(ratio.reshape(-1).argmax())
            w = float(ratio.reshape(-1)[flat])
            if w > self.worst:
                at = [int(i) for i in torch.unravel_index(torch.tensor(flat), tuple(ratio.shape))]
                at[0] += row0 + lo
                self.worst, self.worst_at = w, tuple(at)
                self.worst_err, self.worst_ref = float(err.reshape(-1)[flat]), float(r.reshape(-1)[flat])
        return self

    def finish(self):
        self.worst = max(self.worst, 0.0)
        self.rel = math.sqrt(self._d2 / self._r2) if self._r2 > 0 else self._emax
        self.ok = self.n_over == 0 and (self.rel_max is None or self.rel <= self.rel_max)
        return self

    def where(self):
        at = self.worst_at
        if self.dims:
            return ", ".join(f"{n}={i}" for n, i in zip(self.dims, at))
        return str(at)

    def __str__(self):
        return (f"{self.what}: {self.n_over} elements over the bound, worst err/bound {self.worst:.3g} at ({self.where()}) "
                f"|err|={self.worst_err:.3g} ref={self.worst_ref:.3g}; rel-L2 {self.rel:.3g}"
                + (f" (limit {self.rel_max:g})" if self.rel_max is not None else ""))


class Flag:
    """A boolean finding that is not an element-wise comparison (bytes outside a view, pad frames)."""

    def __init__(self, what, ok, detail=""):
        self.what, self.ok, self.detail = what, bool(ok), detail
        self.n_over, self.worst, self.rel, self.rel_max = (0 if ok else 1), (0.0 if ok else math.inf), 0.0, None

    def __str__(self):
        return f"{self.what}: {self.detail}"


# ------------------------------------------------------------------------------------------------ references (fp64)
def mm_abs(a, w, rows=None, step=None):
    """(a @ w^T, |a| @ |w|^T) in fp64, chunked over rows to bound memory; `a` is a matrix, or a function of (lo, hi)
    that returns those rows of it (then `rows` = M and `step` = rows per chunk)."""
    w = w.to(F64)
    M = a.shape[0] if rows is None else rows
    out = torch.empty((M, w.shape[0]), dtype=F64, device=w.device)
    s = torch.empty_like(out)
    wa = w.abs().t()
    wt = w.t()
    step = step or max(1, (1 << 27) // max(1, w.shape[1]))
    for lo in range(0, M, step):
        blk = a(lo, min(M, lo + step)) if rows is not None else a[lo:lo + step].to(F64)
        out[lo:lo + step] = blk @ wt
        s[lo:lo + step] = blk.abs() @ wa
    return out, s


def epilogue_ref(acc, s, row0=0, bias=None, row_bias=None, rows_per_batch=1, residual=None):
    """acc + bias + row_bias[row // rows_per_batch] + residual for the rows row0.. of a block (residual: those rows);
    the abs-sum S grows by the same terms' magnitudes."""
    if bias is not None:
        acc = acc + bias.to(F64)
        s = s + bias.to(F64).abs()
    if row_bias is not None:
        idx = torch.arange(row0, row0 + acc.shape[0], device=acc.device) // rows_per_batch
        rb = row_bias.to(F64)[idx]
        acc = acc + rb
        s = s + rb.abs()
    if residual is not None:
        acc = acc + residual.to(F64)
        s = s + residual.to(F64).abs()
    return acc, s


def gelu64(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def geglu_ref(h, s, c):
    """Undo interleave_geglu's tiles (128 value columns, then their 128 gate columns, per 256-column tile)."""
    M, N = h.shape
    h = h.reshape(M, N // 256, 2, 128)
    s = s.reshape(M, N // 256, 2, 128)
    v, g = h[:, :, 0], h[:, :, 1]
    sv, sg = s[:, :, 0], s[:, :, 1]
    gg = gelu64(g)
    ref = (v * gg).reshape(M, N // 2)
    # value error c S_v times |gelu(g)|, gate error c S_g through the slope, the fitted GELU's own error times |v|
    extra = (c * (sv * gg.abs() + GELU_SLOPE * v.abs() * sg) + E_GELU * v.abs()).reshape(M, N // 2)
    return ref, extra


def im2col64(x, NF, H, W, stride=1):
    """x [NF*H*W, C] -> [NF*Ho*Wo, 9*C] in fp64, K ordered (kh, kw, c), zero padding 1."""
    C = x.shape[1]
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    xp = F.pad(x.to(F64).reshape(NF, H, W, C), (0, 0, 1, 1, 1, 1))
    taps = [xp[:, kh:kh + stride * (Ho - 1) + 1:stride, kw:kw + stride * (Wo - 1) + 1:stride] for kh in range(3)
            for kw in range(3)]
    return torch.stack(taps, 3).reshape(NF * Ho * Wo, 9 * C)


def conv_mm(x, NF, H, W, stride, w):
    """3x3 pad-1 conv of x [NF*H*W, C] with w [N, 9*C] ((kh, kw, c) order) and its abs-product, chunked over images."""
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    imgs = max(1, (1 << 27) // (Ho * Wo * w.shape[1]))
    o, hw = Ho * Wo, H * W
    return mm_abs(lambda lo, hi: im2col64(x[lo // o * hw:hi // o * hw], (hi - lo) // o, H, W, stride), w,
                  rows=NF * o, step=imgs * o)


def upsample_phase_ref(x, NF, H, W, w_phases):
    """The phase definition of lavie_upsample_conv3x3_bf16 (include/lavie_b200.h): output pixel (2y + py, 2x + px) =
    sum over taps (a, b) of source pixel (y + py - 1 + a, x + px - 1 + b) times w_phases[phase py*2+px, :, a, b, :]."""
    C = x.shape[1]
    N = w_phases.shape[0] // 4
    xp = F.pad(x.to(F64).reshape(NF, H, W, C), (0, 0, 1, 1, 1, 1))
    wp = w_phases.to(F64).reshape(4, N, 4 * C)
    out = torch.empty((NF, H, 2, W, 2, N), dtype=F64, device=x.device)
    s = torch.empty_like(out)
    for py in range(2):
        for px in range(2):
            cols = torch.stack([xp[:, py + a:py + a + H, px + b:px + b + W] for a in range(2) for b in range(2)], 3)
            o, sa = mm_abs(cols.reshape(NF * H * W, 4 * C), wp[py * 2 + px])
            out[:, :, py, :, px] = o.reshape(NF, H, W, N)
            s[:, :, py, :, px] = sa.reshape(NF, H, W, N)
    return out.reshape(NF * 4 * H * W, N), s.reshape(NF * 4 * H * W, N)


def gn_stats64(X, samples, groups):
    """fp64 (mean, var) per (sample, group) of X [rows, C], plus E[x^2] (conditioning of the one-pass variance)."""
    rows, C = X.shape
    v = X.to(F64).reshape(samples, rows // samples, groups, C // groups)
    mean = v.mean((1, 3))
    msq = (v * v).mean((1, 3))
    var = (msq - mean * mean).clamp_min(0)
    return mean, var, msq


def gn_scale_shift64(X, samples, gamma, beta, eps, groups=32):
    """(scale, shift) [samples, C] with GroupNorm(X) = X * scale + shift, and the bounds of the fp32 kernels' values:
    NORM_REL relative, plus the fp32 one-pass variance's conditioning E[x^2] / var times 2^-20."""
    C = X.shape[1]
    mean, var, msq = gn_stats64(X, samples, groups)
    rstd = 1.0 / torch.sqrt(var + eps)
    rep = C // groups
    g, b = gamma.to(F64), beta.to(F64)
    scale = rstd.repeat_interleave(rep, 1) * g
    m = mean.repeat_interleave(rep, 1)
    shift = b - m * scale
    kappa = (msq / (var + eps)).repeat_interleave(rep, 1)
    rel = NORM_REL + kappa * 2.0 ** -20
    b_scale = rel * scale.abs()
    b_shift = rel * (b.abs() + (m * scale).abs()) + scale.abs() * torch.sqrt(msq).repeat_interleave(rep, 1) * 2.0 ** -20
    return scale, shift, b_scale, b_shift


def silu64(x):
    return x * torch.sigmoid(x)


def apply_rows(x, sc, sh, silu):
    """y = act(x * sc + sh) element-wise (sc / sh: the per-row (scale, shift) of each row's sample), and the magnitude
    |x sc| + |sh| the fp32 arithmetic rounds against."""
    x = x.to(F64)
    t = x * sc + sh
    mag = (x * sc).abs() + sh.abs()
    return (silu64(t) if silu else t), mag, t


def apply_ref(X, scale, shift, samples, silu):
    rows = X.shape[0]
    idx = torch.arange(rows, device=X.device) // (rows // samples)
    return apply_rows(X, scale[idx], shift[idx], silu)


def layernorm_ref(x, gamma, beta, eps):
    x = x.to(F64)
    mean = x.mean(1, keepdim=True)
    msq = (x * x).mean(1, keepdim=True)
    var = (msq - mean * mean).clamp_min(0)
    xh = (x - mean) / torch.sqrt(var + eps)
    y = xh * gamma.to(F64) + beta.to(F64)
    kappa = msq / (var + eps)
    small = (NORM_REL + kappa * 2.0 ** -20) * ((xh * gamma.to(F64)).abs() + beta.to(F64).abs() + gamma.to(F64).abs())
    return y, small


def attention_core(Q, K, V, scale, bias=None, causal=False, rho=RHO_F32, c_p=C_ATTN_P, Qr=None, Kr=None):
    """softmax(scale Q K^T + bias) V in fp64 on [batch, heads, S, d] tensors, chunked over the batch, and the bound
    U |o| + c_p sum_j p_j |v_j| + sum_j p_j ds_j (|v_j| + |o|), ds_j = rho scale sum_i |q_i| |k_ji| the score error
    (Qr / Kr: the operands the kernel actually multiplies, when they differ from Q / K)."""
    Bt, Hh, Sq, _ = Q.shape
    Sk = K.shape[2]
    o = torch.empty((Bt, Hh, Sq, V.shape[-1]), dtype=F64, device=Q.device)
    bnd = torch.empty_like(o)
    qstep = max(1, min(Sq, (1 << 25) // max(1, Hh * Sk)))          # score blocks of <= 2^25 elements
    step = max(1, (1 << 25) // max(1, Hh * Sq * Sk)) if qstep == Sq else 1
    Qr = Q if Qr is None else Qr
    Kr = K if Kr is None else Kr
    for lo in range(0, Bt, step):
        k, v = K[lo:lo + step].to(F64), V[lo:lo + step].to(F64)
        kra = Kr[lo:lo + step].to(F64).abs().transpose(-1, -2)
        va = v.abs()
        for q0 in range(0, Sq, qstep):
            q = Q[lo:lo + step, :, q0:q0 + qstep].to(F64)
            s = scale * (q @ k.transpose(-1, -2))
            if bias is not None:
                s = s + bias.to(F64)[..., q0:q0 + qstep, :]
            if causal:
                mask = torch.arange(q0, q0 + q.shape[2], device=s.device)[:, None] < torch.arange(Sk, device=s.device)
                s = s.masked_fill(mask, -math.inf)
            p = torch.softmax(s, -1)
            oo = p @ v
            ds = rho * abs(scale) * (Qr[lo:lo + step, :, q0:q0 + qstep].to(F64).abs() @ kra) + 2.0 ** -20
            pd = p * ds
            bnd[lo:lo + step, :, q0:q0 + qstep] = (U * oo.abs() + c_p * (p @ va) + pd @ va
                                                   + pd.sum(-1, keepdim=True) * oo.abs() + 1e-30)
            o[lo:lo + step, :, q0:q0 + qstep] = oo
    return o, bnd


def rope64(t, table):
    """Rotate adjacent pairs (x0, x1) -> (x0 c - x1 s, x1 c + x0 s) of the first rot_pairs pairs; t [..., F, d],
    table [F, rot_pairs, 2] (cos, sin)."""
    rp = table.shape[1]
    c = table[..., 0].to(F64)
    s = table[..., 1].to(F64)
    a = t[..., :2 * rp].reshape(*t.shape[:-1], rp, 2)
    x0, x1 = a[..., 0], a[..., 1]
    rot = torch.stack([x0 * c - x1 * s, x1 * c + x0 * s], -1).reshape(*t.shape[:-1], 2 * rp)
    return torch.cat([rot, t[..., 2 * rp:]], -1)


def bf16_round(t):
    return t.to(torch.float32).to(BF16).to(F64)


def sparse_causal_key_rows(batch, Sk, F_, sc_halo, device):
    """Key rows [batch, 2*Sk] of SparseCausalAttention: frame f of a video reads [frame 0 | frame max(f-1, 0)] of the same
    video; with sc_halo the key buffer starts with two halo frames [frame 0 | the frame before the first local one]."""
    b = torch.arange(batch, device=device)
    j = torch.arange(Sk, device=device)
    if sc_halo:
        first = torch.zeros_like(b)
        former = torch.where(b == 0, torch.full_like(b, 1 if sc_halo == 1 else 2), b + 1)
    else:
        vid, f = b // F_, b % F_
        first = vid * F_
        former = vid * F_ + (f - 1).clamp_min(0)
    return torch.cat([first[:, None] * Sk + j, former[:, None] * Sk + j], 1)


def heads_of(t, rows_idx, heads, pitch, d):
    """t [rows, >= heads*pitch] gathered at rows_idx [batch, S] -> [batch, heads, S, d]."""
    x = t[rows_idx.reshape(-1)][:, :heads * pitch].reshape(*rows_idx.shape, heads, pitch)[..., :d]
    return x.permute(0, 2, 1, 3)


def attention_layout(a):
    """Query / key row indices of one ops.attention call: ([batch, Sq], [batch, keys])."""
    batch, Sq, Sk = a["batch"], a["Sq"], a["Sk"]
    dev = a["q"].device
    qrows = torch.arange(batch * Sq, device=dev).reshape(batch, Sq)
    if a["sparse_causal_frames"]:
        krows = sparse_causal_key_rows(batch, Sk, a["sparse_causal_frames"], a["sc_halo"], dev)
    else:
        kb = torch.arange(batch, device=dev) // a["kv_batch_div"]
        krows = kb[:, None] * Sk + torch.arange(Sk, device=dev)
    return qrows, krows


def frame_layout(B, F_, HW, device):
    """Rows of the frame sequences of every (video, pixel): [B*HW, F]."""
    b = torch.arange(B, device=device)[:, None, None]
    px = torch.arange(HW, device=device)[None, :, None]
    f = torch.arange(F_, device=device)[None, None, :]
    return (b * F_ * HW + f * HW + px).reshape(B * HW, F_)


# ------------------------------------------------------------------------------------------------ producer statistics
def colsum_expected(out, segs=1, src_rows=None):
    """The col_stats a producer must have written for its bf16 output `out` [M, N], in the kernel layout
    [slabs, N/32, 4, 2], with a mask of the written entries.  Micro-groups of 10 channels when N % 10 == 0 (decades), else
    8 (octets); upsample outputs (segs = 4) keep each output-pixel parity in its own segment of slabs."""
    M, N = out.shape
    x = out.to(F64)
    if segs > 1:
        NF, H, W = src_rows
        x = x.reshape(NF, H, 2, W, 2, N).permute(2, 4, 0, 1, 3, 5).reshape(4 * NF * H * W, N)
        M = x.shape[0]
    slabs = (M + 31) // 32
    pad = torch.zeros((slabs * 32, N), dtype=F64, device=x.device)
    pad[:M] = x
    v = pad.reshape(slabs, 32, N)
    s1, s2, sa = v.sum(1), (v * v).sum(1), v.abs().sum(1)
    mg = 10 if N % 10 == 0 else 8
    sel = torch.zeros((N, N // 32 * 4), dtype=F64, device=x.device)
    for k in range(N // 32):
        d0 = (k * 32) // mg
        for piece in range(4):
            g = d0 + piece
            lo, hi = max(k * 32, g * mg), min(k * 32 + 32, g * mg + mg, N)
            if lo < hi:
                sel[lo:hi, k * 4 + piece] = 1.0
    written = sel.sum(0) > 0
    exp = torch.stack([s1 @ sel, s2 @ sel], -1).reshape(slabs, N // 32, 4, 2)
    mag = torch.stack([sa @ sel, s2 @ sel], -1).reshape(slabs, N // 32, 4, 2)
    return exp, mag, written.reshape(N // 32, 4)


def check_colsums(cs, out, segs=1, src_rows=None):
    exp, mag, written = colsum_expected(out, segs, src_rows)
    got = cs.to(F64)
    assert got.shape == exp.shape, (tuple(got.shape), tuple(exp.shape))
    m = written[None, :, :, None].expand_as(exp)
    return Cmp("producer column sums", got[m], exp[m], COLSUM_REL * mag[m] + 1e-30)


# ------------------------------------------------------------------------------------------------ views
def view_mask(base, view):
    m = torch.zeros(base.shape, dtype=torch.bool, device=base.device)
    m.as_strided(view.shape, view.stride(), view.storage_offset() - base.storage_offset()).fill_(True)
    return m


def check_outside_view(before, after, mask):
    """Every element of the underlying buffer outside the view must keep its bits."""
    bits = {1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[before.element_size()]
    b, a = before.view(bits), after.view(bits)
    changed = (b != a) & ~mask
    n = int(changed.sum())
    where = tuple(int(i) for i in changed.nonzero()[0]) if n else ()
    return Flag("buffer outside the out= view", n == 0, f"{n} elements changed outside the view, first at {where}")


# ------------------------------------------------------------------------------------------------ per-op checks
# Whole-tensor rel-L2, the second check: one bf16 rounding of the output gives ~1.7e-3 on these tensors (B200 audit,
# profiles/r3_launch_audit.log); attention adds the rounding of P (~2.4e-3)
REL_ROUND = 2.5e-3
REL_ATTN = 4e-3


def row_blocks(what, res, step, block, rel_max=None, dims=None):
    """Compare `res` with a reference built block by block: block(lo, hi) -> (ref, bound) of rows lo..hi."""
    cmp = Cmp(what, rel_max=rel_max, dims=dims)
    for lo in range(0, res.shape[0], step):
        hi = min(res.shape[0], lo + step)
        ref, bound = block(lo, hi)
        cmp.add(res[lo:hi], ref, bound, lo)
    return cmp.finish()


def gemm_check(res, rows_fn, w, K, a, splits=1, step=None, rel_max=REL_ROUND, dims=("row", "col")):
    """A GEMM-family launch: rows_fn(lo, hi) gives rows lo..hi of the A operand (fp64), w the [N, K] weights; the fused
    epilogue of `a` (bias, row bias, residual, GEGLU) is applied in fp64."""
    c = c_gemm(K, splits) * (1 + U)
    step = step or max(1, Cmp.STEP // max(w.shape[0], w.shape[1]))
    res_t = a.get("residual")

    def block(lo, hi):
        acc, s = mm_abs(rows_fn(lo, hi), w)
        acc, s = epilogue_ref(acc, s, lo, a.get("bias"), a.get("row_bias"), a.get("rows_per_batch", 1),
                              None if res_t is None else res_t[lo:hi])
        if a.get("geglu"):
            ref, extra = geglu_ref(acc, s, c)
            return ref, U * ref.abs() + extra
        return acc, U * acc.abs() + c * s
    return row_blocks("gemm+geglu" if a.get("geglu") else "gemm", res, step, block, rel_max, dims)


def chk_gemm(a, res, ctx):
    a0, a1 = a["a"], a["a2"]
    K = a["w"].shape[1]

    def rows(lo, hi):
        r = a0[lo:hi].to(F64)
        return r if a1 is None else torch.cat([r, a1[lo:hi].to(F64)], 1)
    return [gemm_check(res, rows, a["w"], K, a, ctx.get("splits", 1))]


def _img_step(per_img, width):
    return max(1, Cmp.STEP // max(1, width * per_img)) * per_img


def chk_conv3x3(a, res, ctx):
    NF, H, W, s_ = a["NF"], a["H"], a["W"], a["stride"]
    Ho, Wo = (H - 1) // s_ + 1, (W - 1) // s_ + 1
    x, o, hw = a["x"], Ho * Wo, H * W
    cmp = gemm_check(res, lambda lo, hi: im2col64(x[lo // o * hw:hi // o * hw], (hi - lo) // o, H, W, s_), a["w"],
                     a["w"].shape[1], a, ctx.get("splits", 1), step=_img_step(o, a["w"].shape[1]),
                     dims=("image", "y", "x", "channel"))
    r, c = cmp.worst_at
    cmp.worst_at = (r // o, r // Wo % Ho, r % Wo, c)
    return [cmp]


def chk_im2col3x3(a, res, ctx):
    ref = im2col64(a["x"], a["NF"], a["H"], a["W"], a["stride"])
    return [Cmp("im2col3x3", res, ref, 1e-300)]


def chk_frame_conv(a, res, ctx):
    xp, taps, tr = a["xpad"], a["taps"], a["tap_rows"]
    out = [gemm_check(res, lambda lo, hi: torch.cat([xp[t * tr + lo:t * tr + hi] for t in range(taps)], 1).to(F64),
                      a["w"], a["w"].shape[1], a, ctx.get("splits", 1), dims=("row", "channel"))]
    pad = (taps // 2) * tr
    z = xp[:pad].abs().sum() + xp[xp.shape[0] - pad:].abs().sum() if pad else 0
    out.append(Flag("zero pad frames of the frame-conv input", float(z) == 0, f"sum |pad| = {float(z)}"))
    return out


def chk_upsample_conv3x3(a, res, ctx):
    NF, H, W, x = a["NF"], a["H"], a["W"], a["x"]
    o = 4 * H * W
    # 4 tap-GEMMs of K = 4C summed per output: the bound counts all 16 C terms
    c = c_gemm(16 * x.shape[1]) * (1 + U)

    def block(lo, hi):
        acc, s = upsample_phase_ref(x[lo // 4:hi // 4], (hi - lo) // o, H, W, a["w_phases"])
        acc, s = epilogue_ref(acc, s, lo, a["bias"])
        return acc, U * acc.abs() + c * s
    cmp = row_blocks("upsample conv", res, _img_step(o, 4 * x.shape[1]), block, REL_ROUND)
    r, ch = cmp.worst_at
    cmp.worst_at, cmp.dims = (r // o, r // (2 * W) % (2 * H), r % (2 * W), ch), ("image", "y", "x", "channel")
    return [cmp]


def chk_groupnorm_scale_shift(a, res, ctx):
    X = a["x"] if a["x2"] is None else torch.cat([a["x"], a["x2"]], 1)
    scale, shift, bs, bsh = gn_scale_shift64(X, a["samples"], a["gamma"], a["beta"], a["eps"], a["groups"])
    d = ("sample", "channel")
    return [Cmp("GroupNorm scale", res[..., 0], scale, bs, None, d),
            Cmp("GroupNorm shift", res[..., 1], shift, bsh, None, d)]


def _norm_rows(a):
    X = a["x"] if a["x2"] is None else torch.cat([a["x"], a["x2"]], 1)
    return X, max(1, Cmp.STEP // X.shape[1]), X.shape[0] // a["samples"]


def chk_groupnorm_apply(a, res, ctx):
    X, step, rps = _norm_rows(a)
    ss = a["scale_shift"].to(F64)

    def block(lo, hi):
        idx = torch.arange(lo, hi, device=X.device) // rps
        y, mag, t = apply_rows(X[lo:hi], ss[idx, :, 0], ss[idx, :, 1], a["silu"])
        # fp32 FMA and the fast SiLU (__expf, __fdividef: 2^-21 relative) against |x scale| + |shift|
        return y, U * y.abs() + 2.0 ** -20 * (SILU_SLOPE * mag + t.abs())
    return [row_blocks("GroupNorm apply", res, step, block, REL_ROUND, ("row", "channel"))]


def chk_groupnorm(a, res, ctx):
    X, step, rps = _norm_rows(a)
    scale, shift, bs, bsh = gn_scale_shift64(X, a["samples"], a["gamma"], a["beta"], a["eps"], a["groups"])

    def block(lo, hi):
        idx = torch.arange(lo, hi, device=X.device) // rps
        y, mag, t = apply_rows(X[lo:hi], scale[idx], shift[idx], a["silu"])
        stat = X[lo:hi].to(F64).abs() * bs[idx] + bsh[idx]
        return y, U * y.abs() + SILU_SLOPE * (stat + 2.0 ** -20 * mag) + 2.0 ** -20 * t.abs()
    return [row_blocks("GroupNorm", res, step, block, REL_ROUND, ("row", "channel"))]


def chk_layernorm(a, res, ctx):
    x = a["x"]

    def block(lo, hi):
        y, small = layernorm_ref(x[lo:hi], a["gamma"], a["beta"], a["eps"])
        return y, U * y.abs() + small
    return [row_blocks("LayerNorm", res, max(1, Cmp.STEP // x.shape[1]), block, REL_ROUND, ("row", "channel"))]


def _attn_out(o, batch, heads, Sq, d):
    return o.permute(0, 2, 1, 3).reshape(batch * Sq, heads * d)


def attention_ref(a, v=None):
    heads, d, pitch = a["heads"], a["d"], a["head_pitch"]
    qrows, krows = attention_layout(a)
    Q = heads_of(a["q"], qrows, heads, pitch, d)
    K = heads_of(a["k"], krows, heads, pitch, d)
    V = heads_of(a["v"] if v is None else v, krows, heads, pitch, d)
    scale = a["scale"] if a["scale"] is not None else d ** -0.5
    o, bnd = attention_core(Q, K, V, scale)
    return o, bnd


def chk_attention(a, res, ctx):
    batch, heads, Sq, d = a["batch"], a["heads"], a["Sq"], a["d"]
    o, bnd = attention_ref(a)
    cmp = Cmp("attention", res, _attn_out(o, batch, heads, Sq, d), _attn_out(bnd, batch, heads, Sq, d), REL_ATTN)
    r, c = cmp.worst_at
    cmp.worst_at, cmp.dims = (r // Sq, c // d, r % Sq, c % d), ("batch", "head", "query", "column")
    out = [cmp]
    if ctx.get("probe") is not None:
        out += ctx["probe"](a, res)
    return out


def frame_attention_ref(qkv, B, F_, HW, heads, d, pitch, rope=None, bias=None):
    hp = heads * pitch
    rows = frame_layout(B, F_, HW, qkv.device)
    Q = heads_of(qkv, rows, heads, pitch, d)
    K = heads_of(qkv[:, hp:], rows, heads, pitch, d)
    V = heads_of(qkv[:, 2 * hp:], rows, heads, pitch, d)
    scale = d ** -0.5
    if rope is None:
        return attention_core(Q, K, V, scale)
    # q scaled before the rotation; the kernel rounds both rotated operands to bf16 before Q K^T
    Qs = rope64(Q.to(F64) * scale, rope)
    Ks = rope64(K.to(F64), rope)
    return attention_core(Qs, Ks, V, 1.0, bias=bias, rho=RHO_ROPE)


def _frame_out(o, B, F_, HW, heads, d):
    return o.reshape(B, HW, heads, F_, d).permute(0, 3, 1, 2, 4).reshape(B * F_ * HW, heads * d)


def _frame_cmp(what, res, o, bnd, a, rel_max):
    B, F_, HW, heads, d = a["B"], a["F"], a["HW"], a["heads"], a["d"]
    cmp = Cmp(what, res, _frame_out(o, B, F_, HW, heads, d), _frame_out(bnd, B, F_, HW, heads, d), rel_max)
    r, c = cmp.worst_at
    cmp.worst_at = (r // (F_ * HW), r // HW % F_, r % HW, c // d, c % d)
    cmp.dims = ("item", "frame", "pixel", "head", "column")
    return cmp


def chk_frame_attention(a, res, ctx):
    o, bnd = frame_attention_ref(a["qkv"], a["B"], a["F"], a["HW"], a["heads"], a["d"], a["head_pitch"])
    out = [_frame_cmp("frame attention", res, o, bnd, a, REL_ATTN)]
    if ctx.get("probe") is not None:
        out += ctx["probe"](a, res)
    return out


def chk_temporal_attention(a, res, ctx):
    o, bnd = frame_attention_ref(a["qkv"], a["B"], a["F"], a["HW"], a["heads"], a["d"], a["head_pitch"], a["rope"],
                                 a["bias"])
    out = [_frame_cmp("temporal attention", res, o, bnd, a, REL_ATTN)]
    if ctx.get("probe") is not None:
        out += ctx["probe"](a, res)
    return out


def chk_causal_attention_small(a, res, ctx):
    B, L, H, d = a["B"], a["L"], a["heads"], a["d"]
    x = a["qkv"].to(F64).reshape(B, L, 3, H, d)
    Q, K, V = (x[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    o, bnd = attention_core(Q, K, V, d ** -0.5, causal=True, c_p=C_ATTN_P_F32)
    return [Cmp("causal attention", res, _attn_out(o, B, H, L, d), _attn_out(bnd, B, H, L, d), REL_ROUND)]


def chk_linear_smallm(a, res, ctx):
    x = a["x"].to(F64)
    if a["silu_in"]:
        x = silu64(x)
    acc, s = mm_abs(x, a["w"])
    if a["bias"] is not None:
        acc, s = acc + a["bias"].to(F64), s + a["bias"].to(F64).abs()
    # fp32 FMA chain over K (the fast SiLU on load adds 2^-21 relative to every term)
    c = (a["x"].shape[1] + 4) * U32 + 2.0 ** -20
    if a["silu_out"]:
        return [Cmp("linear_smallm", res, silu64(acc), SILU_SLOPE * c * s + 2.0 ** -20 * acc.abs() + 1e-30, 1e-5)]
    return [Cmp("linear_smallm", res, acc, c * s + 1e-30, 1e-5)]


def chk_timestep_embedding(a, res, ctx):
    t = a["t"].to(F64)
    half = a["dim"] // 2
    w = 10000.0 ** (-torch.arange(half, dtype=F64, device=t.device) / half)
    ang = t[:, None] * w[None]
    ref = torch.cat([ang.cos(), ang.sin()], 1)
    # fp32 angle: the frequency (2 ulp), the product and the argument reduction of cos / sin (1 ulp each) put it within
    # 2^-21 |angle|; cos / sin themselves add 2^-21
    bound = 2.0 ** -21 * torch.cat([ang.abs(), ang.abs()], 1) + 2.0 ** -21
    return [Cmp("timestep embedding", res, ref, bound)]


def chk_conv_in(a, res, ctx):
    x = a["x"].to(F64)
    B, Cin, Fr, H, W = x.shape
    if a["input_scale"] is not None:
        x = x * float(a["input_scale"])
    xi = x.permute(0, 2, 1, 3, 4).reshape(B * Fr, Cin, H, W)
    w = a["w"].to(F64)
    y = F.conv2d(xi, w, a["bias"].to(F64), padding=1).permute(0, 2, 3, 1).reshape(-1, w.shape[0])
    s = F.conv2d(xi.abs(), w.abs(), a["bias"].to(F64).abs(), padding=1).permute(0, 2, 3, 1).reshape(-1, w.shape[0])
    return [Cmp("conv_in (fp32)", res, y, U * y.abs() + (9 * Cin + 4) * U32 * s, REL_ROUND)]


def chk_conv_in_tc(a, res, ctx):
    x = a["x"]
    B, Cin, Fr, H, W = x.shape
    xs = x if a["input_scale"] is None else x * a["input_scale"]
    xb = xs.to(BF16)                       # im2col rounds the (scaled) fp32 input to bf16 once
    xi = xb.permute(0, 2, 1, 3, 4).reshape(B * Fr, Cin, H, W).to(F64)
    col = F.unfold(xi, 3, padding=1).transpose(1, 2).reshape(B * Fr * H * W, 9 * Cin)   # K index c*9 + kh*3 + kw
    kpad = a["w_pad"].shape[1]
    assert float(a["w_pad"][:, 9 * Cin:].abs().sum()) == 0 or kpad == 9 * Cin
    return [gemm_check(res, lambda lo, hi: col[lo:hi], a["w_pad"][:, :9 * Cin], kpad, {"bias": a["bias"]})]


def chk_conv_out_tc(a, res, ctx):
    """GroupNorm apply + SiLU (bf16 activations: U |h| per tap) -> 3x3 conv -> bf16 rows -> fp32 [B, Cout, F, H, W]."""
    B, Fr, H, W, Cout = a["B"], a["Fr"], a["H"], a["W"], a["Cout"]
    ss = a["scale_shift"].to(F64)
    h, _, _ = apply_ref(a["x"], ss[..., 0], ss[..., 1], B, True)
    acc, s = conv_mm(h, B * Fr, H, W, 1, a["w_pad"][:Cout])
    acc = acc + a["bias_pad"][:Cout].to(F64)
    s = s + a["bias_pad"][:Cout].to(F64).abs()
    ref = acc.reshape(B, Fr, H, W, Cout).permute(0, 4, 1, 2, 3)
    s = s.reshape(B, Fr, H, W, Cout).permute(0, 4, 1, 2, 3)
    K = a["w_pad"].shape[1]
    return [Cmp("conv_out (tensor cores)", res, ref, U * ref.abs() + (U + c_gemm(K)) * (1 + U) * s, REL_ATTN,
                ("item", "channel", "frame", "y", "x"))]


def chk_embedding_add(a, res, ctx):
    lab = a["labels"].clamp(0, a["table"].shape[0] - 1)
    ref = a["emb"].to(F64) + a["table"].to(F64)[lab]
    return [Cmp("embedding_add", res, ref, U32 * ref.abs() + 1e-300)]


def chk_upsample_nearest2x(a, res, ctx):
    NF, H, W = a["NF"], a["H"], a["W"]
    x = a["x"].reshape(NF, H, 1, W, 1, -1).expand(NF, H, 2, W, 2, a["x"].shape[1])
    return [Cmp("upsample_nearest2x", res, x.reshape(NF * 4 * H * W, -1), 1e-300)]


def chk_cfg_ddim_step(a, res, ctx):
    u, t, lat = (a[k].to(F64) for k in ("noise_uncond", "noise_text", "latents"))
    g, at, ap = a["guidance"], a["alpha_t"], a["alpha_prev"]
    eps = u + g * (t - u)
    x0 = (lat - math.sqrt(1 - at) * eps) / math.sqrt(at)
    ref = math.sqrt(ap) * x0 + math.sqrt(1 - ap) * eps
    ea = u.abs() + abs(g) * (t.abs() + u.abs())
    mag = math.sqrt(ap) * (lat.abs() + math.sqrt(1 - at) * ea) / math.sqrt(at) + math.sqrt(1 - ap) * ea
    return [Cmp("cfg_ddim_step", res, ref, 2.0 ** -20 * mag + 1e-300)]


def chk_cfg_linear_step(a, res, ctx):
    u, t, lat = (a[k].to(F64) for k in ("noise_uncond", "noise_text", "latents"))
    g = a["guidance"]
    eps = u + g * (t - u)
    ref = a["a"] * lat + a["b"] * eps
    mag = abs(a["a"]) * lat.abs() + abs(a["b"]) * (u.abs() + abs(g) * (t.abs() + u.abs()))
    if a["noise"] is not None:
        ref = ref + a["c_noise"] * a["noise"].to(F64)
        mag = mag + abs(a["c_noise"]) * a["noise"].to(F64).abs()
    return [Cmp("cfg_linear_step", res, ref, 2.0 ** -21 * mag + 1e-300)]


def chk_cfg_combine(a, res, ctx):
    c, u = a["cond"].to(F64), a["uncond"].to(F64)
    g = u + a["scale"] * (c - u)
    ref = torch.cat([g, g]) if a["duplicate"] else g
    mag = u.abs() + abs(a["scale"]) * (c.abs() + u.abs())
    mag = torch.cat([mag, mag]) if a["duplicate"] else mag
    return [Cmp("cfg_combine", res, ref, 2.0 ** -22 * mag + 1e-300)]


def chk_clip_embed(a, res, ctx):
    L = a["L"]
    rows = a["ids"].numel()
    tok = a["tok"].to(F64)[a["ids"]]
    pos = a["pos"].to(F64)[torch.arange(rows, device=tok.device) % L]
    ref = tok + pos
    return [Cmp("clip_embed", res, ref, U * ref.abs() + U32 * (tok.abs() + pos.abs()) + 1e-300)]


def chk_activation_(a, res, ctx):
    x = a["x"].to(F64)
    ref = x * torch.sigmoid(1.702 * x) if a["kind"] == "quick_gelu" else gelu64(x)
    return [Cmp(f"activation {a['kind']}", res, ref, U * ref.abs() + 2.0 ** -20 * x.abs() + 1e-300, REL_ROUND)]


def chk_softmax_rows_(a, res, ctx):
    s = a["s"].to(F64)
    p = torch.softmax(a["scale"] * s, -1)
    n = s.shape[1]
    # fp32 exponentials (2^-21) and an fp32 row sum of n terms, relative to each probability
    return [Cmp("softmax_rows", res, p, (U + (n + 8) * U32 + 2.0 ** -20) * p + 1e-38, REL_ROUND)]


def chk_image_to_uint8(a, res, ctx):
    y = a["y"][:, :3].to(F64)
    v = ((y / 2 + 0.5) * 255 + 0.5).clamp(0, 255)
    ref = v.floor()
    # the kernel computes in fp32: within 2^-16 of an integer the fp32 value may land on either side
    near = (v - v.round()).abs() < 2.0 ** -16
    bound = torch.where(near, torch.ones_like(v), torch.full_like(v, 1e-300))
    return [Cmp("image_to_uint8", res, ref, bound)]


def chk_pointwise_conv_nchw(a, res, ctx):
    x = a["x"].to(F64) * a["scale"]
    w = a["w"].to(F64)
    ref = torch.einsum("oc,nchw->nohw", w, x) + a["bias"].to(F64)[None, :, None, None]
    mag = torch.einsum("oc,nchw->nohw", w.abs(), x.abs()) + a["bias"].to(F64).abs()[None, :, None, None]
    return [Cmp("pointwise_conv_nchw", res, ref, (x.shape[1] + 2) * U32 * mag + 1e-300)]


CHECKERS = {
    "gemm": chk_gemm, "conv3x3": chk_conv3x3, "im2col3x3": chk_im2col3x3, "frame_conv": chk_frame_conv,
    "upsample_conv3x3": chk_upsample_conv3x3, "groupnorm_scale_shift": chk_groupnorm_scale_shift,
    "groupnorm_apply": chk_groupnorm_apply, "groupnorm": chk_groupnorm, "layernorm": chk_layernorm,
    "attention": chk_attention, "frame_attention": chk_frame_attention, "temporal_attention": chk_temporal_attention,
    "causal_attention_small": chk_causal_attention_small, "linear_smallm": chk_linear_smallm,
    "timestep_embedding": chk_timestep_embedding, "conv_in": chk_conv_in, "conv_in_tc": chk_conv_in_tc,
    "conv_out_tc": chk_conv_out_tc, "embedding_add": chk_embedding_add,
    "upsample_nearest2x": chk_upsample_nearest2x, "cfg_ddim_step": chk_cfg_ddim_step,
    "cfg_linear_step": chk_cfg_linear_step, "cfg_combine": chk_cfg_combine, "clip_embed": chk_clip_embed,
    "activation_": chk_activation_, "softmax_rows_": chk_softmax_rows_, "image_to_uint8": chk_image_to_uint8,
    "pointwise_conv_nchw": chk_pointwise_conv_nchw,
}

# launching functions of `ops` that the model runs below do not issue, with the test that covers each
COVERED_ELSEWHERE = {
    "layernorm_scatter": "tests/test_sharding_gpu.py, tests/test_p2p_gpu.py (frame-sharded temporal attention)",
    "add_gathered": "tests/test_sharding_gpu.py, tests/test_p2p_gpu.py (frame-sharded temporal attention)",
    "groupnorm_sums": "tests/test_sharding_gpu.py (frame-sharded GroupNorm statistics)",
    "groupnorm_finalize_sums": "tests/test_sharding_gpu.py (frame-sharded GroupNorm statistics)",
    "conv_out": "tests/test_kernels_gpu.py::test_conv_in_and_out (fp32 conv_out, used when C % 64 != 0)",
    "im2col3x3": "tests/test_kernels_gpu.py::test_conv3x3_stride_and_explicit_im2col (explicit patch matrix, C % 64 != 0)",
}


def launching_functions():
    """Every public function of `ops` that launches a kernel itself or through another one."""
    from lavie_b200 import ops
    names = set()
    for name, fn in inspect.getmembers(ops, inspect.isfunction):
        if fn.__module__ != ops.__name__ or name.startswith("_"):
            continue
        src = inspect.getsource(fn)
        if "_Launch(" in src:
            names.add(name)
    for name, fn in inspect.getmembers(ops, inspect.isfunction):       # composites: call a launching function
        if fn.__module__ == ops.__name__ and not name.startswith("_") and name not in names:
            src = inspect.getsource(fn).split(":", 1)[1]
            if any(f"{n}(" in src for n in names if n != name):
                names.add(name)
    return names


def ramp_values(rows, seq_len, seq_stride, F_=None):
    """Key-index ramps of the probe V, one column each, exact or nearly exact in bf16: the position inside the key
    sequence (j / seq_len), the same position modulo 64 (exact: adjacent keys always differ), and the index of the
    sequence modulo 64 (tells the key segments / frames apart)."""
    r = torch.arange(rows, dtype=torch.int64)
    pos = r // seq_stride % seq_len
    return torch.stack([pos.to(F64) / seq_len, (pos % 64).to(F64) / 64, (r // (seq_len * seq_stride) % 64).to(F64) / 64],
                       1)


def attention_probes(name, real, a):
    """Launch the attention kernel `real` again on the recorded Q and K with probe values: V = 1 in every real head
    column (every output must be 1 within 2^-7: an extra or missing key or a wrong normalisation moves it by ~1/keys),
    then V = key-index ramps (ramp_values) in the first columns of every head, whose outputs must match the fp64
    expected key index within the attention bound."""
    heads, d, pitch = a["heads"], a["d"], a["head_pitch"]
    out = []
    for kind in ("ones", "ramp"):
        if name == "attention":
            k = a["k"]
            vbuf = torch.zeros((k.shape[0], k.stride(0)), dtype=BF16, device=k.device)
            v = vbuf[:, :k.shape[1]]
            hv = v[:, :heads * pitch].reshape(-1, heads, pitch)
            if kind == "ones":
                hv[..., :d] = 1.0
            else:
                hv[..., :3] = ramp_values(k.shape[0], a["Sk"], 1)[:, None, :].to(device=k.device, dtype=BF16)
            got = real(a["q"], a["k"], v, a["batch"], heads, a["Sq"], a["Sk"], d, pitch, a["kv_batch_div"], a["scale"],
                       None, a["sparse_causal_frames"], a["sc_halo"])
            o, bnd = attention_ref(a, v)
            ref = _attn_out(o, a["batch"], heads, a["Sq"], d)
            bnd = _attn_out(bnd, a["batch"], heads, a["Sq"], d)
            ncol = 3
        else:
            qkv = a["qkv"].clone()
            hp = heads * pitch
            hv = qkv[:, 2 * hp:3 * hp].reshape(-1, heads, pitch)
            hv.zero_()
            if kind == "ones":
                hv[..., :d] = 1.0
            else:
                # rows (b, f, pixel): the key sequence of a pixel runs over the frames, stride HW rows
                hv[..., :2] = ramp_values(qkv.shape[0], a["F"], a["HW"])[:, None, :2].to(device=qkv.device, dtype=BF16)
            if name == "frame_attention":
                got = real(qkv, a["B"], a["F"], a["HW"], heads, d, pitch)
                o, bnd = frame_attention_ref(qkv, a["B"], a["F"], a["HW"], heads, d, pitch)
            else:
                got = real(qkv, a["B"], a["F"], a["HW"], heads, d, pitch, a["rope"], a["bias"])
                o, bnd = frame_attention_ref(qkv, a["B"], a["F"], a["HW"], heads, d, pitch, a["rope"], a["bias"])
            ref = _frame_out(o, a["B"], a["F"], a["HW"], heads, d)
            bnd = _frame_out(bnd, a["B"], a["F"], a["HW"], heads, d)
            ncol = 2
        if got.is_cuda:
            torch.cuda.synchronize()
        if kind == "ones":
            out.append(Cmp(f"{name} probe V=1", got, torch.ones_like(ref), 2.0 ** -7))
        else:
            cols = (torch.arange(heads)[:, None] * d + torch.arange(ncol)).reshape(-1).to(got.device)
            out.append(Cmp(f"{name} probe V=key ramp", got[:, cols], ref[:, cols], bnd[:, cols]))
    return out


# ------------------------------------------------------------------------------------------------ recorder
MODEL_FILES = ("unet.py", "vsr.py", "vae.py", "clip.py")


def model_block():
    """The model block that issued the launch: the nearest caller frame in a model file with a prefix `p`, and the
    geometry (B, Fr, H, W) of its activations when that frame holds it."""
    f = sys._getframe(2)
    fallback = None
    while f is not None:
        fn = os.path.basename(f.f_code.co_filename)
        if fn in MODEL_FILES:
            p = f.f_locals.get("p")
            if isinstance(p, str):
                loc = f.f_locals
                H, W = loc.get("H", loc.get("h")), loc.get("W", loc.get("w"))
                if not isinstance(W, int) and isinstance(loc.get("HW"), int):
                    H, W = loc["HW"], 1
                geom = (loc.get("B"), loc.get("Fr"), H, W)
                return f"{fn[:-3]}:{p}", (geom if all(isinstance(g, int) for g in geom) else None)
            fallback = fallback or f"{fn[:-3]}:{f.f_code.co_name}"
        f = f.f_back
    return fallback or "test", None


def decode_item_frame(r, geom, rows):
    """Rewrite a worst-element position in activation rows, (row, channel) or (image, y, x, channel), as (item, frame,
    y, x, channel) when the issuing block's geometry (B, Fr, H, W) matches the launch."""
    if geom is None or not isinstance(r, Cmp) or not r.dims or not r.worst_at:
        return
    B, Fr, H, W = geom
    if r.dims[0] == "row" and len(r.worst_at) == 2 and rows == B * Fr * H * W:
        row, c = r.worst_at
        r.worst_at = (row // (Fr * H * W), row // (H * W) % Fr, row // W % H, row % W, c)
        r.dims = ("item", "frame", "y", "x", "channel")
    elif r.dims[0] == "image" and len(r.worst_at) == 4:
        img, y, x, c = r.worst_at
        if img < B * Fr:
            r.worst_at, r.dims = (img // Fr, img % Fr, y, x, c), ("item", "frame", "y", "x", "channel")


class OpRow:
    def __init__(self):
        self.launches = 0
        self.worst = 0.0
        self.worst_rel = 0.0
        self.plans = set()
        self.probes = 0


class Recorder:
    """Wraps the launching functions of `ops` for the duration of a `with` block."""

    def __init__(self, log):
        from lavie_b200 import _lib, ops
        self.ops = ops
        self.lib = _lib.load()
        self.log = log
        self.real = {}
        self.probed = set()
        self.calls = 0

    def __enter__(self):
        self.tf32 = tf32_off()
        for name in CHECKERS:
            fn = getattr(self.ops, name)
            self.real[name] = fn
            setattr(self.ops, name, self._wrap(name, fn))
        return self

    def __exit__(self, *exc):
        for name, fn in self.real.items():
            setattr(self.ops, name, fn)
        tf32_restore(self.tf32)
        return False

    def _plan(self, M, N, K, conv, geglu):
        import ctypes
        bn, sp, tt, ts = (ctypes.c_int() for _ in range(4))
        self.lib.lavie_gemm_plan(M, N, K, conv, int(geglu), self.ops.WORKSPACE_BYTES, ctypes.byref(bn), ctypes.byref(sp),
                                 ctypes.byref(tt), ctypes.byref(ts))
        kinds = set()
        kinds.add(f"split-K x{sp.value}" if sp.value > 1 else "full-width")
        if tt.value:
            kinds.add("main+tail window")
        return kinds, max(sp.value, ts.value, 1)

    def _wrap(self, name, fn):
        sig = inspect.signature(fn)
        check = CHECKERS[name]

        def wrapper(*args, **kw):
            bound = sig.bind(*args, **kw)
            bound.apply_defaults()
            a = dict(bound.arguments)
            block, geom = model_block()
            idx = self.calls
            self.calls += 1
            before = {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in a.items()}
            out_view = a.get("out")
            base_before = None
            if torch.is_tensor(out_view) and out_view._base is not None:
                base_before = out_view._base.detach().clone()
            res = fn(*args, **kw)
            torch.cuda.synchronize()
            ctx = {}
            plans = set()
            if name in ("gemm", "conv3x3", "frame_conv"):
                if name == "gemm":
                    K = a["w"].shape[1]
                    M, N = a["a"].shape[0], a["w"].shape[0]
                    plans, splits = self._plan(M, N, K, 0, a["geglu"])
                elif name == "conv3x3":
                    K = a["w"].shape[1]
                    plans, splits = self._plan(res.shape[0], a["w"].shape[0], K, 1, False)
                else:
                    K = a["w"].shape[1]
                    plans, splits = self._plan(res.shape[0], a["w"].shape[0], K, 0, False)
                ctx["splits"] = splits
            if name in ("attention", "frame_attention", "temporal_attention"):
                key = (name,) + tuple((k, tuple(v.shape) if torch.is_tensor(v) else v) for k, v in a.items()
                                      if k not in ("out", "scale"))
                if key not in self.probed:
                    self.probed.add(key)
                    ctx["probe"] = lambda aa, rr, n=name: self._probe(n, aa, rr)
            results = check(before, res, ctx)
            if getattr(res, "_gn_colsums", None) is not None:
                segs = getattr(res, "_gn_segs", 1)
                src = (a["NF"], a["H"], a["W"]) if segs > 1 else None
                results.append(check_colsums(res._gn_colsums, res, segs, src))
            if base_before is not None:
                results.append(check_outside_view(base_before, out_view._base, view_mask(out_view._base, out_view)))
            if geom is not None and name in ("conv3x3", "upsample_conv3x3") and a["NF"] != geom[0] * geom[1]:
                geom = None
            for r in results:
                decode_item_frame(r, geom, res.shape[0] if res.dim() == 2 else -1)
            self._record(name, idx, block, a, results, plans, "probe" in ctx)
            return res

        wrapper.__wrapped__ = fn
        return wrapper

    def _probe(self, name, a, res):
        return attention_probes(name, self.real[name], a)

    def _record(self, name, idx, block, a, results, plans, probed):
        row = self.log.rows[name]
        row.launches += 1
        row.plans |= plans
        row.probes += int(probed)
        for r in results:
            row.worst = max(row.worst, r.worst)
            row.worst_rel = max(row.worst_rel, r.rel if isinstance(r, Cmp) else 0.0)
            if not r.ok:
                shapes = {k: (tuple(v.shape) if torch.is_tensor(v) else v) for k, v in a.items()
                          if torch.is_tensor(v) or isinstance(v, (int, float, bool, str))}
                self.log.failures.append(f"[{self.log.run}] #{idx} ops.{name} from {block}: {r}; args {shapes}"
                                         + (f"; plan {sorted(plans)}" if plans else ""))


class AuditLog:
    def __init__(self):
        self.rows = collections.defaultdict(OpRow)
        self.failures = []
        self.runs = []
        self.run = ""

    def record(self, run_name):
        self.run = run_name
        self.runs.append(run_name)
        return Recorder(self)

    def summary(self):
        lines = [f"{'op':24s} {'launches':>8s} {'probes':>6s} {'worst err/bound':>15s} {'worst rel-L2':>12s}  plans"]
        for name in sorted(self.rows):
            r = self.rows[name]
            lines.append(f"{name:24s} {r.launches:8d} {r.probes:6d} {r.worst:15.3g} {r.worst_rel:12.3g}  "
                         f"{', '.join(sorted(r.plans))}")
        return "\n".join(lines)


# ------------------------------------------------------------------------------------------------ GPU runs
RUNS_DEFAULT = ("base headline", "base ragged", "interpolation 61f", "vsr 16f", "vsr ragged", "clip", "vae 40x64",
                "vae ragged")


@pytest.fixture(scope="session")
def audit_log():
    return AuditLog()


@pytest.fixture(scope="session")
def reference_selfcheck():
    """Each GPU reference helper against the same helper on the CPU in fp64 at a small shape: a reduced-precision default
    (TF32, reduced-precision reductions) turning up in a later torch would show here."""
    saved = tf32_off()
    g = torch.Generator().manual_seed(0)

    def both(fn, *xs, **kw):
        cpu = fn(*xs, **kw)
        gpu = fn(*(x.cuda() if torch.is_tensor(x) else x for x in xs), **kw)
        cpu = cpu if isinstance(cpu, tuple) else (cpu,)
        gpu = gpu if isinstance(gpu, tuple) else (gpu,)
        for c, d in zip(cpu, gpu):
            assert rel_l2(d.cpu(), c) < 1e-6, fn.__name__

    a = torch.randn(300, 320, generator=g).to(BF16)
    w = torch.randn(256, 320, generator=g).to(BF16)
    both(mm_abs, a, w)
    x = torch.randn(2 * 6 * 10, 64, generator=g).to(BF16)
    both(im2col64, x, 2, 6, 10, 2)
    both(upsample_phase_ref, x, 2, 6, 10, torch.randn(4 * 32, 4 * 64, generator=g).to(BF16))
    gam, bet = torch.randn(64, generator=g), torch.randn(64, generator=g)
    both(gn_scale_shift64, x, 2, gam, bet, 1e-6)
    both(layernorm_ref, x, gam, bet, 1e-5)
    q, k, v = (torch.randn(3, 2, 40, 24, generator=g).to(BF16) for _ in range(3))
    both(attention_core, q, k, v, 0.2)
    both(attention_core, q, k, v, 0.2, causal=True)
    y = torch.randn(200, 320, generator=g).to(BF16)
    both(lambda t: colsum_expected(t)[0], y)
    yield True
    tf32_restore(saved)


def _synthetic_base(synthetic_sd, config=None):
    from lavie_b200 import UNet3DConditionModel
    m = UNet3DConditionModel(config, use_cuda_graph=False) if config is not None else \
        UNet3DConditionModel(use_cuda_graph=False)
    m.load_state_dict(synthetic_sd, strict=True)
    return m.to("cuda").eval()


def _finish(log):
    torch.cuda.synchronize()
    if log.failures:
        msg = "\n".join(log.failures[:20])
        n = len(log.failures)
        log.failures.clear()
        pytest.fail(f"{n} audited launches out of bounds:\n{msg}")


def _cfg_ops(ops, out, lat):
    """The caller-side guidance / scheduler updates on the run's own noise predictions."""
    u, t = out[0:1].contiguous(), out[1:2].contiguous()
    ops.cfg_ddim_step(u, t, 7.5, 0.2, 0.35, lat)
    ops.cfg_linear_step(u, t, 7.5, 0.9, -0.3, lat, noise=t * 0.5 + 0.1, c_noise=0.05)
    ops.cfg_combine(t, u, 7.5)


@pytest.fixture(scope="module")
def base_unet(synthetic_sd):
    return _synthetic_base(synthetic_sd)


@pytest.mark.gpu
def test_audit_base_headline(base_unet, audit_log, reference_selfcheck):
    """BASELINE config 1/2: batch 2 x [4, 16, 40, 64], 77 tokens (every launch of one base step)."""
    from lavie_b200 import ops
    from lavie_b200.synthetic import synthetic_inputs
    sample, t, text = synthetic_inputs(2, 16, 40, 64, seed=0)
    with audit_log.record("base headline"):
        out = base_unet(sample.cuda(), t, encoder_hidden_states=text.cuda()).sample
        _cfg_ops(ops, out, out[0:1].contiguous() * 0.5)
    _finish(audit_log)


@pytest.mark.gpu
def test_audit_base_ragged(base_unet, audit_log, reference_selfcheck):
    """3 items x 5 frames x 24x40, 33 tokens: M / N tails, partial key tiles, F < 16 in the temporal kernel."""
    from lavie_b200.synthetic import synthetic_inputs
    sample, t, text = synthetic_inputs(3, 5, 24, 40, seed=11, text_len=33)
    with audit_log.record("base ragged"):
        base_unet(sample.cuda(), t, encoder_hidden_states=text.cuda())
    _finish(audit_log)


@pytest.mark.gpu
def test_audit_interpolation_61_frames(audit_log, reference_selfcheck):
    from lavie_b200.config import INTERP_CONFIG
    from lavie_b200.synthetic import synthetic_state_dict
    m = _synthetic_base(synthetic_state_dict(INTERP_CONFIG, seed=0), INTERP_CONFIG)
    g = torch.Generator().manual_seed(61)
    sample = torch.randn(1, 8, 61, 8, 16, generator=g)
    text = torch.randn(1, 77, 768, generator=g)
    with audit_log.record("interpolation 61f"):
        m(sample.cuda(), 321, encoder_hidden_states=text.cuda())
    _finish(audit_log)


@pytest.fixture(scope="module")
def vsr_unet():
    from lavie_b200.config import VSR_CONFIG
    from lavie_b200.synthetic import synthetic_state_dict
    from lavie_b200.vsr import UNet3DVSRModel
    m = UNet3DVSRModel(use_cuda_graph=False)
    m.load_state_dict(synthetic_state_dict(VSR_CONFIG, seed=0), strict=True)
    return m.to("cuda").eval()


def _vsr_run(m, log, name, B, Fr, H, W, L, seed):
    g = torch.Generator().manual_seed(seed)
    sample, low = torch.randn(B, 4, Fr, H, W, generator=g), torch.randn(B, 3, Fr, H, W, generator=g)
    text = torch.randn(B, L, 1024, generator=g)
    with log.record(name):
        m(sample.cuda(), 321, low.cuda(), encoder_hidden_states=text.cuda(), class_labels=torch.tensor([20] * B))
    _finish(log)


@pytest.mark.gpu
def test_audit_vsr_16_frames(vsr_unet, audit_log, reference_selfcheck):
    _vsr_run(vsr_unet, audit_log, "vsr 16f", 2, 16, 32, 32, 77, 11)


@pytest.mark.gpu
def test_audit_vsr_ragged(vsr_unet, audit_log, reference_selfcheck):
    _vsr_run(vsr_unet, audit_log, "vsr ragged", 1, 3, 24, 8, 20, 5)


@pytest.mark.gpu
@pytest.mark.skipif(os.environ.get("LAVIE_AUDIT_FULL") != "1", reason="full-geometry VSR audit: set LAVIE_AUDIT_FULL=1")
def test_audit_vsr_bench_chunk(vsr_unet, audit_log, reference_selfcheck):
    """bench.py's VSR workload as the reference runs it: one 8-frame chunk of a 320x512 latent (1280x2048 output frames),
    CFG batch 2, 77 tokens.  Gated: several minutes of fp64 references."""
    _vsr_run(vsr_unet, audit_log, "vsr bench chunk", 2, 8, 320, 512, 77, 7)
    print("\nper-launch audit (" + ", ".join(audit_log.runs) + ")\n" + audit_log.summary())


@pytest.mark.gpu
def test_audit_clip(audit_log, reference_selfcheck):
    from lavie_b200.clip import CLIPTextConfig, CLIPTextEncoder, clip_synthetic_state_dict
    cfg = CLIPTextConfig()
    enc = CLIPTextEncoder(cfg)
    enc.load_state_dict(clip_synthetic_state_dict(cfg, seed=0), strict=True)
    enc = enc.to("cuda").eval()
    ids = torch.randint(0, cfg.vocab_size, (2, 77), generator=torch.Generator().manual_seed(0))
    with audit_log.record("clip"):
        enc(ids.cuda())
    _finish(audit_log)


@pytest.fixture(scope="module")
def vae():
    from lavie_b200.vae import VAEDecoder, vae_synthetic_state_dict
    m = VAEDecoder()
    m.load_state_dict(vae_synthetic_state_dict(seed=0), strict=True)
    return m.to("cuda").eval()


@pytest.mark.gpu
def test_audit_vae_production_latent(vae, audit_log, reference_selfcheck):
    z = torch.randn(1, 4, 40, 64, generator=torch.Generator().manual_seed(40))
    with audit_log.record("vae 40x64"):
        vae.decode(z.cuda(), scale=1 / 0.18215)
    _finish(audit_log)


@pytest.mark.gpu
def test_audit_vae_ragged_uint8(vae, audit_log, reference_selfcheck):
    """3 frames of a 12x20 latent (the upsample falls back to nearest x2 + conv at 24x40) through decode_latents."""
    lat = 0.18215 * torch.randn(1, 4, 3, 12, 20, generator=torch.Generator().manual_seed(12))
    with audit_log.record("vae ragged"):
        vae.decode_latents(lat.cuda())
    _finish(audit_log)


@pytest.mark.gpu
def test_coverage_ledger_and_summary(audit_log):
    """Every launching function of ops was audited by the runs above or is named with the test that covers it; prints
    the per-op summary (run with -s)."""
    missing_runs = [r for r in RUNS_DEFAULT if r not in audit_log.runs]
    if missing_runs:
        pytest.skip(f"the ledger needs every default audit run; not run: {missing_runs}")
    print("\nper-launch audit (" + ", ".join(audit_log.runs) + ")\n" + audit_log.summary())
    names = launching_functions()
    audited = {n for n, r in audit_log.rows.items() if r.launches}
    unclassified = sorted(n for n in names if n not in audited and n not in COVERED_ELSEWHERE)
    assert not unclassified, f"ops functions neither audited nor covered by a named test: {unclassified}"
    plans = set().union(*(audit_log.rows[n].plans for n in ("gemm", "conv3x3", "frame_conv")))
    assert "full-width" in plans and "main+tail window" in plans and any(p.startswith("split-K") for p in plans), plans
    for n in ("attention", "frame_attention", "temporal_attention"):
        assert audit_log.rows[n].probes > 0, n


# ------------------------------------------------------------------------------------------------ CPU: the ledger's list
def test_ledger_classifies_every_launching_function():
    names = launching_functions()
    assert {"gemm", "conv3x3", "attention", "pointwise_conv_nchw", "conv_in_tc", "groupnorm"} <= names
    unknown = sorted(n for n in names if n not in CHECKERS and n not in COVERED_ELSEWHERE)
    assert not unknown, f"new ops functions without a reference or a named covering test: {unknown}"


def _fma32(a, b, c):
    """fmaf on float32 arrays: a * b is exact in fp64, a * b + c is formed exactly as a two-term sum (TwoSum) and rounded
    once to fp32 (the fp64 sum is corrected when it sits exactly on an fp32 rounding tie)."""
    import numpy as np
    p = a.astype(np.float64) * b.astype(np.float64)
    c = c.astype(np.float64)
    s = p + c
    bb = s - p
    e = (p - (s - bb)) + (c - bb)                       # s + e == p + c exactly
    r = s.astype(np.float32)
    up = np.nextafter(r, np.float32(np.inf))
    dn = np.nextafter(r, np.float32(-np.inf))
    # a tie: s exactly halfway between r and a neighbour; the residual e decides the side
    tie_up = (s - r.astype(np.float64) == (up.astype(np.float64) - r.astype(np.float64)) / 2) & (e > 0)
    tie_dn = (r.astype(np.float64) - s == (r.astype(np.float64) - dn.astype(np.float64)) / 2) & (e < 0)
    return np.where(tie_up, up, np.where(tie_dn, dn, r))


def test_gelu_fast_error_bound():
    """E_GELU covers gelu_fast_f (lavie_b200/csrc/common.cuh) emulated step by step in fp32: the Horner chain of fmaf
    with the fp32 coefficients, ex2.approx (2^-22 relative on e, times t e <= 0.17), the final fmaf."""
    import numpy as np
    from scipy.special import erf
    f32 = np.float32
    c = [f32(0.0005355844041332603), f32(-0.007474260404706001), f32(0.052688680589199066), f32(0.4591757357120514),
         f32(1.1511057615280151), f32(1.0)]
    x = np.linspace(-30, 30, 1200001).astype(f32)
    t = np.abs(x)
    full = np.full_like

    q = _fma32(t, full(t, c[0]), full(t, c[1]))
    for k in c[2:]:
        q = _fma32(q, t, full(t, k))
    e = np.exp2(-q.astype(np.float64)).astype(f32)
    fast = _fma32(-t, e, np.maximum(x, f32(0))).astype(np.float64)
    ref = 0.5 * x.astype(np.float64) * (1 + erf(x.astype(np.float64) / np.sqrt(2)))
    assert np.abs(fast - ref).max() + 0.17 * 2.0 ** -22 <= E_GELU


def test_fma32_rounds_once():
    import numpy as np
    one, eps = np.float32(1), np.float32(2.0 ** -23)
    # (1 + 2^-23)(1 - 2^-23) + (-1) = -2^-46 exactly; rounding the product first would give 0
    got = _fma32(np.array([one + eps]), np.array([one - eps]), np.array([-one]))
    assert got[0] == np.float32(-(2.0 ** -46))


# ------------------------------------------------------------------------------------------------ CPU: sharpness
def _bf16_result(ref):
    return ref.to(torch.float32).to(BF16)


def _gemm_case(M=100, N=96, K=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(M, K, generator=g).to(BF16)
    w = (torch.randn(N, K, generator=g) * K ** -0.5).to(BF16)
    acc, _ = mm_abs(a, w)
    return a, w, acc


def _gemm_cmp(out, a, w):
    return gemm_check(out, lambda lo, hi: a[lo:hi].to(F64), w, w.shape[1], {}, step=32)


def _four_ulps(out, r, c):
    bad = out.clone()
    v = bad[r, c].float()
    ulp = 2.0 ** (math.floor(math.log2(abs(float(v)))) - 7)
    bad[r, c] = (v + 4 * ulp * (1 if v > 0 else -1)).to(BF16)
    return bad


@pytest.mark.parametrize("K", [64, 11520])
def test_gemm_comparator_flags_defects(K):
    """K = 11520 is the largest K the models issue (3x3 conv over 1280 channels): there the accumulation term c S of the
    bound is larger than U |ref|, and a 4-ulp error must still stand out."""
    a, w, acc = _gemm_case(K=K)
    out = _bf16_result(acc)
    assert _gemm_cmp(out, a, w).ok
    # one element off by 4 bf16 ulps (at the largest output of row 40, past the first comparison block)
    r = 40
    c = int(acc[r].abs().argmax())
    cmp = _gemm_cmp(_four_ulps(out, r, c), a, w)
    assert not cmp.ok and cmp.n_over == 1 and cmp.worst_at == (r, c)
    # the last row of a partial 32-row slab (M = 100: rows 96..99) zeroed
    bad = out.clone()
    bad[99] = 0
    assert not _gemm_cmp(bad, a, w).ok
    # the N-tail column block (columns 64..95 of N = 96) shifted by one column
    bad = out.clone()
    bad[:, 65:96] = out[:, 64:95]
    assert _gemm_cmp(bad, a, w).n_over > 100
    # a sign flip of one element
    bad = out.clone()
    bad[3, 7] = -bad[3, 7]
    assert not _gemm_cmp(bad, a, w).ok


def test_geglu_comparator_flags_defects():
    a, w, acc = _gemm_case(M=64, N=512, K=64, seed=1)
    ref, extra = geglu_ref(acc, mm_abs(a, w)[1], c_gemm(64) * (1 + U))
    out = _bf16_result(ref)
    chk = lambda o: gemm_check(o, lambda lo, hi: a[lo:hi].to(F64), w, 64, {"geglu": True})   # noqa: E731
    assert chk(out).ok
    # value and gate columns paired with the wrong tile half (columns j and j + 128 swapped)
    h = acc.reshape(64, 2, 2, 128)
    swapped = (h[:, :, 1] * gelu64(h[:, :, 0])).reshape(64, 256)
    assert not chk(_bf16_result(swapped)).ok


def _fake_attention(defect=None):
    """A CPU stand-in for ops.attention with the same signature: an honest kernel's bf16 output (fp64 softmax, P V), or
    one that counts an extra zero-score zero-value key, or drops the last key."""
    def run(q, k, v, batch, heads, Sq, Sk, d, pitch, kv_batch_div=1, scale=None, out=None, sparse_causal_frames=0,
            sc_halo=0):
        a = {"q": q, "k": k, "v": v, "batch": batch, "heads": heads, "Sq": Sq, "Sk": Sk, "d": d, "head_pitch": pitch,
             "kv_batch_div": kv_batch_div, "sparse_causal_frames": sparse_causal_frames, "sc_halo": sc_halo}
        qrows, krows = attention_layout(a)
        Q, K, V = (heads_of(t, r, heads, pitch, d).to(F64) for t, r in ((q, qrows), (k, krows), (v, krows)))
        if defect == "extra":
            z = torch.zeros_like(K[:, :, :1])
            K, V = torch.cat([K, z], 2), torch.cat([V, z], 2)
        elif defect == "drop":
            K, V = K[:, :, :-1], V[:, :, :-1]
        p = torch.softmax((scale or d ** -0.5) * Q @ K.transpose(-1, -2), -1)
        return _bf16_result(_attn_out(p @ V, batch, heads, Sq, d))
    return run


def _attn_args(batch=4, heads=2, Sq=9, Sk=20, d=16, pitch=16, div=2, seed=0):
    g = torch.Generator().manual_seed(seed)
    q = torch.randn(batch * Sq, heads * pitch, generator=g).to(BF16)
    k, v = (torch.randn(batch // div * Sk, heads * pitch, generator=g).to(BF16) for _ in range(2))
    return {"q": q, "k": k, "v": v, "batch": batch, "heads": heads, "Sq": Sq, "Sk": Sk, "d": d, "head_pitch": pitch,
            "kv_batch_div": div, "sparse_causal_frames": 0, "sc_halo": 0, "scale": None}


def test_attention_probes_flag_key_mask_defects():
    """The recorder's own probe launches (attention_probes), run against CPU stand-ins of the kernel."""
    a = _attn_args()
    assert all(c.ok for c in attention_probes("attention", _fake_attention(), a))
    o, bnd = attention_ref(a)
    out = _fake_attention()(a["q"], a["k"], a["v"], 4, 2, 9, 20, 16, 16, 2)
    assert Cmp("attn", out, _attn_out(o, 4, 2, 9, 16), _attn_out(bnd, 4, 2, 9, 16)).ok
    ones, ramp = attention_probes("attention", _fake_attention("extra"), a)
    assert not ones.ok                      # one extra zero-score, zero-value key
    ones, ramp = attention_probes("attention", _fake_attention("drop"), a)
    assert not (ones.ok and ramp.ok)        # the last key dropped


def test_key_ramp_tells_adjacent_keys_apart_at_long_sequences():
    """At 2560 keys per sequence (the base model's level-0 self-attention) neighbouring keys still get distinct bf16
    probe values in the position-mod-64 column, and the sequence column tells two key segments apart."""
    v = ramp_values(2 * 2560, 2560, 1).to(torch.float32).to(BF16).to(F64)
    assert bool((v[1:2560, 1] != v[:2559, 1]).all())
    assert float(v[2560, 2] - v[0, 2]) == 1 / 64


def test_sparse_causal_comparator_flags_wrong_key_segment():
    """Frame 3 of a 5-frame video reading frame 1 instead of frame 2 as its former frame."""
    batch, S, heads, pitch, d = 5, 12, 2, 16, 16
    g = torch.Generator().manual_seed(3)
    q, k, v = (torch.randn(batch * S, heads * pitch, generator=g).to(BF16) for _ in range(3))
    a = {"q": q, "k": k, "v": v, "batch": batch, "heads": heads, "Sq": S, "Sk": S, "d": d, "head_pitch": pitch,
         "kv_batch_div": 1, "sparse_causal_frames": batch, "sc_halo": 0, "scale": None}
    o, bnd = attention_ref(a)
    ref, bnd = _attn_out(o, batch, heads, S, d), _attn_out(bnd, batch, heads, S, d)
    assert Cmp("sc", _bf16_result(ref), ref, bnd).ok
    qrows, krows = attention_layout(a)
    assert krows[3, S:].tolist() == list(range(2 * S, 3 * S))         # frame 3: [frame 0 | frame 2]
    wrong = krows.clone()
    wrong[3, S:] -= S
    Q = heads_of(q, qrows, heads, pitch, d)
    o2, _ = attention_core(Q, heads_of(k, wrong, heads, pitch, d), heads_of(v, wrong, heads, pitch, d), d ** -0.5)
    cmp = Cmp("sc", _bf16_result(_attn_out(o2, batch, heads, S, d)), ref, bnd)
    assert not cmp.ok and all(3 * S <= r < 4 * S for r in [cmp.worst_at[0]])


def test_groupnorm_comparator_flags_count_off_by_one():
    g = torch.Generator().manual_seed(4)
    samples, rps, C = 2, 64, 320
    x = (torch.randn(samples * rps, C, generator=g) * 2 + 0.5).to(BF16)
    gamma, beta = torch.randn(C, generator=g) * 0.1 + 1, torch.randn(C, generator=g) * 0.1
    scale, shift, bs, bsh = gn_scale_shift64(x, samples, gamma, beta, 1e-5)
    assert Cmp("s", scale.float(), scale, bs).ok and Cmp("sh", shift.float(), shift, bsh).ok
    # statistics with the element count off by one (sum / (n + 1))
    v = x.to(F64).reshape(samples, rps, 32, C // 32)
    n = rps * C // 32
    mean = v.sum((1, 3)) / (n + 1)
    var = (v * v).sum((1, 3)) / (n + 1) - mean * mean
    rstd = (1 / torch.sqrt(var + 1e-5)).repeat_interleave(C // 32, 1)
    s_bad = rstd * gamma.to(F64)
    sh_bad = beta.to(F64) - mean.repeat_interleave(C // 32, 1) * s_bad
    assert not Cmp("s", s_bad, scale, bs).ok and not Cmp("sh", sh_bad, shift, bsh).ok
    # the normalised output of the apply pass on those statistics
    y, mag, t = apply_ref(x, scale, shift, samples, True)
    yb, _, _ = apply_ref(x, s_bad, sh_bad, samples, True)
    bound = U * y.abs() + 2.0 ** -20 * (SILU_SLOPE * mag + t.abs())
    assert Cmp("apply", _bf16_result(y), y, bound).ok
    assert not Cmp("apply", _bf16_result(yb), y, bound).ok


def test_layernorm_comparator_flags_defects():
    g = torch.Generator().manual_seed(5)
    x = (torch.randn(50, 320, generator=g) * 3 + 1).to(BF16)
    gamma, beta = torch.randn(320, generator=g) * 0.1 + 1, torch.randn(320, generator=g) * 0.1
    y, small = layernorm_ref(x, gamma, beta, 1e-5)
    assert Cmp("ln", _bf16_result(y), y, U * y.abs() + small).ok
    yb, _ = layernorm_ref(x[:, :319], gamma[:319], beta[:319], 1e-5)       # statistics over one channel less
    bad = y.clone()
    bad[:, :319] = yb
    assert not Cmp("ln", _bf16_result(bad), y, U * y.abs() + small).ok


def test_colsum_comparator_flags_missing_slab():
    for N in (320, 256):                    # decades and octets
        g = torch.Generator().manual_seed(N)
        out = torch.randn(100, N, generator=g).to(BF16)
        exp, _, written = colsum_expected(out)
        cs = exp.float().clone()
        cs[:, ~written] = float("nan")     # unwritten pieces are never read
        assert check_colsums(cs, out).ok
        bad = cs.clone()
        bad[2] = 0                          # one slab of column sums missing
        assert not check_colsums(bad, out).ok
    # 4 phase segments of an upsample output (NF = 2, 4x8 source: 32 rows per segment slab)
    out = torch.randn(2 * 4 * 4 * 8, 320, generator=g).to(BF16)
    exp, _, _ = colsum_expected(out, 4, (2, 4, 8))
    assert check_colsums(exp.float(), out, 4, (2, 4, 8)).ok
    flat, _, _ = colsum_expected(out)                                      # slabs in plain row order: wrong layout
    assert not check_colsums(flat.float(), out, 4, (2, 4, 8)).ok


def test_view_check_flags_one_element_outside():
    buf = torch.randn(10, 64).to(BF16)
    view = buf[2:8, 16:48]
    before = buf.clone()
    view.fill_(1.0)
    assert check_outside_view(before, buf, view_mask(buf, view)).ok
    buf[8, 16] = 5.0                        # one element just past the view's last row
    f = check_outside_view(before, buf, view_mask(buf, view))
    assert not f.ok and "(8, 16)" in f.detail
    buf3 = torch.zeros(2, 7 * 4, 8).to(BF16)                              # VSR frame-padded buffer [B, (F+2)*HW, C]
    before = buf3.clone()
    buf3[1, 4:24] = 1.0
    assert check_outside_view(before, buf3, view_mask(buf3, buf3[1, 4:24])).ok
    buf3[1, 24] = 1.0                       # the first trailing pad frame written
    assert not check_outside_view(before, buf3, view_mask(buf3, buf3[1, 4:24])).ok


def test_upsample_phase_reference_is_nearest_upsample_then_conv():
    """The phase reference (from the packed phase weights) equals nearest x2 + the 3x3 conv it was packed from."""
    from lavie_b200.packing import pack_upsample_conv3x3
    g = torch.Generator().manual_seed(6)
    NF, H, W, C, N = 2, 3, 5, 8, 6
    x = torch.randn(NF * H * W, C, generator=g).to(BF16)
    w = torch.randn(N, C, 3, 3, generator=g, dtype=F64)
    got, _ = upsample_phase_ref(x, NF, H, W, pack_upsample_conv3x3(w, dtype=None))
    up = F.interpolate(x.to(F64).reshape(NF, H, W, C).permute(0, 3, 1, 2), scale_factor=2, mode="nearest")
    ref = F.conv2d(up, w, padding=1).permute(0, 2, 3, 1).reshape(-1, N)
    assert rel_l2(got, ref) < 1e-6                 # the packed phase taps are summed in fp32
