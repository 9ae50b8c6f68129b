"""Per-kernel numerics on the B200: every C-ABI entry point against a plain PyTorch fp32 reference of the same
op, on bf16-rounded inputs.  Tolerances are stated per test (bf16 output rounding = 2^-9 relative)."""
import math

import pytest
import torch
import torch.nn.functional as F

from conftest import rel_l2

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(autouse=True, scope="module")
def _exact_fp32_references():
    """The fp32 references (F.conv2d, matmul) run on the GPU: keep TF32 off for cuDNN and cuBLAS, else a reference
    carries ~bf16-sized error of its own."""
    saved = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved


def _ops():
    from lavie_b200 import ops
    return ops


def _bf(t):
    return t.to(torch.bfloat16)


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed + sum(shape))
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


# ------------------------------------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("block_n", [0, 64, 128, 160, 192, 256, 320])
@pytest.mark.parametrize("M,N,K", [(256, 256, 64), (1000, 320, 320), (4096, 1152, 320), (300, 640, 2560)])
def test_gemm_plain(M, N, K, block_n):
    ops = _ops()
    a = _bf(_rand(M, K))
    w = _bf(_rand(N, K, scale=K ** -0.5))
    out = ops.gemm(a, w, block_n=block_n)
    ref = a.float() @ w.float().t()
    assert rel_l2(out.float(), ref) < 4e-3          # bf16 output rounding only


def test_gemm_epilogue_bias_rowbias_residual_strided():
    ops = _ops()
    M, N, K, B = 768, 320, 640, 3
    a = _bf(_rand(M, K))
    w = _bf(_rand(N, K, scale=K ** -0.5))
    bias = _rand(N, seed=1)
    rb = _rand(B, N, seed=2)
    res_full = _bf(_rand(M, N + 64, seed=3))
    res = res_full[:, 64:]                            # strided residual view
    out_full = torch.zeros((M, 2 * N), dtype=torch.bfloat16, device=DEV)
    out = out_full[:, N:]                             # strided output view (writes into a wider buffer)
    ops.gemm(a, w, bias=bias, row_bias=rb, rows_per_batch=M // B, residual=res, out=out)
    ref = a.float() @ w.float().t() + bias + rb.repeat_interleave(M // B, 0) + res.float()
    assert rel_l2(out.float(), ref) < 4e-3
    assert out_full[:, :N].abs().max() == 0           # nothing written outside the view


@pytest.mark.parametrize("N", [320, 640, 200])
def test_gemm_wide_tile_epilogue(N):
    """BLOCK_N = 320: two 160-wide MMAs per K step share the activation stage, single accumulator stage, five
    staging chunks per epilogue warp; several tiles per CTA pair so the accumulator hand-back is exercised."""
    ops = _ops()
    M, K = 256 * 150 + 77, 192
    a = _bf(_rand(M, K))
    w = _bf(_rand(N, K, scale=K ** -0.5))
    bias = _rand(N, seed=1)
    res = _bf(_rand(M, N, seed=3))
    out = ops.gemm(a, w, bias=bias, residual=res, block_n=320)
    ref = a.float() @ w.float().t() + bias + res.float()
    assert rel_l2(out.float(), ref) < 4e-3


def test_gemm_main_plus_splitk_tail_window():
    """More than one wave of tiles with a nearly empty last wave: the planner issues full waves over the leading tile
    rows and a split-K launch over the rest.  Same epilogue on both paths; compare with the single-launch result."""
    ops = _ops()
    from lavie_b200 import _lib
    lib = _lib.load()
    M, N, K, B = 256 * 39 + 100, 640, 2048, 2
    a = _bf(_rand(M, K))
    w = _bf(_rand(N, K, scale=K ** -0.5))
    bias = _rand(N, seed=1)
    rb = _rand(B, N, seed=2)
    res = _bf(_rand(M, N, seed=3))
    rpb = (M + B - 1) // B
    out = ops.gemm(a, w, bias=bias, row_bias=rb, rows_per_batch=rpb, residual=res)
    lib.lavie_debug_set(5, 1)
    try:
        single = ops.gemm(a, w, bias=bias, row_bias=rb, rows_per_batch=rpb, residual=res)
    finally:
        lib.lavie_debug_set(5, 0)
    ref = a.float() @ w.float().t() + bias + rb.repeat_interleave(rpb, 0)[:M] + res.float()
    assert rel_l2(out.float(), ref) < 4e-3
    assert rel_l2(out.float(), single.float()) < 3e-3     # split-K changes the summation order of the tail rows only
    assert torch.equal(out[: 256 * 30], single[: 256 * 30])


def test_conv3x3_main_plus_tail_window():
    ops = _ops()
    from lavie_b200.packing import pack_conv3x3
    NF, H, W, C, N = 32, 10, 16, 128, 1280
    x = _bf(_rand(NF * H * W, C))
    w = _bf(_rand(N, C, 3, 3, scale=(9 * C) ** -0.5))
    res = _bf(_rand(NF * H * W, N, seed=5))
    out = ops.conv3x3(x, NF, H, W, pack_conv3x3(w), residual=res)
    assert rel_l2(out.float(), _conv_ref(x, w, NF, H, W) + res.float()) < 4e-3


def test_conv3x3_wide_tile():
    ops = _ops()
    from lavie_b200.packing import pack_conv3x3
    NF, H, W, C, N = 3, 20, 32, 128, 640
    x = _bf(_rand(NF * H * W, C))
    w = _bf(_rand(N, C, 3, 3, scale=(9 * C) ** -0.5))
    out = ops.conv3x3(x, NF, H, W, pack_conv3x3(w), block_n=320)
    assert rel_l2(out.float(), _conv_ref(x, w, NF, H, W)) < 4e-3


def test_gemm_two_sources_fold_concat():
    ops = _ops()
    M, N, k0, k1 = 640, 320, 640, 320
    a0 = _bf(_rand(M, k0))
    a1 = _bf(_rand(M, k1, seed=5))
    w = _bf(_rand(N, k0 + k1, scale=(k0 + k1) ** -0.5))
    out = ops.gemm(a0, w, a2=a1)
    ref = torch.cat([a0, a1], 1).float() @ w.float().t()
    assert rel_l2(out.float(), ref) < 4e-3


def test_gemm_geglu():
    ops = _ops()
    M, C = 512, 320
    a = _bf(_rand(M, C))
    w = _bf(_rand(8 * C, C, scale=C ** -0.5))          # reference layout: rows [0,4C) value, [4C,8C) gate
    b = _rand(8 * C, seed=7)
    from lavie_b200.packing import interleave_geglu
    wi, bi = interleave_geglu(w, b)
    out = ops.gemm(a, wi, bias=bi, geglu=True)
    hg = a.float() @ w.float().t() + b
    ref = hg[:, : 4 * C] * F.gelu(hg[:, 4 * C:])
    assert out.shape == (M, 4 * C)
    assert rel_l2(out.float(), ref) < 5e-3


# ------------------------------------------------------------------------------------------------ conv
def _conv_ref(x_nhwc, w_oihw, NF, H, W, stride=1):
    x = x_nhwc.float().reshape(NF, H, W, -1).permute(0, 3, 1, 2)
    y = F.conv2d(x, w_oihw.float(), None, stride=stride, padding=1)
    return y.permute(0, 2, 3, 1).reshape(-1, w_oihw.shape[0])


@pytest.mark.parametrize("NF,H,W,C,N", [(4, 8, 64, 64, 64), (3, 20, 32, 128, 320), (5, 10, 16, 320, 128),
                                        (7, 5, 8, 64, 64), (2, 40, 64, 320, 320), (3, 12, 24, 64, 64),
                                        (2, 5, 7, 64, 64), (3, 3, 3, 128, 64), (1, 1, 1, 64, 64)])
def test_conv3x3_tma(NF, H, W, C, N):
    ops = _ops()
    from lavie_b200.packing import pack_conv3x3
    x = _bf(_rand(NF * H * W, C))
    w = _bf(_rand(N, C, 3, 3, scale=(9 * C) ** -0.5))
    assert ops.conv3x3_supported(H, W, C)
    out = ops.conv3x3(x, NF, H, W, pack_conv3x3(w))
    ref = _conv_ref(x, w, NF, H, W)
    assert rel_l2(out.float(), ref) < 4e-3


def test_conv3x3_epilogue_time_bias_and_shortcut():
    ops = _ops()
    from lavie_b200.packing import pack_conv3x3
    B, Fr, H, W, C, N = 2, 3, 10, 16, 64, 128
    NF = B * Fr
    x = _bf(_rand(NF * H * W, C))
    w = _bf(_rand(N, C, 3, 3, scale=(9 * C) ** -0.5))
    bias = _rand(N, seed=3)
    temb = _rand(B, N, seed=4)
    res = _bf(_rand(NF * H * W, N, seed=5))
    out = ops.conv3x3(x, NF, H, W, pack_conv3x3(w), bias=bias, row_bias=temb, rows_per_batch=Fr * H * W, residual=res)
    ref = _conv_ref(x, w, NF, H, W) + bias + temb.repeat_interleave(Fr * H * W, 0) + res.float()
    assert rel_l2(out.float(), ref) < 4e-3


@pytest.mark.parametrize("stride", [1, 2])
@pytest.mark.parametrize("explicit", [False, True])
@pytest.mark.parametrize("NF,H,W,C,N", [(3, 12, 24, 64, 64), (2, 40, 64, 320, 320), (2, 5, 7, 128, 64)])
def test_conv3x3_stride_and_explicit_im2col(NF, H, W, C, N, stride, explicit):
    """stride-2 Downsample3D through im2col-mode TMA, and the explicit patch-matrix path (kept for C % 64 != 0)."""
    ops = _ops()
    from lavie_b200.packing import pack_conv3x3
    x = _bf(_rand(NF * H * W, C))
    w = _bf(_rand(N, C, 3, 3, scale=(9 * C) ** -0.5))
    bias = _rand(N, seed=2)
    out = ops.conv3x3(x, NF, H, W, pack_conv3x3(w), stride=stride, bias=bias, force_im2col=explicit)
    ref = _conv_ref(x, w, NF, H, W, stride) + bias
    assert out.shape == ref.shape
    assert rel_l2(out.float(), ref) < 4e-3


# ------------------------------------------------------------------------------------------------ norms
@pytest.mark.parametrize("C0,C1", [(320, 0), (640, 320), (1280, 1280), (64, 0)])
@pytest.mark.parametrize("per_frame", [False, True])
def test_groupnorm(C0, C1, per_frame):
    ops = _ops()
    B, Fr, HW = 2, 3, 200
    rows = B * Fr * HW
    x0 = _bf(_rand(rows, C0) * 2 + 0.5)
    x1 = _bf(_rand(rows, C1, seed=9) - 1.0) if C1 else None
    C = C0 + C1
    gamma = _rand(C, seed=1) * 0.1 + 1
    beta = _rand(C, seed=2) * 0.1
    samples, rps = (B * Fr, HW) if per_frame else (B, Fr * HW)
    out = ops.groupnorm(x0, samples, rps, gamma, beta, 1e-5, silu=True, x2=x1)
    xc = torch.cat([x0, x1], 1) if C1 else x0
    ref = F.group_norm(xc.float().reshape(samples, rps, C).permute(0, 2, 1), 32, gamma, beta, 1e-5)
    ref = F.silu(ref).permute(0, 2, 1).reshape(rows, C)
    assert rel_l2(out.float(), ref) < 4e-3


@pytest.mark.parametrize("C", [320, 640, 1280])
def test_layernorm(C):
    ops = _ops()
    rows = 1003
    x = _bf(_rand(rows, C) * 3 + 1)
    g = _rand(C, seed=1) * 0.1 + 1
    b = _rand(C, seed=2) * 0.1
    out = ops.layernorm(x, g, b, 1e-5)
    ref = F.layer_norm(x.float(), (C,), g, b, 1e-5)
    assert rel_l2(out.float(), ref) < 4e-3


# ------------------------------------------------------------------------------------------------ attention
def _attn_ref(q, k, v, batch, heads, Sq, Sk, d, pitch, div):
    qh = q.float().reshape(batch, Sq, heads, pitch)[..., :d].permute(0, 2, 1, 3)
    kh = k.float().reshape(batch // div, Sk, heads, pitch)[..., :d].permute(0, 2, 1, 3).repeat_interleave(div, 0)
    vh = v.float().reshape(batch // div, Sk, heads, pitch)[..., :d].permute(0, 2, 1, 3).repeat_interleave(div, 0)
    p = torch.softmax(qh @ kh.transpose(-1, -2) * d ** -0.5, -1)
    return (p @ vh).permute(0, 2, 1, 3).reshape(batch * Sq, heads * d)


def _padded(rows, heads, d, pitch, seed):
    t = torch.zeros(rows, heads, pitch, device=DEV)
    t[..., :d] = _rand(rows, heads, d, seed=seed)
    return _bf(t.reshape(rows, heads * pitch))


@pytest.mark.parametrize("batch,Sq,Sk,d,pitch,div", [
    (4, 256, 256, 40, 48, 1), (2, 640, 640, 80, 80, 1), (2, 160, 160, 160, 160, 1), (3, 40, 40, 160, 160, 1),
    (4, 200, 77, 40, 48, 2), (4, 160, 77, 80, 80, 2), (4, 40, 77, 160, 160, 4), (1, 2560, 2560, 40, 48, 1),
    (2, 64, 154, 40, 48, 1),
    # head dims of the VSR denoiser (512 / 8 and 1024 / 8 channels per head)
    (2, 320, 320, 64, 64, 1), (4, 256, 77, 64, 64, 2), (2, 200, 200, 128, 128, 1), (4, 96, 77, 128, 128, 4)])
def test_attention(batch, Sq, Sk, d, pitch, div):
    ops = _ops()
    heads = 8
    q = _padded(batch * Sq, heads, d, pitch, 1)
    k = _padded(batch // div * Sk, heads, d, pitch, 2)
    v = _padded(batch // div * Sk, heads, d, pitch, 3)
    out = ops.attention(q, k, v, batch, heads, Sq, Sk, d, pitch, div)
    ref = _attn_ref(q, k, v, batch, heads, Sq, Sk, d, pitch, div)
    assert rel_l2(out.float(), ref) < 1e-2          # P is rounded to bf16 before P V


@pytest.mark.parametrize("batch,Sq,Sk,d,pitch,div", [
    (4, 200, 77, 40, 48, 2), (32, 2560, 77, 40, 48, 16), (8, 640, 77, 80, 80, 4), (4, 37, 20, 160, 160, 4),
    (2, 16, 80, 64, 64, 1), (6, 100, 1, 128, 128, 3), (4, 5, 33, 96, 96, 2)])
def test_short_key_attention_single_pass_kernel(batch, Sq, Sk, d, pitch, div):
    """The optional single-pass mma.sync kernel for Sk <= 80 (lavie_debug_set(8, 1); off by default -- it is bound by the
    legacy HMMA rate and not faster): same results as the tcgen05 flash kernel and as the fp32 reference, incl. ragged
    query tiles, 1 key, every head dim."""
    ops = _ops()
    from lavie_b200 import _lib
    lib = _lib.load()
    heads = 8
    q = _padded(batch * Sq, heads, d, pitch, 1)
    k = _padded(batch // div * Sk, heads, d, pitch, 2)
    v = _padded(batch // div * Sk, heads, d, pitch, 3)
    old = ops.attention(q, k, v, batch, heads, Sq, Sk, d, pitch, div)          # default: the tcgen05 flash kernel
    ref = _attn_ref(q, k, v, batch, heads, Sq, Sk, d, pitch, div)
    lib.lavie_debug_set(8, 1)
    try:
        out = ops.attention(q, k, v, batch, heads, Sq, Sk, d, pitch, div)
        # strided views of a fused projection buffer (q | junk) and an output with a wider row stride
        wide = torch.zeros(batch * Sq, heads * pitch + 64, dtype=torch.bfloat16, device=DEV)
        wide[:, :heads * pitch] = q
        o_wide = torch.zeros(batch * Sq, heads * d + 32, dtype=torch.bfloat16, device=DEV)
        ops.attention(wide[:, :heads * pitch], k, v, batch, heads, Sq, Sk, d, pitch, div, out=o_wide[:, :heads * d])
    finally:
        lib.lavie_debug_set(8, 0)
    assert rel_l2(out.float(), ref) < 1e-2
    assert rel_l2(out.float(), old.float()) < 1e-2
    assert torch.equal(o_wide[:, :heads * d], out) and float(o_wide[:, heads * d:].abs().max()) == 0.0


def test_attention_fused_qkv_views():
    """q/k/v as column slices of one fused projection buffer (how the UNet calls it)."""
    ops = _ops()
    batch, S, heads, d, pitch = 2, 384, 8, 40, 48
    hp = heads * pitch
    parts = [_padded(batch * S, heads, d, pitch, s) for s in (1, 2, 3)]
    qkv = torch.cat(parts, 1).contiguous()
    out = ops.attention(qkv[:, :hp], qkv[:, hp:2 * hp], qkv[:, 2 * hp:], batch, heads, S, S, d, pitch)
    ref = _attn_ref(parts[0], parts[1], parts[2], batch, heads, S, S, d, pitch, 1)
    assert rel_l2(out.float(), ref) < 1e-2


@pytest.mark.parametrize("Fr,d,pitch", [(16, 40, 48), (16, 80, 80), (5, 160, 160), (16, 64, 64), (8, 128, 128)])
def test_temporal_attention(Fr, d, pitch):
    ops = _ops()
    from lavie_b200.packing import rope_table
    from oracle import unet3d_oracle as O
    B, HW, heads = 2, 37, 8
    rows = B * Fr * HW
    parts = [_padded(rows, heads, d, pitch, s) for s in (1, 2, 3)]
    qkv = torch.cat(parts, 1).contiguous()
    freqs = 1.0 / (10000.0 ** (torch.arange(0, 32, 2).float() / 32))
    table = torch.randn(32, heads, generator=torch.Generator().manual_seed(3))
    bias = O.rel_pos_bias(table, Fr).contiguous().to(DEV)
    out = ops.temporal_attention(qkv, B, Fr, HW, heads, d, pitch, rope_table(freqs, Fr).to(DEV), bias)

    def heads_of(t):   # [(b f hw), heads*pitch] -> [(b hw), heads, F, d]
        return t.float().reshape(B, Fr, HW, heads, pitch)[..., :d].permute(0, 2, 3, 1, 4).reshape(B * HW, heads, Fr, d)
    q, k, v = (heads_of(t).cpu() for t in parts)
    q = O.rope(q * d ** -0.5, freqs)
    k = O.rope(k, freqs)
    s = q @ k.transpose(-1, -2) + bias.cpu()
    o = torch.softmax(s, -1) @ v                                             # [(b hw), heads, F, d]
    ref = o.reshape(B, HW, heads, Fr, d).permute(0, 3, 1, 2, 4).reshape(rows, heads * d)
    assert rel_l2(out.float().cpu(), ref) < 4e-3


# ------------------------------------------------------------------------------------------------ small kernels
def test_time_embedding_path():
    ops = _ops()
    from oracle import unet3d_oracle as O
    t = torch.tensor([500.0, 981.0, 1.0], device=DEV)
    emb = ops.timestep_embedding(t, 320)
    assert torch.allclose(emb.cpu(), O.timestep_embedding(t.cpu(), 320), atol=2e-4)
    w = _bf(_rand(1280, 320, scale=320 ** -0.5))
    b = _rand(1280, seed=1)
    y = ops.linear_smallm(emb, w, b, silu_in=False, silu_out=True)
    ref = F.silu(emb @ w.float().t() + b)
    assert rel_l2(y, ref) < 1e-4
    y2 = ops.linear_smallm(y, _bf(_rand(640, 1280, scale=1280 ** -0.5)), None, silu_in=True)
    ref2 = F.silu(y) @ _bf(_rand(640, 1280, scale=1280 ** -0.5)).float().t()
    assert rel_l2(y2, ref2) < 1e-4


@pytest.mark.parametrize("rows,C,samples", [(2 * 40 * 64 * 4, 320, 2), (32 * 160, 1280, 32), (2 * 77, 64, 2)])
def test_groupnorm_fused_finalize_matches_two_launch(rows, C, samples):
    """The last-block-finalizes kernel must give the same bits as stats + finalize, call after call (tickets reset)."""
    ops = _ops()
    x = _bf(_rand(rows, C))
    gamma = _rand(C, seed=2) * 0.1 + 1
    beta = _rand(C, seed=3) * 0.1
    ref = ops.groupnorm_scale_shift(x, samples, rows // samples, gamma, beta, 1e-5, fused=False)
    for _ in range(3):
        got = ops.groupnorm_scale_shift(x, samples, rows // samples, gamma, beta, 1e-5)
        assert torch.equal(got, ref)



@pytest.mark.parametrize("H,W", [(10, 16), (5, 7), (3, 1), (40, 64)])
def test_conv_in_and_out(H, W):
    ops = _ops()
    B, Fr = 2, 3
    x = _rand(B, 4, Fr, H, W)
    w = _rand(320, 4, 3, 3, scale=1 / 6.0)
    b = _rand(320, seed=1)
    y = ops.conv_in(x, w, b)
    ref = F.conv2d(x.permute(0, 2, 1, 3, 4).reshape(B * Fr, 4, H, W), w, b, padding=1).permute(0, 2, 3, 1).reshape(-1, 320)
    assert rel_l2(y.float(), ref) < 4e-3
    # the tensor-core route of conv_in: explicit im2col of the 4 input channels + one GEMM (bf16 inputs and filters)
    y_tc = ops.conv_in_tc(x, ops.pack_conv_in(w, DEV), b)
    assert y_tc.shape == y.shape and rel_l2(y_tc.float(), ref) < 6e-3
    sc = torch.full((1,), 0.37, device=DEV)
    assert rel_l2(ops.conv_in_tc(x, ops.pack_conv_in(w, DEV), b, sc).float(),
                  F.conv2d(0.37 * x.permute(0, 2, 1, 3, 4).reshape(B * Fr, 4, H, W), w, b, padding=1).permute(0, 2, 3, 1)
                  .reshape(-1, 320)) < 6e-3
    x7, w7 = _rand(B, 7, Fr, H, W, seed=8), _rand(256, 7, 3, 3, seed=9, scale=1 / 8.0)      # the VSR model's 7 channels
    ref7 = F.conv2d(x7.permute(0, 2, 1, 3, 4).reshape(B * Fr, 7, H, W), w7, None, padding=1).permute(0, 2, 3, 1).reshape(-1, 256)
    assert rel_l2(ops.conv_in_tc(x7, ops.pack_conv_in(w7, DEV), torch.zeros(256, device=DEV)).float(), ref7) < 6e-3
    # conv_norm_out + SiLU + conv_out
    gamma = _rand(320, seed=2) * 0.1 + 1
    beta = _rand(320, seed=3) * 0.1
    ss = ops.groupnorm_scale_shift(y, B, Fr * H * W, gamma, beta, 1e-5)
    wo = _rand(4, 320, 3, 3, scale=(9 * 320) ** -0.5)
    bo = _rand(4, seed=4)
    out = ops.conv_out(y, ss, B, Fr, H, W, wo.permute(0, 2, 3, 1).contiguous(), bo)
    y5 = y.float().reshape(B, Fr, H, W, 320).permute(0, 4, 1, 2, 3)
    h = F.silu(F.group_norm(y5, 32, gamma, beta, 1e-5))
    ref = F.conv2d(h.permute(0, 2, 1, 3, 4).reshape(B * Fr, 320, H, W), wo, bo, padding=1)
    ref = ref.reshape(B, Fr, 4, H, W).permute(0, 2, 1, 3, 4)
    assert out.shape == (B, 4, Fr, H, W)
    assert rel_l2(out, ref) < 2e-3
    # the tensor-core route of the same op (GroupNorm apply + SiLU, implicit-GEMM conv against zero-padded filters, unpack
    # to [B, 4, F, H, W]): bf16 activations and bf16 output rows, hence the looser bound
    from lavie_b200.packing import pack_conv3x3
    wp = torch.zeros(ops.CONV_OUT_PAD, 9 * 320, device="cuda")
    wp[:4] = pack_conv3x3(wo, dtype=None)
    bp = torch.zeros(ops.CONV_OUT_PAD, device="cuda")
    bp[:4] = bo
    out_tc = ops.conv_out_tc(y, ss, B, Fr, H, W, wp.to(torch.bfloat16).contiguous(), bp, 4)
    assert out_tc.shape == (B, 4, Fr, H, W)
    assert rel_l2(out_tc, ref) < 8e-3


def test_upsample_and_cfg_ddim():
    ops = _ops()
    NF, H, W, C = 3, 5, 8, 64
    x = _bf(_rand(NF * H * W, C))
    y = ops.upsample_nearest2x(x, NF, H, W)
    ref = F.interpolate(x.float().reshape(NF, H, W, C).permute(0, 3, 1, 2), scale_factor=2, mode="nearest")
    assert torch.equal(y.float(), ref.permute(0, 2, 3, 1).reshape(-1, C))
    from oracle import unet3d_oracle as O
    acp, ts, ratio = O.ddim_schedule(50)
    lat, nu, nt = _rand(1, 4, 2, 8, 8), _rand(1, 4, 2, 8, 8, seed=1), _rand(1, 4, 2, 8, 8, seed=2)
    t = int(ts[7])
    got = ops.cfg_ddim_step(nu, nt, 7.5, float(acp[t]), float(acp[t - ratio]), lat)
    want = O.ddim_step((nu + 7.5 * (nt - nu)).cpu(), t, lat.cpu(), acp, ratio)
    assert torch.allclose(got.cpu(), want, atol=1e-5, rtol=1e-5)


# ------------------------------------------------------------------------------------------------ split-K
@pytest.mark.parametrize("splits", [0, 1, 2, 5])
def test_gemm_splitk_matches(splits):
    """Small-M / large-K problems (the 5x8 level: 1280 rows, K = 11520) take the deterministic split-K path."""
    ops = _ops()
    from lavie_b200 import _lib
    lib = _lib.load()
    M, N, K = 1280, 1280, 11520
    a = _bf(_rand(M, K))
    w = _bf(_rand(N, K, scale=K ** -0.5))
    bias = _rand(N, seed=1)
    res = _bf(_rand(M, N, seed=2))
    lib.lavie_debug_set(1, splits)
    try:
        out = ops.gemm(a, w, bias=bias, residual=res)
        out2 = ops.gemm(a, w, bias=bias, residual=res)
    finally:
        lib.lavie_debug_set(1, 0)
    ref = a.float() @ w.float().t() + bias + res.float()
    assert rel_l2(out.float(), ref) < 4e-3
    assert torch.equal(out, out2)                      # ordered reduction: bit-reproducible


def test_conv3x3_small_m_large_k():
    ops = _ops()
    from lavie_b200.packing import pack_conv3x3
    NF, H, W, C, N = 32, 5, 8, 1280, 1280
    x = _bf(_rand(NF * H * W, C))
    w = _bf(_rand(N, C, 3, 3, scale=(9 * C) ** -0.5))
    temb = _rand(2, N, seed=4)
    out = ops.conv3x3(x, NF, H, W, pack_conv3x3(w), row_bias=temb, rows_per_batch=16 * H * W)
    ref = _conv_ref(x, w, NF, H, W) + temb.repeat_interleave(16 * H * W, 0)
    assert rel_l2(out.float(), ref) < 4e-3


# ------------------------------------------------------------------------------------------------ GroupNorm statistics from the producer's epilogue
def _colsums_ref(out, M, N):
    """[ceil(M/32), N/10, 2] (sum, sumsq) of the bf16 output per 32-row slab and 10-channel micro-group."""
    slabs = (M + 31) // 32
    pad = torch.zeros(slabs * 32, N, device=out.device)
    pad[:M] = out.float()
    v = pad.reshape(slabs, 32, N // 10, 10)
    return torch.stack([v.sum((1, 3)), (v * v).sum((1, 3))], dim=-1)


def _micro(cs, N):
    """kernel layout [slabs, N/32, 4, 2] (chunk, decade piece) -> [slabs, N/10, 2]; unwritten pieces are ignored."""
    slabs = cs.shape[0]
    out = torch.zeros(slabs, N // 10, 2, device=cs.device)
    for k in range(N // 32):
        d0 = (k * 32) // 10
        for piece in range(4):
            dec = d0 + piece
            lo, hi = max(k * 32, dec * 10), min(k * 32 + 32, dec * 10 + 10, N)
            if lo < hi:
                out[:, dec] += cs[:, k, piece]
    return out


@pytest.mark.parametrize("M,N,K,block_n", [(2560, 320, 320, 0), (1000, 640, 1280, 0), (256 * 150 + 96, 320, 192, 320),
                                           (640, 1280, 2560, 0), (4096, 960, 320, 128)])
def test_gemm_emits_groupnorm_column_sums(M, N, K, block_n):
    """lavie_epilogue.col_stats: the producer's epilogue (or the split-K reduction) writes the consumer's GroupNorm
    statistics; they must equal the sums of the bf16 values actually stored (incl. bias + residual, M tails)."""
    ops = _ops()
    a = _bf(_rand(M, K))
    w = _bf(_rand(N, K, scale=K ** -0.5))
    bias = _rand(N, seed=1)
    res = _bf(_rand(M, N, seed=3))
    out = ops.gemm(a, w, bias=bias, residual=res, stats=True, block_n=block_n)
    plain = ops.gemm(a, w, bias=bias, residual=res, block_n=block_n)
    assert torch.equal(out, plain)                                   # the statistics do not change the output
    cs = _micro(out._gn_colsums, N)
    ref = _colsums_ref(out, M, N)
    assert cs.shape == ref.shape
    assert rel_l2(cs, ref) < 1e-5


def test_splitk_gemm_emits_groupnorm_column_sums():
    ops = _ops()
    from lavie_b200 import _lib
    lib = _lib.load()
    M, N, K = 1280, 1280, 11520
    a = _bf(_rand(M, K))
    w = _bf(_rand(N, K, scale=K ** -0.5))
    lib.lavie_debug_set(1, 4)                                        # force split-K
    try:
        out = ops.gemm(a, w, bias=_rand(N, seed=1), stats=True)
    finally:
        lib.lavie_debug_set(1, 0)
    assert rel_l2(_micro(out._gn_colsums, N), _colsums_ref(out, M, N)) < 1e-5


@pytest.mark.parametrize("NF,H,W,C,N,stride", [(4, 16, 32, 320, 640, 1), (2, 40, 64, 320, 320, 1), (3, 20, 32, 640, 640, 2)])
def test_conv_column_sums_feed_groupnorm(NF, H, W, C, N, stride):
    """conv (stats=True) -> GroupNorm through the column sums == conv -> stand-alone statistics pass, for 5-D statistics
    (sample = all frames) and for the per-frame norm, incl. a two-source concat whose groups straddle the seam."""
    ops = _ops()
    from lavie_b200.packing import pack_conv3x3
    x = _bf(_rand(NF * H * W, C))
    w = pack_conv3x3(_rand(N, C, 3, 3, scale=(9 * C) ** -0.5)).to(DEV)
    y = ops.conv3x3(x, NF, H, W, w, stride=stride, bias=_rand(N, seed=2), stats=True)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    rows = NF * Ho * Wo
    assert rel_l2(_micro(y._gn_colsums, N), _colsums_ref(y, rows, N)) < 1e-5
    gamma, beta = _rand(N, seed=4) * 0.1 + 1, _rand(N, seed=5) * 0.1
    plain = y.clone()                                                # a copy carries no statistics -> stand-alone pass
    for samples in (1, NF):
        ss = ops.groupnorm_scale_shift(y, samples, rows // samples, gamma, beta, 1e-5)
        ss_ref = ops.groupnorm_scale_shift(plain, samples, rows // samples, gamma, beta, 1e-5)
        assert rel_l2(ss, ss_ref) < 1e-5
    # concat [y | y2] with 32 groups over N + N2 channels
    y2 = ops.gemm(_bf(_rand(rows, 64, seed=9)), _bf(_rand(320, 64, seed=10, scale=0.1)), stats=True)
    g2, b2 = _rand(N + 320, seed=6) * 0.1 + 1, _rand(N + 320, seed=7) * 0.1
    ss = ops.groupnorm_scale_shift(y, 1, rows, g2, b2, 1e-5, x2=y2)
    ss_ref = ops.groupnorm_scale_shift(plain, 1, rows, g2, b2, 1e-5, x2=y2.clone())
    assert rel_l2(ss, ss_ref) < 1e-5


@pytest.mark.parametrize("M,N,K,splits", [(2048, 256, 256, 0), (1000, 512, 1536, 0), (640, 1024, 4608, 4)])
def test_column_sums_with_octet_micro_groups(M, N, K, splits):
    """Outputs whose width is not a multiple of 10 (the VSR model: 256 / 512 / 1024 channels, GroupNorm groups of
    8 .. 64 channels) carry statistics per 8-channel micro-group: [slab][chunk][piece] = octet chunk*4 + piece.  They
    must equal the sums of the stored bf16 values and feed the GroupNorm finalize exactly like the stand-alone pass,
    also for a two-source concat whose groups straddle the seam (1024 + 512 channels: groups of 48)."""
    ops = _ops()
    from lavie_b200 import _lib
    lib = _lib.load()
    a = _bf(_rand(M, K))
    w = _bf(_rand(N, K, scale=K ** -0.5))
    lib.lavie_debug_set(1, splits)
    try:
        out = ops.gemm(a, w, bias=_rand(N, seed=1), stats=True)
    finally:
        lib.lavie_debug_set(1, 0)
    slabs = (M + 31) // 32
    pad = torch.zeros(slabs * 32, N, device=DEV)
    pad[:M] = out.float()
    v = pad.reshape(slabs, 32, N // 8, 8)
    ref = torch.stack([v.sum((1, 3)), (v * v).sum((1, 3))], dim=-1)
    got = out._gn_colsums.reshape(slabs, N // 8, 2)                  # [slab][chunk][piece] is octet-major already
    assert rel_l2(got, ref) < 1e-5
    if M % 32 == 0:
        gamma, beta = _rand(N, seed=4) * 0.1 + 1, _rand(N, seed=5) * 0.1
        ss = ops.groupnorm_scale_shift(out, 2, M // 2, gamma, beta, 1e-6)
        ss_ref = ops.groupnorm_scale_shift(out.clone(), 2, M // 2, gamma, beta, 1e-6)
        assert rel_l2(ss, ss_ref) < 1e-5
        y2 = ops.gemm(_bf(_rand(M, 64, seed=9)), _bf(_rand(N // 2, 64, seed=10, scale=0.1)), stats=True)
        g2, b2 = _rand(N + N // 2, seed=6) * 0.1 + 1, _rand(N + N // 2, seed=7) * 0.1
        ss = ops.groupnorm_scale_shift(out, 1, M, g2, b2, 1e-5, x2=y2)
        ss_ref = ops.groupnorm_scale_shift(out.clone(), 1, M, g2, b2, 1e-5, x2=y2.clone())
        assert rel_l2(ss, ss_ref) < 1e-5


@pytest.mark.parametrize("NF,H,W,C,N", [(2, 5, 8, 128, 128), (3, 10, 16, 64, 320), (2, 20, 32, 640, 640), (1, 8, 64, 64, 256),
                                         (4, 4, 4, 128, 72), (1, 3, 2, 64, 64)])
def test_upsample_conv3x3_phase_convs(NF, H, W, C, N):
    """Upsample3D without the 4x copy: four 2x2 phase convs on the low-resolution map == nearest x2 + 3x3 conv (incl.
    borders, tile tails across images, N tails), and the statistics it emits (4 phase segments) feed the next GroupNorm
    like a stand-alone pass."""
    ops = _ops()
    from lavie_b200.packing import pack_upsample_conv3x3
    assert ops.upsample_conv3x3_supported(H, W, C)
    x = _bf(_rand(NF * H * W, C))
    w = _rand(N, C, 3, 3, scale=(9 * C) ** -0.5)
    bias = _rand(N, seed=2)
    y = ops.upsample_conv3x3(x, NF, H, W, pack_upsample_conv3x3(w).to(DEV), bias=bias, stats=True)
    up = F.interpolate(x.float().reshape(NF, H, W, C).permute(0, 3, 1, 2), scale_factor=2, mode="nearest")
    ref = F.conv2d(up, _bf(w).float(), bias, padding=1).permute(0, 2, 3, 1).reshape(NF * 4 * H * W, N)
    assert y.shape == ref.shape
    assert rel_l2(y.float(), ref) < 6e-3                      # tap sums are rounded to bf16 once more than the taps
    rows = NF * 4 * H * W
    gamma, beta = _rand(N, seed=4) * 0.1 + 1, _rand(N, seed=5) * 0.1
    for samples in ((1, NF) if N % 32 == 0 else ()):          # 5-D statistics and per-frame statistics (32 groups)
        ss = ops.groupnorm_scale_shift(y, samples, rows // samples, gamma, beta, 1e-5)      # phase-segment sums if usable
        ss_ref = ops.groupnorm_scale_shift(y.clone(), samples, rows // samples, gamma, beta, 1e-5)   # stand-alone pass
        assert rel_l2(ss, ss_ref) < 1e-5
    assert not ops.upsample_conv3x3_supported(5, 24, 64) and not ops.upsample_conv3x3_supported(5, 8, 40)


def test_out_of_bounds_canaries():
    """compute-sanitizer is closed on this GPU pool (profiles/r2_compute_sanitizer_closed.txt), so the memory-safety
    evidence is canaries: every output lives inside a larger poisoned allocation and the bytes around it must survive
    kernels that run with ragged sizes (M, N and key tails, partial slabs)."""
    ops = _ops()
    from lavie_b200 import _lib
    from lavie_b200._lib import Epilogue, check
    import ctypes
    lib = _lib.load()
    POISON = -7.0

    def guarded(rows, cols, dtype):
        big = torch.full((rows + 16, cols), POISON, dtype=dtype, device=DEV)
        return big, big[8:8 + rows]

    # GEMM with an M tail (not a multiple of 32 / 128 / 256) + column statistics with a partial last slab
    M, N, K = 1000, 320, 320
    a, w = _bf(_rand(M, K)), _bf(_rand(N, K, scale=K ** -0.5))
    big_out, out = guarded(M, N, torch.bfloat16)
    slabs = (M + 31) // 32
    big_cs = torch.full((slabs + 2, N // 32, 4, 2), POISON, device=DEV)
    cs = big_cs[1:1 + slabs]
    ep = Epilogue()
    ep.rows_per_batch = 1
    ep.col_stats = cs.data_ptr()
    ws = ops._workspace(a.device)
    check(lib.lavie_gemm_bf16(a.data_ptr(), K, K, None, 0, 0, w.data_ptr(), out.data_ptr(), N, M, N, ctypes.byref(ep), 0,
                              ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream), "gemm")
    torch.cuda.synchronize()
    assert (big_out[:8].float() == POISON).all() and (big_out[8 + M:].float() == POISON).all()
    assert (big_cs[0] == POISON).all() and (big_cs[-1] == POISON).all()
    assert rel_l2(out.float(), a.float() @ w.float().t()) < 4e-3
    # attention with ragged query / key counts writing into a guarded, strided output
    batch, heads, Sq, Sk, d, pitch = 3, 8, 200, 77, 40, 48
    q = torch.zeros(batch * Sq, heads, pitch, device=DEV)
    q[..., :d] = torch.randn(batch * Sq, heads, d, device=DEV)
    kv = torch.zeros(batch * Sk, 2, heads, pitch, device=DEV)
    kv[..., :d] = torch.randn(batch * Sk, 2, heads, d, device=DEV)
    q, kv = _bf(q.reshape(batch * Sq, -1)), _bf(kv.reshape(batch * Sk, -1))
    big_o, o = guarded(batch * Sq, heads * d + 64, torch.bfloat16)
    ops.attention(q, kv[:, :heads * pitch], kv[:, heads * pitch:], batch, heads, Sq, Sk, d, pitch, out=o[:, :heads * d])
    torch.cuda.synchronize()
    assert (big_o[:8].float() == POISON).all() and (big_o[8 + batch * Sq:].float() == POISON).all()
    assert (o[:, heads * d:].float() == POISON).all()
    # norms on a ragged row count
    rows, C = 2 * 77, 320
    x = _bf(_rand(rows, C))
    g, b = _rand(C, seed=1) * 0.1 + 1, _rand(C, seed=2) * 0.1
    big_y, y = guarded(rows, C, torch.bfloat16)
    ops.layernorm(x, g, b, out=y)
    ss = ops.groupnorm_scale_shift(x, 2, 77, g, b, 1e-5)
    big_z, z = guarded(rows, C, torch.bfloat16)
    ops.groupnorm_apply(x, ss, 2, 77, True, out=z)
    torch.cuda.synchronize()
    for bigt, n in ((big_y, rows), (big_z, rows)):
        assert (bigt[:8].float() == POISON).all() and (bigt[8 + n:].float() == POISON).all()
