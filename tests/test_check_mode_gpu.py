"""The fp32-accumulate CHECK MODE (BASELINE north star: noise-prediction rel-L2 <= 1e-3 against the reference's fp32
forward).  ``UNet3DConditionModel(check_mode=True)`` runs the same launch sequence with split-bf16 triples through the
same tcgen05 GEMM / conv mainloops (fp32 epilogues) and fp32 norm / attention kernels (lavie_b200/check.py,
csrc/check.cu).  Tolerances: 1e-3 for the whole network (stated by BASELINE.json), 2e-5 for single kernels."""
import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden, rel_l2

pytestmark = pytest.mark.gpu
CHECK_TOL = 1e-3
DEV = "cuda"


def _split(x):
    """fp32 [rows, C] -> Triple on the device (host-side split, mirrors check.cu's st_triple)."""
    from lavie_b200.check import Triple
    hi = x.to(torch.bfloat16)
    lo = (x - hi.float()).to(torch.bfloat16)
    return Triple(torch.cat([hi, lo, hi], dim=1).contiguous().to(DEV), x.shape[1])


def _rand(*shape, seed=0, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed + sum(shape))) * scale


def test_check_gemm_epilogues():
    from lavie_b200 import check as K
    M, N, Kd, B = 700, 320, 640, 2
    a, a2 = _rand(M, Kd, seed=1), _rand(M, 320, seed=2)
    w = _rand(N, Kd + 320, seed=3, scale=(Kd + 320) ** -0.5)
    bias, rb, res = _rand(N, seed=4), _rand(B, N, seed=5), _rand(M, N, seed=6)
    out = K.gemm(_split(a), K.weight(w, DEV), a2=_split(a2), bias=bias.to(DEV), row_bias=rb.to(DEV), rows_per_batch=M // B,
                 residual=_split(res))
    ref = (torch.cat([a, a2], 1).double() @ w.double().t() + bias.double() + rb.double().repeat_interleave(M // B, 0)
           + res.double())
    assert rel_l2(out.float().cpu(), ref) < 2e-5
    # GEGLU epilogue (interleaved 128 value / 128 gate columns, exact erf GELU), several 256-row tiles
    from lavie_b200.packing import interleave_geglu
    M, C = 1500, 320
    x, w1, b1 = _rand(M, C, seed=7), _rand(8 * C, C, seed=8, scale=C ** -0.5), _rand(8 * C, seed=9)
    wi, bi = interleave_geglu(w1, b1)
    out = K.gemm(_split(x), K.weight(wi, DEV), bias=bi.to(DEV), geglu=True)
    hg = x.double() @ w1.double().t() + b1.double()
    h, g = hg.chunk(2, dim=-1)
    assert rel_l2(out.float().cpu(), h * F.gelu(g)) < 2e-5


@pytest.mark.parametrize("H,W,C,N,stride", [(8, 16, 64, 128, 1), (12, 20, 128, 64, 2), (5, 8, 320, 320, 1)])
def test_check_conv3x3(H, W, C, N, stride):
    from lavie_b200 import check as K
    from lavie_b200.packing import pack_conv3x3
    NF = 3
    x = _rand(NF, C, H, W, seed=1)
    w = _rand(N, C, 3, 3, seed=2, scale=(9 * C) ** -0.5)
    bias = _rand(N, seed=3)
    xt = _split(x.permute(0, 2, 3, 1).reshape(-1, C))
    out = K.conv3x3(xt, NF, H, W, K.weight(pack_conv3x3(w, dtype=None), DEV), stride=stride, bias=bias.to(DEV))
    ref = F.conv2d(x.double(), w.double(), bias.double(), stride=stride, padding=1)
    ref = ref.permute(0, 2, 3, 1).reshape(-1, N)
    assert rel_l2(out.float().cpu(), ref) < 2e-5


def test_check_norms():
    from lavie_b200 import check as K
    B, rows, C = 2, 600, 640
    x = _rand(B * rows, C, seed=1) * 2 + 0.3
    x2 = _rand(B * rows, 320, seed=2)
    g, b = _rand(C + 320, seed=3) * 0.1 + 1, _rand(C + 320, seed=4) * 0.1
    out = K.groupnorm(_split(x), B, rows, g.to(DEV), b.to(DEV), 1e-5, True, x2=_split(x2))
    cat = torch.cat([x, x2], 1).double().reshape(B, rows, C + 320).permute(0, 2, 1)
    ref = F.silu(F.group_norm(cat, 32, g.double(), b.double(), 1e-5)).permute(0, 2, 1).reshape(B * rows, -1)
    assert rel_l2(out.float().cpu(), ref) < 2e-5
    out = K.layernorm(_split(x), g[:C].to(DEV), b[:C].to(DEV))
    assert rel_l2(out.float().cpu(), F.layer_norm(x.double(), (C,), g[:C].double(), b[:C].double())) < 2e-5


_CHECK_ATTN_SHAPES = [(160, 160, 160, 1, 0), (100, 77, 40, 4, 0), (64, 64, 80, 1, 4)]


@pytest.mark.parametrize("S,Sk,d,div,sc,inputs",
                         [pytest.param(*s, "randn", id="-".join(map(str, s))) for s in _CHECK_ATTN_SHAPES]
                         + [pytest.param(*s, kind, id=f"{kind}-" + "-".join(map(str, s)))
                            for kind in ("sharpened", "flush") for s in _CHECK_ATTN_SHAPES])
def test_check_attention(S, Sk, d, div, sc, inputs):
    """inputs: N(0, 1), or test_attention_rescale's sharpened (q x 16) and flush (the keys from 64 on -- Sk // 2 for
    fewer keys -- lifted by 130 log2 units) scores."""
    from lavie_b200 import check as K
    from lavie_b200.packing import head_pitch
    heads, batch = 8, 8
    pitch = head_pitch(d)
    hp = heads * pitch

    def padded(rows, seed):
        t = torch.zeros(rows, hp)
        for h in range(heads):
            t[:, h * pitch:h * pitch + d] = _rand(rows, d, seed=seed + h)
        return t
    q, k, v = padded(batch * S, 1), padded((batch // div) * Sk, 20), padded((batch // div) * Sk, 40)
    if inputs != "randn":
        from test_attention_rescale import sharpen_heads
        qh = q.reshape(batch, S, heads, pitch).transpose(1, 2)
        kh = k.reshape(batch // div, Sk, heads, pitch).transpose(1, 2)
        qh[..., :d], kh[..., :d] = sharpen_heads(qh[..., :d], kh[..., :d], inputs, d ** -0.5)
    out = K.attention(_split(q), _split(k), _split(v), batch, heads, S, Sk, d, pitch, kv_batch_div=div,
                      sparse_causal_frames=sc)
    qq = q.reshape(batch, S, heads, pitch)[..., :d].permute(0, 2, 1, 3).double()
    kk = k.reshape(batch // div, Sk, heads, pitch)[..., :d].permute(0, 2, 1, 3).double().repeat_interleave(div, 0)
    vv = v.reshape(batch // div, Sk, heads, pitch)[..., :d].permute(0, 2, 1, 3).double().repeat_interleave(div, 0)
    if sc:
        f = torch.arange(batch) % sc
        first, former = torch.arange(batch) - f, torch.where(f > 0, torch.arange(batch) - 1, torch.arange(batch))
        kk, vv = torch.cat([kk[first], kk[former]], dim=2), torch.cat([vv[first], vv[former]], dim=2)
    ref = F.scaled_dot_product_attention(qq, kk, vv).permute(0, 2, 1, 3).reshape(batch * S, heads * d)
    # fp32 scores carry an absolute error proportional to their size (2^-24 per rounding), and the output's relative
    # error follows the score error: the 2e-5 of N(0, 1) inputs (scores of a few units) scales with the largest score
    # past 32 units (flush: ~100)
    s_max = float((qq @ kk.transpose(-1, -2)).abs().max()) * d ** -0.5
    assert rel_l2(out.float().cpu(), ref) < 2e-5 * max(1.0, s_max / 32)


@pytest.fixture(scope="module")
def models(synthetic_sd):
    from lavie_b200 import UNet3DConditionModel
    out = []
    for chk in (True, False):
        m = UNet3DConditionModel(check_mode=chk)
        m.load_state_dict(synthetic_sd, strict=True)
        out.append(m.to(DEV).eval())
    return out


@pytest.mark.parametrize("name", ["b2_f16_8x8", "b1_f3_16x24", "b2_f2_8x8_tvec"])
def test_matches_reference_golden_check(models, name):
    """BASELINE north star: <= 1e-3 against the reference's fp32 forward (goldens produced by the reference itself)."""
    chk, _ = models
    g = load_golden(name)
    out = chk(g["sample"].to(DEV), g["timestep"], encoder_hidden_states=g["text"].to(DEV)).sample
    err = rel_l2(out.cpu(), g["out"])
    print(f"{name} [check mode]: rel-L2 vs reference fp32 = {err:.3e}")
    assert out.shape == g["out"].shape and err <= CHECK_TOL


def test_bf16_error_is_storage_noise_per_tap(models, synthetic_sd):
    """Attribution of the ~1e-2 bf16 figure: at every tap the bf16 path sits ~1e-2 from the oracle while the check mode
    (same launch sequence, same GEMM / conv mainloops, >= 16-bit operands) sits <= 1e-3 -- i.e. the gap is operand /
    activation rounding, not a bug that both modes would share."""
    from lavie_b200.synthetic import synthetic_inputs
    from oracle import unet3d_oracle as O
    chk, bf = models
    sample, t, text = synthetic_inputs(2, 4, 8, 64, seed=3)
    taps_o, taps_c, taps_b = {}, {}, {}
    ref = O.unet_forward(synthetic_sd, sample, t, text, taps=taps_o)
    out_c = chk(sample.to(DEV), t, encoder_hidden_states=text.to(DEV), taps=taps_c).sample
    out_b = bf(sample.to(DEV), t, encoder_hidden_states=text.to(DEV), taps=taps_b).sample
    for k in ("emb", "conv_in", "down0_res0", "down0_attn0", "mid", "up_out"):
        ec, eb = rel_l2(taps_c[k].cpu(), taps_o[k]), rel_l2(taps_b[k].cpu(), taps_o[k])
        print(f"tap {k:12s}: check {ec:.2e}   bf16 {eb:.2e}")
        assert ec <= CHECK_TOL, k
    ec, eb = rel_l2(out_c.cpu(), ref), rel_l2(out_b.cpu(), ref)
    print(f"output          : check {ec:.2e}   bf16 {eb:.2e}")
    assert ec <= CHECK_TOL and eb <= 2e-2 and ec < 0.2 * eb


def test_interp_check_mode():
    from lavie_b200 import UNet3DConditionModel
    from lavie_b200.config import INTERP_CONFIG
    from lavie_b200.synthetic import synthetic_state_dict
    m = UNet3DConditionModel(INTERP_CONFIG, check_mode=True)
    m.load_state_dict(synthetic_state_dict(INTERP_CONFIG, seed=0), strict=True)
    m = m.to(DEV).eval()
    g = load_golden("interp_b2_f7_8x8")
    out = m(g["sample"].to(DEV), g["timestep"], encoder_hidden_states=g["text"].to(DEV)).sample
    err = rel_l2(out.cpu(), g["out"])
    print(f"interp_b2_f7_8x8 [check mode]: rel-L2 vs reference fp32 = {err:.3e}")
    assert err <= CHECK_TOL
