"""The flash kernels' lazy softmax rescale, against the fp64 reference, on scores that move the running maximum.

attn_fwd_kernel (ops.attention, ops.frame_attention) and attn_wide_kernel (vae_attention.attention_wide) keep the
exponent offset m_used baked into O and the row sum, and move it only when a 64-key tile's maximum exceeds m_used + 8 in
log2 units: O and l are then multiplied by alpha = 2^(m_used - m_tile), lanes of the same warp that did not grow by 1,
and the probabilities of that tile reach up to 2^8.  N(0, 1) queries and keys at scale d^-1/2 never get there, so the
inputs here are built to: every family below makes rescale_events (test_launch_audit.py, the kernels' own fp32 walk)
count events at tiles j > 0, and the CPU tests show that the kernels' algorithm (lazy_attention_emulation) stays within
attention_core's bound on them while each injected rescale defect leaves it.

Families (deterministic; queries and keys exact in bf16, scale a power of two, so every score is exact in fp32 whatever
the summation order, and the kernel's m_tile is what rescale_events computes):
  rise           key scores grow by 10 log2 units per tile: every tile rescales
  threshold      the second tile's maximum grows by 8 - 1/64 (even query rows) or 8 + 1/64 (odd rows) log2 units, placed
                 with the kernel's fp32 scale_log2: only the odd rows rescale
  spike63/64     one dominant key (+12 log2 units) at key 63 (the first tile: no rescale) or key 64 (the second tile)
  spike_partial  one dominant key (+136) as the last key of a partial tile: without the rescale p would overflow fp32
  spike_segment  one dominant key (+12) in the second SparseCausal segment (the former frame)
  warp_mixed     even query rows see rising keys, odd rows falling ones: every warp has alpha < 1 and alpha = 1 lanes
  flush          the keys past the first tile grow by 130 log2 units: alpha flushes to 0
  sharp4/16      N(0, 1) q, k with q x 4 or x 16
"""
import math

import pytest
import torch

from test_launch_audit import (BF16, F64, LAZY_DEFECTS, REL_ATTN, WIDE_D, Cmp, _frame_cmp,
                               _wide_cmp, attention_cmp, attention_core, attention_layout, attention_ref,
                               check_outside_view, frame_attention_ref, heads_of, launch_events,
                               lazy_attention_emulation, rescale_events, scale_log2, tf32_off, tf32_restore,
                               view_mask, wide_attention_ref)

FAMILIES = ("rise", "threshold", "spike63", "spike64", "spike_partial", "warp_mixed", "flush", "sharp4", "sharp16")
SC_FAMILIES = ("rise", "threshold", "spike_segment", "warp_mixed", "flush")
RISE = 10.0                 # log2 units per key tile
SPIKE, SPIKE_BIG, FLUSH = 12.0, 136.0, 130.0
ONES_TOL = 2.0 ** -7        # V = 1 probe: every output is 1 within this


def pow2_scale(d):
    """A power of two near d^-1/2: the scores stay exact."""
    return 2.0 ** -round(math.log2(math.sqrt(d)))


def _grid(log2_units, sc):
    """The multiple of 1/64 nearest to a score of `log2_units` (at fp32 scale_log2 sc)."""
    return round(log2_units / float(sc) * 64) / 64


def _encode(v):
    """Scores v (multiples of 1/64, |v| < 2^14) as three bf16-exact key columns that sum to v exactly."""
    n = torch.round(v * 64).to(torch.int64)
    sg, a = n.sign().to(torch.float32), n.abs()
    return torch.stack([sg * (a >> 16) * 2.0 ** 10, sg * ((a >> 8) & 255) * 4.0, sg * (a & 255) * 2.0 ** -6], -1)


def threshold_scores(sc):
    """(below, above): scores of the second tile's key whose fp32 growth over a first-tile maximum of 0 is the grid value
    nearest to 8 - 1/64 and to 8 + 1/64 log2 units."""
    out = []
    for target in (8 - 1 / 64, 8 + 1 / 64):
        v = _grid(target, sc)
        grown = float(torch.tensor(v, dtype=torch.float32) * sc)
        assert abs(grown - target) <= float(sc) / 128 + 1e-6, (target, grown)
        out.append(v)
    return out


def family_heads(family, n_q, Sq, n_k, Sk, d, scale, spiked=None, seed=0):
    """Per-head inputs of one family: Q [n_q, Sq, d], K and V [n_k, Sk, d], fp32 tensors of bf16 values.  The score of a
    query row with a key is sigma_row * v_key + tau_row * w_key + noise: columns 0-2 carry v (q = sigma), column 3
    carries w (q = tau), the rest small noise (multiples of 1/16), sized to about one log2 unit of score spread.
    spiked [n_k]: the key sequences that get spike_segment's spike (default all)."""
    g = torch.Generator().manual_seed(seed)
    V = torch.randn(n_k, Sk, d, generator=g).to(BF16).float()
    if family.startswith("sharp"):
        mult = float(family[len("sharp"):])
        Q = (torch.randn(n_q, Sq, d, generator=g).to(BF16).float() * mult)
        K = torch.randn(n_k, Sk, d, generator=g).to(BF16).float()
        return Q, K, V
    sc = scale_log2(scale)
    pos = torch.arange(Sk)
    rows = torch.arange(Sq)
    v = torch.zeros(n_k, Sk)
    w = torch.zeros(n_k, Sk)
    sigma = torch.ones(Sq)
    tau = torch.zeros(Sq)
    amp = min(1.0, max(1 / 16, round(16 * math.sqrt(3 / (math.sqrt(d - 4) * float(sc)))) / 16))
    if family in ("rise", "warp_mixed"):
        v[:] = (pos // 64).float() * _grid(RISE, sc)
        if family == "warp_mixed":
            sigma = 1.0 - 2.0 * (rows % 2).float()
    elif family == "threshold":
        assert Sk >= 72, Sk
        amp = 0.0
        below, above = threshold_scores(sc)
        v[:] = -(pos % 5).float()
        v[:, 71] = below
        w[:, 71] = above - below
        tau = (rows % 2).float()
    elif family.startswith("spike"):
        at = {"spike63": 63, "spike64": 64, "spike_partial": Sk - 1, "spike_segment": 5}[family]
        assert family != "spike_partial" or Sk % 64, Sk
        sel = torch.ones(n_k, dtype=torch.bool) if spiked is None or family != "spike_segment" else spiked
        v[sel, at] = _grid(SPIKE_BIG if family == "spike_partial" else SPIKE, sc)
    elif family == "flush":
        v[:, 64:] = _grid(FLUSH, sc)
    else:
        raise ValueError(family)
    A = int(amp * 16)
    qn = torch.randint(-A, A + 1, (n_q, Sq, d - 4), generator=g).float() / 16
    kn = torch.randint(-A, A + 1, (n_k, Sk, d - 4), generator=g).float() / 16
    Q = torch.cat([sigma[None, :, None].expand(n_q, Sq, 3), tau[None, :, None].expand(n_q, Sq, 1), qn], -1)
    K = torch.cat([_encode(v), w[..., None], kn], -1)
    assert torch.equal(Q.to(BF16).float(), Q) and torch.equal(K.to(BF16).float(), K)
    return Q, K, V


# ------------------------------------------------------------------------------------------------ launch layouts
def attention_case(family, batch, heads, Sq, Sk, d, pitch, div=1, sc_frames=0, sc_halo=0, seed=0, device="cpu"):
    """The arguments of one ops.attention launch (the audit's recorded-argument dict) holding one family: q [batch*Sq,
    heads*pitch], k / v [kv sequences * Sk, heads*pitch], pad columns zero."""
    n_kv = batch // div + (2 if sc_halo else 0)
    seq = torch.arange(n_kv)
    # the key sequences a SparseCausal launch reads as the former frame only (never as frame 0)
    spiked = (seq >= 1) if sc_halo else (seq % sc_frames >= 1) if sc_frames else torch.ones(n_kv, dtype=torch.bool)
    scale = pow2_scale(d)
    Q, K, V = family_heads(family, batch * heads, Sq, n_kv * heads, Sk, d, scale,
                           spiked.repeat_interleave(heads), seed)

    def lay(t, n):
        buf = torch.zeros(n, t.shape[1], heads, pitch)
        buf[..., :d] = t.reshape(n, heads, t.shape[1], d).permute(0, 2, 1, 3)
        return buf.reshape(n * t.shape[1], heads * pitch).to(BF16).to(device)
    return {"q": lay(Q, batch), "k": lay(K, n_kv), "v": lay(V, n_kv), "batch": batch, "heads": heads, "Sq": Sq,
            "Sk": Sk, "d": d, "head_pitch": pitch, "kv_batch_div": div, "sparse_causal_frames": sc_frames,
            "sc_halo": sc_halo, "scale": scale}


def frame_case(family, B, F_, HW, heads, d, pitch, seed=0, device="cpu"):
    """qkv [B*F*HW, 3*heads*pitch] of ops.frame_attention (rows (video, frame, pixel)) holding one family, the sequences
    running over the frames of a pixel; scale d^-1/2, a power of two for d = 64."""
    assert d ** -0.5 == pow2_scale(d), d
    n = B * HW * heads
    Q, K, V = family_heads(family, n, F_, n, F_, d, d ** -0.5, seed=seed)
    qkv = torch.zeros(B, F_, HW, 3, heads, pitch)
    for i, t in enumerate((Q, K, V)):
        qkv[:, :, :, i, :, :d] = t.reshape(B, HW, heads, F_, d).permute(0, 3, 1, 2, 4)
    return {"qkv": qkv.reshape(B * F_ * HW, 3 * heads * pitch).to(BF16).to(device), "B": B, "F": F_, "HW": HW,
            "heads": heads, "d": d, "head_pitch": pitch}


def wide_case(family, frames, S, seed=0, device="cpu"):
    """q, k, v [frames*S, 512] of attention_wide holding one family (scale 1: the kernel's q carries 512^-1/2)."""
    Q, K, V = family_heads(family, frames, S, frames, S, WIDE_D, 1.0, seed=seed)
    if family.startswith("sharp"):
        Q = (Q * WIDE_D ** -0.5).to(BF16).float()
    return {k: t.reshape(frames * S, WIDE_D).to(BF16).to(device) for k, t in (("q", Q), ("k", K), ("v", V))} | {
        "frames": frames, "S": S}


def _heads(a):
    qrows, krows = attention_layout(a)
    h = (a["heads"], a["head_pitch"], a["d"])
    return heads_of(a["q"], qrows, *h), heads_of(a["k"], krows, *h), heads_of(a["v"], krows, *h)


def _segments(a):
    return 2 if a["sparse_causal_frames"] else 1


def _cpu_case(family, Sk, d=40, pitch=48, **kw):
    kw = {"batch": 2, "heads": 2, "Sq": 200, **kw}
    return attention_case(family, Sk=Sk, d=d, pitch=pitch, **kw)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("batch,Sq,Sk,d", [(4, 256, 256, 40), (2, 640, 640, 80), (2, 160, 160, 160),
                                           (1, 2560, 2560, 40), (2, 320, 320, 64)])
def test_normal_inputs_never_rescale_but_sharpened_do(batch, Sq, Sk, d):
    """The shapes of test_kernels_gpu.py::test_attention with bf16 N(0, 1) q, k at scale d^-1/2 (8 heads): no rescale
    event at a tile j > 0 -- the gap these tests close; q x 4 and q x 16 reach it."""
    g = torch.Generator().manual_seed(batch * Sq + d)
    heads = 8
    q = torch.randn(batch, heads, Sq, d, generator=g).to(BF16)
    k = torch.randn(batch, heads, Sk, d, generator=g).to(BF16)
    S = q.float() @ k.float().transpose(-1, -2)
    assert rescale_events(S, d ** -0.5).events == 0
    assert rescale_events(S * 4, d ** -0.5).events > 0 and rescale_events(S * 16, d ** -0.5).events > 0


@pytest.mark.parametrize("Sk", [77, 2597])
@pytest.mark.parametrize("family", FAMILIES + ("spike_segment",))
def test_every_family_rescales(family, Sk):
    """rescale_events counts events at tiles j > 0 for every family (spike63 excepted: its key sits in the first tile
    and must not count; the N(0, 1) families need the long key sequence to be sure of one); warp_mixed and threshold
    mix growing and non-growing lanes within warps; threshold moves exactly the odd rows, at the tile of key 71."""
    sc = 4 if family == "spike_segment" else 0
    a = _cpu_case(family, Sk, sc_frames=sc, batch=4 if sc else 2)
    Q, K, _ = _heads(a)
    r = rescale_events(Q.float() @ K.float().transpose(-1, -2), a["scale"], _segments(a))
    if family == "spike63":
        assert r.events == 0, r
    elif not (family.startswith("sharp") and Sk < 2048):
        assert r.events > 0, (family, r)
    if family in ("warp_mixed", "threshold"):
        assert r.mixed, (family, r)
    if family == "threshold":
        assert r.events == 2 * 2 * 100 and r.first[-1] == 1 and r.first[-2] == 1, r


@pytest.mark.parametrize("family", FAMILIES + ("spike_segment",))
@pytest.mark.parametrize("d,pitch", [(40, 48), (64, 64)])
def test_lazy_emulation_within_bound(family, d, pitch):
    """The kernels' algorithm (lazy_attention_emulation: fp32 scores, lazy maximum, bf16 P, fp32 or ones-column row sum)
    stays within attention_core's element-wise bound and REL_ATTN on every family, with probabilities up to 2^8."""
    for Sk in (77, 2597):
        sc = 4 if family == "spike_segment" else 0
        a = _cpu_case(family, Sk, d=d, pitch=pitch, batch=4 if sc else 2, sc_frames=sc, Sq=100)
        Q, K, V = _heads(a)
        o, bnd = attention_core(Q, K, V, a["scale"])
        got = lazy_attention_emulation(Q, K, V, a["scale"], ones=d % 16 != 0, segments=_segments(a))
        cmp = Cmp("lazy emulation", got, o, bnd, REL_ATTN)
        assert cmp.ok, (family, Sk, str(cmp))


# the family on which each injected defect must show (spike_partial: the skipped threshold lets p overflow)
DEFECT_FAMILY = {"o": "rise", "l": "rise", "sign": "rise", "warp": "warp_mixed", "partial": "spike_partial",
                 "stale": "rise"}


@pytest.mark.parametrize("defect", LAZY_DEFECTS)
def test_each_rescale_defect_is_flagged(defect):
    """Each defect of the rescale, injected into the emulation, is flagged by Cmp on its family (and, for the defects
    that do not depend on the row-sum path, with the ones column as well)."""
    family = DEFECT_FAMILY[defect]
    for d, pitch in ((48, 48), (40, 48)):
        if d == 40 and defect == "l":
            continue            # the ones column carries the row sum through O: the separate l is not used
        a = _cpu_case(family, 2597, d=d, pitch=pitch, Sq=100)
        Q, K, V = _heads(a)
        o, bnd = attention_core(Q, K, V, a["scale"])
        got = lazy_attention_emulation(Q, K, V, a["scale"], defect, ones=d % 16 != 0)
        cmp = Cmp(defect, got, o, bnd, REL_ATTN)
        assert not cmp.ok, (defect, d, str(cmp))


# ------------------------------------------------------------------------------------------------ GPU
DEV = "cuda"


@pytest.fixture
def exact_refs():
    saved = tf32_off()
    yield
    tf32_restore(saved)


def _lib():
    from lavie_b200 import _lib as L
    return L.load()


def _ops():
    from lavie_b200 import ops
    return ops


def _ones_v(a):
    v = torch.zeros_like(a["v"])
    v.reshape(v.shape[0], a["heads"], a["head_pitch"])[..., :a["d"]] = 1.0
    return v


def _run_attention(a, v=None, out=None):
    return _ops().attention(a["q"], a["k"], a["v"] if v is None else v, a["batch"], a["heads"], a["Sq"], a["Sk"],
                            a["d"], a["head_pitch"], a["kv_batch_div"], a["scale"], out, a["sparse_causal_frames"],
                            a["sc_halo"])


def expect_events(family, ev, keys):
    """The launch's inputs reach the rescale (spike63: must not; the N(0, 1) families: sure only with long keys)."""
    if family == "spike63":
        assert ev.events == 0, ev
    elif not (family.startswith("sharp") and keys < 2048):
        assert ev.events > 0, (family, ev)


def check_attention_case(a, family, worst, out=None):
    """Kernel vs attention_core element by element (and REL_ATTN), then the V = 1 probe; records err/bound."""
    ev = launch_events("attention", a)
    expect_events(family, ev, a["Sk"] * _segments(a))
    got = _run_attention(a, out=out)
    o, bnd = attention_ref(a)
    cmp = attention_cmp(f"attention {family}", got, a, o, bnd)
    ones = _run_attention(a, v=_ones_v(a))
    probe = Cmp(f"attention {family} V=1", ones, torch.ones((), dtype=F64), ONES_TOL)
    worst.append((family, cmp.worst))
    assert cmp.ok, f"{cmp}; first rescale at (sequence, head, row, tile) {ev.first}"
    assert probe.ok, str(probe)
    return got


HEADS = [(40, 48), (48, 48), (64, 64), (72, 80), (80, 80), (96, 96), (128, 128), (160, 160)]


@pytest.mark.gpu
@pytest.mark.parametrize("poly", [0, 4])
@pytest.mark.parametrize("d,pitch", HEADS)
@pytest.mark.parametrize("family", FAMILIES)
def test_attention_families(family, d, pitch, poly, exact_refs):
    """Every dk instantiation (48 .. 160), with the ones-column denominator (d = 40, 72) and without, both exponent paths
    (lavie_debug_set(4, 0): all on the MUFU; (4, 4): every 4th on the FMA pipe), 77 keys (a full and a 13-key tile) and
    2597 keys (40 full tiles and a 37-key one), 200 queries (a partial query tile)."""
    lib = _lib()
    worst = []
    lib.lavie_debug_set(4, poly)
    try:
        for Sk in (77, 2597):
            check_attention_case(attention_case(family, 2, 2, 200, Sk, d, pitch, seed=d + Sk, device=DEV), family,
                                 worst)
    finally:
        lib.lavie_debug_set(4, -1)
    print(f"attention {family} d={d} poly={poly}: worst err/bound {max(w for _, w in worst):.3g}")


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["rise", "threshold", "spike64", "warp_mixed", "flush"])
@pytest.mark.parametrize("d,pitch", [(40, 48), (64, 64)])
def test_attention_families_shared_kv(family, d, pitch, exact_refs):
    """kv_batch_div = 2: two query batches read one key sequence."""
    worst = []
    for Sk in (77, 2597):
        check_attention_case(attention_case(family, 4, 2, 130, Sk, d, pitch, div=2, seed=Sk, device=DEV), family,
                             worst)


@pytest.mark.gpu
@pytest.mark.parametrize("sc_halo", [0, 1, 2])
@pytest.mark.parametrize("family", SC_FAMILIES)
@pytest.mark.parametrize("d,pitch", [(40, 48), (64, 64)])
def test_sparse_causal_families(family, sc_halo, d, pitch, exact_refs):
    """SparseCausal attention: two key segments [frame 0 | former frame], each walked in its own tiles (a partial one
    per segment at 77 keys); spike_segment puts the dominant key in the second segment only; sc_halo 1 / 2: the
    frame-sharded key buffer with two halo frames."""
    frames = 4
    worst = []
    for Sk in (77, 200):
        a = attention_case(family, frames, 2, Sk, Sk, d, pitch, sc_frames=frames, sc_halo=sc_halo, seed=Sk,
                           device=DEV)
        check_attention_case(a, family, worst)


@pytest.mark.gpu
@pytest.mark.parametrize("family", ["rise", "spike_partial", "warp_mixed", "flush"])
def test_attention_families_out_view(family, exact_refs):
    """out= a column view of a wider buffer: the rescaled results land in the view and nothing outside it changes."""
    a = attention_case(family, 2, 2, 200, 2597, 72, 80, seed=5, device=DEV)
    base = torch.randn(2 * 200, 2 * 72 + 40, device=DEV).to(BF16)
    view = base[:, 8:8 + 2 * 72]
    before = base.clone()
    got = check_attention_case(a, family, [], out=view)
    assert got.data_ptr() == view.data_ptr()
    flag = check_outside_view(before, base, view_mask(base, view))
    assert flag.ok, flag.detail


@pytest.mark.gpu
@pytest.mark.parametrize("family", FAMILIES)
def test_frame_attention_families(family, exact_refs):
    """ops.frame_attention at F = 130 frames: three key tiles (64, 64, 2) on the swapped-dimension tensor maps (the
    pixels are the batch, the frames the sequence), d = 64 so that d^-1/2 is a power of two."""
    a = frame_case(family, 1, 130, 12, 2, 64, 64, seed=3, device=DEV)
    ev = launch_events("frame_attention", a)
    expect_events(family, ev, 130)
    ops = _ops()
    got = ops.frame_attention(a["qkv"], a["B"], a["F"], a["HW"], a["heads"], a["d"], a["head_pitch"])
    o, bnd = frame_attention_ref(a["qkv"], a["B"], a["F"], a["HW"], a["heads"], a["d"], a["head_pitch"])
    cmp = _frame_cmp(f"frame attention {family}", got, o, bnd, a, REL_ATTN)
    assert cmp.ok, f"{cmp}; first rescale at (sequence, head, row, tile) {ev.first}"
    qkv = a["qkv"].clone()
    hp = a["heads"] * a["head_pitch"]
    qkv[:, 2 * hp:] = _ones_v({"v": qkv[:, 2 * hp:].contiguous(), "heads": a["heads"], "head_pitch": a["head_pitch"],
                               "d": a["d"]})
    ones = ops.frame_attention(qkv, a["B"], a["F"], a["HW"], a["heads"], a["d"], a["head_pitch"])
    probe = Cmp(f"frame attention {family} V=1", ones, torch.ones((), dtype=F64), ONES_TOL)
    assert probe.ok, str(probe)
    print(f"frame_attention {family}: worst err/bound {cmp.worst:.3g}")


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1317, 4133])
@pytest.mark.parametrize("family", FAMILIES)
def test_wide_attention_families(family, S, exact_refs):
    """attention_wide (one head, d = 512, S keys per frame in 64-key tiles with a partial last one, double-buffered S
    and the parity wait on the previous P V before the O rescale), 2 frames."""
    from lavie_b200.vae_attention import attention_wide
    if family == "spike_partial":
        assert S % 64
    a = wide_case(family, 2, S, seed=S, device=DEV)
    ev = launch_events("attention_wide", a)
    expect_events(family, ev, S)
    got = attention_wide(a["q"], a["k"], a["v"], 2, S)
    ref, bnd = wide_attention_ref(a["q"], a["k"], a["v"], 2, S)
    cmp = _wide_cmp(f"attention_wide {family}", got, a, None, ref, bnd)
    assert cmp.ok, f"{cmp}; first rescale at (frame, head, row, tile) {ev.first}"
    ones = attention_wide(a["q"], a["k"], torch.ones_like(a["v"]), 2, S)
    probe = Cmp(f"attention_wide {family} V=1", ones, torch.ones((), dtype=F64), ONES_TOL)
    assert probe.ok, str(probe)
    print(f"attention_wide {family} S={S}: worst err/bound {cmp.worst:.3g}")


# ------------------------------------------------------------------------------------------------ shared with other tests
def sharpen_heads(q, k, kind, scale):
    """The sharpened and flush inputs for per-head q [..., Sq, d], k [..., Sk, d] (fp32 or bf16, modified copies
    returned): "sharpened" q x 16; "flush" column 0 of q set to 16 and column 0 of the keys from key 64 on (Sk // 2 for
    fewer keys) to a bf16 value that lifts their scores by ~130 log2 units, column 0 of the others to 0."""
    if kind == "sharpened":
        return q * 16, k
    q, k = q.clone(), k.clone()
    Sk = k.shape[-2]
    at = 64 if Sk > 64 else Sk // 2
    c = float(torch.tensor(FLUSH / (16 * scale * math.log2(math.e))).to(BF16))
    q[..., 0] = 16
    k[..., 0] = 0
    k[..., at:, 0] = c
    return q, k
