"""Every tile plan of the tcgen05 GEMM (lavie_b200/csrc/gemm.cu), checked element by element against fp64.

For each call `make_plan` picks a tile width bn (64 .. 320), a split-K factor (1 .. 16) and, optionally, a main window
of full waves plus a split-K tail window over the last 1 .. 16 pair-tile rows.  The choice depends only on (M, N, K),
the mode and the SM count, so a test reaches only the plans its shapes happen to plan to.  This file searches shapes of
a few model-like families for each plan class `(mode, bn, splits, tail_splits)` (tail_splits 0: no tail window) with
the host-side planner query `lavie_gemm_plan`, pins which classes the search reaches (CPU tests), and runs the real op
on the cheapest shape of each class, with every epilogue at once, against the audit's fp64 references and bounds
(GPU tests).  The plans are those of a 148-SM B200 (the host fallback of lavie_num_sms); the GPU tests re-query the
plan on the device and fail if it differs.

The CPU tests at the end inject single defects into an fp64-correct bf16 result of a tail plan and show that the
element-wise check flags each one, and whether a whole-tensor rel-L2 < 4e-3 would have.
"""
import collections
import ctypes
import functools

import pytest
import torch

from conftest import rel_l2
from test_launch_audit import (BF16, F64, REL_ROUND, U, Cmp, c_gemm, check_colsums, check_outside_view,
                               chk_upsample_conv3x3, colsum_expected, conv_out_size, conv_rows, conv_step,
                               epilogue_ref, gemm_check, mm_abs, tf32_off, tf32_restore, view_mask)

WORKSPACE_BYTES = 128 << 20          # ops.WORKSPACE_BYTES: the split-K workspace every op passes
TICKET_BYTES = 64 << 10              # gemm.cu: lavie_debug_set(7, 1) keeps the workspace's last 64 KiB for tickets
BNS = (64, 128, 160, 192, 256, 320)
MODES = ("gemm", "conv3x3", "frame_conv")
CONV = {"gemm": 0, "conv3x3": 1, "frame_conv": 0}     # frame_conv plans as a plain GEMM (frame_conv_impl)


def _lib():
    from lavie_b200 import _lib as L
    return L.load()


def plan_of(mode, M, N, K, ws=WORKSPACE_BYTES, geglu=False):
    """(bn, splits, tail_tiles, tail_splits) the library plans for this launch; tail_splits is 1 without a tail."""
    out = [ctypes.c_int() for _ in range(4)]
    rc = _lib().lavie_gemm_plan(M, N, K, CONV[mode], int(geglu), ws, *(ctypes.byref(o) for o in out))
    assert rc == 0, (mode, M, N, K)
    return tuple(o.value for o in out)


def class_of(mode, M, N, K):
    bn, s, tt, ts = plan_of(mode, M, N, K)
    return (mode, bn, s, ts if tt else 0)


# ------------------------------------------------------------------------------------------------ shape finder
# A shape: mode, M, N, K and the geometry the op needs (gemm: nothing; conv3x3: NF, H, W, C; frame_conv: F, HW, C,
# taps).  M is never a multiple of 32: every 32-row statistics slab and 256-row pair tile of the last row ends early.
Shape = collections.namedtuple("Shape", "mode M N K geo")

GEMM_N = (256, 320, 512, 640, 1024, 1280)
GEMM_K = (320, 512, 640, 1280, 2560, 5120, 10240)
CONV_C = (256, 320, 512, 640, 1280, 1920, 2560)     # 1920 / 2560: the up blocks' concatenated inputs
CONV_N = (256, 320, 512, 640, 1280)
CONV_HW = ((5, 7), (10, 16), (15, 9), (20, 32))      # Ho * Wo = 35, 160, 135, 640
FRAME_C = (256, 320, 512, 640, 1280)
FRAME_HW = (35, 40, 160, 290)


def candidates(mode):
    if mode == "gemm":
        for N in GEMM_N:
            for K in GEMM_K:
                for t in range(1, 400):
                    yield Shape(mode, 256 * t - 44, N, K, ())
    elif mode == "conv3x3":
        for C in CONV_C:
            for N in CONV_N:
                for H, W in CONV_HW:
                    for NF in range(1, 129):
                        if NF * H * W % 32:
                            yield Shape(mode, NF * H * W, N, 9 * C, (NF, H, W, C))
    else:
        for C in FRAME_C:
            for taps in (3, 5):
                for HW in FRAME_HW:
                    for F_ in range(1, 129):
                        if F_ * HW % 32:
                            yield Shape(mode, F_ * HW, C, taps * C, (F_, HW, C, taps))


@functools.lru_cache(maxsize=None)
def reachable(mode):
    """{class: the cheapest shape (fewest M N K) of the search that plans to it}."""
    best = {}
    for sh in candidates(mode):
        cls = class_of(mode, sh.M, sh.N, sh.K)
        if cls not in best or sh.M * sh.N * sh.K < best[cls].M * best[cls].N * best[cls].K:
            best[cls] = sh
    return best


# The (mode, bn) classes the search does NOT reach, pinned: split-K factors 2..16 of plans without a tail window, and
# tail_splits 1..16 of tail plans.  A tail window with tail_splits == 1 is unreachable by construction: two unsplit
# launches never take fewer waves than one (ceil(a) + ceil(b) >= ceil(a + b)) and the second costs a launch more.
# When the planner changes this test fails until the matrix below has been looked at again.
UNREACHED_SPLITS = {
    ('gemm', 64): (3, 6, 7, 8, 11, 12, 13, 15),
    ('gemm', 128): (11, 13, 15),
    ('gemm', 160): (8, 10, 11, 13, 14, 15),
    ('gemm', 192): (3, 4, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('gemm', 256): (11, 13, 14, 15, 16),
    ('gemm', 320): (6, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('conv3x3', 64): (2, 6, 8, 11, 12, 13),
    ('conv3x3', 128): (11, 13),
    ('conv3x3', 160): (8, 11, 13, 14),
    ('conv3x3', 192): (4, 7, 8, 9, 10, 11, 13, 14, 15, 16),
    ('conv3x3', 256): (11, 13, 15),
    ('conv3x3', 320): (11, 13, 15, 16),
    ('frame_conv', 64): (7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('frame_conv', 128): (8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('frame_conv', 160): (6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('frame_conv', 192): (3, 4, 6, 7, 8, 9, 11, 12, 13, 14, 15, 16),
    ('frame_conv', 256): (4, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('frame_conv', 320): (2, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
}
UNREACHED_TAILS = {
    ('gemm', 64): (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('gemm', 128): (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15),
    ('gemm', 160): (1, 2, 3, 4, 5, 6, 8, 11, 13, 14, 15, 16),
    ('gemm', 192): (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15),
    ('gemm', 256): (1, 11, 13, 15),
    ('gemm', 320): (1, 11, 13, 15),
    ('conv3x3', 64): (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('conv3x3', 128): (1, 2, 3, 4, 5, 8, 10, 11, 13, 14),
    ('conv3x3', 160): (1, 2, 3, 4, 8, 11, 12, 13, 14, 15),
    ('conv3x3', 192): (1, 2, 3, 4, 5, 6, 8, 10, 11, 13, 14),
    ('conv3x3', 256): (1, 8, 11, 13, 14),
    ('conv3x3', 320): (1, 8, 11, 13, 14),
    ('frame_conv', 64): (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('frame_conv', 128): (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('frame_conv', 160): (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('frame_conv', 192): (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('frame_conv', 256): (1, 2, 3, 4, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16),
    ('frame_conv', 320): (1, 9, 11, 12, 13, 14, 15, 16),
}


def matrix_classes():
    """The classes the GPU matrix runs: per (mode, bn) no split, s = 2, the smallest odd s and the largest s reached, and
    the smallest and the largest tail_splits reached."""
    out = []
    for mode in MODES:
        r = reachable(mode)
        for bn in BNS:
            splits = sorted(c[2] for c in r if c[1] == bn and c[3] == 0)
            tails = sorted(c[3] for c in r if c[1] == bn and c[3] > 0)
            odd = [s for s in splits if s % 2 and s > 1]
            want = {1, splits[-1], *odd[:1], *(s for s in splits if s == 2)}
            out += [(mode, bn, s, 0) for s in sorted(want)]
            out += [(mode, bn, 1, ts) for ts in sorted({*tails[:1], *tails[-1:]})]
    return out


def _cls_id(cls):
    mode, bn, s, ts = cls
    return f"{mode}-bn{bn}-" + (f"tail-x{ts}" if ts else (f"split-x{s}" if s > 1 else "full"))


# ------------------------------------------------------------------------------------------------ CPU: the finder
def test_finder_reaches_every_class_but_the_pinned():
    for mode in MODES:
        r = reachable(mode)
        for bn in BNS:
            splits = {c[2] for c in r if c[1] == bn and c[3] == 0}
            tails = {c[3] for c in r if c[1] == bn and c[3] > 0}
            assert 1 in splits, (mode, bn)
            assert tuple(s for s in range(2, 17) if s not in splits) == UNREACHED_SPLITS[(mode, bn)], (mode, bn, splits)
            assert tuple(t for t in range(1, 17) if t not in tails) == UNREACHED_TAILS[(mode, bn)], (mode, bn, tails)
    # the targets: every width with a split (s = 2, an odd s; the largest >= 14 where the families reach it), and
    # split-K tail windows for the 160- and 320-wide tiles
    for mode in MODES:
        for bn in BNS:
            reached = set(range(2, 17)) - set(UNREACHED_SPLITS[(mode, bn)])
            assert any(s % 2 for s in reached) and (2 in reached or (mode, bn) in {("conv3x3", 64), ("frame_conv", 320)})
    for mode in ("gemm", "conv3x3"):
        assert max(set(range(2, 17)) - set(UNREACHED_SPLITS[(mode, 64 if mode == "gemm" else 128)])) >= 14
        for bn in (160, 320):
            assert len(UNREACHED_TAILS[(mode, bn)]) < 16, (mode, bn)
    assert max(16 - len(UNREACHED_TAILS[("frame_conv", 320)]), 0) > 0
    assert all(1 in t for t in UNREACHED_TAILS.values())     # tail_splits == 1: never planned (see above)


def test_matrix_classes_cover_the_targets():
    classes = matrix_classes()
    assert len(set(classes)) == len(classes)
    for mode in MODES:
        mine = [c for c in classes if c[0] == mode]
        assert {c[1] for c in mine} == set(BNS)
        assert any(c[3] > 1 for c in mine if c[1] == 320)
    # frame convs with 3 and 5 taps on split and on tail plans
    frames = [(reachable("frame_conv")[c].geo[3], c) for c in classes if c[0] == "frame_conv"]
    for taps in (3, 5):
        assert any(t == taps and c[2] > 1 for t, c in frames) and any(t == taps and c[3] for t, c in frames), taps


def test_tail_plans_without_the_tail_switch_are_unsplit():
    """lavie_debug_set(5, 1) plans the same shape as one unsplit launch: so its rows of the main window run the same
    K-block order as the tail plan's main window, and must come out bit-identical (GPU test below)."""
    lib = _lib()
    for cls in matrix_classes():
        if cls[3]:
            sh = reachable(cls[0])[cls]
            lib.lavie_debug_set(5, 1)
            try:
                p = plan_of(sh.mode, sh.M, sh.N, sh.K)
            finally:
                lib.lavie_debug_set(5, 0)
            assert p[1:] == (1, 0, 1), (cls, p)
            # and the in-kernel split-K reduction plans with 64 KiB less workspace: the same classes
            assert class_of(sh.mode, sh.M, sh.N, sh.K) == cls
            assert plan_of(sh.mode, sh.M, sh.N, sh.K, ws=WORKSPACE_BYTES - TICKET_BYTES) == plan_of(sh.mode, sh.M, sh.N, sh.K)


# ------------------------------------------------------------------------------------------------ extra shapes
def _first(mode, N, K, pred, Ms):
    for M in Ms:
        if pred(plan_of(mode, M, N, K)):
            return M
    raise AssertionError(f"no {mode} shape N={N} K={K} with the wanted plan")


def ragged_shapes():
    """Plain GEMMs at N, K not multiples of 32 / 64, and two sources whose seam sits inside a K split."""
    out = []
    for N in (8, 72, 200):
        out.append((f"N{N}", Shape("gemm", 1000, N, 320, ())))
    for K in (8, 72, 200):
        out.append((f"K{K}", Shape("gemm", 2020, 320, K, ())))
    # K = 2888: 46 K blocks, the last 8 columns wide and inside the last split
    M = _first("gemm", 320, 2888, lambda p: p[1] > 1 and p[2] == 0, range(20, 4000, 32))
    out.append(("K2888-split", Shape("gemm", M, 320, 2888, ())))
    out.append(("K2888", Shape("gemm", 9700, 320, 2888, ())))
    # two sources: k0 = 640 (10 K blocks), k1 = 1000 (a partial last block): a split whose K range straddles block 10
    M = _first("gemm", 320, 1640, lambda p: p[1] > 1 and 10 % -(-26 // p[1]) != 0 and p[2] == 0, range(20, 4000, 32))
    out.append(("two-sources-split", Shape("gemm", M, 320, 1640, (640, 1000))))
    out.append(("two-sources", Shape("gemm", 3000, 320, 1640, (640, 1000))))
    return out


# conv3x3: (stride, padding) with NF * Ho * Wo not a multiple of 128; a time bias per item of F frames
CONV_EXTRA = [(stride, pad, NF, C, N) for stride in (1, 2) for pad in ((1, 1), (0, 1))
              for NF, C, N in ((6, 320, 320), (2, 1280, 640))]
CONV_EXTRA_HW = (19, 27)

GEGLU_M = (212, 1000, 256 * 75 - 44, 256 * 150 + 20)


def upsample_shapes():
    """(NF, H, W, C, N) of the fused upsample conv, one per tile width the planner gives it (planned as 4M rows, never
    split), with row counts that end inside a 256-row tile."""
    best = {}
    for H, W in ((5, 8), (10, 16), (20, 32), (3, 4), (10, 32)):
        for C in (128, 320, 640):
            for N in (256, 320, 640, 1280):
                for NF in range(1, 33):
                    M = NF * H * W
                    if (4 * M) % 256 == 0 or M % 32:
                        continue
                    bn = plan_of("conv3x3", 4 * M, N, 4 * C, ws=0)[0]
                    if bn not in best or M * N * C < best[bn][0]:
                        best[bn] = (M * N * C, (NF, H, W, C, N))
    return {bn: v[1] for bn, v in sorted(best.items())}


def test_extra_shapes_plan_what_they_are_for():
    shapes = dict(ragged_shapes())
    M = shapes["K2888-split"].M
    bn, s, tt, ts = plan_of("gemm", M, 320, 2888)
    assert s > 1 and (46 - 1) // -(-46 // s) == s - 1           # the partial last K block is in the last split
    bn, s, tt, ts = plan_of("gemm", shapes["two-sources-split"].M, 320, 1640)
    kbps = -(-26 // s)
    assert s > 1 and 10 % kbps != 0                              # a split straddles the seam of the two sources
    for M in GEGLU_M:
        assert plan_of("gemm", M, 1280, 320, geglu=True) == (256, 1, 0, 1)
    up = upsample_shapes()
    assert len(up) >= 4, up
    for stride, pad, NF, C, N in CONV_EXTRA:
        Ho, Wo = (conv_out_size(n, stride, pad) for n in CONV_EXTRA_HW)
        assert NF * Ho * Wo % 128, (stride, pad)


# ------------------------------------------------------------------------------------------------ GPU cases
DEV = "cuda"
RPB = 97                                 # time-bias rows per batch item of the GEMM cases: a boundary inside every tile
POISON = 0x7FA5                          # a NaN bit pattern around the out= views


def _g(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


class Case:
    """Inputs of one launch of `sh` with every epilogue: bias, a time bias whose batch boundaries fall inside tiles, a
    residual and an out= view inside a poisoned wider buffer (strided), and column statistics when N % 32 == 0."""

    def __init__(self, sh, seed=0, stride=1, padding=(1, 1), rows_per_batch=None, epilogue=True):
        self.sh, self.stride, self.padding, self.epilogue = sh, stride, padding, epilogue
        g = _g(seed)
        M, N, K = sh.M, sh.N, sh.K
        self.w = (torch.randn(N, K, generator=g, device=DEV) * K ** -0.5).to(BF16)
        if sh.mode == "gemm":
            k0, k1 = sh.geo or (K, 0)
            self.a = torch.randn(M, k0, generator=g, device=DEV).to(BF16)
            self.a2 = torch.randn(M, k1, generator=g, device=DEV).to(BF16) if k1 else None
            self.rows = lambda lo, hi: (self.a[lo:hi].to(F64) if self.a2 is None else
                                        torch.cat([self.a[lo:hi].to(F64), self.a2[lo:hi].to(F64)], 1))
            self.step = None
        elif sh.mode == "conv3x3":
            NF, H, W, C = sh.geo
            self.x = torch.randn(NF * H * W, C, generator=g, device=DEV).to(BF16)
            Ho, Wo = conv_out_size(H, stride, padding), conv_out_size(W, stride, padding)
            assert NF * Ho * Wo == M
            self.rows = conv_rows(self.x, NF, H, W, stride, padding)
            self.step = conv_step(Ho, Wo, K)
            F_ = NF // 2 if NF % 2 == 0 else 1                 # items of F frames: one time bias per item
            rows_per_batch = rows_per_batch or F_ * Ho * Wo
        else:
            F_, HW, C, taps = sh.geo
            pad = taps // 2 * HW
            self.xpad = torch.randn((F_ + taps - 1) * HW, C, generator=g, device=DEV).to(BF16)
            self.xpad[:pad] = 0
            self.xpad[self.xpad.shape[0] - pad:] = 0
            self.rows = lambda lo, hi: torch.cat([self.xpad[t * HW + lo:t * HW + hi] for t in range(taps)], 1).to(F64)
            self.step = None
        self.ep = {}
        if epilogue:
            self.rpb = rows_per_batch or RPB
            B = -(-M // self.rpb)
            self.ep["bias"] = torch.randn(N, generator=g, device=DEV)
            self.ep["row_bias"] = torch.randn(B, N, generator=g, device=DEV)
            self.ep["rows_per_batch"] = self.rpb
            res_full = torch.randn(M, N + 72, generator=g, device=DEV).to(BF16)
            self.ep["residual"] = res_full[:, 64:64 + N]
        self.stats = epilogue and N % 32 == 0

    def new_out(self):
        """A poisoned [M + 2, N + 96] buffer and the [M, N] view at (1, 32) the op writes."""
        M, N = self.sh.M, self.sh.N
        base = torch.empty((M + 2, N + 96), dtype=BF16, device=DEV)
        base.view(torch.int16).fill_(POISON)
        return base, base[1:M + 1, 32:32 + N]

    def run(self):
        """(out view, its buffer before and after, column sums or None)."""
        from lavie_b200 import ops
        base, out = self.new_out() if self.epilogue else (None, None)
        before = base.clone() if base is not None else None
        kw = dict(self.ep, out=out, stats=self.stats)
        sh = self.sh
        if sh.mode == "gemm":
            res = ops.gemm(self.a, self.w, a2=self.a2, **kw)
        elif sh.mode == "conv3x3":
            NF, H, W, C = sh.geo
            res = ops.conv3x3(self.x, NF, H, W, self.w, stride=self.stride, padding=self.padding, **kw)
        else:
            F_, HW, C, taps = sh.geo
            res = ops.frame_conv(self.xpad, taps, HW, self.w, **kw)
        torch.cuda.synchronize()
        return res, before, base, getattr(res, "_gn_colsums", None)

    def check(self, run, splits):
        res, before, base, cs = run
        a = {k: v for k, v in self.ep.items()}
        out = [gemm_check(res, self.rows, self.w, self.sh.K, a, splits, step=self.step)]
        if self.stats:
            assert cs is not None
            out.append(check_colsums(cs, res))
        if base is not None:
            out.append(check_outside_view(before, base, view_mask(base, res)))
        return out


@pytest.fixture(scope="module")
def fp64_refs():
    saved = tf32_off()
    yield
    tf32_restore(saved)


def _assert_ok(results, what):
    bad = [str(r) for r in results if not r.ok]
    assert not bad, f"{what}: " + "; ".join(bad)


def _report(what, results, extra=""):
    worst = max(r.worst for r in results)
    print(f"\n[gemm-plans] {what:44s} worst err/bound {worst:.3f} {extra}", end="")


def _written_stats(cs, N):
    """The entries of a col_stats buffer the producer writes (the others are never read and stay as allocated)."""
    written = colsum_expected(torch.zeros(1, N))[2]
    return cs[:, written]


@pytest.mark.gpu
@pytest.mark.parametrize("cls", matrix_classes(), ids=_cls_id)
def test_plan_class_against_fp64(cls, fp64_refs):
    from lavie_b200 import _lib as L
    lib = L.load()
    mode, bn, s, ts = cls
    sh = reachable(mode)[cls]
    plan = plan_of(mode, sh.M, sh.N, sh.K)          # on the device: planned with its SM count
    assert class_of(mode, sh.M, sh.N, sh.K) == cls, (cls, plan)
    splits = max(s, ts)
    case = Case(sh, seed=bn + s + ts)
    first = case.run()
    results = case.check(first, splits)
    _assert_ok(results, _cls_id(cls))
    # split-K order is fixed: a second run gives the same bits, outputs and column sums
    again = case.run()
    assert torch.equal(first[0], again[0])
    if case.stats:
        assert torch.equal(_written_stats(first[3], sh.N), _written_stats(again[3], sh.N))
    notes = []
    if ts:
        # one unsplit launch: within the bound, and the main window's rows bit for bit those of the tail plan
        main_rows = (-(-sh.M // 256) - plan[2]) * 256
        lib.lavie_debug_set(5, 1)
        try:
            assert plan_of(mode, sh.M, sh.N, sh.K)[1:] == (1, 0, 1)
            single = case.run()
        finally:
            lib.lavie_debug_set(5, 0)
        r5 = case.check(single, 1)
        _assert_ok(r5, _cls_id(cls) + " without the tail window")
        assert torch.equal(single[0][:main_rows], first[0][:main_rows]), "main window rows differ without the tail"
        results += r5
        notes.append(f"no-tail ok, {main_rows} main rows equal")
    if splits > 1:
        # in-kernel split-K reduction: the same planes summed in the same order
        # the tickets (one int per 128-row block and column tile) must fit their 64 KiB, else apply_plan falls back to
        # the reduction kernel and the comparison below would compare that kernel with itself
        assert -(-sh.M // 256) * 2 * -(-sh.N // bn) * 4 <= TICKET_BYTES
        lib.lavie_debug_set(7, 1)
        try:
            assert plan_of(mode, sh.M, sh.N, sh.K, ws=WORKSPACE_BYTES - TICKET_BYTES) == plan
            ik = case.run()
        finally:
            lib.lavie_debug_set(7, 0)
        r7 = case.check(ik, splits)
        _assert_ok(r7, _cls_id(cls) + " with the in-kernel split-K reduction")
        # the outputs are the same bits; the column sums are summed in the epilogue's order, not the statistics
        # reduction kernel's, so they only agree within the bound checked above
        assert torch.equal(ik[0], first[0]), "in-kernel split-K reduction output differs from the reduction kernel's"
        notes.append("in-kernel reduce: same output bits")
        if case.stats:
            # without statistics the split-K planes go through splitk_reduce_kernel instead of
            # splitk_reduce_stats_kernel: the same sum in the same order
            case.stats = False
            try:
                plain = case.run()
                rp = case.check(plain, splits)
            finally:
                case.stats = True
            _assert_ok(rp, _cls_id(cls) + " without column statistics")
            assert torch.equal(plain[0], first[0]), "the two split-K reduction kernels differ"
            results += rp
    _report(f"{_cls_id(cls)} M={sh.M} N={sh.N} K={sh.K}", results, "; ".join(notes))


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n, _ in ragged_shapes()])
def test_ragged_shapes_against_fp64(name, fp64_refs):
    sh = dict(ragged_shapes())[name]
    bn, s, tt, ts = plan_of("gemm", sh.M, sh.N, sh.K)
    case = Case(sh, seed=sh.N + sh.K)
    first = case.run()
    results = case.check(first, max(s, ts))
    _assert_ok(results, name)
    again = case.run()
    assert torch.equal(first[0], again[0])
    _report(f"ragged {name} M={sh.M} N={sh.N} K={sh.K} bn{bn} s{s} t{tt}x{ts}", results)


@pytest.mark.gpu
@pytest.mark.parametrize("stride,pad,NF,C,N", CONV_EXTRA)
def test_conv3x3_stride_padding_against_fp64(stride, pad, NF, C, N, fp64_refs):
    H, W = CONV_EXTRA_HW
    Ho, Wo = conv_out_size(H, stride, pad), conv_out_size(W, stride, pad)
    sh = Shape("conv3x3", NF * Ho * Wo, N, 9 * C, (NF, H, W, C))
    bn, s, tt, ts = plan_of("conv3x3", sh.M, N, sh.K)
    case = Case(sh, seed=stride + NF, stride=stride, padding=pad)
    first = case.run()
    results = case.check(first, max(s, ts))
    _assert_ok(results, f"conv3x3 stride {stride} pad {pad}")
    assert torch.equal(first[0], case.run()[0])
    _report(f"conv3x3 s{stride} pad{pad} NF={NF} C={C} N={N} bn{bn} s{s} t{tt}x{ts}", results)


@pytest.mark.gpu
@pytest.mark.parametrize("M", GEGLU_M)
def test_geglu_row_tails_against_fp64(M, fp64_refs):
    from lavie_b200 import ops
    N, K = 1280, 320
    assert plan_of("gemm", M, N, K, geglu=True) == (256, 1, 0, 1)
    g = _g(M)
    a = torch.randn(M, K, generator=g, device=DEV).to(BF16)
    w = (torch.randn(N, K, generator=g, device=DEV) * K ** -0.5).to(BF16)
    bias = torch.randn(N, generator=g, device=DEV)
    out = ops.gemm(a, w, bias=bias, geglu=True)
    results = [gemm_check(out, lambda lo, hi: a[lo:hi].to(F64), w, K, {"bias": bias, "geglu": True})]
    _assert_ok(results, f"geglu M={M}")
    assert torch.equal(out, ops.gemm(a, w, bias=bias, geglu=True))
    _report(f"geglu M={M} N={N} K={K} bn256", results)


@pytest.mark.gpu
@pytest.mark.parametrize("bn", sorted(upsample_shapes()))
def test_upsample_conv3x3_every_width_against_fp64(bn, fp64_refs):
    from lavie_b200 import ops
    NF, H, W, C, N = upsample_shapes()[bn]
    assert plan_of("conv3x3", 4 * NF * H * W, N, 4 * C, ws=0)[0] == bn
    g = _g(bn)
    x = torch.randn(NF * H * W, C, generator=g, device=DEV).to(BF16)
    w_ph = (torch.randn(4 * N, 4 * C, generator=g, device=DEV) * (4 * C) ** -0.5).to(BF16)
    bias = torch.randn(N, generator=g, device=DEV)
    out = ops.upsample_conv3x3(x, NF, H, W, w_ph, bias=bias, stats=True)
    a = {"NF": NF, "H": H, "W": W, "x": x, "w_phases": w_ph, "bias": bias}
    results = chk_upsample_conv3x3(a, out, {})
    if getattr(out, "_gn_colsums", None) is not None:
        results.append(check_colsums(out._gn_colsums, out, 4, (NF, H, W)))
    _assert_ok(results, f"upsample conv bn{bn}")
    again = ops.upsample_conv3x3(x, NF, H, W, w_ph, bias=bias, stats=True)
    assert torch.equal(out, again)
    _report(f"upsample_conv3x3 bn{bn} NF={NF} {H}x{W} C={C} N={N}", results)


# ------------------------------------------------------------------------------------------------ CPU: defects
# A large tail plan besides the cheapest: a defect confined to one row moves the whole-tensor rel-L2 by ~1 / sqrt(M)
LARGE_TAIL = Shape("gemm", 57300, 256, 2560, ())


def _tail_case(which):
    """A gemm tail plan (the cheapest of the search, or LARGE_TAIL), its fp64 result with every epilogue (on the CPU),
    and its bf16 rounding: the output a correct kernel could have written."""
    if which == "cheapest":
        r = reachable("gemm")
        sh = r[min((c for c in r if c[3]), key=lambda c: r[c].M * r[c].N * r[c].K)]
    else:
        sh = LARGE_TAIL
    bn, s, tt, ts = plan_of("gemm", sh.M, sh.N, sh.K)
    assert tt > 0 and ts > 1, (sh, bn, s, tt, ts)
    g = torch.Generator().manual_seed(1)
    M, N, K = sh.M, sh.N, sh.K
    a = torch.randn(M, K, generator=g).to(BF16)
    w = (torch.randn(N, K, generator=g) * K ** -0.5).to(BF16)
    ep = {"bias": torch.randn(N, generator=g), "row_bias": torch.randn(-(-M // RPB), N, generator=g),
          "rows_per_batch": RPB, "residual": torch.randn(M, N, generator=g).to(BF16)}
    acc, S = mm_abs(a, w, step=4096)
    ref, S = epilogue_ref(acc, S, 0, ep["bias"], ep["row_bias"], RPB, ep["residual"])
    bound = U * ref.abs() + c_gemm(K, ts) * (1 + U) * S
    row0 = (-(-M // 256) - tt) * 256
    return dict(sh=sh, a=a, w=w, ep=ep, acc=acc, ref=ref, bound=bound, row0=row0, splits=ts, which=which)


@pytest.fixture(scope="module", params=["cheapest", "large"])
def tail_case(request):
    return _tail_case(request.param)


def _flags(c, out, cs=None):
    """(element-wise check ok, rel-L2 < 4e-3 ok) of an output (or of column sums `cs` of the correct output)."""
    if cs is not None:
        exp = colsum_expected(c["out"])[0]
        return check_colsums(cs, c["out"]).ok, rel_l2(cs, exp) < 4e-3
    cmp = Cmp("gemm", out, c["ref"], c["bound"], rel_max=REL_ROUND)
    return cmp.ok, rel_l2(out.to(F64), c["ref"]) < 4e-3


# defect -> whether rel-L2 < 4e-3 alone passes it (the whole-tensor check of tests/test_kernels_gpu.py), at the
# cheapest tail plan (M = 19156) and at LARGE_TAIL (M = 57300).  The wrong-batch row moves one row by O(1) of the
# output's scale and one slab of column sums is one of M / 32: rel-L2 sees both at the smaller M, not at the larger one.
# The other two move a whole window or every element.
DEFECTS = {"row bias of the wrong batch at the tail window's first row": (False, True),
           "last 8 K columns dropped": (False, False),
           "residual added twice in one split plane of the tail window": (False, False),
           "one column-statistics slab shifted by one": (False, True)}


def test_correct_tail_result_passes(tail_case):
    c = tail_case
    c["out"] = c["ref"].to(BF16)
    assert _flags(c, c["out"]) == (True, True)
    cs = colsum_expected(c["out"])[0].float()
    assert _flags(c, None, cs) == (True, True)


@pytest.mark.parametrize("defect", list(DEFECTS))
def test_each_plan_defect_is_flagged(defect, tail_case):
    c = tail_case
    out = c["ref"].to(BF16)
    c["out"] = out
    row0, rpb = c["row0"], RPB
    rb = c["ep"]["row_bias"].to(F64)
    cs = None
    bad = c["ref"].clone()
    if defect.startswith("row bias"):
        # row0 dropped from the batch index: row row0 takes the bias of batch 0
        bad[row0] += rb[0] - rb[row0 // rpb]
    elif defect.startswith("last 8 K"):
        K = c["sh"].K
        bad -= c["a"][:, K - 8:].to(F64) @ c["w"][:, K - 8:].to(F64).t()
    elif defect.startswith("residual"):
        # one split plane of the tail window carries the residual too: added twice over the window's rows
        bad[row0:] += c["ep"]["residual"][row0:].to(F64)
    else:
        cs = colsum_expected(out)[0].float()
        slab = row0 // 32 + 1
        cs[slab] = cs[slab + 1]
        bad = None
    if bad is not None:
        elem_ok, rel_ok = _flags(c, bad.to(BF16))
    else:
        elem_ok, rel_ok = _flags(c, None, cs)
    print(f"\n[gemm-plans] defect '{defect}' (M={c['sh'].M}): element-wise {'PASSES' if elem_ok else 'flagged'}, "
          f"rel-L2 < 4e-3 {'passes' if rel_ok else 'flags'}", end="")
    assert not elem_ok
    assert rel_ok == DEFECTS[defect][c["which"] == "large"]
