"""Element-by-element grading of the tensor-core kernels against fp64 products of the exact bf16 operands they consume.

The other tensor-core tests compare with fp64 on the UNROUNDED inputs, so their tolerances must absorb the bf16 rounding of
the operands, and they normalise the worst error by max|ref|.  Here the reference is built from the operand planes the
kernel read (bf16x3: hi_a hi_b + hi_a lo_b + lo_a hi_b, the lo lo term is dropped by design; bf16: hi_a hi_b), and every
element is held to its own bound, so that an error confined to a tail tile, one CTA of a pair or one epilogue addend
cannot hide behind the largest elements.  The split into planes is pinned bit for bit first.
"""
import math

import pytest
import torch

from dostransformer_b200 import _lib as L
from dostransformer_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda"

# fp32 accumulation of exact bf16 products: ~50x the expected accumulation error at K = 1024, and smaller than one
# dropped hi*lo term on a single 64-wide k-tile (which is ~2^-8 of that tile's share of |A||B|)
C_PROD = 2.0 ** -18
# one fp32 rounding (2^-24) per epilogue addend, with a factor 2 for the rounding of the sum it is added to
C_ADD = 2.0 ** -23
TINY = 1e-30
# hi + lo of an fp32 value v: two round-to-nearest steps to 8 significant bits, |v - hi - lo| <= 2^-8 |v - hi| <= 2^-16 |v|;
# hi alone: |v - hi| <= 2^-8 |v|
SPLIT_REP = {"bf16x3": 2.0 ** -16, "bf16": 2.0 ** -8}
PRECS = ["bf16x3", "bf16"]
MODES = [(L.KC, L.KC), (L.KC, L.MC), (L.MC, L.MC)]
ACTS = [L.ACT_NONE, L.ACT_RELU, L.ACT_LEAKY, L.ACT_PRELU]

# GEMM shapes (M, N, K).  Boundaries: BM = 128, BK = 64, bn = 64 / 128 / 256 for N <= 64 / <= 128 / larger, CTA pairs
# (256 x 256 tiles) when M > 128 and N > 128 (M = 129: the second CTA holds one row), TMA-store epilogue only for M, N >= 32.
# Every M meets an N on both sides of 128; every K appears in a pair launch and in a single-CTA launch.
GEMM_SHAPES = [
    (1, 4, 8), (1, 260, 1024),
    (32, 32, 56), (32, 132, 64),
    (127, 60, 72), (127, 256, 192),
    (128, 64, 1024), (128, 516, 8),
    (129, 68, 56), (129, 260, 1024), (129, 132, 192),
    (255, 128, 64), (255, 132, 8),
    (256, 4, 192), (256, 256, 56),
    (257, 32, 8), (257, 516, 72),
    (511, 60, 1024), (511, 260, 64),
]
# per-problem row counts of the ragged GEMMs (tails around the 32-row epilogue warps and the 64 / 128-row tiles)
RAGGED_COUNTS = [1, 31, 32, 33, 64, 65, 128, 129]
# fused attention, dense: (S, Lq, Lk, H, q scale).  128-query tiles, phase-A MMA width NB in {32, 64, 128, 256} chosen by
# the key count, 32-key phase-B chunks, at most 256 keys; a case with more work items than SMs; peaked scores (q x8 .. x16)
FUSED_DENSE = [
    (3, 1, 1, 64, 1.0), (2, 127, 31, 128, 1.0), (2, 128, 32, 192, 1.0), (2, 129, 33, 256, 1.0), (2, 201, 63, 64, 1.0),
    (1, 300, 64, 128, 1.0), (2, 127, 65, 192, 1.0), (2, 128, 127, 256, 1.0), (2, 129, 128, 64, 1.0), (2, 201, 129, 128, 1.0),
    (1, 300, 255, 192, 1.0), (2, 201, 256, 256, 1.0), (300, 129, 33, 128, 1.0),
    (2, 201, 129, 64, 12.0), (2, 129, 256, 128, 16.0), (2, 127, 33, 256, 8.0),
]
# fused attention, ragged (make_edos_batch sizes: a crystal has size + 1 atoms and size + 2 keys with the phantom):
# key counts straddling 32, 64 and 128 in one batch, a 1-atom crystal, the largest crystal (phantom multiplicity 0)
FUSED_RAGGED = [
    ([29, 30, 31, 61, 62, 63, 125, 126, 127, 0], 70, 128, 1, 1.0),
    ([0, 254, 40, 100], 129, 64, 2, 1.0),
    ([29, 30, 31, 61, 62, 63, 125, 126, 127, 0], 33, 256, 2, 12.0),
    ([5, 0, 93, 17], 201, 192, 1, 16.0),
]


# ----------------------------------------------------------------------------------------------------------------- helpers
def _rand(*shape, seed, scale=1.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randn(*shape, generator=g, device=DEV) * scale


def split_ref(x):
    """Round-to-nearest-even hi / lo split of fp32 x, as torch computes it."""
    hi = x.to(torch.bfloat16)
    return hi, (x - hi.float()).to(torch.bfloat16)


def bits(t):
    return t.contiguous().view(torch.int16)


def feed(hi, lo, prec):
    """The fp64 operand the tensor cores see: (hi, lo) of bf16x3, hi of bf16 (lo is None or ignored)."""
    return hi.double(), (lo.double() if (prec == "bf16x3" and lo is not None) else None)


def feed_product(a, b, prec):
    """(fp64 product the kernel computes, fp64 |A| |B|) for feeds a = (hi, lo) [M, K], b = (hi, lo) [K, N]."""
    (ah, al), (bh, bl) = a, b
    prod = ah @ bh
    if prec == "bf16x3":
        prod = prod + ah @ bl + al @ bh
        return prod, (ah + al).abs() @ (bh + bl).abs()
    return prod, ah.abs() @ bh.abs()


def planes_feed(pl, prec, cols=None):
    cols = pl.cols if cols is None else cols
    return feed(pl.hi[:, :cols], pl.lo[:, :cols] if pl.lo is not None else None, prec)


def pair_t(pair):
    return pair[0].t(), (pair[1].t() if pair[1] is not None else None)


def pair_rows(pair, rows):
    return pair[0][rows], (pair[1][rows] if pair[1] is not None else None)


def logical_feed(pl, mode, prec):
    """Feed of a GEMM operand stored in `mode` layout, as its logical [rows, K] matrix."""
    f = planes_feed(pl, prec)
    return f if mode == L.KC else pair_t(f)


def bound(absprod=None, addends=()):
    """Per-element bound of a contraction: 2^-18 (|A| |B|)_ij + 2^-23 sum |epilogue addends_ij| + 1e-30."""
    b = TINY
    if absprod is not None:
        b = b + C_PROD * absprod
    for t in addends:
        b = b + C_ADD * t.double().abs()
    return b


def check(name, got, ref, bnd):
    """Asserts |got - ref| <= bnd element by element; names the worst element and its ratio to the bound."""
    got, ref = got.double(), ref.double()
    bnd = torch.as_tensor(bnd, dtype=torch.float64, device=got.device).expand_as(ref)
    ratio = ((got - ref).abs() / bnd).nan_to_num(nan=float("inf"))
    worst = ratio.max().item() if ratio.numel() else 0.0
    if worst > 1.0:
        idx = tuple(int(i) for i in torch.unravel_index(ratio.argmax(), ratio.shape))
        raise AssertionError(f"{name}: worst element {idx}: got {got[idx].item():.9g}, ref {ref[idx].item():.9g}, "
                             f"bound {bnd[idx].item():.3g}, ratio {worst:.3g}; {(ratio > 1).sum().item()} elements over")


def check_planes_of(name, pl, x, with_lo):
    """Planes of fp32 x [rows, cols] must be its RNE split bit for bit."""
    hi, lo = split_ref(x)
    c = x.shape[1]
    assert torch.equal(bits(pl.hi[:, :c]), bits(hi)), f"{name}: hi plane differs from bf16(x) at " \
        f"{(bits(pl.hi[:, :c]) != bits(hi)).nonzero()[:4].tolist()}"
    if with_lo:
        assert torch.equal(bits(pl.lo[:, :c]), bits(lo)), f"{name}: lo plane differs from bf16(x - hi) at " \
            f"{(bits(pl.lo[:, :c]) != bits(lo)).nonzero()[:4].tolist()}"


def _act_ref(v, act, slope):
    if act == L.ACT_NONE:
        return v
    return torch.where(v > 0, v, (0.0 if act == L.ACT_RELU else slope) * v)


def _stored(rows, cols, mode, seed):
    """A GEMM operand of logical shape [rows, K=cols] in its storage layout (KC: [rows, K], MC: [K, rows])."""
    return _rand(rows, cols, seed=seed) if mode == L.KC else _rand(cols, rows, seed=seed)


def _logical(t, mode):
    return t if mode == L.KC else t.t()


@pytest.fixture
def small_on_tc(monkeypatch):
    """gemm_raw sends small fp32 problems to the FMA pipe; switched off so that the tensor-core kernel is graded."""
    monkeypatch.setenv("DOST_NO_SMALL_FMA", "1")
    L.reload_switches()
    yield
    monkeypatch.delenv("DOST_NO_SMALL_FMA")
    L.reload_switches()


def _raw_on_tc(M, N, K):
    """gemm_tc.cu's own predicate: smaller problems stay on the FMA pipe."""
    return M >= 64 and N >= 16 and M * N * K >= (1 << 21)


# ------------------------------------------------------------------------------------------- 1. the split, bit for bit
SPECIALS = [0.0, -0.0, 1e-40, -1e-40, 1.4e-45, -2.9e-39, 1.1754942e-38, 3.3e38, -3.3e38, 1e38, 1.0 + 2 ** -8,
            -(1.0 + 3 * 2 ** -8), 1.0 + 2 ** -16 + 2 ** -8, 65504.0, -7.0e-20]


def _special_matrix(rows, cols, seed):
    x = _rand(rows, cols, seed=seed) * torch.exp2(_rand(rows, cols, seed=seed + 1) * 8)
    sp = torch.tensor(SPECIALS, device=DEV)
    flat = x.view(-1)
    flat[: min(flat.numel(), 3 * sp.numel())] = sp.repeat(3)[: min(flat.numel(), 3 * sp.numel())]
    return x


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("rows,cols,ld", [(37, 1, 1), (5, 7, 7), (64, 13, 40), (300, 101, 104), (17, 256, 259), (1, 9, 9)])
def test_split_planes_bitwise(prec, rows, cols, ld):
    base = _special_matrix(rows, ld, seed=rows + cols)
    x = base[:, :cols]                                  # row-strided view: ld > cols
    with_lo = prec == "bf16x3"
    with ops.precision(prec):
        pl = ops.split_planes(x)
        plc, _ = ops.split_planes_colsum(x)
        w = base.clone()[:, :cols]
        ops.refresh_weight_planes([w])
        plm = ops.weight_planes(w)
    for name, p in (("split_planes", pl), ("split_planes_colsum", plc), ("split_planes_multi", plm)):
        assert (p.lo is not None) == with_lo, name
        check_planes_of(name, p, x, with_lo)
        pad = p.hi[:, cols:]
        assert torch.all(bits(pad) == 0), f"{name}: hi pad columns [cols, ld) not zero"
        if with_lo:
            assert torch.all(bits(p.lo[:, cols:]) == 0), f"{name}: lo pad columns [cols, ld) not zero"


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("W,prelu", [(128, False), (256, True), (512, False), (1024, True)])
def test_ln_planes_equal_split_of_fp32(prec, W, prelu):
    """ln_fwd_planes / ln_bwd_planes write planes and fp32 of the same values: the planes are split(y), split(dx)."""
    M = 333
    x = _rand(M, W, seed=W) * 2 + 0.3
    g, b, dy, dres = _rand(W, seed=1), _rand(W, seed=2), _rand(M, W, seed=3), _rand(M, W, seed=4)
    slope = torch.tensor([0.25], device=DEV) if prelu else None
    with ops.precision(prec):
        y, pl, stats = ops.ln_fwd_planes(x, g, b, slope, want_y=True)
        dx, dxp, *_ = ops.ln_bwd_planes(dy, x, stats, g, b, slope, dres=dres, want_planes=True)
    check_planes_of("ln_fwd_planes", pl, y, prec == "bf16x3")
    check_planes_of("ln_bwd_planes", dxp, dx, prec == "bf16x3")


# ------------------------------------------------------------------------------------------------------- 2. GEMM sweep
def _gemm_planes_case(M, N, K, prec, am, bm, act, tma, seed):
    lo = prec == "bf16x3"
    a_st, b_st = _stored(M, K, am, seed), _stored(N, K, bm, seed + 1)
    bias, res = _rand(N, seed=seed + 2), _rand(M, N, seed=seed + 3)
    div = 3
    rb = _rand((M + div - 1) // div, N, seed=seed + 4)
    slope = 0.3
    pslope = torch.tensor([slope], device=DEV)
    saved = _rand(M, N, seed=seed + 5)
    c0 = _rand(M, N, seed=seed + 6)
    ldc = N + 4
    with ops.precision(prec):
        ap, bp, sp = ops.split_planes(a_st), ops.split_planes(b_st), ops.split_planes(saved)
        # (1) every output of a forward Linear in one launch: fp32 result, pre-activation copy, planes, gate bits
        out = torch.full((M, ldc), float("nan"), device=DEV)
        pre = torch.full((M, N), float("nan"), device=DEV)
        op = ops.empty_planes(M, N, DEV, with_lo=lo)
        for t in op.tensors():
            if t is not None:
                t.fill_(float("nan"))
        gate = None
        if tma and M >= 32 and N % 32 == 0:
            gate = torch.full((N // 32, M), -1, dtype=torch.int32, device=DEV)
        ops.gemm_planes(M=M, N=N, K=K, a=[ap], a_mode=am, b=bp, b_mode=bm, out=out[:, :N], bias=bias, rowbias=rb, rowbias_div=div,
                        act=act, act_slope=slope if act == L.ACT_LEAKY else 0.0,
                        prelu_slope=pslope if act == L.ACT_PRELU else None, out_pre=pre, residual=res, out_planes=op,
                        out_gate=gate)
        # (2) accumulate into an existing output with the act' mask read from a saved plane
        out2 = torch.full((M, ldc), float("nan"), device=DEV)
        out2[:, :N] = c0
        ops.gemm_planes(M=M, N=N, K=K, a=[ap], a_mode=am, b=bp, b_mode=bm, out=out2[:, :N], accumulate=True, dact=sp,
                        dact_slope=0.25)
        # (3) the FFN input-gradient shape: act' mask, fp32 + planes + fused column sums
        out3 = torch.full((M, N), float("nan"), device=DEV)
        op3 = ops.empty_planes(M, N, DEV, with_lo=lo)
        cs = torch.full((N,), float("nan"), device=DEV)
        ops.gemm_planes(M=M, N=N, K=K, a=[ap], a_mode=am, b=bp, b_mode=bm, out=out3, out_planes=op3, dact=sp, dact_slope=0.0,
                        colsum_out=cs)
    tag = f"planes {prec} M={M} N={N} K={K} a={'KC' if am == L.KC else 'MC'} b={'KC' if bm == L.KC else 'MC'} " \
          f"{'tma' if tma else 'reg'}-epi"
    prod, absprod = feed_product(logical_feed(ap, am, prec), pair_t(logical_feed(bp, bm, prec)), prec)
    rbe = rb.double().repeat_interleave(div, 0)[:M]
    v = prod + bias.double() + rbe
    check(f"{tag}: out_pre", pre, v, bound(absprod, (bias.expand(M, N), rbe)))
    ref = _act_ref(v, act, slope) + res.double()
    check(f"{tag}: out", out[:, :N], ref, bound(absprod, (bias.expand(M, N), rbe, res)))
    assert torch.isnan(out[:, N:]).all(), f"{tag}: out columns past N were written"
    check_planes_of(f"{tag}: out_planes vs out", op, out[:, :N], lo)
    # plane pad columns [N, ld): the register epilogue leaves them alone; with N % 8 == 4 the TMA store fills them with the
    # zeros of the out-of-range columns, up to the 16-byte row end (the zero-filled pad of dost_split_planes).  Anything
    # else there is a stray write.
    for t in op.tensors():
        if t is not None and t.shape[1] > N:
            pad = t[:, N:].float()
            assert (torch.isnan(pad) | (pad == 0)).all(), f"{tag}: plane pad columns hold values other than 0"
    if gate is not None:
        got = ((gate.t().reshape(M, N // 32, 1) >> torch.arange(32, device=DEV, dtype=torch.int32)) & 1).reshape(M, N).bool()
        assert torch.equal(got, pre > 0), f"{tag}: gate bits differ from (pre-activation > 0)"
    mask = torch.where(sp.hi[:, :N].float() > 0, 1.0, 0.25).double()
    check(f"{tag}: accumulate + dact", out2[:, :N], c0.double() + prod * mask, bound(absprod, (c0,)))
    assert torch.isnan(out2[:, N:]).all(), f"{tag}: accumulating store wrote past N"
    mask0 = torch.where(sp.hi[:, :N].float() > 0, 1.0, 0.0).double()
    check(f"{tag}: dact (relu')", out3, prod * mask0, bound(absprod))
    check_planes_of(f"{tag}: dact planes vs out", op3, out3, lo)
    # fixed-order fp32 column sums of the stored values: 32-row partials, then a reduction over <= 16 of them (< 64 roundings)
    check(f"{tag}: colsum_out", cs, out3.double().sum(0), 2.0 ** -18 * out3.double().abs().sum(0) + TINY)


def _gemm_raw_case(M, N, K, prec, am, bm, act, seed):
    a_st, b_st = _stored(M, K, am, seed), _stored(N, K, bm, seed + 1)
    bias, res, c0 = _rand(N, seed=seed + 2), _rand(M, N, seed=seed + 3), _rand(M, N, seed=seed + 6)
    slope = 0.3
    pslope = torch.tensor([slope], device=DEV)
    P = L.PRECISIONS[prec]
    ldc = N + 4
    out = torch.full((M, ldc), float("nan"), device=DEV)
    pre = torch.full((M, N), float("nan"), device=DEV)
    ops.gemm_raw(M=M, N=N, K=K, a=[(a_st, None)], a_mode=am, b=b_st, b_mode=bm, out=out[:, :N], ldc=ldc, bias=bias, act=act,
                 act_slope=slope if act == L.ACT_LEAKY else 0.0, prelu_slope=pslope if act == L.ACT_PRELU else None,
                 out_pre=pre, residual=res, prec=P)
    out2 = c0.clone()
    ops.gemm_raw(M=M, N=N, K=K, a=[(a_st, None)], a_mode=am, b=b_st, b_mode=bm, out=out2, accumulate=True, prec=P)
    tag = f"raw {prec} M={M} N={N} K={K} a={'KC' if am == L.KC else 'MC'} b={'KC' if bm == L.KC else 'MC'}"
    # the split the producer warps do (convert4): hi = RNE bf16(x), lo = RNE bf16(x - hi)
    A = feed(*split_ref(_logical(a_st, am)), prec)
    B = feed(*split_ref(_logical(b_st, bm).t()), prec)
    prod, absprod = feed_product(A, B, prec)
    v = prod + bias.double()
    check(f"{tag}: out_pre", pre, v, bound(absprod, (bias.expand(M, N),)))
    check(f"{tag}: out", out[:, :N], _act_ref(v, act, slope) + res.double(), bound(absprod, (bias.expand(M, N), res)))
    assert torch.isnan(out[:, N:]).all(), f"{tag}: out columns past N were written"
    check(f"{tag}: accumulate", out2, c0.double() + prod, bound(absprod, (c0,)))


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
def test_gemm_sweep(M, N, K, monkeypatch, small_on_tc):
    for i, prec in enumerate(PRECS):
        for j, (am, bm) in enumerate(MODES):
            act = ACTS[(i + j + M + N) % 4]
            seed = 1000 * i + 100 * j + M + N + K
            for tma in (True, False):
                monkeypatch.setenv("DOST_GEMM_TMA_EPI", "1" if tma else "0")
                for epi16 in (("2", "0") if (tma and M > 128 and N > 128) else ("1",)):
                    monkeypatch.setenv("DOST_GEMM_EPI16", epi16)
                    _gemm_planes_case(M, N, K, prec, am, bm, act, tma, seed)
            if _raw_on_tc(M, N, K):
                _gemm_raw_case(M, N, K, prec, am, bm, act, seed)


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("M,N,K", [(129, 132, 72), (256, 260, 1024), (64, 68, 200), (300, 64, 3001)])
def test_gemm_split_k(prec, M, N, K, small_on_tc):
    """Deterministic split-K: slices end on 64-wide k-tiles, so K = 72 in 3 or 7 slices gives a slice shorter than a k-tile
    and empty trailing slices."""
    for am, bm in MODES:
        a_st, b_st = _stored(M, K, am, M + K), _stored(N, K, bm, N + K)
        c0 = _rand(M, N, seed=7)
        with ops.precision(prec):
            ap, bp = ops.split_planes(a_st), ops.split_planes(b_st)
        A = feed(*split_ref(_logical(a_st, am)), prec)
        B = feed(*split_ref(_logical(b_st, bm).t()), prec)
        prod, absprod = feed_product(A, B, prec)
        for split in (1, 3, 7):
            tag = f"split_k={split} {prec} M={M} N={N} K={K} a={am} b={bm}"
            out = torch.full((M, N), float("nan"), device=DEV)
            with ops.precision(prec):
                ops.gemm_planes(M=M, N=N, K=K, a=[ap], a_mode=am, b=bp, b_mode=bm, out=out, split_k=split)
            check(f"planes {tag}", out, prod, bound(absprod))
            acc = c0.clone()
            with ops.precision(prec):
                ops.gemm_planes(M=M, N=N, K=K, a=[ap], a_mode=am, b=bp, b_mode=bm, out=acc, split_k=split, accumulate=True)
            check(f"planes accumulate {tag}", acc, c0.double() + prod, bound(absprod, (c0,)))
            if _raw_on_tc(M, N, K):
                out = torch.full((M, N), float("nan"), device=DEV)
                ops.gemm_raw(M=M, N=N, K=K, a=[(a_st, None)], a_mode=am, b=b_st, b_mode=bm, out=out, split_k=split,
                             prec=L.PRECISIONS[prec])
                check(f"raw {tag}", out, prod, bound(absprod))


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("M,N,K", [(201, 68, 72), (201, 260, 192), (129, 4, 64)])
def test_gemm_batched_tails(prec, M, N, K, small_on_tc):
    """Independent problems with M and N tails (3-D tensor maps; a box never spans two problems), bias + residual, an
    output pitch wider than N whose extra columns must stay untouched."""
    S = 5
    lo = prec == "bf16x3"
    a, b = _rand(S * M, K, seed=1), _rand(S * N, K, seed=2)
    bias, res = _rand(N, seed=3), _rand(S * M, N, seed=4)
    ldc = N + 4
    with ops.precision(prec):
        ap, bp = ops.split_planes(a), ops.split_planes(b)
        out = torch.full((S * M, ldc), float("nan"), device=DEV)
        ops.gemm_planes(M=M, N=N, K=K, a=[ap], a_mode=L.KC, b=bp, b_mode=L.KC, out=out, ldc=ldc, bias=bias, residual=res,
                        batch=S, a_bstride=M * ap.ld, b_bstride=N * bp.ld, c_bstride=M * ldc, res_bstride=M * N, ld_res=N)
    A, B = planes_feed(ap, prec), planes_feed(bp, prec)
    for z in range(S):
        rs, ns = slice(z * M, (z + 1) * M), slice(z * N, (z + 1) * N)
        prod, absprod = feed_product(pair_rows(A, rs), pair_t(pair_rows(B, ns)), prec)
        ref = prod + bias.double() + res[rs].double()
        check(f"batched {prec} M={M} N={N} K={K} problem {z}", out[rs, :N], ref, bound(absprod, (bias.expand(M, N), res[rs])))
    assert torch.isnan(out[:, N:]).all(), "batched: columns past N were written"
    if _raw_on_tc(M, N, K):
        out = torch.full((S, M, N), float("nan"), device=DEV)
        ops.gemm_raw(M=M, N=N, K=K, a=[(a, None)], a_mode=L.KC, b=b, b_mode=L.KC, out=out, batch=S, a_bstride=M * K,
                     b_bstride=N * K, c_bstride=M * N, prec=L.PRECISIONS[prec])
        A, B = feed(*split_ref(a), prec), feed(*split_ref(b), prec)
        for z in range(S):
            rs, ns = slice(z * M, (z + 1) * M), slice(z * N, (z + 1) * N)
            prod, absprod = feed_product(pair_rows(A, rs), pair_t(pair_rows(B, ns)), prec)
            check(f"raw batched {prec} M={M} N={N} K={K} problem {z}", out[z], prod, bound(absprod))


@pytest.mark.parametrize("prec", PRECS)
def test_gemm_ragged(prec):
    """Ragged problems of the cross attention: per-problem row offsets into one B plane (K-major and MN-major use) and a
    per-problem output row offset / row limit; nothing past a problem's row limit is written."""
    lo = prec == "bf16x3"
    n = torch.tensor(RAGGED_COUNTS)
    S = len(RAGGED_COUNTS)
    off = torch.cat([torch.zeros(1, dtype=torch.long), n.cumsum(0)])
    Ntot = int(off[-1])
    npad = ops._pad8(int(n.max()))
    Mq, H = 70, 64
    keys, q = _rand(Ntot, H, seed=1), _rand(S * Mq, H, seed=2)
    p = torch.rand(S, Mq, npad, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
    for z in range(S):
        p[z, :, n[z]:] = 0
    offd, nd = off[:-1].to(torch.int32).to(DEV), n.to(torch.int32).to(DEV)
    with ops.precision(prec):
        kp, qp, pp = ops.split_planes(keys), ops.split_planes(q), ops.split_planes(p.view(S * Mq, npad))
        sc = torch.full((S * Mq, npad), float("nan"), device=DEV)
        ops.gemm_planes(M=Mq, N=npad, K=H, a=[qp], a_mode=L.KC, b=kp, b_mode=L.KC, b_rows=Ntot, out=sc, batch=S,
                        a_bstride=Mq * qp.ld, c_bstride=Mq * npad, b_rowoff=offd)
        o = torch.full((S * Mq, H), float("nan"), device=DEV)
        ops.gemm_planes(M=Mq, N=H, K=npad, a=[pp], a_mode=L.KC, b=kp, b_mode=L.MC, b_rows=Ntot, out=o, batch=S,
                        a_bstride=Mq * pp.ld, c_bstride=Mq * H, b_rowoff=offd)
        extra = 5
        dk = torch.full((Ntot + extra, H), 7.0, device=DEV)
        ops.gemm_planes(M=npad, N=H, K=Mq, a=[pp], a_mode=L.MC, b=qp, b_mode=L.MC, out=dk, batch=S, a_bstride=Mq * pp.ld,
                        b_bstride=Mq * qp.ld, c_rowoff=offd, c_rowlim=nd)
    Kh, Kl = planes_feed(kp, prec)
    Qh, Ql = planes_feed(qp, prec)
    Ph, Pl = planes_feed(pp, prec)
    zpad = torch.zeros(npad, H, dtype=torch.float64, device=DEV)
    Khp, Klp = torch.cat([Kh, zpad]), (torch.cat([Kl, zpad]) if lo else None)     # rows past the plane read as zero
    for z in range(S):
        rs = slice(z * Mq, (z + 1) * Mq)
        kr = slice(int(off[z]), int(off[z]) + npad)
        kz = (Khp[kr], Klp[kr] if lo else None)
        prod, absprod = feed_product((Qh[rs], Ql[rs] if lo else None), (kz[0].t(), kz[1].t() if lo else None), prec)
        check(f"ragged scores {prec} problem {z} (n={int(n[z])})", sc[rs], prod, bound(absprod))
        prod, absprod = feed_product((Ph[rs], Pl[rs] if lo else None), kz, prec)
        check(f"ragged P K {prec} problem {z} (n={int(n[z])})", o[rs], prod, bound(absprod))
        prod, absprod = feed_product((Ph[rs].t(), Pl[rs].t() if lo else None), (Qh[rs], Ql[rs] if lo else None), prec)
        nz = int(n[z])
        check(f"ragged dK {prec} problem {z} (n={nz})", dk[int(off[z]):int(off[z]) + nz], prod[:nz], bound(absprod[:nz]))
    assert torch.all(dk[Ntot:] == 7.0), "ragged output: rows past the last problem's row limit were written"


@pytest.mark.parametrize("prec", PRECS)
def test_gemm_concat_segments(prec, small_on_tc):
    """Concatenated A segments (64-aligned widths) with a row-group bias, on both tensor-core GEMMs."""
    lo = prec == "bf16x3"
    M, N, widths = 257, 132, (64, 128, 64)
    K = sum(widths)
    segs = [_rand(M, w, seed=10 + i) for i, w in enumerate(widths)]
    w = _rand(N, K, seed=20)
    rb = _rand((M + 4) // 5, N, seed=21)
    with ops.precision(prec):
        sp = [ops.split_planes(s) for s in segs]
        wp = ops.split_planes(w)
        out = torch.full((M, N), float("nan"), device=DEV)
        op = ops.empty_planes(M, N, DEV, with_lo=lo)
        ops.gemm_planes(M=M, N=N, K=K, a=sp, a_mode=L.KC, b=wp, b_mode=L.KC, out=out, rowbias=rb, rowbias_div=5,
                        act=L.ACT_RELU, out_planes=op)
    fa = [planes_feed(p, prec) for p in sp]
    A = (torch.cat([f[0] for f in fa], 1), torch.cat([f[1] for f in fa], 1) if lo else None)
    Wh, Wl = planes_feed(wp, prec)
    prod, absprod = feed_product(A, (Wh.t(), Wl.t() if lo else None), prec)
    rbe = rb.double().repeat_interleave(5, 0)[:M]
    check(f"concat planes {prec}", out, torch.relu(prod + rbe), bound(absprod, (rbe,)))
    check_planes_of(f"concat planes {prec}: out_planes vs out", op, out, lo)
    out = torch.full((M, N), float("nan"), device=DEV)
    ops.gemm_raw(M=M, N=N, K=K, a=[(s, None) for s in segs], a_mode=L.KC, b=w, b_mode=L.KC, out=out, prec=L.PRECISIONS[prec])
    A = feed(*split_ref(torch.cat(segs, 1)), prec)
    prod, absprod = feed_product(A, feed(*split_ref(w.t().contiguous()), prec), prec)
    check(f"concat raw {prec}", out, prod, bound(absprod))


# ----------------------------------------------------------------------------------------------- 3. fused attention
def _softmax_ref(scores, weight):
    """fp64 softmax of scaled scores [R, C] whose columns carry multiplicities `weight` [R, C] (0 = not taking part); the
    result is the total probability of each column."""
    s = scores.masked_fill(weight == 0, -math.inf)
    mx = s.max(1, keepdim=True).values
    e = torch.exp(s - mx) * weight
    return e / e.sum(1, keepdim=True)


def _p_bound(p_ref, prec, eps_s):
    # the hi (+ lo) representation of p (2^-16 / 2^-8), doubled for ex2.approx (2^-22 relative) and the fp32 sum and
    # reciprocal (< 2^-20 for <= 256 terms); a score error of at most eps_s moves p by a factor within exp(+-2 eps_s)
    return p_ref * (2 * SPLIT_REP[prec] + 2 * eps_s) + TINY


def _grade_fused(tag, prec, qp, kp, k_first, k_count, ncol, weight_of, scale, pp, out, resid, S, Lq, H):
    """(a) P against the fp64 softmax of the fed scores, zeros past the key count; (b) out against resid + P K from the
    saved planes."""
    lo = prec == "bf16x3"
    Qh, Ql = planes_feed(qp, prec)
    Kh, Kl = planes_feed(kp, prec)
    Ph, Pl = planes_feed(pp, prec)
    cols = pp.cols
    zpad = torch.zeros(cols, H, dtype=torch.float64, device=DEV)
    Khp = torch.cat([Kh, zpad])                      # rows past the plane read as zero
    Klp = torch.cat([Kl, zpad]) if lo else None
    for s in range(S):
        rs = slice(s * Lq, (s + 1) * Lq)
        ks = slice(k_first[s], k_first[s] + k_count[s])
        q = (Qh[rs], Ql[rs] if lo else None)
        k = (Kh[ks], Kl[ks] if lo else None)
        sc, abs_sc = feed_product(q, (k[0].t(), k[1].t() if lo else None), prec)
        nc = ncol[s]
        w = weight_of(s, k_count[s]).to(DEV).double()[None].expand(Lq, -1)
        p_ref = torch.zeros(Lq, cols, dtype=torch.float64, device=DEV)
        if nc > 0:
            p_ref[:, :k_count[s]] = _softmax_ref(sc * scale, w)
        eps_s = C_PROD * scale * abs_sc[:, :max(nc, 1)].max(1, keepdim=True).values
        p_got = Ph[rs] + (Pl[rs] if lo else 0.0)
        check(f"{tag} seq {s}: P", p_got[:, :cols], p_ref, _p_bound(p_ref, prec, eps_s))
        assert torch.all(p_got[:, nc:cols] == 0), f"{tag} seq {s}: P columns past the key count are not 0"
        # (b) the output from exactly the P planes the P K product consumed
        kk = slice(k_first[s], k_first[s] + cols)
        prod, absprod = feed_product((Ph[rs], Pl[rs] if lo else None), (Khp[kk], Klp[kk] if lo else None), prec)
        r = resid[rs] if resid is not None else torch.zeros(Lq, H, device=DEV)
        check(f"{tag} seq {s}: out", out[rs], r.double() + prod, bound(absprod, (r,)))


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("S,Lq,Lk,H,qscale", FUSED_DENSE)
def test_fused_attention_dense_stages(prec, S, Lq, Lk, H, qscale):
    q, k, resid = _rand(S * Lq, H, seed=Lq, scale=qscale), _rand(S * Lk, H, seed=Lk + 1), _rand(S * Lq, H, seed=3)
    scale = float(H) ** -0.5
    with ops.precision(prec):
        assert ops.fused_attention_ok(H, Lk, 0.0)
        qp, kp = ops.split_planes(q), ops.split_planes(k)
        pp = ops.empty_planes(S * Lq, Lk, DEV, with_lo=prec == "bf16x3")
        for t in pp.tensors():
            if t is not None:
                t.fill_(float("nan"))
        out = torch.full((S * Lq, H), float("nan"), device=DEV)
        ops._fused_attention_fwd(qp, kp, S * Lk, S, Lq, Lk, H, None, None, None, Lk, resid, Lq * H, out, pp)
        maps = torch.empty(S * Lq, Lk, device=DEV)
        ops._maps_from_planes(pp, maps, S * Lq, None)
    tag = f"fused dense {prec} S={S} Lq={Lq} Lk={Lk} H={H} q x{qscale:g}"
    rec = pp.hi[:, :Lk].double() + (pp.lo[:, :Lk].double() if pp.lo is not None else 0.0)
    assert torch.equal(maps.double(), rec), f"{tag}: recorded maps are not hi + lo of the saved planes"
    _grade_fused(tag, prec, qp, kp, [s * Lk for s in range(S)], [Lk] * S, [Lk] * S, lambda s, c: torch.ones(c), scale, pp,
                 out, resid, S, Lq, H)


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("sizes,T,H,reps,qscale", FUSED_RAGGED)
def test_fused_attention_ragged_stages(prec, sizes, T, H, reps, qscale):
    """Ragged key sets of the energy -> atom cross attention: one extended key plane with a phantom-key row after every
    crystal's atoms, weighted by nmax - n_b inside the softmax.  Query 0 of every sequence is aligned with the phantom key
    so that its row maximum is the phantom column."""
    from dostransformer_b200.synthetic import make_edos_batch
    g = make_edos_batch(len(sizes), seed=5, sizes=torch.tensor(sizes))
    n_b = torch.bincount(g.batch, minlength=len(sizes))
    B = len(sizes)
    S = reps * B
    nmax = int(n_b.max())
    N = int(n_b.sum())
    ptr = torch.cat([torch.zeros(1, dtype=torch.long), n_b.cumsum(0)])
    kv = _rand(N, H, seed=1)
    phantom = _rand(H, seed=2, scale=2.0)
    ext = torch.cat([torch.cat([kv[int(ptr[b]):int(ptr[b + 1])], phantom[None]]) for b in range(B)])
    q = _rand(S, T, H, seed=3, scale=qscale)
    q[:, 0] = phantom * 3.0
    q = q.view(S * T, H)
    resid = _rand(S * T, H, seed=4)
    first = [int(ptr[s % B]) + s % B for s in range(S)]
    count = [int(n_b[s % B]) + 1 for s in range(S)]
    nph = [max(nmax - int(n_b[s % B]), 0) for s in range(S)]
    ncol = [c - 1 + (1 if m > 0 else 0) for c, m in zip(count, nph)]
    npad = ops._pad8(nmax + 1)
    scale = float(H) ** -0.5
    with ops.precision(prec):
        assert ops.fused_attention_ok(H, nmax + 1, 0.0)
        qp, kp = ops.split_planes(q), ops.split_planes(ext)
        pp = ops.empty_planes(S * T, npad, DEV, with_lo=prec == "bf16x3")
        for t in pp.tensors():
            if t is not None:
                t.fill_(float("nan"))
        out = torch.full((S * T, H), float("nan"), device=DEV)
        i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=DEV)
        ops._fused_attention_fwd(qp, kp, N + B, S, T, 0, H, i32(first), i32(count), i32([nmax]), nmax + 1, resid, T * H, out, pp)

    def weight(s, c):
        w = torch.ones(c, dtype=torch.float64)
        w[c - 1] = nph[s]                 # the phantom column stands for nph zero-padded keys (0: the largest crystal)
        return w

    tag = f"fused ragged {prec} sizes={sizes} T={T} H={H} reps={reps} q x{qscale:g}"
    _grade_fused(tag, prec, qp, kp, first, count, ncol, weight, scale, pp, out, resid, S, T, H)
    # the phantom column is the row maximum of query 0 wherever it takes part
    for s in range(S):
        if nph[s] > 0:
            assert pp.hi[s * T, count[s] - 1].float() > 0, f"{tag} seq {s}: phantom column lost"


# ------------------------------------------------------------------ 4. unfused tensor-core attention, softmax backward
def _ds_ref(P, dP, scale):
    """fp64 dS = scale * P (dP - rowsum(P dP)) from the probability planes (a phantom column holds its total probability)."""
    return scale * P * (dP - (P * dP).sum(1, keepdim=True))


def _ds_bound(P, dP, ref, scale, prec, eps_p):
    # fp32 row dot over <= 514 columns and the (dP - dot) difference: 2^-18 of scale P (|dP| + sum P |dP|) (the C_PROD
    # convention); a relative error eps_p of the kernel's own P against the planes enters P and the dot once each; the output
    # planes represent dS to SPLIT_REP
    mag = dP.abs() + (P * dP.abs()).sum(1, keepdim=True)
    return scale * P * mag * (C_PROD + 2 * eps_p) + SPLIT_REP[prec] * ref.abs() + TINY


def _dP_with_cancellation(rows, cols, P, seed):
    """dP with large cancellation: in odd rows sum_c P dP is ~0 for values of size 1000, in rows = 2 mod 4 dP has a large
    common offset (dP - dot is small against |dP|)."""
    dP = _rand(rows, cols, seed=seed)
    u = 1000.0 * _rand(rows, cols, seed=seed + 1)
    Pf = P.float()
    u = u - (Pf * u).sum(1, keepdim=True) / Pf.sum(1, keepdim=True).clamp_min(1e-30)
    dP[1::2] = u[1::2]
    dP[2::4] += 1000.0
    return dP


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("rows,cols", [(300, 1), (257, 13), (129, 33), (64, 200), (77, 256), (40, 7)])
def test_ds_from_planes(prec, rows, cols):
    """dost_softmax_bwd_from_planes (the dS of the fused attention's backward) against fp64 from the same P planes and dP."""
    scale = 0.0883883
    x = _rand(rows, cols, seed=cols, scale=3.0)
    x[::5, cols // 2 + 1:] = -math.inf             # rows whose trailing columns are masked (exact zeros in P)
    p = torch.softmax(x, 1)
    Lp = (cols + 3) // 4 * 4
    with ops.precision(prec):
        pp = ops.split_planes(p)
        dP = torch.full((rows, Lp), float("nan"), device=DEV)
        dP[:, :cols] = _dP_with_cancellation(rows, cols, pp.hi[:, :cols], seed=rows)
        dsp = ops.empty_planes(rows, cols, DEV, with_lo=prec == "bf16x3")
        ops._ds_from_planes(pp, dP, rows, cols, scale, dsp)
    Ph, Pl = planes_feed(pp, prec)
    P = Ph + (Pl if Pl is not None else 0.0)
    d = dP[:, :cols].double()
    ref = _ds_ref(P, d, scale)
    got = dsp.hi[:, :cols].double() + (dsp.lo[:, :cols].double() if dsp.lo is not None else 0.0)
    check(f"ds_from_planes {prec} rows={rows} cols={cols}", got, ref, _ds_bound(P, d, ref, scale, prec, 0.0))
    assert torch.all(got[P == 0] == 0), "ds_from_planes: dS is not 0 where P is 0"


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("sizes,T,reps", [([256, 3, 299], 70, 1), ([512, 0, 127, 40], 33, 2)])
def test_xattn_softmax_planes(prec, sizes, T, reps):
    """Over 256 keys the cross attention runs unfused (xattn_tc.cu): the probability planes against the fp64 softmax of
    the kernel's own fp32 scores with the phantom weighting, and the dS planes against scale P (dP - rowsum(P dP))."""
    from dostransformer_b200.synthetic import make_edos_batch
    g = make_edos_batch(len(sizes), seed=9, sizes=torch.tensor(sizes))
    n_b = torch.bincount(g.batch, minlength=len(sizes))
    B, H = len(sizes), 128
    S = reps * B
    nmax = int(n_b.max())
    assert nmax + 1 > 256
    N = int(n_b.sum())
    ptr = torch.cat([torch.zeros(1, dtype=torch.long), n_b.cumsum(0)])
    kv, phantom = _rand(N, H, seed=1), _rand(H, seed=2, scale=2.0)
    ext = torch.cat([torch.cat([kv[int(ptr[b]):int(ptr[b + 1])], phantom[None]]) for b in range(B)])
    q = _rand(S, T, H, seed=3, scale=2.0)
    q[:, 0] = phantom * 3.0
    q = q.view(S * T, H)
    npad = ops._pad8(nmax + 1)
    scale = float(H) ** -0.5
    first = torch.tensor([int(ptr[s % B]) + s % B for s in range(S)], dtype=torch.int32, device=DEV)
    ptr_d, nmax_d = ptr.to(torch.int32).to(DEV), torch.tensor([nmax], dtype=torch.int32, device=DEV)
    lib = L.lib()
    with ops.precision(prec):
        lo = prec == "bf16x3"
        qp, kp = ops.split_planes(q), ops.split_planes(ext)
        scores = torch.empty(S * T, npad, device=DEV)
        ops.gemm_planes(M=T, N=npad, K=H, a=[qp], a_mode=L.KC, b=kp, b_mode=L.KC, b_rows=N + B, out=scores, batch=S,
                        a_bstride=T * qp.ld, c_bstride=T * npad, b_rowoff=first)
        pp = ops.empty_planes(S * T, npad, DEV, with_lo=lo)
        lse = torch.empty(S * T, device=DEV)
        L.check(lib.dost_xattn_softmax_fwd(L.p(scores), L.p(ptr_d), L.p(nmax_d), S * T, B, T, npad, scale, L.p(pp.hi),
                                           L.p(pp.lo), pp.ld, L.p(lse), 0.0, 0, L.stream()), "xattn_softmax_fwd")
        Ph, Pl = planes_feed(pp, prec)
        P = Ph + (Pl if lo else 0.0)
        dP = _dP_with_cancellation(S * T, npad, P, seed=11)
        dsp = ops.empty_planes(S * T, npad, DEV, with_lo=lo)
        L.check(lib.dost_xattn_softmax_bwd(L.p(scores), L.p(lse), L.p(dP), L.p(ptr_d), L.p(nmax_d), S * T, B, T, npad, scale,
                                           L.p(dsp.hi), L.p(dsp.lo), dsp.ld, 0.0, 0, L.stream()), "xattn_softmax_bwd")
    tag = f"xattn_tc {prec} sizes={sizes} T={T} reps={reps}"
    w = torch.zeros(S * T, npad, dtype=torch.float64, device=DEV)
    for s in range(S):
        nb = int(n_b[s % B])
        w[s * T:(s + 1) * T, :nb] = 1.0
        w[s * T:(s + 1) * T, nb] = max(nmax - nb, 0)
    v = scores.double() * scale
    p_ref = _softmax_ref(v, w).nan_to_num(0.0)
    mx = v.masked_fill(w == 0, -math.inf).max(1, keepdim=True).values
    # fp32 scale multiply and (v - max) (2^-24 of |v| + |v - max| in the exponent), expf (2 ulp), the fp32 sum over
    # <= 17 terms per lane and 5 shuffles (< 2^-19), reciprocal and weight products (3 roundings)
    eps_p = 2.0 ** -23 * (v.abs() + (v - mx).abs()).masked_fill(w == 0, 0).amax(1, keepdim=True) + 2.0 ** -18
    check(f"{tag}: P", P, p_ref, p_ref * (2 * SPLIT_REP[prec] + 2 * eps_p) + TINY)
    assert torch.all(P[w == 0] == 0), f"{tag}: P columns that take no part are not 0"
    ref = _ds_ref(P, dP.double(), scale)
    got = dsp.hi[:, :npad].double() + (dsp.lo[:, :npad].double() if lo else 0.0)
    # the backward recomputes P in fp32 from the log-sum-exp: within eps_p + the planes' own representation of P
    check(f"{tag}: dS", got, ref, _ds_bound(P, dP.double(), ref, scale, prec, eps_p + SPLIT_REP[prec]))
