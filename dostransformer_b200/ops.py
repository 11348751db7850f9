"""Host-side operators: torch.autograd.Function wrappers around the C ABI (include/dost.h).

Every device computation below is a kernel of libdost_b200.so launched on torch's current stream; torch
only provides device memory (torch.empty) and the autograd graph.  No CPU fallback, no torch math on the
forward or backward path.
"""
from __future__ import annotations

import ctypes as C
import math
from contextlib import nullcontext
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib as L

NUM_SMS = 148

# GEMM precision: "fp32" = FMA pipe (bit-for-bit fp32 arithmetic), "bf16x3" = tcgen05 tensor cores with error-compensated
# bf16 operand splits (fp32 parity), "bf16" = tcgen05 with bf16 operands (fp32 accumulate; stated looser tolerance).
_PRECISION = L.PREC_FMA


def set_precision(name: str) -> None:
    global _PRECISION
    _PRECISION = L.PRECISIONS[name]


def get_precision() -> int:
    return _PRECISION


class precision:
    """Context manager: ``with ops.precision("bf16x3"): ...``"""

    def __init__(self, name: str):
        self.new = L.PRECISIONS[name]

    def __enter__(self):
        global _PRECISION
        self.old, _PRECISION = _PRECISION, self.new
        return self

    def __exit__(self, *exc):
        global _PRECISION
        _PRECISION = self.old
        return False


class precision_value:
    """Context manager restoring a saved precision enum (used by backward passes)."""

    def __init__(self, value: int):
        self.new = value

    def __enter__(self):
        global _PRECISION
        self.old, _PRECISION = _PRECISION, self.new
        return self

    def __exit__(self, *exc):
        global _PRECISION
        _PRECISION = self.old
        return False


def _ws(nbytes: int, device) -> Optional[torch.Tensor]:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _ld(t: torch.Tensor) -> int:
    """Leading dimension (elements) of a 2-D row-strided view with unit column stride."""
    assert t.dim() == 2 and (t.shape[1] == 1 or t.stride(1) == 1), "need a row-major (possibly row-strided) 2-D view"
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1])


# =====================================================================================================
# graph structure (integer work)
# =====================================================================================================
@dataclass
class CSR:
    rowptr: torch.Tensor      # int32 [size+1]
    perm: Optional[torch.Tensor]  # int32 [n] or None (identity)
    key: torch.Tensor         # int32 [n]  (the index the segments were built from)
    size: int


def to_i32(t: torch.Tensor) -> torch.Tensor:
    if t.dtype == torch.int32:
        return t.contiguous()
    assert t.dtype == torch.int64, f"index tensor must be int64/int32, got {t.dtype}"
    t = t.contiguous()
    out = torch.empty(t.shape, dtype=torch.int32, device=t.device)
    L.check(L.lib().dost_cast_i64_i32(L.p(t), L.p(out), t.numel(), L.stream()), "cast_i64_i32")
    return out


def csr_build(key32: torch.Tensor, size: int, want_max: bool = False) -> Tuple[CSR, Optional[torch.Tensor]]:
    n = key32.numel()
    dev = key32.device
    rowptr = torch.empty(size + 1, dtype=torch.int32, device=dev)
    perm = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    mx = torch.empty(1, dtype=torch.int32, device=dev) if want_max else None
    lib = L.lib()
    nb = lib.dost_csr_workspace_bytes(n, size)
    ws = _ws(nb, dev)
    L.check(lib.dost_csr_build(L.p(key32), n, size, L.p(rowptr), L.p(perm), L.p(mx), L.p(ws), nb, L.stream()), "csr_build")
    return CSR(rowptr, perm[:n], key32, size), mx


@dataclass
class CrystalGraph:
    """Integer structure of one batch, built once and shared by all layers and the backward pass."""
    N: int
    E: int
    B: int
    row: torch.Tensor
    col: torch.Tensor
    batch: torch.Tensor
    system: torch.Tensor
    by_dst: CSR          # edges grouped by destination (col): scatter_sum / scatter_mean order
    by_src: CSR          # edges grouped by source (row): adjoint of x[row]
    by_system: CSR       # crystals grouped by crystal system: adjoint of promt_token[g.system]
    crystals: CSR        # nodes grouped by crystal (contiguous): ptr = crystals.rowptr
    nmax: torch.Tensor   # int32 [1] on device: max nodes per crystal (to_dense_batch padding length)
    nmax_host: Optional[int] = None   # the same number on the host when the collate / sharder knows it (no device sync)
    # this batch's OWN largest crystal (<= nmax_host, which may be the data-parallel global padding length): sizes the
    # attention's key-side buffers, so that a rank's work does not grow with the other ranks' crystals; the phantom-key
    # multiplicity always uses `nmax`
    nmax_local: Optional[int] = None
    _trows: dict = field(default_factory=dict)

    @property
    def nkeys_host(self) -> Optional[int]:
        """Host-side bound on the keys of one sequence: the crystal's atoms + the phantom column."""
        n = self.nmax_local if self.nmax_local is not None else self.nmax_host
        return None if n is None else n + 1

    def ragged(self, reps: int = 1):
        """(ptr_ext, n_ext): first row and row count of every crystal in the extended key plane (atoms + 1 phantom row),
        repeated ``reps`` times (sequence s of S = reps * B attends to crystal s % B)."""
        key = ("ragged", reps)
        if key not in self._trows:
            if reps == 1:
                ar = torch.arange(self.B, dtype=torch.int32, device=self.row.device)
                ptr = self.crystals.rowptr
                self._trows[key] = ((ptr[:-1] + ar).contiguous(), (ptr[1:] - ptr[:-1] + 1).contiguous())
            else:
                p1, n1 = self.ragged(1)
                self._trows[key] = (p1.repeat(reps), n1.repeat(reps))
        return self._trows[key]

    @property
    def ptr(self) -> torch.Tensor:
        return self.crystals.rowptr

    def token_mod(self, T: int) -> torch.Tensor:
        """int32 [B*T]: t = i % T (row map that repeats a [T, H] block for every crystal)."""
        key = ("mod", T)
        if key not in self._trows:
            self._trows[key] = (torch.arange(self.B * T, dtype=torch.int32, device=self.row.device) % T).contiguous()
        return self._trows[key]

    def token_rowptr(self, T: int) -> torch.Tensor:
        """rowptr of the [B*T] token rows grouped by crystal (T contiguous rows each)."""
        if T not in self._trows:
            self._trows[T] = torch.arange(0, (self.B + 1) * T, T, dtype=torch.int32, device=self.row.device)
        return self._trows[T]


def build_graph(edge_index: torch.Tensor, batch: torch.Tensor, system: torch.Tensor, *, nmax_override: Optional[int] = None,
                need_backward: bool = True, nmax_hint: Optional[int] = None, phantoms: bool = True) -> CrystalGraph:
    """edge_index int64 [2,E] (row = centre atom, col = neighbour), batch int64 [N] sorted, system int64 [B]."""
    assert edge_index.is_cuda, "dostransformer_b200 has no CPU path: move the batch to a CUDA device"
    L.lib()
    L.poll_device_errors()        # invalid input skipped by the kernels of an earlier step (no synchronisation)
    N, E, B = batch.numel(), edge_index.shape[1], system.numel()
    ei = to_i32(edge_index)
    row, col = ei[0], ei[1]
    b32, s32 = to_i32(batch), to_i32(system)
    by_dst, _ = csr_build(col, N)
    by_src = by_sys = None
    if need_backward:
        by_src, _ = csr_build(row, N)
        by_sys, _ = csr_build(s32, 7)
    crystals, nmax = csr_build(b32, B, want_max=True)
    crystals.perm = None
    # Padding length (to_dense_batch's Nmax).  `nmax_override` is the data-parallel global value set by the sharder; it
    # may exceed this batch's own maximum but must never undercut it: a crystal with more atoms than the padding length
    # would get a negative phantom-key count and, on the tensor-core attention path, more score columns than were
    # allocated.  The batch's own maximum is known on the host when the collate recorded it (`nmax_hint`); otherwise the
    # device value max(override, measured) is used and the host-sized tensor-core path is only taken with a hint.
    host = None
    if not phantoms:
        # per-crystal evaluation (the reference's batch_size-1 loaders): no padding, hence no phantom keys and no use for
        # a data-parallel padding length; buffers are sized by the batch's own maximum when the collate recorded it
        nmax = torch.zeros(1, dtype=torch.int32, device=batch.device)
        host = int(nmax_hint) if nmax_hint is not None else None
    elif nmax_override is not None:
        if nmax_hint is not None and int(nmax_override) < int(nmax_hint):
            raise ValueError(f"max_num_nodes={int(nmax_override)} (model.max_num_nodes / sharder) is smaller than this "
                             f"batch's largest crystal ({int(nmax_hint)} nodes): stale data-parallel padding length")
        L.check(L.lib().dost_imax_scalar(L.p(nmax), int(nmax_override), L.stream()), "imax_scalar")   # nmax = max(nmax, override)
        host = int(nmax_override) if nmax_hint is not None else None
    elif nmax_hint is not None:
        host = int(nmax_hint)
    if host is None and phantoms and B > 0 and not L.switch("DOST_NO_NMAX_SYNC") and not torch.cuda.is_current_stream_capturing():
        # A batch collated elsewhere (a stock PyG Batch from main_eDOS.py:54 carries no max_num_nodes): ONE device->host
        # read of the padding length buys the tensor-core attention path, whose buffers are sized on the host.  (The
        # reference reads back twice per forward: len(batch.unique()) DOSTransformer.py:118 and to_dense_batch's max().)
        # Batches from this package's collate / sharder / synthetic generators carry the hint and never get here.
        host = int(nmax.item())
    local = int(nmax_hint) if (nmax_hint is not None and host is not None) else host
    return CrystalGraph(N, E, B, row, col, b32, s32, by_dst, by_src, by_sys, crystals, nmax, host, local)


# =====================================================================================================
# raw kernel wrappers (no autograd)
# =====================================================================================================
@dataclass
class RowMap:
    """How A-operand row m of a GEMM maps to a row of ``tensor``: row = idx[m // div] (idx optional)."""
    idx: Optional[torch.Tensor] = None
    div: int = 1
    # adjoint information (needed for the backward of the mapped operand)
    csr: Optional[CSR] = None            # groups target rows by source row (for idx maps)
    div_rowptr: Optional[torch.Tensor] = None  # contiguous groups of `div` rows


def _seg(t: torch.Tensor, m: Optional[RowMap], width: int) -> L.Seg:
    s = L.Seg()
    s.base = t.data_ptr()
    s.ld = _ld(t)
    s.idx = m.idx.data_ptr() if (m is not None and m.idx is not None) else None
    s.div = m.div if m is not None else 1
    s.width = width
    return s


def gemm_raw(*, M: int, N: int, K: int, a: Sequence[Tuple[torch.Tensor, Optional[RowMap]]], a_mode: int,
             b: torch.Tensor, b_mode: int, b_map: Optional[RowMap] = None, out: torch.Tensor,
             bias: Optional[torch.Tensor] = None, act: int = L.ACT_NONE, act_slope: float = 0.0,
             prelu_slope: Optional[torch.Tensor] = None, out_pre: Optional[torch.Tensor] = None,
             dact_saved: Optional[torch.Tensor] = None, dact_kind: int = L.ACT_NONE, dact_slope: float = 0.0,
             residual: Optional[torch.Tensor] = None, accumulate: bool = False, split_k: int = 1,
             batch: int = 1, a_bstride: int = 0, b_bstride: int = 0, c_bstride: int = 0,
             ldb: Optional[int] = None, ldc: Optional[int] = None, lda: Optional[int] = None,
             prec: Optional[int] = None) -> None:
    g = L.Gemm()
    g.dtype = L.dt(out)
    g.M, g.N, g.K, g.batch = M, N, K, batch
    g.a_mode, g.a_nseg = a_mode, len(a)
    for i, (t, m) in enumerate(a):
        width = t.shape[-1] if (a_mode == L.KC and len(a) > 1) else K
        g.a[i] = _seg(t if t.dim() == 2 else t.reshape(-1, t.shape[-1]), m, width)
        if lda is not None:
            g.a[i].ld = lda
    g.a_bstride = a_bstride
    g.b_mode = b_mode
    g.b = _seg(b if b.dim() == 2 else b.reshape(-1, b.shape[-1]), b_map, 0)
    if ldb is not None:
        g.b.ld = ldb
    g.b_bstride = b_bstride
    g.bias = bias.data_ptr() if bias is not None else None
    g.act, g.act_slope = act, act_slope
    g.prelu_slope = prelu_slope.data_ptr() if prelu_slope is not None else None
    if out_pre is not None:
        g.out_pre, g.ld_pre = out_pre.data_ptr(), _ld(out_pre.reshape(-1, out_pre.shape[-1]))
    if dact_saved is not None:
        g.dact_saved, g.ld_dact = dact_saved.data_ptr(), _ld(dact_saved.reshape(-1, dact_saved.shape[-1]))
        g.dact_kind, g.dact_slope = dact_kind, dact_slope
    if residual is not None:
        g.residual, g.ld_res = residual.data_ptr(), _ld(residual.reshape(-1, residual.shape[-1]))
    g.out = out.data_ptr()
    g.ldc = ldc if ldc is not None else _ld(out if out.dim() == 2 else out.reshape(-1, out.shape[-1]))
    g.c_bstride = c_bstride
    g.accumulate = 1 if accumulate else 0
    precision = _PRECISION if prec is None else prec
    # Small fp32 problems (the per-crystal Linears of the DOS heads: [B, 2H] x [2H, H] and their adjoints) are latency-bound:
    # a few tiles whose K loop runs serially - 44 us on the converting tensor-core kernel at ANY batch size.  They go to the
    # FMA pipe (exact fp32) with the reduction split over up to 8 blocks when the epilogue is a plain store.
    if (precision != L.PREC_FMA and out.dtype == torch.float32 and batch == 1 and M * N * K < (1 << 27)
            and not L.switch("DOST_NO_SMALL_FMA")):
        precision = L.PREC_FMA
        if (split_k == 1 and K >= 256 and bias is None and act == L.ACT_NONE and out_pre is None and dact_saved is None
                and residual is None):
            split_k = min(8, K // 64)
    g.split_k = split_k
    g.precision = precision
    lib = L.lib()
    ws, nb = None, 0
    if split_k > 1:
        nb = lib.dost_gemm_workspace_bytes(C.byref(g))
        ws = _ws(nb, out.device)
    L.check(lib.dost_gemm(C.byref(g), L.p(ws), nb, L.stream()), "gemm")


# =====================================================================================================
# bf16 operand planes + TMA-fed tcgen05 GEMM (dost_gemm_bf16)
# =====================================================================================================
@dataclass
class Planes:
    """A GEMM operand stored as bf16 planes: hi = bf16(x), lo = bf16(x - hi) (None in plain-bf16 mode)."""
    hi: torch.Tensor
    lo: Optional[torch.Tensor]
    rows: int
    cols: int

    @property
    def ld(self) -> int:
        return self.hi.stride(0)

    def tensors(self):
        return (self.hi, self.lo)


def _pad8(n: int) -> int:
    return (n + 7) // 8 * 8


def empty_planes(rows: int, cols: int, device, with_lo: bool = True) -> Planes:
    ld = _pad8(cols)
    hi = torch.empty(rows, ld, dtype=torch.bfloat16, device=device)
    lo = torch.empty(rows, ld, dtype=torch.bfloat16, device=device) if with_lo else None
    return Planes(hi, lo, rows, cols)


def split_planes(x2d: torch.Tensor, with_lo: Optional[bool] = None) -> Planes:
    """fp32 [rows, cols] -> bf16 planes (one pass; padded columns are zero)."""
    assert x2d.dtype == torch.float32 and x2d.dim() == 2
    if x2d.stride(1) != 1:
        x2d = x2d.contiguous()
    if with_lo is None:
        with_lo = _PRECISION != L.PREC_BF16
    rows, cols = x2d.shape
    pl = empty_planes(rows, cols, x2d.device, with_lo)
    L.check(L.lib().dost_split_planes(L.p(x2d), _ld(x2d), rows, cols, L.p(pl.hi), L.p(pl.lo), pl.ld, L.stream()), "split_planes")
    return pl


def split_planes_colsum(x2d: torch.Tensor) -> Tuple[Planes, torch.Tensor]:
    """split_planes(x) and x.sum(0) in one pass over x (operand planes of an output gradient + its bias gradient)."""
    assert x2d.dtype == torch.float32 and x2d.dim() == 2
    if x2d.stride(1) != 1:
        x2d = x2d.contiguous()
    rows, cols = x2d.shape
    pl = empty_planes(rows, cols, x2d.device, _with_lo())
    cs = torch.empty(cols, dtype=torch.float32, device=x2d.device)
    lib = L.lib()
    nb = lib.dost_split_planes_colsum_workspace_bytes(rows, cols, pl.ld)
    ws = _ws(nb, x2d.device)
    L.check(lib.dost_split_planes_colsum(L.p(x2d), _ld(x2d), rows, cols, L.p(pl.hi), L.p(pl.lo), pl.ld, L.p(cs), L.p(ws), nb,
                                         L.stream()), "split_planes_colsum")
    return pl, cs


_PLANES_GENERATION = 0


def invalidate_weight_planes(model=None) -> None:
    """Drops the cached bf16 operand planes of the weights (all of them, or those of ``model`` / an iterable of
    parameters).  The cache is keyed on the parameter's autograd version counter and storage address, so optimizers that
    update through ``p.add_()`` / ``p.copy_()`` / this package's fused AdamW are seen automatically; writes that BYPASS
    the version counter are not - ``p.data.copy_()``, ``p.data.mul_()``, ``dist.broadcast(p.data)``, EMA swaps through
    ``.data``, raw-pointer or graph-captured updates.  Call this after any such write (``dp.broadcast_parameters`` and
    ``graphed.GraphedStep`` do).  ``DOST_CHECK_PLANES=1`` re-splits on every cache hit and raises on a stale entry."""
    global _PLANES_GENERATION
    if model is None:
        _PLANES_GENERATION += 1
        return
    params = model.parameters() if hasattr(model, "parameters") else model
    for p in params:
        base = p._base if p._base is not None else p
        base.__dict__.pop("_dost_weight_planes", None)


def _planes_key(w: torch.Tensor):
    return (w.storage_offset(), tuple(w.shape), tuple(w.stride()), _PRECISION != L.PREC_BF16)


def weight_planes(w: torch.Tensor) -> Planes:
    """Planes of a parameter (or of a strided view of one), cached ON the parameter object until it is modified in
    place (optimizer step).  Keying on the object - not on its address - keeps the cache exact across models.  A column
    slice of a parameter whose full planes are cached (refresh_weight_planes) is served as a view of those."""
    base = w._base if w._base is not None else w
    cache = base.__dict__.setdefault("_dost_weight_planes", {})
    key = _planes_key(w)
    # the address too: `p.data = other` swaps storage without a version bump
    ver = (base._version, base.data_ptr(), _PLANES_GENERATION)
    hit = cache.get(key)
    if hit is not None and hit[0] == ver:
        if L.switch("DOST_CHECK_PLANES"):
            fresh = split_planes(w.detach())
            same = torch.equal(fresh.hi, hit[1].hi) and (fresh.lo is None or torch.equal(fresh.lo, hit[1].lo))
            if not same:
                raise RuntimeError("stale weight planes: a parameter was written without bumping its version counter "
                                   "(p.data.*, raw pointers); call ops.invalidate_weight_planes(model) after such writes")
        return hit[1]
    if base is not w and base.dim() == 2 and w.dim() == 2 and w.stride() == base.stride() and w.shape[0] == base.shape[0]:
        full = cache.get(_planes_key(base))
        c0 = w.storage_offset() - base.storage_offset()
        if full is not None and full[0] == ver and 0 <= c0 < base.stride(0) and c0 % 8 == 0 and \
                (w.shape[1] % 8 == 0 or c0 + w.shape[1] == base.shape[1]):
            pl = cols_view(full[1], c0, c0 + w.shape[1])
            cache[key] = (ver, pl)
            return pl
    pl = split_planes(w.detach())
    cache[key] = (ver, pl)
    return pl


def refresh_weight_planes(weights: Sequence[torch.Tensor]) -> None:
    """Splits all of ``weights`` (2-D fp32 parameters) into operand planes with ONE launch per 24 tensors and fills the
    cache of weight_planes: the once-per-step refresh after an optimizer update, and the first node of a captured step
    (graphed.GraphedStep), where the cache cannot be trusted across replays."""
    ws = [w for w in weights if w.dim() == 2 and w.dtype == torch.float32 and w.is_cuda and w.stride(1) == 1]
    if not ws:
        return
    with_lo = _with_lo()
    dev = ws[0].device
    sizes = [w.shape[0] * _pad8(w.shape[1]) for w in ws]
    offs, total = [], 0
    for n in sizes:
        offs.append(total)
        total += (n + 7) // 8 * 8                   # every plane starts 16-byte aligned
    flat_hi = torch.empty(total, dtype=torch.bfloat16, device=dev)
    flat_lo = torch.empty(total, dtype=torch.bfloat16, device=dev) if with_lo else None
    n = len(ws)
    his, los = [], []
    for w, o, sz in zip(ws, offs, sizes):
        ldp = _pad8(w.shape[1])
        hi = flat_hi[o:o + sz].view(w.shape[0], ldp)
        lo = flat_lo[o:o + sz].view(w.shape[0], ldp) if with_lo else None
        his.append(hi)
        los.append(lo)
    vp = lambda xs: (C.c_void_p * n)(*xs)
    ll = lambda xs: (C.c_longlong * n)(*xs)
    L.check(L.lib().dost_split_planes_multi(
        n, vp([w.data_ptr() for w in ws]), ll([w.stride(0) for w in ws]), ll([w.shape[0] for w in ws]),
        (C.c_int * n)(*[w.shape[1] for w in ws]), vp([h.data_ptr() for h in his]),
        vp([(l.data_ptr() if l is not None else None) for l in los]), ll([_pad8(w.shape[1]) for w in ws]), L.stream()),
        "split_planes_multi")
    for w, hi, lo in zip(ws, his, los):
        base = w._base if w._base is not None else w
        cache = base.__dict__.setdefault("_dost_weight_planes", {})
        cache[_planes_key(w)] = ((base._version, base.data_ptr(), _PLANES_GENERATION), Planes(hi, lo, w.shape[0], w.shape[1]))


def _planes_c(pl: Planes, width: int) -> L.PlanesC:
    c = L.PlanesC()
    c.hi = pl.hi.data_ptr()
    c.lo = pl.lo.data_ptr() if pl.lo is not None else None
    c.ld = pl.ld
    c.rows = pl.rows
    c.width = width
    return c


def gemm_planes(*, M: int, N: int, K: int, a: Sequence[Planes], a_mode: int, b: Planes, b_mode: int,
                out: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None,
                rowbias: Optional[torch.Tensor] = None, rowbias_div: int = 1, act: int = L.ACT_NONE, act_slope: float = 0.0,
                prelu_slope: Optional[torch.Tensor] = None, out_pre: Optional[torch.Tensor] = None,
                dact: Optional[Planes] = None, dact_slope: float = 0.0, residual: Optional[torch.Tensor] = None,
                accumulate: bool = False, split_k: int = 1, out_planes: Optional[Planes] = None,
                ldc: Optional[int] = None, prec: Optional[int] = None, batch: int = 1, a_bstride: int = 0, b_bstride: int = 0,
                c_bstride: int = 0, res_bstride: int = 0, ld_res: Optional[int] = None, b_rows: Optional[int] = None,
                b_rowoff: Optional[torch.Tensor] = None, c_rowoff: Optional[torch.Tensor] = None,
                c_rowlim: Optional[torch.Tensor] = None, colsum_out: Optional[torch.Tensor] = None,
                out_gate: Optional[torch.Tensor] = None, dact_gate: Optional[torch.Tensor] = None) -> None:
    """C = epi(A B^T) on the TMA-fed tcgen05 kernel; operands are bf16 planes (see include/dost.h).
    b_rows: valid rows of a K-major B per problem when N is padded beyond them (the rest reads as zero).
    out_gate / dact_gate: int32 [N / 32, M] activation gate bits written / read by the epilogue (see `gate_bits_ok`)."""
    g = L.GemmBf16()
    g.M, g.N, g.K = M, N, K
    g.a_mode, g.a_nseg = a_mode, len(a)
    for i, pl in enumerate(a):
        g.a[i] = _planes_c(pl, pl.cols if a_mode == L.KC else K)
    g.b_mode = b_mode
    g.b = _planes_c(b, 0)
    g.b.rows = b_rows if b_rows is not None else 0
    g.bias = bias.data_ptr() if bias is not None else None
    if rowbias is not None:
        g.rowbias, g.ld_rowbias, g.rowbias_div = rowbias.data_ptr(), _ld(rowbias), rowbias_div
    g.act, g.act_slope = act, act_slope
    g.prelu_slope = prelu_slope.data_ptr() if prelu_slope is not None else None
    if out_pre is not None:
        g.out_pre, g.ld_pre = out_pre.data_ptr(), _ld(out_pre)
    if dact is not None:
        g.dact_hi, g.ld_dact, g.dact_slope = dact.hi.data_ptr(), dact.ld, dact_slope
    if residual is not None:
        g.residual, g.ld_res = residual.data_ptr(), (ld_res if ld_res is not None else _ld(residual))
    if out is not None:
        g.out = out.data_ptr()
        g.ldc = ldc if ldc is not None else _ld(out)
    g.accumulate = 1 if accumulate else 0
    g.batch, g.a_bstride, g.b_bstride, g.c_bstride, g.res_bstride = batch, a_bstride, b_bstride, c_bstride, res_bstride
    g.b_rowoff = b_rowoff.data_ptr() if b_rowoff is not None else None
    g.c_rowoff = c_rowoff.data_ptr() if c_rowoff is not None else None
    g.c_rowlim = c_rowlim.data_ptr() if c_rowlim is not None else None
    if out_planes is not None:
        g.out_hi = out_planes.hi.data_ptr()
        g.out_lo = out_planes.lo.data_ptr() if out_planes.lo is not None else None
        g.ld_op = out_planes.ld
    g.split_k = split_k
    g.precision = _PRECISION if prec is None else prec
    g.colsum = colsum_out.data_ptr() if colsum_out is not None else None
    if out_gate is not None:
        g.out_gate, g.ld_gate = out_gate.data_ptr(), out_gate.stride(0)
    if dact_gate is not None:
        g.dact_gate, g.ld_gate, g.dact_slope = dact_gate.data_ptr(), dact_gate.stride(0), dact_slope
    lib = L.lib()
    ws, nb = None, 0
    if split_k > 1 or colsum_out is not None:
        nb = lib.dost_gemm_bf16_workspace_bytes(C.byref(g))
        ws = _ws(nb, b.hi.device)
    L.check(lib.dost_gemm_bf16(C.byref(g), L.p(ws), nb, L.stream()), "gemm_bf16")


def gate_bits_ok(M: int, N: int) -> bool:
    """The FFN keeps its ReLU gates as 1 bit per hidden activation (written by fc1's epilogue, read by the epilogue of the fc2
    input-gradient GEMM instead of the 16-bit hi plane): needs the TMA-store epilogue (M >= 32, N % 32 == 0, not disabled)."""
    return M >= 32 and N % 32 == 0 and os.environ.get("DOST_GEMM_TMA_EPI", "1") != "0" and not L.switch("DOST_NO_FFN_GATE")


def tc_active(t: torch.Tensor) -> bool:
    """True when `t`'s Linear stacks run on the tensor cores (bf16x3 / bf16 planes) rather than the FMA pipe."""
    return _PRECISION != L.PREC_FMA and t.dtype == torch.float32


def _with_lo() -> bool:
    return _PRECISION != L.PREC_BF16


def ln_fwd_planes(x2d: torch.Tensor, gamma, beta, slope=None, *, want_y: bool = False, want_planes: bool = True,
                  gather_add=None):
    """LayerNorm(+PReLU) of fp32 rows, written directly as operand planes (and/or fp32).  Returns (y, planes, stats).

    gather_add = (ga, ia, gb, ib): x2d[r] += ga[ia[r]] + gb[ib[r]] first, IN PLACE (x2d then holds the LayerNorm input)."""
    M, W = x2d.shape
    ga = ia = gb = ib = None
    ldg = 0
    if gather_add is not None:
        ga, ia, gb, ib = gather_add
        ldg = _ld(ga)
        assert _ld(gb) == ldg
    dev = x2d.device
    y = torch.empty(M, W, dtype=torch.float32, device=dev) if want_y else None
    pl = empty_planes(M, W, dev, _with_lo()) if want_planes else None
    stats = torch.empty(M, 2, dtype=torch.float32, device=dev)
    L.check(L.lib().dost_ln_fwd_planes(L.p(x2d), _ld(x2d), L.p(ga), L.p(ia), L.p(gb), L.p(ib), ldg, L.p(gamma), L.p(beta),
                                       L.p(slope), L.p(y),
                                       L.p(pl.hi) if pl else None, L.p(pl.lo) if (pl and pl.lo is not None) else None,
                                       pl.ld if pl else 0, L.p(stats), M, W, L.stream()), "ln_fwd_planes")
    return y, pl, stats


def ln_bwd_planes(dy2d, x2d, stats, gamma, beta, slope=None, *, dres=None, want_dx: bool = True, want_planes: bool = False,
                  want_xsum: bool = False):
    """Backward of ln_fwd_planes.  Returns (dx fp32|None, dx planes|None, dgamma, dbeta, dslope|None, colsum(dx)|None)."""
    M, W = x2d.shape
    dev = x2d.device
    dx = torch.empty(M, W, dtype=torch.float32, device=dev) if want_dx else None
    pl = empty_planes(M, W, dev, _with_lo()) if want_planes else None
    dg = torch.empty(W, dtype=torch.float32, device=dev)
    db = torch.empty(W, dtype=torch.float32, device=dev)
    ds = torch.empty(1, dtype=torch.float32, device=dev) if slope is not None else None
    xs = torch.empty(W, dtype=torch.float32, device=dev) if want_xsum else None
    lib = L.lib()
    nb = lib.dost_ln_bwd_planes_workspace_bytes(M, W)
    ws = _ws(nb, dev)
    L.check(lib.dost_ln_bwd_planes(L.p(dy2d), _ld(dy2d), L.p(x2d), _ld(x2d), L.p(stats), L.p(gamma), L.p(beta), L.p(slope),
                                   L.p(dres), _ld(dres) if dres is not None else 0, L.p(dx),
                                   L.p(pl.hi) if pl else None, L.p(pl.lo) if (pl and pl.lo is not None) else None,
                                   pl.ld if pl else 0, L.p(dg), L.p(db), L.p(ds), L.p(xs), M, W, L.p(ws), nb, L.stream()),
            "ln_bwd_planes")
    return dx, pl, dg, db, ds, xs


def colsum_planes(pl: Planes) -> torch.Tensor:
    out = torch.empty(pl.cols, dtype=torch.float32, device=pl.hi.device)
    lib = L.lib()
    nb = lib.dost_colsum_planes_workspace_bytes(pl.rows, pl.cols)
    ws = _ws(nb, pl.hi.device)
    L.check(lib.dost_colsum_planes(L.p(pl.hi), L.p(pl.lo), pl.ld, pl.rows, pl.cols, L.p(out), L.p(ws), nb, L.stream()),
            "colsum_planes")
    return out


def _split_for(M_out: int, N_out: int, K_red: int) -> int:
    """Split-K factor of a weight-gradient GEMM on the planes kernel (128 x 256 tiles, 148 SMs)."""
    bn = 64 if N_out <= 64 else (128 if N_out <= 128 else 256)
    tiles = math.ceil(M_out / 128) * math.ceil(N_out / bn)
    want = max(1, (2 * NUM_SMS) // tiles)
    return int(max(1, min(want, math.ceil(K_red / 512), 256)))


def _planes_save(pl: Planes):
    return [pl.hi, pl.lo]


def _planes_load(hi, lo, rows, cols) -> Planes:
    return Planes(hi, lo, rows, cols)


class _FFNBlock(torch.autograd.Function):
    """out = y + fc2(relu(fc1(LN(y))))  (layers/transformer.py:141-148) on the tensor cores.

    The normalised input and the 4H-wide hidden activation exist only as bf16 operand planes (written by the
    LayerNorm kernel and by fc1's epilogue); the backward fuses relu' into the epilogue of the fc2 input-gradient GEMM
    and the residual gradient into the LayerNorm backward.
    """

    @staticmethod
    def forward(ctx, y_nd, ln_w, ln_b, w1, b1, w2, b2):
        H = y_nd.shape[-1]
        y = y_nd.reshape(-1, H)
        if y.stride(-1) != 1 or (y.shape[0] > 1 and y.stride(0) != H):
            y = y.contiguous()
        M = y.shape[0]
        F = w1.shape[0]
        dev = y.device
        _, h0p, stats = ln_fwd_planes(y, ln_w, ln_b)
        w1p, w2p = weight_planes(w1), weight_planes(w2)
        h1p = empty_planes(M, F, dev, _with_lo())
        gate = torch.empty(F // 32, M, dtype=torch.int32, device=dev) if (gate_bits_ok(M, F) and any(ctx.needs_input_grad)) else None
        gemm_planes(M=M, N=F, K=H, a=[h0p], a_mode=L.KC, b=w1p, b_mode=L.KC, bias=b1, act=L.ACT_RELU, out_planes=h1p, out_gate=gate)
        out = torch.empty(M, H, dtype=torch.float32, device=dev)
        gemm_planes(M=M, N=H, K=F, a=[h1p], a_mode=L.KC, b=w2p, b_mode=L.KC, bias=b2, residual=y, out=out)
        ctx.save_for_backward(y, stats, ln_w, ln_b, w1, w2, *_planes_save(h0p), *_planes_save(h1p), gate)
        ctx.prec = _PRECISION
        ctx.shape = y_nd.shape
        # y is the output of an attention op whose backward wants this block's input gradient as GEMM operand planes
        ctx.emit_grad_planes = bool(getattr(y_nd, "_dost_attn_out", False))
        return out.view(y_nd.shape)

    @staticmethod
    def backward(ctx, d_out_nd):
        y, stats, ln_w, ln_b, w1, w2, h0h, h0l, h1h, h1l, gate = ctx.saved_tensors
        M, H = y.shape
        F = w1.shape[0]
        dev = y.device
        with precision_value(ctx.prec):
            h0p, h1p = _planes_load(h0h, h0l, M, H), _planes_load(h1h, h1l, M, F)
            w1p, w2p = weight_planes(w1), weight_planes(w2)
            # the LayerNorm backward that produced this gradient may already have written its operand planes and column
            # sums in the same pass (_LayerNorm.backward, `emit_grad_planes`): one pass over d_out saved
            dop = getattr(d_out_nd, "_dost_planes", None)
            db2 = getattr(d_out_nd, "_dost_colsum", None)
            d_out = d_out_nd.reshape(M, H)
            if d_out.stride(-1) != 1 or (M > 1 and d_out.stride(0) != H):
                d_out, dop = d_out.contiguous(), None
            if dop is None or db2 is None or dop.rows != M or dop.cols != H or (dop.lo is not None) != _with_lo() or \
                    getattr(d_out_nd, "_dost_planes_version", -1) != d_out_nd._version:
                dop, db2 = split_planes_colsum(d_out)
            dw2 = torch.empty(H, F, dtype=torch.float32, device=dev)
            gemm_planes(M=H, N=F, K=M, a=[dop], a_mode=L.MC, b=h1p, b_mode=L.MC, out=dw2, split_k=_split_for(H, F, M))
            # d(relu input) = (d_out W2) * relu'(h1): relu' from the sign of the saved hi plane, result as planes only
            dv1p = empty_planes(M, F, dev, _with_lo())
            db1 = torch.empty(F, dtype=torch.float32, device=dev)      # bias gradient from the epilogue that writes dv1
            # (the gates: 1 bit per element from fc1's epilogue when it wrote them, else the sign of the saved hi plane)
            gemm_planes(M=M, N=F, K=H, a=[dop], a_mode=L.KC, b=w2p, b_mode=L.MC, dact=h1p if gate is None else None,
                        dact_gate=gate, dact_slope=0.0, out_planes=dv1p, colsum_out=db1)
            dw1 = torch.empty(F, H, dtype=torch.float32, device=dev)
            gemm_planes(M=F, N=H, K=M, a=[dv1p], a_mode=L.MC, b=h0p, b_mode=L.MC, out=dw1, split_k=_split_for(F, H, M))
            dh0 = torch.empty(M, H, dtype=torch.float32, device=dev)
            gemm_planes(M=M, N=H, K=F, a=[dv1p], a_mode=L.KC, b=w1p, b_mode=L.MC, out=dh0)
            dy, dyp, dg, db, _, _ = ln_bwd_planes(dh0, y, stats, ln_w, ln_b, dres=d_out, want_planes=ctx.emit_grad_planes)
        dy = dy.view(ctx.shape)
        if dyp is not None:      # read by the attention backward when this very tensor reaches it unmodified (single consumer)
            dy._dost_planes, dy._dost_planes_version = dyp, dy._version
        return dy, dg, db, dw1, db1, dw2, db2


def ffn_block(y, ln_w, ln_b, w1, b1, w2, b2):
    """y [..., H] -> y + fc2(relu(fc1(LN(y)))) in y's shape.  The result is tagged so that a LayerNorm that consumes it
    (the next layer's LN0 / the stack's final LayerNorm) emits its input gradient as operand planes + column sums too."""
    out = _FFNBlock.apply(y, ln_w, ln_b, w1, b1, w2, b2)
    out._dost_ffn_out = True
    return out


def cols_view(pl: Planes, a: int, b: int) -> Planes:
    """Column range [a, b) of an operand (a, b multiples of 8): a strided view, nothing is copied."""
    return Planes(pl.hi[:, a:b], pl.lo[:, a:b] if pl.lo is not None else None, pl.rows, b - a)


def get_planes(t: torch.Tensor) -> Planes:
    """Planes attached to `t` by the kernel that produced it, else one conversion pass."""
    pl = getattr(t, "_dost_planes", None)
    if pl is not None and pl.rows == t.shape[0] and pl.cols == t.shape[1] and (pl.lo is not None) == _with_lo():
        return pl
    return split_planes(t)


class _EdgeBlock(torch.autograd.Function):
    """Edge update of one Processor (DOSTransformer.py:139-143,171-175 and the residual of :59):

        v = W2 PReLU(LN(W1 [x[row] | x[col] | e] + b1)) + b2 ;  e_new = e + v

    restructured with split weights W1 = [Ws | Wd | We]: the node terms P = x [Ws; Wd]^T are computed once per node
    ([N, 2W]) and gathered per edge inside the LayerNorm kernel, so the first GEMM over the E edges has K = H instead of
    3H, no [E, 3H] concatenation or gather is ever materialised, and every GEMM runs on the TMA-fed planes kernel.
    Backward: the adjoints of the two gathers are CSR segment sums (by source / by destination) of d_pre.
    Returns (e_new, v, e_new.hi, e_new.lo) or (v,) for the last layer.
    """

    @staticmethod
    def forward(ctx, x, e, w1, b1, ln_w, ln_b, slope, w2, b2, graph, last):
        N, H = x.shape
        E = e.shape[0]
        W = w1.shape[0]
        dev = x.device
        xp, ep = get_planes(x), get_planes(e)
        w1p, w2p = weight_planes(w1), weight_planes(w2)
        w_s, w_d, w_e = cols_view(w1p, 0, H), cols_view(w1p, H, 2 * H), cols_view(w1p, 2 * H, 3 * H)
        P = torch.empty(N, 2 * W, dtype=torch.float32, device=dev)
        gemm_planes(M=N, N=W, K=H, a=[xp], a_mode=L.KC, b=w_s, b_mode=L.KC, out=P[:, :W])
        gemm_planes(M=N, N=W, K=H, a=[xp], a_mode=L.KC, b=w_d, b_mode=L.KC, out=P[:, W:])
        pre = torch.empty(E, W, dtype=torch.float32, device=dev)
        gemm_planes(M=E, N=W, K=H, a=[ep], a_mode=L.KC, b=w_e, b_mode=L.KC, bias=b1, out=pre)
        _, h2p, stats = ln_fwd_planes(pre, ln_w, ln_b, slope, gather_add=(P[:, :W], graph.row, P[:, W:], graph.col))
        v = torch.empty(E, H, dtype=torch.float32, device=dev)
        ctx.graph, ctx.last, ctx.prec = graph, last, _PRECISION
        ctx.save_for_backward(w1, ln_w, ln_b, slope, w2, pre, stats, *_planes_save(xp), *_planes_save(ep), *_planes_save(h2p))
        if last:
            gemm_planes(M=E, N=H, K=W, a=[h2p], a_mode=L.KC, b=w2p, b_mode=L.KC, bias=b2, out=v)
            return v
        e_new = torch.empty(E, H, dtype=torch.float32, device=dev)
        enp = empty_planes(E, H, dev, _with_lo())
        gemm_planes(M=E, N=H, K=W, a=[h2p], a_mode=L.KC, b=w2p, b_mode=L.KC, bias=b2, out_pre=v, residual=e, out=e_new,
                    out_planes=enp)
        lo = enp.lo if enp.lo is not None else enp.hi
        ctx.mark_non_differentiable(enp.hi, lo)
        ctx.set_materialize_grads(False)
        return e_new, v, enp.hi, lo

    @staticmethod
    def backward(ctx, *grads):
        w1, ln_w, ln_b, slope, w2, pre, stats, xh, xl, eh, el, hh, hl = ctx.saved_tensors
        g: CrystalGraph = ctx.graph
        E, W = pre.shape
        N, H = xh.shape[0], w2.shape[0]
        dev = pre.device
        if ctx.last:
            d_e_new, d_v = None, grads[0]
        else:
            d_e_new, d_v = grads[0], grads[1]
        with precision_value(ctx.prec):
            xp, ep, h2p = _planes_load(xh, xl, N, H), _planes_load(eh, el, E, H), _planes_load(hh, hl, E, W)
            w1p, w2p = weight_planes(w1), weight_planes(w2)
            w_s, w_d, w_e = cols_view(w1p, 0, H), cols_view(w1p, H, 2 * H), cols_view(w1p, 2 * H, 3 * H)
            # gradient wrt v: from the aggregation path and (through e_new = e + v) from the residual stream
            if d_v is None:
                dv = d_e_new.contiguous()
            elif d_e_new is None:
                dv = d_v.contiguous()
            else:
                dv = torch.empty(E, H, dtype=torch.float32, device=dev)
                _axpy2(d_v.contiguous(), d_e_new.contiguous(), dv)
            dvp, db2 = split_planes_colsum(dv)
            dw2 = torch.empty(H, W, dtype=torch.float32, device=dev)
            gemm_planes(M=H, N=W, K=E, a=[dvp], a_mode=L.MC, b=h2p, b_mode=L.MC, out=dw2, split_k=_split_for(H, W, E))
            dh2 = torch.empty(E, W, dtype=torch.float32, device=dev)
            gemm_planes(M=E, N=W, K=H, a=[dvp], a_mode=L.KC, b=w2p, b_mode=L.MC, out=dh2)
            d_pre, dpp, dgam, dbet, dslope, db1 = ln_bwd_planes(dh2, pre, stats, ln_w, ln_b, slope, want_dx=True,
                                                                want_planes=True, want_xsum=True)
            dw1 = torch.empty(W, 3 * H, dtype=torch.float32, device=dev)
            gemm_planes(M=W, N=H, K=E, a=[dpp], a_mode=L.MC, b=ep, b_mode=L.MC, out=dw1[:, 2 * H:], split_k=_split_for(W, H, E))
            d_e = torch.empty(E, H, dtype=torch.float32, device=dev)
            gemm_planes(M=E, N=H, K=W, a=[dpp], a_mode=L.KC, b=w_e, b_mode=L.MC, out=d_e, residual=d_e_new)
            # adjoint of the two gathers: fixed-order CSR segment sums of d_pre by source and by destination node
            dP = torch.empty(N, 2 * W, dtype=torch.float32, device=dev)
            segment_reduce_raw(d_pre, g.by_src.rowptr, g.by_src.perm, N, out=dP[:, :W])
            segment_reduce_raw(d_pre, g.by_dst.rowptr, g.by_dst.perm, N, out=dP[:, W:])
            dPp = split_planes(dP)
            dps, dpd = cols_view(dPp, 0, W), cols_view(dPp, W, 2 * W)
            gemm_planes(M=W, N=H, K=N, a=[dps], a_mode=L.MC, b=xp, b_mode=L.MC, out=dw1[:, :H], split_k=_split_for(W, H, N))
            gemm_planes(M=W, N=H, K=N, a=[dpd], a_mode=L.MC, b=xp, b_mode=L.MC, out=dw1[:, H:2 * H], split_k=_split_for(W, H, N))
            dx = torch.empty(N, H, dtype=torch.float32, device=dev)
            gemm_planes(M=N, N=H, K=W, a=[dps], a_mode=L.KC, b=w_s, b_mode=L.MC, out=dx)
            gemm_planes(M=N, N=H, K=W, a=[dpd], a_mode=L.KC, b=w_d, b_mode=L.MC, out=dx, accumulate=True)
        return dx, d_e, dw1, db1, dgam, dbet, dslope, dw2, db2, None, None


def edge_block(x, e, seq, graph: CrystalGraph, last: bool):
    """seq = nn.Sequential(Linear(3H, 2H), LayerNorm(2H), PReLU, Linear(2H, H)).  Returns (e_new, v) or v (last layer)."""
    args = (x, e, seq[0].weight, seq[0].bias, seq[1].weight, seq[1].bias, seq[2].weight, seq[3].weight, seq[3].bias, graph, last)
    if last:
        return _EdgeBlock.apply(*args)
    e_new, v, hi, lo = _EdgeBlock.apply(*args)
    e_new._dost_planes = Planes(hi, lo if _with_lo() else None, e_new.shape[0], e_new.shape[1])
    return e_new, v


def planes_ok(width: int) -> bool:
    """Row widths the vectorised LayerNorm/planes kernels support."""
    return width in (128, 256, 512, 1024)


def _pick_split(M_out: int, N_out: int, K_red: int, elem: int) -> int:
    tile = 128 if elem == 4 else 64
    tiles = math.ceil(M_out / tile) * math.ceil(N_out / tile)
    want = max(1, (4 * NUM_SMS) // tiles)
    return int(max(1, min(want, math.ceil(K_red / 256), 512)))


def colsum(x2d: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    M, W = x2d.shape
    if out is None:
        out = torch.empty(W, dtype=x2d.dtype, device=x2d.device)
    lib = L.lib()
    nb = lib.dost_colsum_workspace_bytes(L.dt(x2d), M, W)
    ws = _ws(nb, x2d.device)
    L.check(lib.dost_colsum(L.dt(x2d), L.p(x2d), _ld(x2d), M, W, L.p(out), L.p(ws), nb, L.stream()), "colsum")
    return out


def segment_reduce_raw(src: torch.Tensor, rowptr: torch.Tensor, perm: Optional[torch.Tensor], nseg: int, *,
                       mean: bool = False, out: Optional[torch.Tensor] = None, accumulate: bool = False) -> torch.Tensor:
    W = src.shape[1]
    if out is None:
        assert not accumulate
        out = torch.empty(nseg, W, dtype=src.dtype, device=src.device)
    L.check(L.lib().dost_segment_reduce(L.dt(src), L.p(src), _ld(src), L.p(rowptr), L.p(perm), nseg, W,
                                        1 if mean else 0, 1 if accumulate else 0, L.p(out), _ld(out), L.stream()),
            "segment_reduce")
    return out


def gather_rows_raw(src: torch.Tensor, idx: torch.Tensor, *, deg_rowptr: Optional[torch.Tensor] = None,
                    add: Optional[torch.Tensor] = None) -> torch.Tensor:
    R, W = idx.numel(), src.shape[1]
    out = torch.empty(R, W, dtype=src.dtype, device=src.device)
    L.check(L.lib().dost_gather_rows(L.dt(src), L.p(src), _ld(src), L.p(idx), L.p(deg_rowptr), L.p(add),
                                     _ld(add) if add is not None else 0, R, W, L.p(out), _ld(out), L.stream()),
            "gather_rows")
    return out


# =====================================================================================================
# Linear with gather/concat prologue and fused epilogue
# =====================================================================================================
@dataclass
class LinearSpec:
    maps: List[Optional[RowMap]]     # one per A segment
    tensor_of_seg: List[int]         # which input tensor each segment reads (lets x feed two segments)
    M: int
    act: int = L.ACT_NONE
    act_slope: float = 0.0
    want_pre: bool = False           # also return the pre-activation / pre-residual value
    rowbias_div: int = 0             # > 0: a [M / div, N] row-group bias input follows the residual (planes path only)
    out_buf: Optional[torch.Tensor] = None   # write the result into this [M, N] row block of a larger buffer (stack2)


class _Linear(torch.autograd.Function):
    """y = act(cat_s(X_s[map_s]) @ W^T + b) (+ residual); optionally also returns the pre-activation value.

    args: spec, weight [N,K], bias [N]|None, prelu_slope [1]|None, residual [M,N]|None, *tensors
    """

    @staticmethod
    def forward(ctx, spec: LinearSpec, weight, bias, slope, residual, rowbias, *tensors):
        N, K = weight.shape
        M = spec.M
        dev = weight.device
        out = spec.out_buf if spec.out_buf is not None else torch.empty(M, N, dtype=weight.dtype, device=dev)
        assert out.shape == (M, N) and out.stride(1) == 1
        need_pre = spec.want_pre or spec.act == L.ACT_PRELU
        pre = torch.empty(M, N, dtype=weight.dtype, device=dev) if need_pre else None
        ctx.use_planes = _linear_on_planes(spec, weight, tensors)
        saved_in = tensors
        if ctx.use_planes:
            xps = [get_planes(tensors[ti]) for ti in spec.tensor_of_seg]
            gemm_planes(M=M, N=N, K=K, a=xps, a_mode=L.KC, b=weight_planes(weight), b_mode=L.KC, out=out, bias=bias,
                        rowbias=rowbias, rowbias_div=max(spec.rowbias_div, 1), act=spec.act, act_slope=spec.act_slope,
                        prelu_slope=slope, out_pre=pre, residual=residual)
            saved_in = [t for pl in xps for t in _planes_save(pl)]     # only the operand planes are needed again
        else:
            assert rowbias is None, "row-group bias needs the tensor-core path"
            segs = [(tensors[ti], spec.maps[si]) for si, ti in enumerate(spec.tensor_of_seg)]
            gemm_raw(M=M, N=N, K=K, a=segs, a_mode=L.KC, b=weight, b_mode=L.KC, out=out, bias=bias, act=spec.act,
                     act_slope=spec.act_slope, prelu_slope=slope, out_pre=pre, residual=residual)
        # (the output buffer is a view whose base is the stacked tensor that _Stack2 returns with THIS node behind it:
        # keeping it on the ctx would close a reference cycle that only the cyclic GC could free, a [2 B T, H] tensor each)
        spec.out_buf = None
        ctx.spec = spec
        ctx.prec = _PRECISION
        ctx.n_tensors = len(tensors)
        ctx.in_rows = [t.shape[0] for t in tensors]
        ctx.in_cols = [t.shape[-1] for t in tensors]
        ctx.has_bias, ctx.has_res, ctx.has_rowbias = bias is not None, residual is not None, rowbias is not None
        saved_act = None
        if spec.act in (L.ACT_RELU, L.ACT_LEAKY):
            saved_act = out
        elif spec.act == L.ACT_PRELU:
            saved_act = pre
        ctx.save_for_backward(weight, slope, saved_act, *saved_in)
        if spec.want_pre:
            return out, pre
        return out

    @staticmethod
    def backward(ctx, d_out, d_pre=None):
        spec: LinearSpec = ctx.spec
        weight, slope, saved_act, *tensors = ctx.saved_tensors
        if ctx.use_planes:
            with precision_value(ctx.prec):
                return _Linear._backward_planes(ctx, spec, weight, slope, saved_act, tensors, d_out, d_pre)
        N, K = weight.shape
        M = spec.M
        dev, dtype = weight.device, weight.dtype
        d_out = d_out.contiguous()
        d_res = d_out if ctx.has_res else None
        d_slope = None
        # ---- gradient wrt the pre-activation value v
        if spec.act == L.ACT_PRELU:
            dv = torch.empty_like(d_out)
            d_slope = torch.empty(1, dtype=dtype, device=dev)
            lib = L.lib()
            nb = lib.dost_prelu_bwd_workspace_bytes(L.dt(d_out), d_out.numel())
            ws = _ws(nb, dev)
            L.check(lib.dost_prelu_bwd(L.dt(d_out), L.p(d_out), L.p(saved_act), L.p(slope), L.p(dv), L.p(d_slope),
                                       d_out.numel(), L.p(ws), nb, L.stream()), "prelu_bwd")
            dact = None
        elif spec.act in (L.ACT_RELU, L.ACT_LEAKY):
            # dv = d_out * act'(out): the PReLU-backward kernel with a constant slope (sign(out) == sign(v) here)
            dv = torch.empty_like(d_out)
            cslope = _const(spec.act_slope if spec.act == L.ACT_LEAKY else 0.0, dtype, dev)
            junk = torch.empty(1, dtype=dtype, device=dev)
            lib = L.lib()
            nb = lib.dost_prelu_bwd_workspace_bytes(L.dt(d_out), d_out.numel())
            ws = _ws(nb, dev)
            L.check(lib.dost_prelu_bwd(L.dt(d_out), L.p(d_out), L.p(saved_act), L.p(cslope), L.p(dv), L.p(junk),
                                       d_out.numel(), L.p(ws), nb, L.stream()), "act_bwd")
            dact = None
        else:
            dv = d_out
            if spec.want_pre and d_pre is not None:
                # v feeds both outputs: out = v + residual and pre = v
                dv = torch.empty_like(d_out)
                _axpy2(d_out, d_pre.contiguous(), dv)
        needs = ctx.needs_input_grad
        # ---- bias
        d_bias = colsum(dv) if (ctx.has_bias and needs[2]) else None
        # ---- weight: dW[:, kseg] = dv^T @ X_s[map]   (reduction over the M rows, deterministic split-K)
        d_weight = None
        if needs[1]:
            d_weight = torch.empty(N, K, dtype=dtype, device=dev)
            k0 = 0
            for si, ti in enumerate(spec.tensor_of_seg):
                t = tensors[ti]
                w = t.shape[-1]
                split = _pick_split(N, w, M, weight.element_size())
                gemm_raw(M=N, N=w, K=M, a=[(dv, None)], a_mode=L.MC, b=t, b_mode=L.MC, b_map=spec.maps[si],
                         out=d_weight[:, k0:k0 + w], ldc=K, split_k=split, prec=ctx.prec)
                k0 += w
        # ---- inputs: dA = dv @ W  [M, K], then the adjoint of each row map
        d_tensors: List[Optional[torch.Tensor]] = [None] * ctx.n_tensors
        tens_needs = needs[6:]
        if any(tens_needs):
            dA = torch.empty(M, K, dtype=dtype, device=dev)
            gemm_raw(M=M, N=K, K=N, a=[(dv, None)], a_mode=L.KC, b=weight, b_mode=L.MC, out=dA, prec=ctx.prec)
            k0 = 0
            for si, ti in enumerate(spec.tensor_of_seg):
                t = tensors[ti]
                w = t.shape[-1]
                if tens_needs[ti]:
                    piece = dA[:, k0:k0 + w]
                    d_tensors[ti] = _map_adjoint(piece, spec.maps[si], t.shape[0], d_tensors[ti])
                k0 += w
        return (None, d_weight, d_bias, d_slope, d_res, None, *d_tensors)

    @staticmethod
    def _dv(ctx, spec, slope, saved_act, d_out, d_pre):
        """Gradient wrt the pre-activation value (fp32) and the PReLU slope gradient."""
        dev, dtype = d_out.device, d_out.dtype
        d_slope = None
        lib = L.lib()
        if spec.act == L.ACT_PRELU:
            dv = torch.empty_like(d_out)
            d_slope = torch.empty(1, dtype=dtype, device=dev)
            nb = lib.dost_prelu_bwd_workspace_bytes(L.dt(d_out), d_out.numel())
            ws = _ws(nb, dev)
            L.check(lib.dost_prelu_bwd(L.dt(d_out), L.p(d_out), L.p(saved_act), L.p(slope), L.p(dv), L.p(d_slope),
                                       d_out.numel(), L.p(ws), nb, L.stream()), "prelu_bwd")
        elif spec.act in (L.ACT_RELU, L.ACT_LEAKY):
            dv = torch.empty_like(d_out)
            cslope = _const(spec.act_slope if spec.act == L.ACT_LEAKY else 0.0, dtype, dev)
            junk = torch.empty(1, dtype=dtype, device=dev)
            nb = lib.dost_prelu_bwd_workspace_bytes(L.dt(d_out), d_out.numel())
            ws = _ws(nb, dev)
            L.check(lib.dost_prelu_bwd(L.dt(d_out), L.p(d_out), L.p(saved_act), L.p(cslope), L.p(dv), L.p(junk),
                                       d_out.numel(), L.p(ws), nb, L.stream()), "act_bwd")
        else:
            dv = d_out
            if spec.want_pre and d_pre is not None:
                dv = torch.empty_like(d_out)
                _axpy2(d_out, d_pre.contiguous(), dv)
        return dv, d_slope

    @staticmethod
    def _backward_planes(ctx, spec, weight, slope, saved_act, saved_planes, d_out, d_pre):
        N, K = weight.shape
        M = spec.M
        dev = weight.device
        if d_out is None:                      # only the pre-activation output was used downstream
            d_out = torch.zeros(M, N, dtype=weight.dtype, device=dev)
        d_out = d_out.contiguous()
        d_res = d_out if ctx.has_res else None
        dv, d_slope = _Linear._dv(ctx, spec, slope, saved_act, d_out, d_pre)
        needs = ctx.needs_input_grad
        if ctx.has_bias and needs[2]:
            dvp, d_bias = split_planes_colsum(dv)
        else:
            dvp, d_bias = split_planes(dv), None
        d_rowbias = None
        if ctx.has_rowbias and needs[5]:
            div = spec.rowbias_div
            groups = (M + div - 1) // div
            rp = torch.arange(0, (groups + 1) * div, div, dtype=torch.int32, device=dev).clamp_(max=M)
            d_rowbias = segment_reduce_raw(dv, rp, None, groups)
        xps = []
        for si, ti in enumerate(spec.tensor_of_seg):
            xps.append(_planes_load(saved_planes[2 * si], saved_planes[2 * si + 1], ctx.in_rows[ti], ctx.in_cols[ti]))
        d_weight = None
        Kp = _pad8(K)          # K % 8 != 0 only for a single segment: gradients are computed at the zero-padded width
        if needs[1]:
            d_weight = torch.empty(N, Kp, dtype=torch.float32, device=dev)
            k0 = 0
            for si, ti in enumerate(spec.tensor_of_seg):
                w = ctx.in_cols[ti]
                wp_ = _pad8(w)
                xb = xps[si] if wp_ == w else Planes(xps[si].hi, xps[si].lo, xps[si].rows, wp_)
                gemm_planes(M=N, N=wp_, K=M, a=[dvp], a_mode=L.MC, b=xb, b_mode=L.MC, out=d_weight[:, k0:k0 + wp_],
                            split_k=_split_for(N, wp_, M))
                k0 += w
            if Kp != K:
                d_weight = d_weight[:, :K].contiguous()
        d_tensors: List[Optional[torch.Tensor]] = [None] * ctx.n_tensors
        tens_needs = needs[6:]
        if any(tens_needs):
            dA = torch.empty(M, Kp, dtype=torch.float32, device=dev)
            wpl = weight_planes(weight)
            if Kp != K:
                wpl = Planes(wpl.hi, wpl.lo, wpl.rows, Kp)
            gemm_planes(M=M, N=Kp, K=N, a=[dvp], a_mode=L.KC, b=wpl, b_mode=L.MC, out=dA)
            if Kp != K:
                dA = dA[:, :K].contiguous()
            k0 = 0
            for si, ti in enumerate(spec.tensor_of_seg):
                w = ctx.in_cols[ti]
                if tens_needs[ti]:
                    d_tensors[ti] = _map_adjoint(dA[:, k0:k0 + w], None, ctx.in_rows[ti], d_tensors[ti])
                k0 += w
        return (None, d_weight, d_bias, d_slope, d_res, d_rowbias, *d_tensors)


def planes_gemm_ok(M: int, N: int, K: int, single_segment: bool = False) -> bool:
    """Problem sizes worth a 128 x N tensor-core tile whose operands satisfy the TMA alignment rules.  A single-segment
    operand may have any width: its planes are zero-padded to a multiple of 8 columns (e.g. the 41 Gaussian distance
    features of the edge encoder) and the gradients are computed at the padded width."""
    return M >= 128 and N % 8 == 0 and (K % 8 == 0 or single_segment) and M * N * max(K, 32) >= (1 << 22)


def _linear_on_planes(spec: LinearSpec, weight: torch.Tensor, tensors) -> bool:
    """Plain (un-mapped) fp32 segments of TMA-friendly widths go to the TMA-fed tensor-core kernel."""
    if not tc_active(weight) or L.switch("DOST_NO_LINPLANES"):
        return False
    N, K = weight.shape
    if not planes_gemm_ok(spec.M, N, K, single_segment=len(spec.maps) == 1):
        return False
    if any(m is not None and (m.idx is not None or m.div != 1) for m in spec.maps):
        return False
    if len(spec.maps) > 1 and any(tensors[ti].shape[-1] % 64 != 0 for ti in spec.tensor_of_seg):
        return False
    return len(spec.maps) <= 3


def _axpy2(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor) -> None:
    """out = a + b through the row-gather kernel (identity rows), keeping elementwise math in our kernels."""
    R, W = a.shape
    idx = _arange_i32(R, a.device)
    L.check(L.lib().dost_gather_rows(L.dt(a), L.p(a), _ld(a), L.p(idx), None, L.p(b), _ld(b), R, W, L.p(out), _ld(out),
                                     L.stream()), "add")


_ARANGE_CACHE = {}
_CONST_CACHE = {}


def _const(value: float, dtype, device) -> torch.Tensor:
    key = (float(value), dtype, str(device))
    if key not in _CONST_CACHE:
        _CONST_CACHE[key] = torch.full((1,), float(value), dtype=dtype, device=device)
    return _CONST_CACHE[key]


_ARANGE_RETIRED = []     # outgrown index tensors stay alive: captured CUDA graphs (graphed.GraphedStep) hold their addresses


def _arange_i32(n: int, device) -> torch.Tensor:
    key = (str(device), )
    cur = _ARANGE_CACHE.get(key)
    if cur is None or cur.numel() < n:
        if cur is not None:
            # never free the old one: a graph captured while it was current replays kernels that read it (a freed block is
            # re-used by the allocator and the graph then gathers through garbage indices: an illegal address in the
            # large-cell bench, where the second batch has more edges than the first)
            _ARANGE_RETIRED.append(cur)
        cur = torch.arange(max(2 * n, 1 << 20), dtype=torch.int32, device=device)
        _ARANGE_CACHE[key] = cur
    return cur[:n]


def _map_adjoint(piece: torch.Tensor, m: Optional[RowMap], n_src_rows: int, acc: Optional[torch.Tensor]) -> torch.Tensor:
    """Adjoint of row gather/broadcast: reduce the [M, w] gradient onto the source rows (fixed order)."""
    if m is None or (m.idx is None and m.div == 1):
        if acc is None:
            return piece
        out = torch.empty_like(acc)
        _axpy2(acc, piece, out)
        return out
    cur = piece
    if m.div > 1:
        assert m.div_rowptr is not None
        groups = m.div_rowptr.numel() - 1
        if m.idx is None:
            return segment_reduce_raw(cur, m.div_rowptr, None, groups, out=acc, accumulate=acc is not None)
        cur = segment_reduce_raw(cur, m.div_rowptr, None, groups)
    assert m.csr is not None, "row map used in a differentiable position needs its CSR"
    if acc is None:
        return segment_reduce_raw(cur, m.csr.rowptr, m.csr.perm, n_src_rows)
    return segment_reduce_raw(cur, m.csr.rowptr, m.csr.perm, n_src_rows, out=acc, accumulate=True)


class _RowDot(torch.autograd.Function):
    """Linear(H -> 1): y[m] = x[m, :] . w + b as streaming kernels (out_layer, DOSTransformer.py:75,89)."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        M, K = x.shape
        out = torch.empty(M, 1, dtype=torch.float32, device=x.device)
        L.check(L.lib().dost_rowdot_fwd(L.p(x), _ld(x), L.p(weight), L.p(bias), L.p(out), M, K, L.stream()), "rowdot_fwd")
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return out

    @staticmethod
    def backward(ctx, d_out):
        x, weight = ctx.saved_tensors
        M, K = x.shape
        dev = x.device
        d_out = d_out.contiguous()
        dx = torch.empty(M, K, dtype=torch.float32, device=dev) if ctx.needs_input_grad[0] else None
        dwb = torch.empty(K + 1, dtype=torch.float32, device=dev)
        lib = L.lib()
        nb = lib.dost_rowdot_bwd_workspace_bytes(M, K)
        ws = _ws(nb, dev)
        L.check(lib.dost_rowdot_bwd(L.p(d_out), L.p(x), _ld(x), L.p(weight), L.p(dx), L.p(dwb), M, K, L.p(ws), nb, L.stream()),
                "rowdot_bwd")
        return dx, dwb[:K].view(1, K), (dwb[K:].view(1) if ctx.has_bias else None)


def linear(segments: Sequence[Tuple[torch.Tensor, Optional[RowMap]]], weight: torch.Tensor,
           bias: Optional[torch.Tensor], *, M: Optional[int] = None, act: int = L.ACT_NONE, act_slope: float = 0.0,
           prelu_slope: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
           want_pre: bool = False, rowbias: Optional[torch.Tensor] = None, rowbias_div: int = 0,
           out_buf: Optional[torch.Tensor] = None):
    """Fused Linear.  ``segments`` are concatenated along the feature axis; a tensor may appear in several.
    ``rowbias`` [ceil(M / rowbias_div), N] is added to row m as rowbias[m // rowbias_div] (tensor-core path only).
    ``out_buf``: a [M, N] row block of a larger buffer to write the result into (see stack2)."""
    if (weight.shape[0] == 1 and len(segments) == 1 and segments[0][1] is None and act == L.ACT_NONE and residual is None
            and not want_pre and rowbias is None and out_buf is None and weight.dtype == torch.float32 and weight.shape[1] in (128, 256, 512)
            and weight.is_contiguous()):
        x = segments[0][0]
        if x.dim() == 2 and x.stride(1) == 1 and x.stride(0) % 4 == 0 and x.data_ptr() % 16 == 0:
            return _RowDot.apply(x, weight, bias)
    tensors: List[torch.Tensor] = []
    tos: List[int] = []
    for t, _ in segments:
        for i, u in enumerate(tensors):
            if u is t:
                tos.append(i)
                break
        else:
            tensors.append(t)
            tos.append(len(tensors) - 1)
    if M is None:
        t0, m0 = segments[0]
        assert m0 is None or (m0.idx is None and m0.div == 1)
        M = t0.shape[0]
    spec = LinearSpec([m for _, m in segments], tos, M, act, act_slope, want_pre, rowbias_div if rowbias is not None else 0,
                      out_buf)
    return _Linear.apply(spec, weight, bias, prelu_slope, residual, rowbias, *tensors)


class _Box:
    """Keeps a tensor out of autograd's sight when passed to Function.apply."""

    def __init__(self, t):
        self.t = t


class _Stack2(torch.autograd.Function):
    """[a; b] along the rows WITHOUT a copy: a and b are the two row blocks of ``buf`` already (their producers wrote
    there through ``linear(out_buf=...)``).  Backward hands each producer its row block of the gradient (views)."""

    @staticmethod
    def forward(ctx, a, b, box):
        buf = box.t
        ra = a.shape[0]
        assert a.data_ptr() == buf.data_ptr() and b.data_ptr() == buf[ra:].data_ptr() and ra + b.shape[0] == buf.shape[0]
        ctx.ra = ra
        return buf

    @staticmethod
    def backward(ctx, d):
        return d[:ctx.ra], d[ctx.ra:], None


def stack2_buffer(rows_a: int, rows_b: int, cols: int, like: torch.Tensor):
    """(buf, view_a, view_b): one [rows_a + rows_b, cols] buffer and its two row blocks, to be filled by two
    ``linear(..., out_buf=view)`` calls and then joined with ``stack2``."""
    buf = torch.empty(rows_a + rows_b, cols, dtype=like.dtype, device=like.device)
    return buf, buf[:rows_a], buf[rows_a:]


def stack2(a: torch.Tensor, b: torch.Tensor, buf: torch.Tensor) -> torch.Tensor:
    return _Stack2.apply(a, b, _Box(buf))


# =====================================================================================================
# LayerNorm (+PReLU)
# =====================================================================================================
class _LayerNorm(torch.autograd.Function):
    """outputs: y [, planes hi, lo] [, x passed through].  The pass-through output lets a residual block
    ``out = x + f(LN(x))`` hand BOTH uses of x to this node: backward then adds the residual gradient inside the LayerNorm
    backward kernel (``dres``) instead of autograd launching a separate add over the [S, T, H] stream."""

    @staticmethod
    def forward(ctx, x, gamma, beta, slope, want_planes=False, with_residual=False):
        x2 = x.reshape(-1, x.shape[-1])
        if x2.stride(-1) != 1:
            x2 = x2.contiguous()
        M, W = x2.shape
        ctx.vec = x.dtype == torch.float32 and planes_ok(W) and x2.stride(0) % 4 == 0 and x2.data_ptr() % 16 == 0 \
            and not L.switch("DOST_NO_LNVEC")
        ctx.n_planes = 0
        ctx.with_residual = with_residual
        ctx.shape = x.shape
        # x is the output of an FFN block whose backward wants this node's dx as GEMM operand planes + its column sums
        ctx.emit_grad_planes = bool(getattr(x, "_dost_ffn_out", False)) and _PRECISION != L.PREC_FMA
        ctx.prec = _PRECISION
        outs = []
        if ctx.vec:       # 16-byte vectorised fp32 kernels (rows_bf.cu)
            y, pl, stats = ln_fwd_planes(x2, gamma, beta, slope, want_y=True, want_planes=want_planes)
            outs.append(y.view(x.shape))
            if want_planes:
                ctx.n_planes = 2
                lo = pl.lo if pl.lo is not None else pl.hi
                ctx.mark_non_differentiable(pl.hi, lo)
                outs += [pl.hi, lo]
        else:
            assert not want_planes
            y = torch.empty(M, W, dtype=x.dtype, device=x.device)
            stats = torch.empty(M, 2, dtype=x.dtype, device=x.device)
            L.check(L.lib().dost_ln_fwd(L.dt(x), L.p(x2), _ld(x2), L.p(gamma), L.p(beta), L.p(slope), L.p(y), L.p(stats), M, W,
                                        L.stream()), "ln_fwd")
            outs.append(y.view(x.shape))
        ctx.save_for_backward(x2, gamma, beta, slope, stats)
        ctx.set_materialize_grads(False)
        if with_residual:
            outs.append(x.view_as(x))
        return outs[0] if len(outs) == 1 else tuple(outs)

    @staticmethod
    def backward(ctx, dy, *rest):
        x2, gamma, beta, slope, stats = ctx.saved_tensors
        M, W = x2.shape
        d_res = rest[ctx.n_planes] if ctx.with_residual else None
        if d_res is not None:
            d_res = d_res.reshape(M, W)
            if d_res.stride(-1) != 1:
                d_res = d_res.contiguous()
        if dy is None:                    # only the pass-through was used downstream
            return (d_res.view(ctx.shape) if d_res is not None else None), None, None, None, None, None
        dy2 = dy.reshape(M, W)
        if dy2.stride(-1) != 1:
            dy2 = dy2.contiguous()
        if ctx.vec and dy2.stride(0) % 4 == 0 and dy2.data_ptr() % 16 == 0 and \
                (d_res is None or (d_res.stride(0) % 4 == 0 and d_res.data_ptr() % 16 == 0)):
            if ctx.emit_grad_planes:
                with precision_value(ctx.prec):
                    dx, pl, dg, db, ds, xs = ln_bwd_planes(dy2, x2, stats, gamma, beta, slope, dres=d_res, want_planes=True,
                                                           want_xsum=True)
                out = dx.view(ctx.shape)
                # read by _FFNBlock.backward when this very tensor object reaches it unmodified (single consumer; an
                # in-place accumulation by autograd would bump the version counter)
                out._dost_planes, out._dost_colsum, out._dost_planes_version = pl, xs, out._version
                return out, dg, db, ds, None, None
            dx, _, dg, db, ds, _ = ln_bwd_planes(dy2, x2, stats, gamma, beta, slope, dres=d_res)
            return dx.view(ctx.shape), dg, db, ds, None, None
        dev, dtype = x2.device, x2.dtype
        dx = torch.empty(M, W, dtype=dtype, device=dev)
        dg = torch.empty(W, dtype=dtype, device=dev)
        db = torch.empty(W, dtype=dtype, device=dev)
        ds = torch.empty(1, dtype=dtype, device=dev) if slope is not None else None
        lib = L.lib()
        nb = lib.dost_ln_bwd_workspace_bytes(L.dt(x2), M, W)
        ws = _ws(nb, dev)
        L.check(lib.dost_ln_bwd(L.dt(x2), L.p(dy2), _ld(dy2), L.p(x2), _ld(x2), L.p(stats), L.p(gamma), L.p(beta),
                                L.p(slope), L.p(dx), L.p(dg), L.p(db), L.p(ds), M, W, L.p(ws), nb, L.stream()), "ln_bwd")
        if d_res is not None:
            out = torch.empty_like(dx)
            _axpy2(dx, d_res, out)
            dx = out
        return dx.view(ctx.shape), dg, db, ds, None, None


def layer_norm(x, gamma, beta, prelu_slope=None, want_planes: bool = False, with_residual: bool = False):
    """LayerNorm (+PReLU).  want_planes: also emit the result as GEMM operand planes (attached to the returned tensor as
    ``_dost_planes``; only on the vectorised fp32 path).  with_residual: returns (LN(x), x) where the second output is x
    routed through this node, to be used as the residual operand of the block (see _LayerNorm)."""
    planes = False
    if want_planes and x.dtype == torch.float32 and planes_ok(x.shape[-1]) and tc_active(x) and \
            not L.switch("DOST_NO_LNVEC"):
        x2 = x.reshape(-1, x.shape[-1])
        planes = x2.stride(-1) == 1 and x2.stride(0) % 4 == 0 and x2.data_ptr() % 16 == 0
    res = _LayerNorm.apply(x, gamma, beta, prelu_slope, planes, with_residual)
    if not planes and not with_residual:
        return res
    y = res[0]
    if planes:
        y._dost_planes = Planes(res[1], res[2] if _with_lo() else None, x.numel() // x.shape[-1], x.shape[-1])
    return (y, res[-1]) if with_residual else y


# =====================================================================================================
# segmented reduction (scatter_sum / scatter_mean / pooling)
# =====================================================================================================
class _SegmentReduce(torch.autograd.Function):
    @staticmethod
    def forward(ctx, src, csr: CSR, mean: bool):
        ctx.csr, ctx.mean = csr, mean
        return segment_reduce_raw(src.contiguous(), csr.rowptr, csr.perm, csr.size, mean=mean)

    @staticmethod
    def backward(ctx, d_out):
        csr: CSR = ctx.csr
        d_src = gather_rows_raw(d_out.contiguous(), csr.key, deg_rowptr=csr.rowptr if ctx.mean else None)
        return d_src, None, None


def segment_reduce(src, csr: CSR, mean: bool = False):
    return _SegmentReduce.apply(src, csr, mean)


# =====================================================================================================
# cross attention energy tokens -> atoms (ragged, phantom keys)
# =====================================================================================================
class _CrossAttention(torch.autograd.Function):
    """out = resid + softmax(q kv^T / sqrt(H)) kv over the atoms of each sequence's crystal plus
    (nmax - n_b) phantom keys equal to ``phantom``.  q/resid: [S,T,H] or [T,H] (broadcast over S).
    seed_offset: optional 1-element int64 device tensor added to ``seed`` by the kernels (dost.h, ``_dseed`` entry points)."""

    @staticmethod
    def forward(ctx, q, kv, phantom, resid, graph: CrystalGraph, S: int, drop_p: float, seed: int, seed_offset=None, maps_out=None):
        H = kv.shape[1]
        T = q.shape[-2]
        q, resid = q.contiguous(), resid.contiguous()
        q_ss = T * H if q.dim() == 3 else 0
        r_ss = T * H if resid.dim() == 3 else 0
        out = torch.empty(S, T, H, dtype=kv.dtype, device=kv.device)
        lse = torch.empty(S, T, dtype=torch.float32, device=kv.device)
        scale = float(H) ** -0.5
        L.check(L.lib().dost_xattn_fwd_dseed(L.dt(kv), L.p(q), q_ss, L.p(kv), L.p(phantom), L.p(graph.ptr), L.p(graph.nmax),
                                             L.p(resid), r_ss, L.p(out), L.p(lse), S, graph.B, T, H, scale, drop_p, seed,
                                             L.p(seed_offset), L.stream()), "xattn_fwd")
        if maps_out is not None:      # the probabilities once more, from the log-sum-exp
            L.check(L.lib().dost_xattn_probs(L.dt(kv), L.p(q), q_ss, L.p(kv), L.p(phantom), L.p(graph.ptr), L.p(graph.nmax), L.p(lse),
                                             L.p(maps_out), maps_out.shape[-1], S, graph.B, T, H, scale, drop_p, seed,
                                             L.p(seed_offset), L.stream()), "xattn_probs")
        ctx.save_for_backward(q, kv, phantom, resid, out, lse)
        ctx.graph, ctx.S, ctx.drop_p, ctx.seed, ctx.seed_offset = graph, S, drop_p, seed, seed_offset
        ctx.q_ss, ctx.r_ss = q_ss, r_ss
        return out

    @staticmethod
    def backward(ctx, d_out):
        q, kv, phantom, resid, out, lse = ctx.saved_tensors
        g: CrystalGraph = ctx.graph
        S = ctx.S
        H, T = kv.shape[1], out.shape[1]
        d_out = d_out.contiguous()
        dev, dtype = kv.device, kv.dtype
        dq = torch.empty(S, T, H, dtype=dtype, device=dev)
        dkv = torch.empty_like(kv)
        dph = torch.empty(H, dtype=dtype, device=dev)
        lib = L.lib()
        nb = lib.dost_xattn_bwd_workspace_bytes(L.dt(kv), S, T, H)
        ws = _ws(nb, dev)
        L.check(lib.dost_xattn_bwd_dseed(L.dt(kv), L.p(d_out), L.p(q), ctx.q_ss, L.p(kv), L.p(phantom), L.p(g.ptr),
                                         L.p(g.batch), L.p(g.nmax), L.p(out), L.p(resid), ctx.r_ss, L.p(lse), L.p(dq), L.p(dkv),
                                         L.p(dph), S, g.B, T, H, g.N, float(H) ** -0.5, ctx.drop_p, ctx.seed,
                                         L.p(ctx.seed_offset), L.p(ws), nb, L.stream()), "xattn_bwd")
        d_q = dq if ctx.q_ss else colsum(dq.view(S, T * H)).view(T, H)
        d_resid = d_out if ctx.r_ss else colsum(d_out.view(S, T * H)).view(T, H)
        return d_q, dkv, dph, d_resid, None, None, None, None, None, None


def _grad_planes(d_out: torch.Tensor, rows: int, cols: int) -> Planes:
    """Operand planes of an incoming gradient: those its producer attached (the FFN block's LayerNorm backward writes them in
    the same pass, `_FFNBlock.backward`), if the tensor arrived unmodified; else one conversion pass."""
    pl = getattr(d_out, "_dost_planes", None)
    if (pl is not None and pl.rows == rows and pl.cols == cols and (pl.lo is not None) == _with_lo() and d_out.is_contiguous()
            and getattr(d_out, "_dost_planes_version", -1) == d_out._version):
        return pl
    return split_planes(d_out.reshape(rows, cols))


def fused_attention_ok(H: int, max_keys: int, drop_p: float = 0.0) -> bool:
    """True when the single-kernel attention forward (csrc/attn_fused.cu: QK^T -> fp32 softmax -> PK with the scores in
    TMEM) covers this call: at most 256 keys per sequence, H in {64, 128, 192, 256}.  Attention dropout is applied inside
    the kernel (same counter-based mask as the unfused kernels).  DOST_NO_ATTN_FUSED=1 switches it off."""
    return (H % 64 == 0 and 64 <= H <= 256 and 1 <= max_keys <= 256 and _PRECISION != L.PREC_FMA
            and not L.switch("DOST_NO_ATTN_FUSED"))


def _fused_attention_fwd(qp: Planes, kp: Planes, k_rows: int, S: int, Lq: int, Lk: int, H: int, rowoff, count, nmax, max_keys: int,
                         resid2d, res_seq_stride: int, out2d, pp: Optional[Planes], drop_p: float = 0.0, seed: int = 0, lse=None,
                         seed_offset=None):
    L.check(L.lib().dost_attn_fused_fwd_dseed(L.p(qp.hi), L.p(qp.lo), qp.ld, L.p(kp.hi), L.p(kp.lo), kp.ld, k_rows, S, Lq, Lk, H,
                                              L.p(rowoff), L.p(count), L.p(nmax), max_keys, float(H) ** -0.5, L.p(resid2d),
                                              res_seq_stride, L.p(out2d), L.p(pp.hi) if pp is not None else None,
                                              L.p(pp.lo) if pp is not None else None, pp.ld if pp is not None else 0, _PRECISION,
                                              float(drop_p), int(seed), L.p(seed_offset), L.p(lse), L.stream()), "attn_fused_fwd")


def _ds_from_planes(pp: Planes, dP2d: torch.Tensor, rows: int, cols: int, scale: float, dsp: Planes):
    L.check(L.lib().dost_softmax_bwd_from_planes(L.p(pp.hi), L.p(pp.lo), pp.ld, L.p(dP2d), dP2d.stride(0), rows, cols, scale,
                                                 L.p(dsp.hi), L.p(dsp.lo), dsp.ld, L.stream()), "softmax_bwd_from_planes")


class _CrossAttentionTC(torch.autograd.Function):
    """The same attention with its contractions on the tensor cores: ragged batched GEMMs (one problem per sequence, the
    keys of its crystal addressed by a row offset into one extended key plane that carries a phantom-key row per
    crystal), fp32 softmax in between (csrc/xattn_tc.cu).  S = reps * B sequences (sequence s attends to crystal s % B: the
    global and the system branch of DOSTransformer.py:71-91 batched together); attention dropout is applied by the softmax
    kernel when it writes the probability planes.  Needs the padding length on the host."""

    @staticmethod
    def forward(ctx, q, kv, phantom, resid, graph: CrystalGraph, qpl: Optional[Planes], S: int, drop_p: float = 0.0, seed: int = 0,
                seed_offset=None, maps_out=None):
        N, H = kv.shape
        B = graph.B
        T = q.shape[-2]
        reps = S // B
        dev = kv.device
        lib = L.lib()
        npad = _pad8(graph.nkeys_host)
        ptr_ext, n_ext = graph.ragged(reps)
        q, resid = q.contiguous(), resid.contiguous()
        bcast_q = q.dim() == 2
        if bcast_q:                       # first layer of the first stack: every crystal shares the energy embeddings
            q3 = gather_rows_raw(q, graph.token_mod(T))
            qp = split_planes(q3)
        else:
            qp = qpl if qpl is not None else split_planes(q.view(S * T, H))
        kvp = empty_planes(N + B, H, dev, _with_lo())
        L.check(lib.dost_xattn_kv_ext_build(L.p(kv), L.p(phantom), L.p(graph.batch), L.p(graph.ptr), N, B, H, L.p(kvp.hi), L.p(kvp.lo),
                                            kvp.ld, L.stream()), "xattn_kv_ext_build")
        out = torch.empty(S, T, H, dtype=torch.float32, device=dev)
        r2 = resid.view(-1, H)
        ctx.graph, ctx.prec, ctx.npad = graph, _PRECISION, npad
        ctx.bcast_q, ctx.bcast_r, ctx.T, ctx.S = bcast_q, resid.dim() == 2, T, S
        ctx.drop_p, ctx.seed, ctx.seed_offset = drop_p, seed, seed_offset
        ctx.fused = fused_attention_ok(H, graph.nkeys_host, drop_p)
        if ctx.fused:
            # one kernel: scores stay in TMEM, the probabilities leave only as the operand planes the backward needs
            need = any(ctx.needs_input_grad[:4])
            pp = empty_planes(S * T, npad, dev, _with_lo()) if (need or maps_out is not None) else None
            # with dropout the planes hold the dropped-out probabilities; the backward recomputes P from the log-sum-exp
            lse = torch.empty(S * T, dtype=torch.float32, device=dev) if (need and drop_p > 0) else None
            _fused_attention_fwd(qp, kvp, N + B, S, T, 0, H, ptr_ext, n_ext, graph.nmax, graph.nkeys_host, r2,
                                 0 if resid.dim() == 2 else T * H, out.view(S * T, H), pp, drop_p, seed, lse, seed_offset)
            if maps_out is not None:
                _maps_from_planes(pp, maps_out, S * T, graph, T, drop_p, seed, seed_offset)
            if need:
                ctx.save_for_backward(kv, phantom, None, lse, *_planes_save(qp), *_planes_save(kvp), *_planes_save(pp))
            return out
        scores = torch.empty(S * T, npad, dtype=torch.float32, device=dev)
        gemm_planes(M=T, N=npad, K=H, a=[qp], a_mode=L.KC, b=kvp, b_mode=L.KC, b_rows=N + B, out=scores, batch=S,
                    a_bstride=T * qp.ld, c_bstride=T * npad, b_rowoff=ptr_ext)
        pp = empty_planes(S * T, npad, dev, _with_lo())
        lse = torch.empty(S * T, dtype=torch.float32, device=dev)
        scale = float(H) ** -0.5
        L.check(lib.dost_xattn_softmax_fwd_dseed(L.p(scores), L.p(graph.ptr), L.p(graph.nmax), S * T, B, T, npad, scale, L.p(pp.hi),
                                                 L.p(pp.lo), pp.ld, L.p(lse), drop_p, seed, L.p(seed_offset), L.stream()),
                "xattn_softmax_fwd")
        if maps_out is not None:
            _maps_from_planes(pp, maps_out, S * T, graph, T, drop_p, seed, seed_offset)
        gemm_planes(M=T, N=H, K=npad, a=[pp], a_mode=L.KC, b=kvp, b_mode=L.MC, b_rows=N + B, out=out.view(S * T, H), residual=r2,
                    batch=S, a_bstride=T * pp.ld, c_bstride=T * H, res_bstride=(0 if resid.dim() == 2 else T * H),
                    b_rowoff=ptr_ext)
        ctx.save_for_backward(kv, phantom, scores, lse, *_planes_save(qp), *_planes_save(kvp), *_planes_save(pp))
        return out

    @staticmethod
    def backward(ctx, d_out):
        kv, phantom, scores, lse, qh, ql, kh, kl, ph, pl_ = ctx.saved_tensors
        g: CrystalGraph = ctx.graph
        N, H = kv.shape
        B, T, npad = g.B, ctx.T, ctx.npad
        S = ctx.S
        reps = S // B
        dev = kv.device
        lib = L.lib()
        with precision_value(ctx.prec):
            ptr_ext, n_ext = g.ragged(reps)
            qp, kvp, pp = Planes(qh, ql, S * T, H), Planes(kh, kl, N + B, H), Planes(ph, pl_, S * T, npad)
            dop = _grad_planes(d_out, S * T, H)
            d_out = d_out.contiguous()
            # dP = dO k^T
            dP = torch.empty(S * T, npad, dtype=torch.float32, device=dev)
            gemm_planes(M=T, N=npad, K=H, a=[dop], a_mode=L.KC, b=kvp, b_mode=L.KC, b_rows=N + B, out=dP, batch=S,
                        a_bstride=T * dop.ld, c_bstride=T * npad, b_rowoff=ptr_ext)
            dsp = empty_planes(S * T, npad, dev, _with_lo())
            if ctx.fused and ctx.drop_p > 0:      # the scores once more (one ragged GEMM), then the softmax backward below
                scores = torch.empty(S * T, npad, dtype=torch.float32, device=dev)
                gemm_planes(M=T, N=npad, K=H, a=[qp], a_mode=L.KC, b=kvp, b_mode=L.KC, b_rows=N + B, out=scores, batch=S,
                            a_bstride=T * qp.ld, c_bstride=T * npad, b_rowoff=ptr_ext)
            if ctx.fused and ctx.drop_p == 0:      # probabilities from their saved planes (the phantom column behaves like one key of its total mass)
                _ds_from_planes(pp, dP, S * T, npad, float(H) ** -0.5, dsp)
            else:
                L.check(lib.dost_xattn_softmax_bwd_dseed(L.p(scores), L.p(lse), L.p(dP), L.p(g.ptr), L.p(g.nmax), S * T, B, T, npad,
                                                         float(H) ** -0.5, L.p(dsp.hi), L.p(dsp.lo), dsp.ld, ctx.drop_p, ctx.seed,
                                                         L.p(ctx.seed_offset), L.stream()), "xattn_softmax_bwd")
            # dQ = dS k
            dq = torch.empty(S, T, H, dtype=torch.float32, device=dev)
            gemm_planes(M=T, N=H, K=npad, a=[dsp], a_mode=L.KC, b=kvp, b_mode=L.MC, b_rows=N + B, out=dq.view(S * T, H), batch=S,
                        a_bstride=T * dsp.ld, c_bstride=T * H, b_rowoff=ptr_ext)
            # d(extended keys) = dS^T q + P^T dO, written at each crystal's rows of the extended plane
            # (sequences s and s + B write the same crystal's rows: one launch per repetition, accumulating in order)
            dkv = torch.empty(N, H, dtype=torch.float32, device=dev)
            dbrows = torch.empty(B, H, dtype=torch.float32, device=dev)
            if not L.switch("DOST_NO_XATTN_PADDED_DK"):
                # per SEQUENCE into a padded buffer: plain batched problems (TMA store, then a TMA reduction store for the
                # second product) instead of ragged accumulating ones per repetition; the split kernel sums the repetitions
                dpad = torch.empty(S * npad, H, dtype=torch.float32, device=dev)
                gemm_planes(M=npad, N=H, K=T, a=[dsp], a_mode=L.MC, b=qp, b_mode=L.MC, out=dpad, batch=S, a_bstride=T * dsp.ld,
                            b_bstride=T * qp.ld, c_bstride=npad * H)
                gemm_planes(M=npad, N=H, K=T, a=[pp], a_mode=L.MC, b=dop, b_mode=L.MC, out=dpad, accumulate=True, batch=S,
                            a_bstride=T * pp.ld, b_bstride=T * dop.ld, c_bstride=npad * H)
                L.check(lib.dost_xattn_kv_pad_split(L.p(dpad), npad, reps, L.p(g.batch), L.p(g.ptr), N, B, H, L.p(dkv), L.p(dbrows),
                                                    L.stream()), "xattn_kv_pad_split")
                dph = colsum(dbrows)
                d_q = colsum(dq.view(S, T * H)).view(T, H) if ctx.bcast_q else dq
                d_resid = colsum(d_out.view(S, T * H)).view(T, H) if ctx.bcast_r else d_out
                return d_q, dkv, dph, d_resid, None, None, None, None, None, None, None
            dext = torch.empty(N + B, H, dtype=torch.float32, device=dev)
            p1, n1 = g.ragged(1)
            for rep in range(reps):
                r0, r1 = rep * B * T, (rep + 1) * B * T
                gemm_planes(M=npad, N=H, K=T, a=[_rows(dsp, r0, r1)], a_mode=L.MC, b=_rows(qp, r0, r1), b_mode=L.MC, out=dext,
                            accumulate=rep > 0, batch=B, a_bstride=T * dsp.ld, b_bstride=T * qp.ld, c_rowoff=p1, c_rowlim=n1)
                gemm_planes(M=npad, N=H, K=T, a=[_rows(pp, r0, r1)], a_mode=L.MC, b=_rows(dop, r0, r1), b_mode=L.MC, out=dext,
                            accumulate=True, batch=B, a_bstride=T * pp.ld, b_bstride=T * dop.ld, c_rowoff=p1, c_rowlim=n1)
            L.check(lib.dost_xattn_kv_ext_split(L.p(dext), L.p(g.batch), L.p(g.ptr), N, B, H, L.p(dkv), L.p(dbrows), L.stream()),
                    "xattn_kv_ext_split")
            dph = colsum(dbrows)
            d_q = colsum(dq.view(S, T * H)).view(T, H) if ctx.bcast_q else dq
            d_resid = colsum(d_out.view(S, T * H)).view(T, H) if ctx.bcast_r else d_out
        return d_q, dkv, dph, d_resid, None, None, None, None, None, None, None


def _maps_from_planes(pp: Planes, maps_out: torch.Tensor, rows: int, graph: Optional[CrystalGraph], T: int = 0, drop_p: float = 0.0,
                      seed: int = 0, seed_offset=None) -> None:
    """Attention maps from probability planes (dost_attn_maps_from_planes): ragged with the graph (phantom column expanded into
    the padded key slots, the dropout mask of the forward regenerated there), dense without."""
    B = graph.B if graph is not None else 0
    L.check(L.lib().dost_attn_maps_from_planes(L.p(pp.hi), L.p(pp.lo), pp.ld, rows, maps_out.shape[-1], T, B,
                                               L.p(graph.ptr) if graph is not None else None,
                                               L.p(graph.nmax) if graph is not None else None, L.p(maps_out), float(drop_p), int(seed),
                                               L.p(seed_offset), L.stream()), "attn_maps_from_planes")


def _rows(pl: Planes, r0: int, r1: int) -> Planes:
    """Row range [r0, r1) of an operand (a view)."""
    return Planes(pl.hi[r0:r1], pl.lo[r0:r1] if pl.lo is not None else None, r1 - r0, pl.cols)


def _check_seed_offset(seed_offset) -> None:
    if seed_offset is not None and (seed_offset.dtype != torch.int64 or seed_offset.numel() != 1):
        raise ValueError("seed_offset must be a 1-element int64 CUDA tensor")


def _check_maps_out(maps_out, lead, like: torch.Tensor) -> None:
    if maps_out is not None and (maps_out.dim() != 3 or tuple(maps_out.shape[:2]) != tuple(lead) or maps_out.dtype != like.dtype
                                 or maps_out.device != like.device or not maps_out.is_contiguous()):
        raise ValueError(f"maps_out must be a contiguous [{lead[0]}, {lead[1]}, keys] {like.dtype} tensor on {like.device}")


def cross_attention(q, kv, phantom, resid, graph: CrystalGraph, S: int, drop_p: float = 0.0, seed: int = 0, seed_offset=None,
                    maps_out=None):
    """Energy -> atom cross attention (see _CrossAttention).  Dropout masks with ``seed``, plus the value of ``seed_offset``
    (optional 1-element int64 CUDA tensor) read on the device when the kernels run: a captured step rewrites it per replay.
    ``maps_out`` (optional, contiguous [S, T, Nmax] in kv's dtype, Nmax = the padding length on the device ``graph.nmax``)
    receives the attention probabilities in the reference's padded layout: atom j of the crystal in column j, the
    probability of one zero-padded key in each of the columns n_b .. Nmax - 1, with dropout the dropped-out values."""
    _check_seed_offset(seed_offset)
    H = kv.shape[1]
    _check_maps_out(maps_out, (S, q.shape[-2]), kv)
    if (tc_active(kv) and H % 128 == 0 and S % graph.B == 0 and graph.nmax_host is not None
            and graph.nkeys_host <= 1016 and q.shape[-2] >= 64 and not L.switch("DOST_NO_XATTN_TC")
            and (q.dim() == 3 or S == graph.B)):
        out = _CrossAttentionTC.apply(q, kv, phantom, resid, graph, _planes3(q), S, drop_p, seed, seed_offset, maps_out)
        out._dost_attn_out = True        # (its backward takes the incoming gradient as operand planes, see _grad_planes)
        return out
    return _CrossAttention.apply(q, kv, phantom, resid, graph, S, drop_p, seed, seed_offset, maps_out)


# =====================================================================================================
# dense self attention over the T energy tokens of each sequence
# =====================================================================================================
class _SelfAttention(torch.autograd.Function):
    """out = resid + softmax_fp32(q k^T / sqrt(H)) k, per sequence; q, resid: [S,Lq,H], k (= v): [S,Lk,H]."""

    @staticmethod
    def forward(ctx, q, k, resid, drop_p: float, seed: int, seed_offset=None, maps_out=None):
        S, Lq, H = q.shape
        Lk = k.shape[1]
        qpl, kpl = _planes3(q), _planes3(k)
        q, k, resid = q.contiguous(), k.contiguous(), resid.contiguous()
        dev, dtype = q.device, q.dtype
        Lp = (Lk + 3) // 4 * 4          # padded row length of the score matrices: keeps 16-byte vector loads legal
        ctx.on_planes = tc_active(q) and H % 8 == 0 and Lq * Lk * H >= (1 << 18) and not L.switch("DOST_NO_ATTNPLANES")
        if ctx.on_planes:
            # the four batched contractions on the TMA-fed tensor-core kernel (3-D tensor maps, one batch per sequence)
            qp = qpl if qpl is not None else split_planes(q.view(S * Lq, H))
            kp = kpl if kpl is not None else split_planes(k.view(S * Lk, H))
            ctx.drop_p, ctx.seed, ctx.seed_offset, ctx.prec = drop_p, seed, seed_offset, _PRECISION
            ctx.dims = (S, Lq, Lk, H, Lp)
            ctx.fused = fused_attention_ok(H, Lk, drop_p)
            if ctx.fused:
                out = torch.empty(S, Lq, H, dtype=dtype, device=dev)
                need = any(ctx.needs_input_grad[:3])
                pdp = empty_planes(S * Lq, Lk, dev, _with_lo()) if (need or maps_out is not None) else None
                _fused_attention_fwd(qp, kp, S * Lk, S, Lq, Lk, H, None, None, None, Lk, resid.view(S * Lq, H), Lq * H,
                                     out.view(S * Lq, H), pdp, drop_p, seed, seed_offset=seed_offset)
                if maps_out is not None:
                    _maps_from_planes(pdp, maps_out, S * Lq, None)
                if need:
                    ctx.save_for_backward(None, None, *_planes_save(qp), *_planes_save(kp), *_planes_save(pdp))
                return out
            scores = torch.empty(S, Lq, Lp, dtype=dtype, device=dev)
            gemm_planes(M=Lq, N=Lp, K=H, a=[qp], a_mode=L.KC, b=kp, b_mode=L.KC, b_rows=Lk, out=scores.view(S * Lq, Lp),
                        batch=S, a_bstride=Lq * qp.ld, b_bstride=Lk * kp.ld, c_bstride=Lq * Lp)
            pd = torch.empty_like(scores) if drop_p > 0 else scores
            pdp = empty_planes(S * Lq, Lk, dev, _with_lo())      # probabilities straight into operand planes
            L.check(L.lib().dost_softmax_fwd_planes_dseed(L.p(scores), L.p(scores), L.p(pd), S * Lq, Lk, Lp, float(H) ** -0.5,
                                                          drop_p, seed, L.p(seed_offset), L.p(pdp.hi), L.p(pdp.lo), pdp.ld,
                                                          L.stream()), "softmax_fwd_planes")
            if maps_out is not None:
                _maps_from_planes(pdp, maps_out, S * Lq, None)
            out = torch.empty(S, Lq, H, dtype=dtype, device=dev)
            gemm_planes(M=Lq, N=H, K=Lk, a=[pdp], a_mode=L.KC, b=kp, b_mode=L.MC, out=out.view(S * Lq, H),
                        residual=resid.view(S * Lq, H), batch=S, a_bstride=Lq * pdp.ld, b_bstride=Lk * kp.ld, c_bstride=Lq * H,
                        res_bstride=Lq * H)
            ctx.save_for_backward(scores, pd if drop_p > 0 else None, *_planes_save(qp), *_planes_save(kp), *_planes_save(pdp))
            return out
        scores = torch.empty(S, Lq, Lp, dtype=dtype, device=dev)
        gemm_raw(M=Lq, N=Lk, K=H, a=[(q.view(S * Lq, H), None)], a_mode=L.KC, b=k.view(S * Lk, H), b_mode=L.KC,
                 out=scores, batch=S, a_bstride=Lq * H, b_bstride=Lk * H, c_bstride=Lq * Lp, ldc=Lp)
        pd = torch.empty_like(scores) if drop_p > 0 else scores
        L.check(L.lib().dost_softmax_fwd_dseed(L.dt(q), L.p(scores), L.p(scores), L.p(pd), S * Lq, Lk, Lp, float(H) ** -0.5,
                                               drop_p, seed, L.p(seed_offset), L.stream()), "softmax_fwd")
        if maps_out is not None:      # the softmax wrote P (and the dropped-out P) into row-padded score buffers
            maps_out.copy_(pd[:, :, :Lk])
        out = torch.empty(S, Lq, H, dtype=dtype, device=dev)
        gemm_raw(M=Lq, N=H, K=Lk, a=[(pd.view(S * Lq, Lp), None)], a_mode=L.KC, b=k.view(S * Lk, H), b_mode=L.MC,
                 out=out, residual=resid, batch=S, a_bstride=Lq * Lp, b_bstride=Lk * H, c_bstride=Lq * H, ldc=H, lda=Lp)
        ctx.save_for_backward(q, k, scores, pd if drop_p > 0 else None)
        ctx.drop_p, ctx.seed, ctx.seed_offset, ctx.prec = drop_p, seed, seed_offset, _PRECISION
        return out

    @staticmethod
    def backward(ctx, d_out):
        if ctx.on_planes:
            with precision_value(ctx.prec):
                return _SelfAttention._backward_planes(ctx, d_out)
        q, k, prob, pd = ctx.saved_tensors
        if pd is None:
            pd = prob
        S, Lq, H = q.shape
        Lk, Lp = k.shape[1], prob.shape[2]
        d_out = d_out.contiguous()
        dev, dtype = q.device, q.dtype
        scale = float(H) ** -0.5
        # dPd = dO k^T
        dpd = torch.empty(S, Lq, Lp, dtype=dtype, device=dev)
        gemm_raw(M=Lq, N=Lk, K=H, a=[(d_out.view(S * Lq, H), None)], a_mode=L.KC, b=k.view(S * Lk, H), b_mode=L.KC,
                 out=dpd, batch=S, a_bstride=Lq * H, b_bstride=Lk * H, c_bstride=Lq * Lp, ldc=Lp, prec=ctx.prec)
        ds = dpd  # in place
        L.check(L.lib().dost_softmax_bwd_dseed(L.dt(q), L.p(prob), L.p(dpd), L.p(ds), S * Lq, Lk, Lp, scale, ctx.drop_p,
                                               ctx.seed, L.p(ctx.seed_offset), L.stream()), "softmax_bwd")
        # dQ = dS k
        dq = torch.empty(S, Lq, H, dtype=dtype, device=dev)
        gemm_raw(M=Lq, N=H, K=Lk, a=[(ds.view(S * Lq, Lp), None)], a_mode=L.KC, b=k.view(S * Lk, H), b_mode=L.MC,
                 out=dq, batch=S, a_bstride=Lq * Lp, b_bstride=Lk * H, c_bstride=Lq * H, ldc=H, lda=Lp, prec=ctx.prec)
        # dK = dS^T q + Pd^T dO   (reduction over the Lq queries)
        dk = torch.empty(S, Lk, H, dtype=dtype, device=dev)
        gemm_raw(M=Lk, N=H, K=Lq, a=[(ds.view(S * Lq, Lp), None)], a_mode=L.MC, b=q.view(S * Lq, H), b_mode=L.MC,
                 out=dk, batch=S, a_bstride=Lq * Lp, b_bstride=Lq * H, c_bstride=Lk * H, ldc=H, lda=Lp, prec=ctx.prec)
        gemm_raw(M=Lk, N=H, K=Lq, a=[(pd.view(S * Lq, Lp), None)], a_mode=L.MC, b=d_out.view(S * Lq, H), b_mode=L.MC,
                 out=dk, accumulate=True, batch=S, a_bstride=Lq * Lp, b_bstride=Lq * H, c_bstride=Lk * H, ldc=H, lda=Lp,
                 prec=ctx.prec)
        return dq, dk, d_out, None, None, None, None


def _self_attention_backward_planes(ctx, d_out):
    prob, pd, qh, ql, kh, kl, ph, pl_ = ctx.saved_tensors
    S, Lq, Lk, H, Lp = ctx.dims
    dev = qh.device
    scale = float(H) ** -0.5
    qp, kp = Planes(qh, ql, S * Lq, H), Planes(kh, kl, S * Lk, H)
    pdp = Planes(ph, pl_, S * Lq, Lk)
    dop = _grad_planes(d_out, S * Lq, H)
    d_out = d_out.contiguous()
    # dPd = dO k^T
    dpd = torch.empty(S, Lq, Lp, dtype=torch.float32, device=dev)
    gemm_planes(M=Lq, N=Lp, K=H, a=[dop], a_mode=L.KC, b=kp, b_mode=L.KC, b_rows=Lk, out=dpd.view(S * Lq, Lp), batch=S,
                a_bstride=Lq * dop.ld, b_bstride=Lk * kp.ld, c_bstride=Lq * Lp)
    dsp = empty_planes(S * Lq, Lk, dev, _with_lo())              # dS only ever feeds GEMMs: planes, no fp32 copy
    if ctx.fused and ctx.drop_p > 0:
        # dropout: the saved planes hold the dropped-out probabilities; P itself is recomputed (scores GEMM + softmax)
        prob = torch.empty(S, Lq, Lp, dtype=torch.float32, device=dev)
        gemm_planes(M=Lq, N=Lp, K=H, a=[qp], a_mode=L.KC, b=kp, b_mode=L.KC, b_rows=Lk, out=prob.view(S * Lq, Lp), batch=S,
                    a_bstride=Lq * qp.ld, b_bstride=Lk * kp.ld, c_bstride=Lq * Lp)
        L.check(L.lib().dost_softmax_fwd(L.F32, L.p(prob), L.p(prob), None, S * Lq, Lk, Lp, scale, 0.0, 0, L.stream()), "softmax_fwd")
    if ctx.fused and ctx.drop_p == 0:
        _ds_from_planes(pdp, dpd.view(S * Lq, Lp), S * Lq, Lk, scale, dsp)
    else:
        L.check(L.lib().dost_softmax_bwd_planes_dseed(L.p(prob), L.p(dpd), None, S * Lq, Lk, Lp, scale, ctx.drop_p, ctx.seed,
                                                      L.p(ctx.seed_offset), L.p(dsp.hi), L.p(dsp.lo), dsp.ld, L.stream()),
                "softmax_bwd_planes")
    # dQ = dS k
    dq = torch.empty(S, Lq, H, dtype=torch.float32, device=dev)
    gemm_planes(M=Lq, N=H, K=Lk, a=[dsp], a_mode=L.KC, b=kp, b_mode=L.MC, out=dq.view(S * Lq, H), batch=S,
                a_bstride=Lq * dsp.ld, b_bstride=Lk * kp.ld, c_bstride=Lq * H)
    # dK = dS^T q + Pd^T dO   (reduction over the Lq queries)
    dk = torch.empty(S, Lk, H, dtype=torch.float32, device=dev)
    gemm_planes(M=Lk, N=H, K=Lq, a=[dsp], a_mode=L.MC, b=qp, b_mode=L.MC, out=dk.view(S * Lk, H), batch=S,
                a_bstride=Lq * dsp.ld, b_bstride=Lq * qp.ld, c_bstride=Lk * H)
    gemm_planes(M=Lk, N=H, K=Lq, a=[pdp], a_mode=L.MC, b=dop, b_mode=L.MC, out=dk.view(S * Lk, H), accumulate=True, batch=S,
                a_bstride=Lq * pdp.ld, b_bstride=Lq * dop.ld, c_bstride=Lk * H)
    return dq, dk, d_out, None, None, None, None


_SelfAttention._backward_planes = staticmethod(_self_attention_backward_planes)


def _cols(pl: Planes, cols: int) -> Planes:
    """Same storage, fewer valid columns (the padded tail is excluded from the tensor-map extent)."""
    return Planes(pl.hi, pl.lo, pl.rows, cols)


def _planes3(t: torch.Tensor) -> Optional[Planes]:
    """Planes attached to a [S, L, H] tensor by the LayerNorm that produced it."""
    pl = getattr(t, "_dost_planes", None)
    if pl is not None and t.dim() == 3 and pl.rows == t.shape[0] * t.shape[1] and pl.cols == t.shape[2] and \
            (pl.lo is not None) == _with_lo():
        return pl
    return None


def self_attention(q, k, resid, drop_p: float = 0.0, seed: int = 0, seed_offset=None, maps_out=None):
    """Dense self attention (see _SelfAttention); ``seed_offset`` as in cross_attention.  ``maps_out`` (optional, contiguous
    [S, Lq, Lk] in q's dtype) receives the attention probabilities that multiply k (with dropout the dropped-out ones)."""
    _check_seed_offset(seed_offset)
    _check_maps_out(maps_out, q.shape[:2], q)
    if maps_out is not None and maps_out.shape[2] != k.shape[1]:
        raise ValueError(f"maps_out must have {k.shape[1]} columns (one per key)")
    out = _SelfAttention.apply(q, k, resid, drop_p, seed, seed_offset, maps_out)
    if tc_active(q) and q.shape[-1] % 8 == 0:
        out._dost_attn_out = True
    return out


# =====================================================================================================
# loss
# =====================================================================================================
class _DosLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred_g, pred_s, target, mode: int, beta: float):
        B, T = pred_g.shape
        pred_g, pred_s = pred_g.contiguous(), pred_s.contiguous()
        target = target.reshape(B, T).contiguous()
        loss = torch.empty(1, dtype=pred_g.dtype, device=pred_g.device)
        saved = torch.empty(4 * B, dtype=pred_g.dtype, device=pred_g.device)
        L.check(L.lib().dost_loss_fwd(L.dt(pred_g), mode, L.p(pred_g), L.p(pred_s), L.p(target), beta, B, T, L.p(loss),
                                      L.p(saved), L.stream()), "loss_fwd")
        ctx.save_for_backward(pred_g, pred_s, target, saved)
        ctx.mode, ctx.beta = mode, beta
        return loss.view(())

    @staticmethod
    def backward(ctx, g):
        pred_g, pred_s, target, saved = ctx.saved_tensors
        B, T = pred_g.shape
        g = g.contiguous()
        dg, ds = torch.empty_like(pred_g), torch.empty_like(pred_s)
        L.check(L.lib().dost_loss_bwd(L.dt(pred_g), ctx.mode, L.p(pred_g), L.p(pred_s), L.p(target), ctx.beta, B, T,
                                      L.p(saved), L.p(g), L.p(dg), L.p(ds), L.stream()), "loss_bwd")
        return dg, ds, None, None, None


def dos_loss(pred_global, pred_system, target, *, mode: str = "edos", beta: float = 1.0):
    """mode 'edos': main_eDOS.py:111-123 (targets clamped at 0, per-crystal RMSE); 'phonon': main_phDOS.py:109-114."""
    return _DosLoss.apply(pred_global, pred_system, target, 0 if mode == "edos" else 1, float(beta))


def eval_metrics(pred: torch.Tensor, target: torch.Tensor, clamp_pred: bool = True):
    """(per_crystal [B,4] = mse, rmse, mae, r2; mean [4]) as utils.test computes them with batch_size 1 (utils.py:74-88)."""
    B, T = pred.shape
    pred = pred.contiguous()
    target = target.reshape(B, T).contiguous()
    per = torch.empty(B, 4, dtype=pred.dtype, device=pred.device)
    mean = torch.empty(4, dtype=pred.dtype, device=pred.device)
    L.check(L.lib().dost_eval_metrics(L.dt(pred), L.p(pred), L.p(target), 1 if clamp_pred else 0, B, T, L.p(per), L.p(mean),
                                      L.stream()), "eval_metrics")
    return per, mean


class _PhononEdgeEncode(torch.autograd.Function):
    """First Linear + PReLU of the phonon model's edge encoder with the edge features (smooth cutoff x l <= 1 spherical
    harmonics of edge_vec, DOSTransformer_phonon.py:74-77) computed inside the same kernel: the [E, 4] feature tensor never
    exists in the forward.  The backward recomputes it once for the weight gradient."""

    @staticmethod
    def forward(ctx, edge_vec, weight, bias, slope):
        ev = edge_vec.contiguous()
        w = weight.contiguous()
        E, H = ev.shape[0], w.shape[0]
        need = any(ctx.needs_input_grad[1:])
        pre = torch.empty(E, H, dtype=ev.dtype, device=ev.device) if need else None
        out = torch.empty(E, H, dtype=ev.dtype, device=ev.device)
        L.check(L.lib().dost_phonon_edge_encode(L.dt(ev), L.p(ev), E, L.p(w), L.p(bias), L.p(slope), H, L.p(pre), L.p(out),
                                                L.stream()), "phonon_edge_encode")
        if need:
            ctx.save_for_backward(ev, slope, pre)
        ctx.has_bias = bias is not None
        return out

    @staticmethod
    def backward(ctx, d_out):
        ev, slope, pre = ctx.saved_tensors
        E, H = pre.shape
        dev, dtype = pre.device, pre.dtype
        d_out = d_out.contiguous()
        lib = L.lib()
        dv = torch.empty_like(d_out)
        d_slope = torch.empty(1, dtype=dtype, device=dev)
        nb = lib.dost_prelu_bwd_workspace_bytes(L.dt(d_out), d_out.numel())
        ws = _ws(nb, dev)
        L.check(lib.dost_prelu_bwd(L.dt(d_out), L.p(d_out), L.p(pre), L.p(slope), L.p(dv), L.p(d_slope), d_out.numel(), L.p(ws), nb,
                                   L.stream()), "prelu_bwd")
        feat = phonon_edge_features(ev)
        d_w = torch.empty(H, 4, dtype=dtype, device=dev)
        gemm_raw(M=H, N=4, K=E, a=[(dv, None)], a_mode=L.MC, b=feat, b_mode=L.MC, out=d_w,
                 split_k=_pick_split(H, 4, E, dv.element_size()), prec=L.PREC_FMA)
        d_b = colsum(dv) if ctx.has_bias else None
        return None, d_w, d_b, d_slope


def phonon_edge_encode(edge_vec: torch.Tensor, weight: torch.Tensor, bias, slope: torch.Tensor) -> torch.Tensor:
    """PReLU(Linear(phonon_edge_features(edge_vec))) in one kernel (weight [H, 4])."""
    return _PhononEdgeEncode.apply(edge_vec, weight, bias, slope)


def phonon_edge_features(edge_vec: torch.Tensor) -> torch.Tensor:
    ev = edge_vec.contiguous()
    out = torch.empty(ev.shape[0], 4, dtype=ev.dtype, device=ev.device)
    L.check(L.lib().dost_phonon_edge_feat(L.dt(ev), L.p(ev), ev.shape[0], L.p(out), L.stream()), "phonon_edge_feat")
    return out
