"""Sparsity-pattern descriptors and their cache.

The reference rebuilds index structure on every call: a Python block-diagonal assembly for batched
inputs (``utils/utils.py:474-645``), a ``repeat_interleave`` row expansion in every backward
(``sparse_matmul.py:190-192``) and an implicit CSC->CSR re-sort inside ``torch.sparse.mm(A.t(), .)``
(``sparse_matmul.py:229``).  Training loops keep the pattern fixed and only update the values
(``tests/test_sparse_matmul.py:295-338``), so here every derived structure (COO->CSR order, the
transpose) is built once per pattern by the index-builder kernels and cached.

Cache contract.  An entry is keyed on the *identity of the index memory*: data pointer, element count,
shape, strides, storage offset, dtype and version counter of every index tensor, plus the sparse shape.  It
keeps a reference to those tensors, so their storage cannot be recycled for a different pattern while the
entry lives.  What the key cannot see is an in-place write through an *unrelated alias* of the same storage
(``idx.copy_(new)`` on the buffer a sparse tensor was built from: torch gives ``_indices()`` /
``crow_indices()`` their own version counters): while a pattern is cached its index memory is **frozen**;
call ``clear_pattern_cache()`` after rewriting index buffers in place.  A violation does not go unnoticed: every
entry stores a checksum of its index arrays (``tsgu_fingerprint``) which is re-checked on cache hits number 1, 2, 4,
8, ... and a mismatch raises -- by a deferred comparison on a following hit, so that no call synchronises with the
device because of it.  ``TSGU_B200_VERIFY_PATTERN=1`` checks every hit on the spot (a host read per call), ``=0`` never.  Entries are evicted LRU under both an entry cap and a byte cap (``set_pattern_cache_capacity``,
``TSGU_B200_PATTERN_CACHE_BYTES``); ``clear_pattern_cache()`` drops everything.  Objects that must not lose
their pattern to eviction (``GraphedSparseMM``) pin it with :func:`pin_pattern`.
"""
from __future__ import annotations

import ctypes
import os
import threading
import weakref
from collections import OrderedDict
from dataclasses import dataclass, field
from typing import Optional

import torch

from . import _native as nat
from . import _ops

_CACHE_CAPACITY = 16
_CACHE_BYTES = int(os.environ.get("TSGU_B200_PATTERN_CACHE_BYTES", str(8 << 30)))  # derived structures + kept index tensors
_VERIFY = os.environ.get("TSGU_B200_VERIFY_PATTERN", "sampled")  # "1": every hit, "0": never, else hits 1, 2, 4, 8, ...
_cache: "OrderedDict[tuple, object]" = OrderedDict()
_pinned: "weakref.WeakValueDictionary[tuple, object]" = weakref.WeakValueDictionary()
_cache_lock = threading.Lock()
_I32_MAX = 2**31 - 1


def clear_pattern_cache() -> None:
    with _cache_lock:
        _cache.clear()
        _pinned.clear()


def set_pattern_cache_capacity(n: int, max_bytes: Optional[int] = None) -> None:
    """Cap the cache at `n` patterns and (optionally) `max_bytes` of device memory held by them."""
    global _CACHE_CAPACITY, _CACHE_BYTES
    _CACHE_CAPACITY = max(int(n), 0)
    if max_bytes is not None:
        _CACHE_BYTES = max(int(max_bytes), 0)
    with _cache_lock:
        _evict_locked()


def aligned_contiguous(t: torch.Tensor) -> torch.Tensor:
    """`t` itself if it is contiguous with a 16-byte aligned base, else a fresh (aligned) contiguous copy."""
    if t.is_contiguous() and t.data_ptr() % 16 == 0:
        return t
    return t.clone(memory_format=torch.contiguous_format)


def _index_key(t: torch.Tensor) -> tuple:
    """Identity of an index tensor's memory (not of its contents -- see the module docstring)."""
    return (t.data_ptr(), t.numel(), tuple(t.shape), tuple(t.stride()), t.storage_offset(), t.dtype, t._version)


def _tensor_bytes(t) -> int:
    return t.numel() * t.element_size() if isinstance(t, torch.Tensor) else 0


def pattern_nbytes(p) -> int:
    """Device bytes a cached pattern keeps alive (index tensors it was built from included)."""
    if p is None:
        return 0
    if isinstance(p, CooPattern):
        return (pattern_nbytes(p.csr) + sum(_tensor_bytes(t) for t in (p.grad_indices, p.seg, p.sort_perm))
                + (_tensor_bytes(p.out_index) if p.out_index is not p.csr.perm else 0))
    total = sum(_tensor_bytes(t) for t in (p.rowptr, p.colind, p.perm))
    total += sum(_tensor_bytes(t) for t in p.keep if isinstance(t, torch.Tensor) and t is not p.rowptr and t is not p.colind)
    if p.window is not None:
        total += _tensor_bytes(p.window.lcol) + _tensor_bytes(p.window.desc)
    for extra in p.extras.values():
        if isinstance(extra, TriPlan):
            extra = (extra.order, extra.rowptr, extra.col, extra.pos, extra.diag)
        total += sum(_tensor_bytes(t) for t in (extra if isinstance(extra, (tuple, list)) else (extra,)))
    return total + pattern_nbytes(p._transpose)


def _evict_locked() -> None:
    while len(_cache) > _CACHE_CAPACITY:
        _cache.popitem(last=False)
    if len(_cache) > 1:  # the byte cap never evicts the most recent entry (it is the one in use)
        sizes = {k: pattern_nbytes(v) for k, v in _cache.items()}
        total = sum(sizes.values())
        while total > _CACHE_BYTES and len(_cache) > 1:
            k, _ = _cache.popitem(last=False)
            total -= sizes[k]


def _fingerprint(*tensors: torch.Tensor) -> torch.Tensor:
    """Position-weighted checksums of index arrays, one int64 per array, on the device (``tsgu_fingerprint``: one small
    kernel per array, no host sync)."""
    dev = tensors[0].device
    if not tensors[0].is_cuda:  # host-side unit tests
        return torch.stack([(t.reshape(-1).long() * (torch.arange(t.numel()) % 65521 + 1)).sum() for t in tensors])
    out = torch.zeros(len(tensors), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        for k, t in enumerate(tensors):
            if t.dim() > 1 and t.stride(0) == 0:
                t = t[0]  # an expanded batch view (PairwiseValueAssembler): every item is the same memory
            t = t if t.is_contiguous() else t.contiguous()
            nat.check(nat.lib().tsgu_fingerprint(t.data_ptr(), t.numel(), nat.idx_enum(t.dtype), out[k:].data_ptr(),
                                                 nat.stream_ptr(dev)), "tsgu_fingerprint")
    return out


def _verify_due(hits: int) -> bool:
    """Which cache hits re-check the fingerprint: all of them ("1"), none ("0"), or -- the default -- hits number
    1, 2, 4, 8, ...: the usual mistake (a static index buffer refilled for the next step) is caught on the first
    reuse, and a long training run pays a logarithmic number of checks (each: two small kernels and one host read)."""
    if _VERIFY == "1":
        return True
    return _VERIFY != "0" and (hits & (hits - 1)) == 0


def pin_pattern(key, pattern) -> None:
    """Keep `pattern` reachable under `key` for as long as the caller holds a reference to it, whatever the LRU
    does (weak registry: the entry dies with its owner)."""
    with _cache_lock:
        _pinned[key] = pattern


@dataclass
class CsrPattern:
    """A batch of CSR matrices as the kernels consume it (see include/tsgu_b200.h conventions)."""

    rowptr: torch.Tensor
    colind: torch.Tensor
    perm: Optional[torch.Tensor]  # value of entry e is vals.flatten()[perm[e]]
    batch: int
    n: int
    m: int
    rowptr_bstride: int
    nnz_bstride: int
    nnz_total: int
    idx: int  # nat.I32 / nat.I64
    algo: int = nat.ALGO_AUTO  # kernel family chosen once per pattern from its row-length skew
    keep: tuple = ()  # tensors whose storage must outlive this pattern (cache-key owners)
    row_map: Optional[torch.Tensor] = None  # rows were permuted: CSR row s of item t is output row row_map[t*n + s]
    padded: bool = False  # perm holds -1 entries (explicit zeros): the values MUST go through gather_values, never the in-kernel perm path
    window: Optional["WindowPlan"] = field(default=None, repr=False)  # column-window plan, decided when the pattern is built
    extras: dict = field(default_factory=dict, repr=False)  # per-pattern plans built lazily (triangular-solve plans, ...)
    fingerprint: Optional[torch.Tensor] = field(default=None, repr=False)
    cache_key: Optional[tuple] = field(default=None, repr=False)
    _transpose: Optional["CsrPattern"] = field(default=None, repr=False)
    _transpose_uses: int = field(default=0, repr=False)
    _uniform: Optional[bool] = field(default=None, repr=False)
    _lock: threading.Lock = field(default_factory=threading.Lock, repr=False)

    # operand view of a CSR tensor's pattern (see pattern_of): values in storage order, gradient on A's own crow/col
    out_index = None
    grad_indices = None

    @property
    def csr(self) -> "CsrPattern":
        return self

    @property
    def nnz_out(self) -> int:
        return self.nnz_total

    def values(self, A: torch.Tensor) -> torch.Tensor:
        return aligned_contiguous(A.values())

    @property
    def device(self) -> torch.device:
        return self.rowptr.device

    @property
    def uniform_rows(self) -> bool:
        """True when no row is much longer than the mean (longest <= 1.25 x mean + 1).  Evaluated lazily, once per
        pattern (one host sync), and only asked for when the dense operand exceeds L2: it gates the K-sliced
        forward SpMM (``TSGU_ALGO_FLAG_KSLICE``), which loses on ragged rows (DESIGN.md section 3.1)."""
        if self._uniform is None:
            rows = self.batch * self.n
            if rows == 0 or self.nnz_total == 0:
                self._uniform = False
            else:
                rp = self.rowptr.reshape(self.batch, -1) if self.rowptr_bstride == self.n + 1 else self.rowptr.reshape(1, -1)
                longest = nat.host_read((rp[:, 1:] - rp[:, :-1]).max())[0]
                self._uniform = _uniform_from(longest, rows, self.nnz_total)
        return self._uniform

    def transpose(self, optimise: Optional[bool] = None) -> "CsrPattern":
        """CSR of the transposes (flat over batch*m rows), built once by tsgu_csr_transpose.

        The first request returns the plain transposed structure; the layout optimisations of the row-tile kernels
        (rows sorted by length inside blocks, rows padded to whole gather groups: ~0.5 ms of index work that saves
        ~0.02 ms per backward on a 1M-entry pattern) are applied from request number ``_LAYOUT_AFTER_USES`` (2) on, so
        a pattern that is used once -- a new graph every step -- does not pay for them.  ``optimise=True`` applies
        them now (GraphedSparseMM before capture, tests), ``False`` never upgrades on this call."""
        t = self._transpose
        if t is not None and "layout_pending" not in t.extras:
            return t
        with self._lock:
            if self._transpose is None:
                self._transpose = _build_transpose(self)
            t = self._transpose
            if "layout_pending" in t.extras:
                if optimise is None:
                    self._transpose_uses += 1
                    optimise = self._transpose_uses >= _LAYOUT_AFTER_USES
                if optimise and not torch.cuda.is_current_stream_capturing():
                    t = self._transpose = _optimise_layout(t)
        return t


_ALGO_ENV = {"auto": None, "rowsplit": nat.ALGO_ROWSPLIT, "merge": nat.ALGO_MERGE}


def choose_algo(max_row: Optional[int], batch: int, n: int, nnz_total: int) -> int:
    """Row-split (regular rows) or merge-path (skewed rows) -- decided once per pattern from its longest row (None: not
    read, as for a batch of matrices, which always takes the row-tile kernels).

    Merge-path pays a fix-up pass and per-entry row bookkeeping, so it is only picked when one row
    is both long in absolute terms (> 256 entries: it would keep one lane group busy for dozens of gather batches
    while the rest of its tile idles) and far above the mean (> 16 x).  Power-law graphs qualify, and so does every
    row block of one: the tail rows of an R-MAT matrix handed to a rank by row sharding still hold rows of several
    hundred entries among rows of 8 (with the round-1 thresholds, 1024 / 32 x, that shard fell to the row-tile
    kernels and its rank took 25 ms per step).  ``TSGU_B200_ALGO=auto|rowsplit|merge`` overrides the heuristic
    (benchmarking only).
    """
    forced = _ALGO_ENV.get(os.environ.get("TSGU_B200_ALGO", "auto").lower())
    if forced is not None:
        return forced
    if max_row is None or batch != 1 or nnz_total == 0 or n == 0:
        return nat.ALGO_AUTO
    return nat.ALGO_MERGE if (max_row > 256 and max_row > 16 * (nnz_total / n)) else nat.ALGO_AUTO


def _new_pattern(rowptr: torch.Tensor, colind: torch.Tensor, perm: Optional[torch.Tensor], batch: int, n: int, m: int,
                 rowptr_bstride: int, nnz_bstride: int, nnz_total: int, idx: int, keep=(), extra=None):
    """The CsrPattern of a new structure, with everything the host must know about it gathered in ONE host read: the
    longest row (kernel family, uniform_rows), the verdict of a speculatively launched column-window plan, and optional
    extra device scalars of the caller.  Returns (pattern, host values of `extra`)."""
    launched = _window_plan_launch(rowptr, colind, batch, n, m, rowptr_bstride, nnz_bstride, nnz_total, idx)
    # the longest row picks the kernel family of a single matrix, and rides along whenever something is read anyway (it
    # also answers CsrPattern.uniform_rows, which would otherwise cost the first forward a host sync of its own)
    with_rows = nnz_total > 0 and n > 0 and (batch == 1 or launched is not None or extra is not None)
    parts = []
    if with_rows:
        flat = rowptr.reshape(-1)  # differences across item boundaries of a (b, n+1) rowptr are <= 0: harmless for a max
        parts.append((flat[1:] - flat[:-1]).max().reshape(1).long())
    if launched is not None:
        parts.append(launched[2].long())
    if extra is not None:
        parts.append(extra.reshape(-1).long())
    host = nat.host_read(torch.cat(parts)) if parts else []  # the one host sync
    max_row = host[0] if with_rows else None
    pos = 1 if with_rows else 0
    algo = choose_algo(max_row, batch, n, nnz_total)
    window = None
    if launched is not None:
        failed, max_w, max_runs, max_entries = host[pos:pos + 4]
        pos += 4
        if failed == 0 and algo == nat.ALGO_AUTO:
            window = WindowPlan(launched[0], launched[1], launched[3], max_w, max_runs, max_entries)
    pat = CsrPattern(rowptr, colind, perm, batch, n, m, rowptr_bstride, nnz_bstride, nnz_total, idx, algo=algo, keep=keep,
                     window=window)
    pat._uniform = _uniform_from(max_row, batch * n, nnz_total)
    return pat, host[pos:]


def _uniform_from(max_row: Optional[int], rows: int, nnz_total: int) -> Optional[bool]:
    """CsrPattern.uniform_rows from an already known longest row (None: not known, read lazily)."""
    if rows == 0 or nnz_total == 0:
        return False
    return None if max_row is None else max_row <= 1.25 * (nnz_total / rows) + 1


def _internal_idx(batch: int, rows: int, cols: int, nnz: int) -> int:
    """Index width for structures we build ourselves: int32 whenever everything fits."""
    return nat.I32 if max(batch * rows + 1, batch * cols + 1, nnz) < _I32_MAX else nat.I64


# ------------------------------------------------------------------------------ column-window plans
@dataclass
class WindowPlan:
    """Per-pattern plan of the column-window kernels (csrc/window.cu): a 16-bit window slot per stored entry and a
    run descriptor per tile of `tile_rows` rows."""

    lcol: torch.Tensor   # int16 storage of the uint16 slots, same indexing as colind
    desc: torch.Tensor   # int32 (num_tiles, 32)
    tile_rows: int
    max_window_rows: int
    max_runs: int
    max_entries: int


_WINDOW_ON = os.environ.get("TSGU_B200_WINDOW", "1") != "0"
_WINDOW_MIN_NNZ = int(os.environ.get("TSGU_B200_WINDOW_MIN_NNZ", str(1 << 18)))
_WINDOW_MIN_ROWS = int(os.environ.get("TSGU_B200_WINDOW_MIN_ROWS", str(64 * 2 * 148)))
_window_limits = None


def window_limits():
    global _window_limits
    if _window_limits is None:
        v = [ctypes.c_int(0) for _ in range(4)]
        nat.check(nat.lib().tsgu_window_limits(*[ctypes.byref(x) for x in v]), "tsgu_window_limits")
        _window_limits = dict(tile_rows=v[0].value, entries=v[1].value, window_rows=v[2].value, runs=v[3].value)
    return _window_limits


def _window_plan_launch(rowptr, colind, batch, n, m, rowptr_bstride, nnz_bstride, nnz_total, idx):
    """Launch tsgu_window_plan if the pattern is large enough to be worth it; returns (lcol, desc, stats, tile_rows) with
    the verdict still on the device, or None."""
    rows = batch * n
    if not (_WINDOW_ON and idx == nat.I32 and nnz_total >= _WINDOW_MIN_NNZ and rows >= _WINDOW_MIN_ROWS and m < _I32_MAX):
        return None
    lim = window_limits()
    avg = nnz_total / rows
    tile_rows = next((t for t in (32, 16, 8) if t <= lim["tile_rows"] and t * avg <= lim["entries"]), 0)
    if not tile_rows:
        return None
    dev = rowptr.device
    tiles = batch * (-(-n // tile_rows))
    lcol = torch.empty(colind.numel(), dtype=torch.int16, device=dev)
    desc = torch.empty((tiles, 32), dtype=torch.int32, device=dev)
    stats = torch.empty(4, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        nat.check(nat.lib().tsgu_window_plan(nat.ptr(rowptr), nat.ptr(colind), batch, n, rowptr_bstride, nnz_bstride, idx,
                                             tile_rows, nat.ptr(lcol), nat.ptr(desc), nat.ptr(stats), nat.stream_ptr(dev)),
                  "tsgu_window_plan")
    return lcol, desc, stats, tile_rows


def window_plan(p: "CsrPattern") -> Optional[WindowPlan]:
    """Column-window plan of a pattern, or None when the pattern is not structured enough (some tile of consecutive
    rows touches more distinct columns / runs than a shared-memory window holds).  Decided together with the kernel
    family when the pattern is built (`_new_pattern`: one host read for both)."""
    return p.window


# ------------------------------------------------------------------------------ triangular-solve plans
@dataclass
class TriPlan:
    """Per-pattern plan of the level-scheduled triangular solve (csrc/trisolve.cu), one per solved triangle and
    transpose flag: rows in level order and, per slot, the dependencies (flat row, value position) and the diagonal's
    value position (-1: none).  Kept in ``CsrPattern.extras``."""

    order: torch.Tensor   # (rows,) flat row of each slot
    rowptr: torch.Tensor  # (rows + 1,) dependency offsets per slot
    col: torch.Tensor     # (deps,) flat row of each dependency
    pos: torch.Tensor     # (deps,) position of its value in the value array the solve reads
    diag: torch.Tensor    # (rows,) position of the diagonal value, -1 if none
    levels: int
    idx: int


def _transpose_csr(p: CsrPattern):
    """Plain CSR of the transposes of `p` (flat over batch*m rows, stable, no length sorting or padding) from
    tsgu_csr_transpose, its perm composed to point into p's value storage.  Returns (rowptr, colind, perm, idx)."""
    dev = p.device
    idx = _internal_idx(p.batch, p.m, p.n, p.nnz_total)
    odt = nat.IDX_TORCH[idx]
    rowptr = torch.empty(p.batch * p.m + 1, dtype=odt, device=dev)
    colind = torch.empty(p.nnz_total, dtype=odt, device=dev)
    perm = torch.empty(p.nnz_total, dtype=odt, device=dev)
    L = nat.lib()
    with torch.cuda.device(dev):
        ws = nat.workspace(L.tsgu_csr_transpose_workspace_bytes(p.batch, p.m, p.nnz_total, idx), dev)
        nat.check(L.tsgu_csr_transpose(nat.ptr(p.rowptr), nat.ptr(p.colind), p.batch, p.n, p.m, p.rowptr_bstride,
                                       p.nnz_bstride, p.nnz_total, p.idx, nat.ptr(rowptr), nat.ptr(colind),
                                       nat.ptr(perm), idx, nat.ptr(ws), ws.numel(), nat.stream_ptr(dev)),
                  "tsgu_csr_transpose")
    if p.perm is not None and p.nnz_total > 0:
        # entries of p are themselves a permutation of the caller's value storage: compose once
        perm = p.perm.to(odt).index_select(0, perm.long())
    return rowptr, colind, perm, idx


def _build_transpose(p: CsrPattern) -> CsrPattern:
    rowptrT, colindT, permT, out_idx = _transpose_csr(p)
    lensT = (rowptrT[1:] - rowptrT[:-1]).long()
    padded_total = ((lensT + (_ROW_PAD - 1)) // _ROW_PAD * _ROW_PAD).sum()  # device scalar, read with the other verdicts
    patT, (padded_total,) = _new_pattern(rowptrT, colindT, permT, p.batch, p.m, p.n, p.m, 0, p.nnz_total, out_idx,
                                         extra=padded_total)
    if patT.algo == nat.ALGO_AUTO and patT.nnz_total >= _PAD_MIN_NNZ and patT.window is None:
        # no column-window structure: the row-tile kernels take it, and two layout optimisations of a structure WE own
        # apply -- later, if the pattern turns out to be reused (CsrPattern.transpose).  No further host sync then: the
        # padded size came with the verdicts above.
        patT.extras["layout_pending"] = padded_total
    return patT


_LAYOUT_AFTER_USES = int(os.environ.get("TSGU_B200_LAYOUT_AFTER_USES", "2"))


def _optimise_layout(patT: CsrPattern) -> CsrPattern:
    """Rows sorted by length inside blocks (the 4 rows a warp works on together then hold the same number of entries:
    Poisson-distributed lengths otherwise cost max-of-4 instead of the mean), and rows padded to whole gather groups
    (skipped if the padding would overflow a 32-bit rowptr).  Returns a new pattern; `patT` is left untouched for
    whoever still holds it."""
    padded_total = patT.extras["layout_pending"]
    rowptrT, colindT, permT = patT.rowptr, patT.colind, patT.perm
    cur = torch.cuda.current_stream(patT.device)
    for t in (rowptrT, colindT, permT):
        t.record_stream(cur)  # the caller drops patT right after; it may have been built under another stream
    rowptrT, colindT, permT, row_map = _sort_rows_by_length(rowptrT, colindT, permT, patT.batch, patT.n)
    if (patT.idx == nat.I64 or padded_total < _I32_MAX) and padded_total > patT.nnz_total:
        rowptrT, colindT, permT = _pad_rows(rowptrT, colindT, permT, _ROW_PAD, padded_total)
    new = CsrPattern(rowptrT, colindT, permT, patT.batch, patT.n, patT.m, patT.n, 0, permT.numel(), patT.idx,
                     algo=patT.algo, row_map=row_map, padded=permT.numel() > patT.nnz_total)
    new._uniform = patT._uniform
    return new


_SORT_BLOCK = 64  # rows per sorting block: a multiple of the rows one pass of a CTA's lane groups covers (32 or 64)


def _sort_rows_by_length(rowptr: torch.Tensor, colind: torch.Tensor, perm: torch.Tensor, batch: int, rows_per_item: int):
    """Reorder the rows of a flat CSR (batch * rows_per_item rows) by length inside blocks of _SORT_BLOCK consecutive rows,
    alternately descending and ascending ("snake"); returns the reordered (rowptr, colind, perm) and
    row_map[t * rows + s] = original row (local to the item) at slot s.

    The kernels give a warp 4 (or 8) CONSECUTIVE rows per pass and the warp advances in lock step, so a warp costs
    the longest of its rows: with Poisson-distributed lengths (a transposed uniform pattern) max-of-4 is ~30 % above
    the mean.  After the block sort a warp's rows are neighbours in length.  Sorting inside small blocks -- instead of
    globally -- keeps every tile's entry count at the average (a globally sorted structure puts all long rows into the
    first tiles, which then overflow the staging buffers), and the alternating direction gives every warp long rows in
    one pass and short ones in the next.  One-off per pattern, no host sync (the entry count does not change)."""
    dev, idt = rowptr.device, rowptr.dtype
    rows = batch * rows_per_item
    lens = (rowptr[1:] - rowptr[:-1]).long()
    r = torch.arange(rows, device=dev)
    local = r % rows_per_item
    block = (r // rows_per_item) * (-(-rows_per_item // _SORT_BLOCK)) + local // _SORT_BLOCK
    longest = lens.max()  # stays on the device
    sub = torch.where(block % 2 == 0, longest - lens, lens)
    order = torch.argsort(block * (longest + 1) + sub, stable=True)
    new_lens = lens[order]
    new_rowptr = torch.zeros(rows + 1, dtype=torch.int64, device=dev)
    new_rowptr[1:] = new_lens.cumsum(0)
    nnz = colind.numel()
    slot = torch.repeat_interleave(r, new_lens, output_size=nnz)
    pos = torch.arange(nnz, device=dev) - new_rowptr[slot] + rowptr.long()[order][slot]
    return new_rowptr.to(idt), colind[pos], perm[pos], (order % rows_per_item).to(idt)


_ROW_PAD = 4          # the row-split kernels consume a row in groups of >= 4 entries
_PAD_MIN_NNZ = 1 << 18


def _pad_rows(rowptr: torch.Tensor, colind: torch.Tensor, perm: torch.Tensor, mult: int, total: int):
    """Pad every row of a structure WE own (a transpose) to a multiple of `mult` entries; `total` is the padded entry
    count (known to the caller: no host sync here).

    Rows of a transposed matrix have Poisson-like lengths, so most rows end in a partly filled group of
    gathers; that ragged path costs the transposed SpMM 20-60 % (profiles/r1_gather_ceilings.txt).
    Padding entries repeat the row's last column (an L1-hot dense row) and carry perm = -1, which the
    value gather turns into an explicit 0, so the product is unchanged.  One-off, cached with the pattern.
    """
    dev = rowptr.device
    lens = (rowptr[1:] - rowptr[:-1]).long()
    plen = (lens + (mult - 1)) // mult * mult
    rows = lens.numel()
    nnz = colind.numel()
    new_rowptr = torch.zeros(rows + 1, dtype=torch.int64, device=dev)
    new_rowptr[1:] = plen.cumsum(0)
    row_of = torch.repeat_interleave(torch.arange(rows, device=dev), lens, output_size=nnz)
    new_pos = new_rowptr[row_of] + (torch.arange(nnz, device=dev) - rowptr.long()[row_of])
    last_col = colind[(rowptr[1:].long() - 1).clamp_(min=0)]  # unused for empty rows (plen == 0)
    colind_p = torch.repeat_interleave(last_col, plen, output_size=total)
    colind_p[new_pos] = colind
    perm_p = torch.full((total,), -1, dtype=perm.dtype, device=dev)
    perm_p[new_pos] = perm
    return new_rowptr.to(rowptr.dtype), colind_p, perm_p


def _cache_get(key, index_tensors=()):
    with _cache_lock:
        hit = _cache.get(key)
        if hit is not None:
            _cache.move_to_end(key)
        else:
            hit = _pinned.get(key)
    if hit is not None and index_tensors and getattr(hit, "fingerprint", None) is not None:
        _check_fingerprint(hit, index_tensors)
    return hit


_REWRITTEN = ("torchsparsegradutils_b200: the index memory of a cached sparsity pattern was rewritten in place "
              "(pattern memory is frozen while cached); call clear_pattern_cache() after editing index buffers")


def _check_fingerprint(hit, index_tensors) -> None:
    """Re-check the checksum of a cached pattern's index arrays on the hits _verify_due() selects.  In the default mode
    the check is asynchronous -- two small kernels plus a 32-byte copy now, the comparison on a later hit -- so no call
    ever synchronises with the device because of it (a host read on the first reuse stalled a loader pipeline that
    prepares patterns ahead: bench.py's end-to-end leg, +1.5 ms per step); TSGU_B200_VERIFY_PATTERN=1 checks on the spot."""
    hits = hit.hits = getattr(hit, "hits", 0) + 1
    pending = getattr(hit, "pending_check", None)
    if pending is None and not _verify_due(hits):
        return
    if index_tensors[0].is_cuda and torch.cuda.is_current_stream_capturing():
        return  # nothing here may run during a graph capture (an event query alone invalidates it)
    if pending is not None and pending[0].query():
        hit.pending_check = None
        got = pending[1].tolist()
        if got[:len(got) // 2] != got[len(got) // 2:]:
            raise RuntimeError(_REWRITTEN + " (detected by a deferred check: results since the rewrite used the old pattern)")
    if not _verify_due(hits):
        return
    pair = torch.cat([hit.fingerprint, _fingerprint(*index_tensors)])
    if _VERIFY == "1" or not pair.is_cuda:
        got = nat.host_read(pair)
        if got[:len(got) // 2] != got[len(got) // 2:]:
            raise RuntimeError(_REWRITTEN)
    elif getattr(hit, "pending_check", None) is None:
        landed = torch.empty(pair.numel(), dtype=torch.int64, pin_memory=True)
        landed.copy_(pair, non_blocking=True)
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream(pair.device))
        hit.pending_check = (done, landed)


def _cache_put(key, value, index_tensors=()):
    if _VERIFY != "0" and index_tensors:
        value.fingerprint = _fingerprint(*index_tensors)
    if _CACHE_CAPACITY == 0:
        return
    with _cache_lock:
        _cache[key] = value
        _evict_locked()


# ------------------------------------------------------------------------------------------ CSR
def csr_pattern(A: torch.Tensor) -> CsrPattern:
    """Pattern of a (batched) torch CSR tensor: a zero-copy view of its crow/col arrays."""
    crow, col = A.crow_indices(), A.col_indices()
    key = ("csr", _index_key(crow), _index_key(col), tuple(A.shape), crow.device)
    hit = _cache_get(key, (crow, col))
    if hit is not None:
        return hit
    batched = A.dim() == 3
    batch = A.shape[0] if batched else 1
    n, m = A.shape[-2], A.shape[-1]
    # the staged (bulk-copy) kernels need 16-byte aligned array bases; torch allocations are, views into them
    # (crow[lo:hi], col[s:e] of a row block) need not be: take an aligned copy once per pattern rather than let the
    # dispatcher fall to the non-staged kernels (measured on a row block of config 4: 15.7 ms instead of 0.93 ms)
    crow_c, col_c = aligned_contiguous(crow), aligned_contiguous(col)
    nnz_item = col_c.shape[-1]
    idx = nat.idx_enum(crow.dtype)
    pat, _ = _new_pattern(crow_c, col_c, None, batch, n, m, n + 1, nnz_item, batch * nnz_item, idx, keep=(crow, col))
    pat.cache_key = key
    _cache_put(key, pat, (crow, col))
    return pat


# ------------------------------------------------------------------------------------------ COO
@dataclass
class CooPattern:
    """Derived structure of a COO tensor: a flat CSR over batch*n rows plus how to map values/grads."""

    csr: CsrPattern
    # unbatched: gradient values go back to storage order through out_index (= csr.perm) or identity
    out_index: Optional[torch.Tensor]
    # batched: gradient lives on the sorted unique pattern
    grad_indices: Optional[torch.Tensor]  # int64 (3, nnz_unique)
    seg: Optional[torch.Tensor]  # (nnz_unique + 1) run offsets into the sorted order when duplicates exist
    sort_perm: Optional[torch.Tensor]  # sorted position -> storage position (for segment sums)
    nnz_unique: int
    fingerprint: Optional[torch.Tensor] = field(default=None, repr=False)
    cache_key: Optional[tuple] = field(default=None, repr=False)

    @property
    def nnz_out(self) -> int:
        return self.nnz_unique

    def values(self, A: torch.Tensor) -> torch.Tensor:
        vals = aligned_contiguous(A._values())
        return vals if self.seg is None else _ops.segment_sum_values(vals, self.sort_perm, self.seg, self.nnz_unique)


def _sort_coo(indices: torch.Tensor, dims, key_dims: int, perm_idx: int, want_sorted: bool):
    """Run tsgu_coo_sort; returns (perm, sorted_indices or None)."""
    dev = indices.device
    ndim, nnz = indices.shape
    perm = torch.empty(nnz, dtype=nat.IDX_TORCH[perm_idx], device=dev)
    sorted_idx = torch.empty((ndim, nnz), dtype=torch.int64, device=dev) if want_sorted else None
    if nnz == 0:
        return perm, sorted_idx
    L = nat.lib()
    dims_c = (ctypes.c_int64 * 3)(*([int(d) for d in dims] + [1] * (3 - len(dims))))
    with torch.cuda.device(dev):
        ws = nat.workspace(L.tsgu_coo_sort_workspace_bytes(ndim, nnz, perm_idx), dev)
        nat.check(L.tsgu_coo_sort(nat.ptr(indices), ndim, nnz, indices.stride(0), dims_c, key_dims,
                                  nat.ptr(sorted_idx), nat.ptr(perm), perm_idx, nat.ptr(ws), ws.numel(),
                                  nat.stream_ptr(dev)), "tsgu_coo_sort")
    return perm, sorted_idx


def _coo_to_flat_csr(indices: torch.Tensor, batch: int, n: int, m: int, perm: Optional[torch.Tensor], idx: int,
                     keep=()) -> CsrPattern:
    dev = indices.device
    ndim, nnz = indices.shape
    odt = nat.IDX_TORCH[idx]
    rowptr = torch.empty(batch * n + 1, dtype=odt, device=dev)
    colind = torch.empty(nnz, dtype=odt, device=dev)
    with torch.cuda.device(dev):
        nat.check(nat.lib().tsgu_coo_to_csr(nat.ptr(indices), ndim, nnz, indices.stride(0), batch, n, nat.ptr(perm),
                                            nat.ptr(rowptr), nat.ptr(colind), idx, nat.stream_ptr(dev)),
                  "tsgu_coo_to_csr")
    return _new_pattern(rowptr, colind, perm, batch, n, m, n, 0, nnz, idx, keep=keep)[0]


def coo_pattern(A: torch.Tensor, unique: bool = False) -> CooPattern:
    """COO -> kernel-ready structure (sort + rowptr), cached per index tensor.

    Duplicates of a batched tensor are coalesced onto its sorted unique pattern, as the reference does.  Those of an
    uncoalesced 2-D tensor stay separate entries, which a product may keep, unless `unique`: a triangular solve may not,
    its diagonal must be one value."""
    ind = A._indices()
    coalesced = A.is_coalesced()
    batched = A.dim() == 3
    unique = unique and not (batched or coalesced)
    if unique:
        key = ("coo-unique", _index_key(ind), tuple(A.shape), ind.device)
    else:
        key = ("coo", _index_key(ind), tuple(A.shape), coalesced, ind.device)
    hit = _cache_get(key, (ind,))
    if hit is not None:
        return hit
    ind_key = ind
    if ind.stride(1) != 1:
        ind = ind.contiguous()
    batch = A.shape[0] if batched else 1
    n, m = A.shape[-2], A.shape[-1]
    nnz = ind.shape[1]
    idx = _internal_idx(batch, n, m, nnz)
    if coalesced:  # already sorted and unique: no sort, identity value map
        csr = _coo_to_flat_csr(ind, batch, n, m, None, idx, keep=(ind,))
        pat = CooPattern(csr, None, ind if batched else None, None, None, nnz)
    elif batched or unique:
        pat = _coo_unique(ind, (batch, n, m) if batched else (n, m), batch, n, m, idx)
    else:  # stable sort by row only: entries of a row keep storage order, duplicates just add up
        perm, _ = _sort_coo(ind, (n, m), 1, idx, False)
        csr = _coo_to_flat_csr(ind, 1, n, m, perm, idx, keep=(ind,))
        pat = CooPattern(csr, perm, None, None, None, nnz)
    pat.cache_key = key
    _cache_put(key, pat, (ind_key,))
    return pat


def _coo_unique(ind: torch.Tensor, dims, batch: int, n: int, m: int, idx: int) -> CooPattern:
    """Full lexicographic sort of uncoalesced coordinates; duplicates, if any, are coalesced onto the sorted unique
    pattern (seg / sort_perm sum their values), otherwise the CSR reads values through the sort permutation."""
    nnz = ind.shape[1]
    perm, srt = _sort_coo(ind, dims, len(dims), idx, True)
    dup = False
    if nnz > 1:
        first = torch.ones(nnz, dtype=torch.bool, device=ind.device)
        first[1:] = (srt[:, 1:] != srt[:, :-1]).any(dim=0)
        dup = not nat.host_read(first.all())[0]  # one-off host sync per pattern (sizes the gradient)
    if not dup:
        csr = _coo_to_flat_csr(ind, batch, n, m, perm, idx, keep=(ind,))
        return CooPattern(csr, None, srt, None, perm, nnz)
    # the reference coalesces every item before multiplying (utils/utils.py:580), so both
    # the product and the gradient live on the sorted unique pattern
    uniq = srt[:, first].contiguous()
    starts = torch.nonzero(first).flatten()
    seg = torch.cat([starts, starts.new_tensor([nnz])]).to(nat.IDX_TORCH[idx])
    csr = _coo_to_flat_csr(uniq, batch, n, m, None, idx, keep=(ind,))
    return CooPattern(csr, None, uniq, seg, perm, uniq.shape[1])


# ------------------------------------------------------------------------------------------ operands
def pattern_of(A: torch.Tensor, unique: bool = False):
    """A's cached pattern (built on first use): a CsrPattern for CSR input, a CooPattern for COO (``unique``: see
    :func:`coo_pattern`).  Both answer what an operator needs without looking at A's layout again:

    * ``.csr`` -- the flat CsrPattern the kernels read;
    * ``.values(A)`` -- A's values in the order those kernels index them: aligned and contiguous, in storage order
      (a kernel reads them through ``csr.perm`` where the pattern has one), summed onto the unique pattern where
      duplicates were coalesced;
    * ``.out_index`` / ``.nnz_out`` -- where the SDDMM over ``.csr`` writes entry e and how many values it writes,
      and ``.grad_indices`` -- the COO indices those values sit on (None: A's own), for :func:`sparse_like`."""
    if A.layout == torch.sparse_csr:
        return csr_pattern(A)
    if A.layout == torch.sparse_coo:
        return coo_pattern(A, unique)
    raise ValueError("A should be in either COO or CSR sparse format")


def sparse_values(A: torch.Tensor) -> torch.Tensor:
    """The stored values of a CSR or COO tensor, in storage order."""
    return A.values() if A.layout == torch.sparse_csr else A._values()


def sparse_like(A: torch.Tensor, values: torch.Tensor, indices: Optional[torch.Tensor] = None,
                is_coalesced: Optional[bool] = None) -> torch.Tensor:
    """A sparse tensor with A's layout and shape holding `values`: on A's own crow/col (CSR), or on A's indices or the
    given ones (COO, with the given coalesced flag)."""
    if A.layout == torch.sparse_csr:
        return torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(), values.view(A.values().shape), A.shape)
    return torch.sparse_coo_tensor(A._indices() if indices is None else indices, values, A.shape,
                                   is_coalesced=is_coalesced)


def prepare_pattern(A: torch.Tensor, backward: bool = True, reuse: bool = True) -> None:
    """Build (and cache) everything that depends only on A's sparsity pattern -- COO order / flat CSR, the kernel-family
    choice, column-window plans and, with `backward`, the transpose -- ahead of the first ``sparse_mm(A, .)``.

    The builds need only A's index tensors, so a data loader can issue them as soon as those have arrived on the device,
    while the dense operands are still in flight (bench.py's end-to-end leg does exactly that); ``sparse_mm`` then finds
    the pattern in the cache.  Purely an optimisation: ``sparse_mm`` builds whatever is missing on first use.

    `reuse` says the pattern will serve many steps, so the transposed structure gets its layout optimisations right
    away (``CsrPattern.transpose``); pass False for a pattern that lives for a single step."""
    csr = pattern_of(A).csr
    if backward:
        csr.transpose(optimise=True if reuse else False)
