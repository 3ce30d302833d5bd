"""Thin launchers: torch tensors in, C-ABI calls on the current stream, torch tensors out."""
from __future__ import annotations

import os
from typing import Optional

import torch

from . import _native as nat
from ._pattern import CsrPattern, WindowPlan, window_plan

_VEC_ELEMS = {torch.float32: 4, torch.float64: 2, torch.bfloat16: 8}
_PREGATHER_MIN_NNZ = 1 << 18


class KernelTimer:
    """Optional per-kernel CUDA-event timing on the launching stream (bench.py's roofline numbers).

    ``with KernelTimer() as kt: ...`` brackets every SpMM / SDDMM launch issued by this module with
    events; ``kt.summary()`` (after a synchronize) gives mean milliseconds and launch count per kernel
    tag.  Inactive by default: the hot path then records nothing.
    """

    active = None

    def __init__(self):
        self.records = []

    def __enter__(self):
        KernelTimer.active = self
        return self

    def __exit__(self, *exc):
        KernelTimer.active = None

    def summary(self):
        out = {}
        for tag, e0, e1 in self.records:
            ms, cnt = out.get(tag, (0.0, 0))
            out[tag] = (ms + e0.elapsed_time(e1), cnt + 1)
        return {k: {"ms": v[0] / v[1], "launches": v[1]} for k, v in out.items()}


class _Null:
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False


_NULL = _Null()


def _on(dev: torch.device):
    """Device guard only when `dev` is not already current (the guard costs ~10 us of host time per call)."""
    return _NULL if torch.cuda.current_device() == dev.index else torch.cuda.device(dev)


_NVTX = os.environ.get("TSGU_B200_NVTX", "0") == "1"


class _nvtx_range:
    """NVTX range around one entry point (SURVEY.md section 5: profiler hooks); TSGU_B200_NVTX=1 turns them on."""

    def __init__(self, tag, inner):
        self.tag, self.inner = tag, inner

    def __enter__(self):
        torch.cuda.nvtx.range_push("tsgu_b200::" + self.tag)
        return self.inner.__enter__()

    def __exit__(self, *exc):
        r = self.inner.__exit__(*exc)
        torch.cuda.nvtx.range_pop()
        return r


def _timer(tag: str, dev: torch.device):
    t = _timed(tag, dev) if KernelTimer.active is not None else _NULL
    return _nvtx_range(tag, t) if _NVTX else t


class _timed:
    def __init__(self, tag, device):
        self.kt = KernelTimer.active
        self.tag, self.device = tag, device

    def __enter__(self):
        if self.kt is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record(torch.cuda.current_stream(self.device))

    def __exit__(self, *exc):
        if self.kt is not None:
            self.e1.record(torch.cuda.current_stream(self.device))
            self.kt.records.append((self.tag, self.e0, self.e1))


def _epv(dtype: torch.dtype) -> int:
    try:
        return _VEC_ELEMS[dtype]
    except KeyError:
        nat.val_enum(dtype)  # raises the documented RuntimeError for unsupported dtypes
        raise


def _vector_ready(x: torch.Tensor) -> bool:
    """Can the 128-bit kernels read this (batch, rows, K) operand in place?"""
    epv = _epv(x.dtype)
    bs, rs, cs = x.stride()
    K = x.shape[-1]
    if K % epv:
        return False
    ok_rs = rs % epv == 0 or x.shape[1] <= 1
    ok_bs = bs % epv == 0 or x.shape[0] <= 1
    return (cs == 1 or K == 1) and ok_rs and ok_bs and x.data_ptr() % 16 == 0


def copy_dense(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    """dst[...] = src[...] for two (batch, rows, K) tensors of any strides, through tsgu_pack_dense."""
    b, r, k = src.shape
    if src.numel():
        with _on(src.device):
            nat.check(nat.lib().tsgu_pack_dense(src.data_ptr(), dst.data_ptr(), b, r, k, *src.stride(), *dst.stride(),
                                                nat.val_enum(src.dtype), nat.stream_ptr(src.device)), "tsgu_pack_dense")
    return dst


def pack_dense(x: torch.Tensor) -> torch.Tensor:
    """Strided (batch, rows, K) -> contiguous (coalesced on both sides)."""
    return copy_dense(x, torch.empty(x.shape, dtype=x.dtype, device=x.device))


def restride_like(x: torch.Tensor, shape, strides) -> torch.Tensor:
    """Return x's values in a tensor with the given (dense, non-overlapping) strides.

    Autograd re-strides a gradient to its leaf's layout with a generic copy (1.2 ms for config 3's
    column-major B); doing it here with the tiled kernel costs a tenth of that.
    """
    out = torch.empty_strided(tuple(shape), tuple(strides), dtype=x.dtype, device=x.device)
    x3 = x.reshape((1,) * (3 - len(shape)) + tuple(shape)) if len(shape) < 3 else x
    o3 = out.unsqueeze(0) if len(shape) < 3 else out
    copy_dense(x3, o3)
    return out


def is_dense_non_overlapping(t: torch.Tensor) -> bool:
    """True if t's strides are a permutation of a contiguous layout (torch's gradient-layout rule)."""
    order = sorted(range(t.dim()), key=lambda d: (-t.stride(d), -t.size(d)))
    return t.permute(order).is_contiguous()


def prepare_dense(x: torch.Tensor) -> torch.Tensor:
    """Return a (batch, rows, K) operand the kernels can address.

    Vectorisable K: make it 128-bit readable (pack once if it is a transposed / permuted / expanded
    view, which is what ``_batch_sparse_mv`` hands us, distributions/sparse_multivariate_normal.py:96,100).
    Other K: the scalar kernels take arbitrary element strides, no copy.
    """
    if x.shape[-1] % _epv(x.dtype) == 0 and not _vector_ready(x):
        return pack_dense(x)
    return x


def _as3d(x: torch.Tensor) -> torch.Tensor:
    return x if x.dim() == 3 else x.unsqueeze(0)


def _strides(x: torch.Tensor):
    """Element strides with size-1 dims normalised, so they never disqualify the 128-bit path."""
    bs, rs, cs = x.stride()
    return (bs if x.shape[0] > 1 else 0, rs if x.shape[1] > 1 else 0, cs if x.shape[2] > 1 else 1)


_L2_BYTES = {}


def _l2_bytes(dev: torch.device) -> int:
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    if key not in _L2_BYTES:
        _L2_BYTES[key] = int(torch.cuda.get_device_properties(key).L2_cache_size)
    return _L2_BYTES[key]


_WINDOW_ROW_BYTES = (64, 128, 256)  # dense row widths the column-window kernels are built for (csrc/window.cu)


def _window_for(pat: CsrPattern, algo: int, *dense: torch.Tensor) -> Optional[WindowPlan]:
    """The pattern's column-window plan if the window kernels can take these operands, else None."""
    if algo != nat.ALGO_AUTO:
        return None
    d0 = dense[0]
    if d0.dtype not in (torch.float32, torch.bfloat16) or d0.shape[-1] * d0.element_size() not in _WINDOW_ROW_BYTES:
        return None
    if not all(_vector_ready(x) for x in dense):
        return None
    return window_plan(pat)


def _spmm_window(pat: CsrPattern, wp: WindowPlan, vals: torch.Tensor, dense: torch.Tensor, tag: str,
                 out_strides=None) -> torch.Tensor:
    dev = dense.device
    K = dense.shape[-1]
    colmajor = out_strides is not None and tuple(out_strides) == (pat.n * K, 1, pat.n) and K > 1 and pat.n > 1
    if colmajor:  # every item column-major: written directly by the kernel's transposing epilogue
        out = torch.empty_strided((pat.batch, pat.n, K), (pat.n * K, 1, pat.n), dtype=dense.dtype, device=dev)
    else:
        out = torch.empty((pat.batch, pat.n, K), dtype=dense.dtype, device=dev)
    if pat.perm is not None:
        with _timer(tag + "_gather", dev):
            vals = gather_values(vals.reshape(-1), pat.perm)
    bs, rs, _ = _strides(dense)
    with _on(dev), _timer(tag, dev):
        nat.check(nat.lib().tsgu_spmm_window(nat.ptr(pat.rowptr), nat.ptr(wp.lcol), nat.ptr(wp.desc), nat.ptr(vals),
                                             dense.data_ptr(), out.data_ptr(), pat.batch, pat.n, K,
                                             pat.rowptr_bstride, pat.nnz_bstride, pat.colind.numel(), wp.tile_rows,
                                             bs, rs if pat.m > 1 else K, pat.n * K, 1 if colmajor else K,
                                             pat.n if colmajor else 1, nat.val_enum(dense.dtype), pat.idx,
                                             nat.stream_ptr(dev)), "tsgu_spmm_window")
    return out


def spmm(pat: CsrPattern, vals: torch.Tensor, dense: torch.Tensor, algo: Optional[int] = None,
         tag: str = "spmm", out_strides=None) -> torch.Tensor:
    """out[t] = A[t] @ dense[t]; dense is (batch, m, K) (any strides); returns contiguous (batch, n, K).
    `out_strides`: a layout the caller would like the (batch, n, K) result in; honoured where a kernel can write it
    directly (column-major items from the column-window kernels), otherwise the result is contiguous and the caller
    re-strides it."""
    algo = pat.algo if algo is None else algo
    dense = prepare_dense(_as3d(dense))
    K = dense.shape[-1]
    if pat.batch * pat.n * K and pat.nnz_total:
        wp = _window_for(pat, algo, dense)
        if wp is not None:
            return _spmm_window(pat, wp, vals, dense, tag, out_strides)
    out = torch.empty((pat.batch, pat.n, K), dtype=dense.dtype, device=dense.device)
    if out.numel() == 0:
        return out
    dev = dense.device
    L = nat.lib()
    vdt = nat.val_enum(dense.dtype)
    perm = pat.perm
    if perm is not None and (pat.nnz_total >= _PREGATHER_MIN_NNZ or pat.padded):
        # one streaming pass that puts the values in the structure's own order is cheaper than a
        # divergent 4-byte gather per entry inside the bandwidth-critical SpMM (0.37 -> 0.25+0.03 ms on config 2)
        with _timer(tag + "_gather", dev):
            vals = gather_values(vals.reshape(-1), perm)
        perm = None
    if (algo == nat.ALGO_AUTO and pat.m * K * dense.element_size() > (_l2_bytes(dev) * 3) // 5
            and pat.uniform_rows):
        algo |= nat.ALGO_FLAG_KSLICE  # dense operand exceeds L2 and the rows are uniform: L2-resident K slices
    if pat.row_map is not None:  # a transpose with length-sorted rows
        with _on(dev), _timer(tag, dev):
            nat.check(L.tsgu_spmm_csr_rowmap(nat.ptr(pat.rowptr), nat.ptr(pat.colind), nat.ptr(vals), nat.ptr(perm),
                                             nat.ptr(pat.row_map), dense.data_ptr(), out.data_ptr(), pat.batch, pat.n, pat.m,
                                             K, pat.rowptr_bstride, pat.nnz_bstride, pat.nnz_total, *_strides(dense),
                                             pat.n * K, K, vdt, pat.idx, algo, nat.stream_ptr(dev)), "tsgu_spmm_csr_rowmap")
        return out
    with _on(dev), _timer(tag, dev):
        ws_bytes = L.tsgu_spmm_workspace_bytes(pat.batch, pat.n, K, pat.nnz_total, vdt, algo) if algo == nat.ALGO_MERGE else 0
        ws = nat.workspace(ws_bytes, dev) if ws_bytes else None
        nat.check(L.tsgu_spmm_csr(nat.ptr(pat.rowptr), nat.ptr(pat.colind), nat.ptr(vals), nat.ptr(perm),
                                  dense.data_ptr(), out.data_ptr(), pat.batch, pat.n, pat.m, K,
                                  pat.rowptr_bstride, pat.nnz_bstride, pat.nnz_total,
                                  *_strides(dense), pat.n * K, K,
                                  vdt, pat.idx, algo, nat.ptr(ws), ws.numel() if ws is not None else 0,
                                  nat.stream_ptr(dev)), "tsgu_spmm_csr")
    return out


def sddmm(pat: CsrPattern, G: torch.Tensor, B: torch.Tensor, out_index: Optional[torch.Tensor], nnz_out: int,
          algo: Optional[int] = None) -> torch.Tensor:
    """values[dst(e)] = <G[t, r_e], B[t, c_e]> for every stored entry of the pattern."""
    algo = pat.algo if algo is None else algo
    G = prepare_dense(_as3d(G))
    B = prepare_dense(_as3d(B))
    out = torch.empty(nnz_out, dtype=B.dtype, device=B.device)
    if nnz_out == 0:
        return out
    dev = B.device
    L = nat.lib()
    wp = _window_for(pat, algo, B, G) if pat.nnz_total else None
    if wp is not None:
        K = B.shape[-1]
        gbs, grs, _ = _strides(G)
        bbs, brs, _ = _strides(B)
        with _on(dev), _timer("sddmm", dev):
            nat.check(L.tsgu_sddmm_window(nat.ptr(pat.rowptr), nat.ptr(wp.lcol), nat.ptr(wp.desc), nat.ptr(out_index),
                                          G.data_ptr(), B.data_ptr(), out.data_ptr(), pat.batch, pat.n, K,
                                          pat.rowptr_bstride, pat.nnz_bstride, pat.colind.numel(), wp.tile_rows,
                                          gbs, grs if pat.n > 1 else K, bbs, brs if pat.m > 1 else K,
                                          nat.val_enum(B.dtype), pat.idx, nat.stream_ptr(dev)), "tsgu_sddmm_window")
        return out
    with _on(dev), _timer("sddmm", dev):
        ws_bytes = L.tsgu_sddmm_workspace_bytes(pat.batch, pat.n, pat.nnz_total, algo) if algo == nat.ALGO_MERGE else 0
        ws = nat.workspace(ws_bytes, dev) if ws_bytes else None
        nat.check(L.tsgu_sddmm_csr(nat.ptr(pat.rowptr), nat.ptr(pat.colind), nat.ptr(out_index),
                                           G.data_ptr(), B.data_ptr(), out.data_ptr(), pat.batch, pat.n, pat.m,
                                           B.shape[-1], pat.rowptr_bstride, pat.nnz_bstride, pat.nnz_total,
                                           *_strides(G), *_strides(B),
                                           nat.val_enum(B.dtype), pat.idx, algo, nat.ptr(ws),
                                           ws.numel() if ws is not None else 0, nat.stream_ptr(dev)),
                  "tsgu_sddmm_csr")
    return out


def sddmm_coo(row: torch.Tensor, col: torch.Tensor, G: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    """Order-agnostic SDDMM on raw int64 COO coordinates (2-D operands)."""
    G = prepare_dense(_as3d(G))[0]
    B = prepare_dense(_as3d(B))[0]
    nnz = row.shape[0]
    out = torch.empty(nnz, dtype=B.dtype, device=B.device)
    if nnz == 0:
        return out
    row, col = row.contiguous(), col.contiguous()
    with _on(B.device):
        nat.check(nat.lib().tsgu_sddmm_coo(row.data_ptr(), col.data_ptr(), G.data_ptr(), B.data_ptr(), out.data_ptr(),
                                           nnz, B.shape[-1], G.stride(0), G.stride(1), B.stride(0), B.stride(1),
                                           nat.val_enum(B.dtype), nat.stream_ptr(B.device)), "tsgu_sddmm_coo")
    return out


def segment_sum_values(vals: torch.Tensor, perm: torch.Tensor, seg: torch.Tensor, nseg: int) -> torch.Tensor:
    out = torch.empty(nseg, dtype=vals.dtype, device=vals.device)
    if nseg:
        with _on(vals.device):
            nat.check(nat.lib().tsgu_segment_sum_values(vals.data_ptr(), nat.ptr(perm), seg.data_ptr(), out.data_ptr(),
                                                        nseg, nat.val_enum(vals.dtype), nat.idx_enum(seg.dtype),
                                                        nat.stream_ptr(vals.device)), "tsgu_segment_sum_values")
    return out


def gather_values(vals: torch.Tensor, perm: torch.Tensor) -> torch.Tensor:
    out = torch.empty(perm.shape, dtype=vals.dtype, device=vals.device)
    if out.numel():
        with _on(vals.device):
            nat.check(nat.lib().tsgu_gather_values(vals.data_ptr(), perm.data_ptr(), out.data_ptr(), perm.numel(),
                                                   nat.val_enum(vals.dtype), nat.idx_enum(perm.dtype),
                                                   nat.stream_ptr(vals.device)), "tsgu_gather_values")
    return out


def scatter_values(vals: torch.Tensor, perm: torch.Tensor, out_count: int) -> torch.Tensor:
    """out[perm[k]] = vals[k], zeros elsewhere (adjoint of gather_values for an injective perm)."""
    out = torch.empty(out_count, dtype=vals.dtype, device=vals.device)
    with _on(vals.device):
        nat.check(nat.lib().tsgu_scatter_values(vals.data_ptr(), perm.data_ptr(), out.data_ptr(), perm.numel(), out_count,
                                                nat.val_enum(vals.dtype), nat.idx_enum(perm.dtype),
                                                nat.stream_ptr(vals.device)), "tsgu_scatter_values")
    return out


def block_diag_csr(crow: torch.Tensor, col: torch.Tensor, m: int):
    """Batched CSR index tensors (b, n+1) / (b, nnz) -> block-diagonal (b*n+1,), (b*nnz,) in one kernel."""
    b, n1 = crow.shape
    nnz = col.shape[1]
    crow, col = crow.contiguous(), col.contiguous()
    crow_out = torch.empty(b * (n1 - 1) + 1, dtype=crow.dtype, device=crow.device)
    col_out = torch.empty(b * nnz, dtype=col.dtype, device=col.device)
    with _on(crow.device):
        nat.check(nat.lib().tsgu_block_diag_csr(crow.data_ptr(), col.data_ptr(), b, n1 - 1, m, nnz, crow_out.data_ptr(),
                                                col_out.data_ptr(), nat.idx_enum(crow.dtype), nat.stream_ptr(crow.device)),
                  "tsgu_block_diag_csr")
    return crow_out, col_out
