"""GPU: the column-window kernels (csrc/window.cu) -- plan structure, and SpMM / SDDMM / transposed SpMM through the
public op against the CPU oracle, on stencil and banded patterns small enough for the whole oracle."""
import os
import sys

import numpy as np
import pytest
import torch

from helpers import TOL
from oracle import oracle as orc

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import workloads as W  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(autouse=True)
def _small_patterns_get_windows(monkeypatch):
    """Oracle-sized inputs: lift the size gates of the window path, clean cache either side."""
    import torchsparsegradutils_b200 as tsgu
    from torchsparsegradutils_b200 import _pattern

    monkeypatch.setattr(_pattern, "_WINDOW_MIN_NNZ", 0)
    monkeypatch.setattr(_pattern, "_WINDOW_MIN_ROWS", 0)
    tsgu.clear_pattern_cache()
    yield
    tsgu.clear_pattern_cache()


def _banded_csr(n, m, offsets, keep_prob=1.0, seed=0, dtype=torch.float32):
    """Rows r hold columns r + o (in range) for o in offsets, each kept with keep_prob -> ragged rows, some empty."""
    g = torch.Generator().manual_seed(seed)
    r = torch.arange(n).unsqueeze(1)
    c = r + torch.tensor(sorted(offsets)).unsqueeze(0)
    ok = (c >= 0) & (c < m)
    if keep_prob < 1.0:
        ok &= torch.rand(c.shape, generator=g) < keep_prob
    crow = torch.zeros(n + 1, dtype=torch.int64)
    crow[1:] = ok.sum(1).cumsum(0)
    col = c[ok]
    vals = torch.rand(col.numel(), generator=g, dtype=torch.float64).to(dtype)
    return torch.sparse_csr_tensor(crow.int().to(DEV), col.int().to(DEV), vals.to(DEV), (n, m))


def _np(t):
    return t.detach().to(torch.float64 if t.dtype == torch.bfloat16 else t.dtype).cpu().numpy()


def _check_against_oracle(A, K, dtype, expect_window=True, b_colmajor=False):
    from torchsparsegradutils_b200 import sparse_mm
    from torchsparsegradutils_b200._pattern import coo_pattern, csr_pattern, window_plan

    batched = A.dim() == 3
    lead = (A.shape[0],) if batched else ()
    n, m = A.shape[-2], A.shape[-1]
    g = torch.Generator().manual_seed(7)
    B = torch.rand(lead + (m, K), generator=g, dtype=torch.float64).to(dtype).to(DEV)
    G = torch.rand(lead + (n, K), generator=g, dtype=torch.float64).to(dtype).to(DEV)
    if b_colmajor:
        B = B.transpose(-1, -2).contiguous().transpose(-1, -2)
    A = A.detach().requires_grad_(True)
    Bd = B.detach().requires_grad_(True)
    C = sparse_mm(A, Bd)
    C.backward(G)
    pat = csr_pattern(A) if A.layout == torch.sparse_csr else coo_pattern(A).csr
    if expect_window is not None:
        assert (window_plan(pat) is not None) == expect_window
    if expect_window:
        assert window_plan(pat.transpose()) is not None
    odt = np.float32
    if A.layout == torch.sparse_csr:
        ref = orc.sparse_mm_fwd_bwd("csr", tuple(A.shape), _np(B).astype(odt), _np(G).astype(odt), crow=_np(A.crow_indices()),
                                    col=_np(A.col_indices()), values=_np(A.values()).astype(odt))
        gv = A.grad.values()
    else:
        ref = orc.sparse_mm_fwd_bwd("coo", tuple(A.shape), _np(B).astype(odt), _np(G).astype(odt), indices=_np(A._indices()),
                                    values=_np(A._values()).astype(odt))
        gv = A.grad._values()
    tol = TOL[dtype]
    np.testing.assert_allclose(_np(C), ref["C"], **tol)
    np.testing.assert_allclose(_np(gv).reshape(ref["gradA_values"].shape), ref["gradA_values"], **tol)
    np.testing.assert_allclose(_np(Bd.grad), ref["gradB"], **tol)


def test_window_plan_reconstructs_every_column():
    """Slots + run descriptors are a lossless re-encoding of colind: column(run containing slot) == colind[e]."""
    from torchsparsegradutils_b200._pattern import csr_pattern, window_limits, window_plan

    A = W.stencil27_csr(14, torch.float32, torch.int32, DEV, seed=3)
    pat = csr_pattern(A)
    wp = window_plan(pat)
    assert wp is not None and wp.tile_rows == 32 and wp.max_runs <= window_limits()["runs"]
    crow, col = A.crow_indices().cpu().numpy().astype(np.int64), A.col_indices().cpu().numpy().astype(np.int64)
    lcol = wp.lcol.cpu().numpy().view(np.uint16).astype(np.int64)
    desc = wp.desc.cpu().numpy()
    n = A.shape[0]
    for t in range(desc.shape[0]):
        r0, r1 = t * wp.tile_rows, min((t + 1) * wp.tile_rows, n)
        s, e = crow[r0], crow[r1]
        nruns, distinct = desc[t, 0], desc[t, 1]
        assert 0 <= nruns <= window_limits()["runs"]
        slot_to_col = np.full(distinct, -1, dtype=np.int64)
        nxt = 0
        for r in range(nruns):
            c0 = int(desc[t, 2 + 2 * r])
            sl = int(desc[t, 3 + 2 * r]) & 0xFFFFFFFF
            slot, ln = sl & 0xFFFF, sl >> 16
            assert slot == nxt and ln > 0  # runs tile the window densely, in column order
            slot_to_col[slot:slot + ln] = np.arange(c0, c0 + ln)
            nxt = slot + ln
        assert nxt == distinct >= len(np.unique(col[s:e]))
        np.testing.assert_array_equal(slot_to_col[lcol[s:e]], col[s:e])
    assert int(desc[:, 1].max()) == wp.max_window_rows <= window_limits()["window_rows"]


@pytest.mark.parametrize("K,dtype", [(16, torch.float32), (32, torch.float32), (64, torch.float32),
                                     (32, torch.bfloat16), (64, torch.bfloat16), (128, torch.bfloat16)])
def test_stencil_window_kernels_vs_oracle(K, dtype):
    A = W.stencil27_csr(20, dtype, torch.int32, DEV, seed=3)
    _check_against_oracle(A, K, dtype)


def test_stencil_window_column_major_B():
    A = W.stencil27_csr(16, torch.float32, torch.int32, DEV, seed=3)
    _check_against_oracle(A, 32, torch.float32, b_colmajor=True)


@pytest.mark.parametrize("D,K,dtype", [(15, 32, torch.float32), (13, 16, torch.float32), (12, 64, torch.float32),
                                       (14, 64, torch.bfloat16), (11, 32, torch.bfloat16)])
def test_column_major_epilogue_shapes(D, K, dtype):
    """grad_B is written column-major by the SpMM's transposing epilogue: row counts that are not multiples of the
    rows per warp / per tile, 4- and 8-lane groups, 64 / 128 / 256-byte rows, fp32 and bf16."""
    from torchsparsegradutils_b200 import sparse_mm

    A = W.stencil27_csr(D, dtype, torch.int32, DEV, seed=3)
    _check_against_oracle(A, K, dtype, b_colmajor=True)
    n = A.shape[0]
    B = torch.rand(K, n, device=DEV).to(dtype).t().requires_grad_(True)  # column-major leaf
    C = sparse_mm(A, B)
    C.backward(torch.rand(n, K, device=DEV).to(dtype))
    assert B.grad.stride() == B.stride()


def test_batched_column_major_epilogue():
    As = [W.stencil27_csr(11, torch.float32, torch.int32, DEV, seed=s) for s in (1, 2)]
    A = torch.sparse_csr_tensor(torch.stack([a.crow_indices() for a in As]), torch.stack([a.col_indices() for a in As]),
                                torch.stack([a.values() for a in As]), (2,) + tuple(As[0].shape))
    _check_against_oracle(A, 32, torch.float32, b_colmajor=True)


def test_lower_triangular_stencil_window():
    A = W.stencil27_csr(18, torch.float32, torch.int32, DEV, seed=3, lower=True)
    _check_against_oracle(A, 32, torch.float32)


@pytest.mark.parametrize("keep", [1.0, 0.6, 0.15])
def test_banded_ragged_rows_window(keep):
    """2-D banded pattern with entries dropped at random: ragged rows, empty rows, runs with holes."""
    A = _banded_csr(3000, 2800, [-120, -119, -61, -60, -59, -1, 0, 1, 2, 59, 60, 61, 119, 120, 121], keep, seed=5)
    # holes in the runs are bridged by the planner (WIN_CLOSE); very sparse bands may still not fit -> row-tile kernels
    _check_against_oracle(A, 32, torch.float32, expect_window=True if keep >= 0.5 else None)


def test_rectangular_and_long_rows_window():
    """~60 entries per row -> 16-row tiles; rectangular shape."""
    offs = list(range(-30, 30))
    A = _banded_csr(2500, 4000, offs, 1.0, seed=6)
    _check_against_oracle(A, 64, torch.float32)
    from torchsparsegradutils_b200._pattern import csr_pattern, window_plan

    assert window_plan(csr_pattern(A)).tile_rows == 16


def test_batched_csr_window():
    As = [W.stencil27_csr(12, torch.float32, torch.int32, DEV, seed=s) for s in (1, 2, 3)]
    A = torch.sparse_csr_tensor(torch.stack([a.crow_indices() for a in As]), torch.stack([a.col_indices() for a in As]),
                                torch.stack([a.values() for a in As]), (3,) + tuple(As[0].shape))
    _check_against_oracle(A, 32, torch.float32)


def test_uncoalesced_coo_stencil_window():
    """COO in shuffled storage order: the flat CSR carries a value permutation (values pre-gathered into pattern
    order before the window SpMM)."""
    Ac = W.stencil27_csr(12, torch.float32, torch.int32, DEV, seed=3).to_sparse_coo()
    idx, v = Ac._indices(), Ac._values()
    sh = torch.randperm(v.numel(), generator=torch.Generator().manual_seed(1)).to(DEV)
    A = torch.sparse_coo_tensor(idx[:, sh].contiguous(), v[sh].contiguous(), Ac.shape)
    _check_against_oracle(A, 32, torch.float32)


def test_random_pattern_is_not_windowed_and_still_correct():
    A = W.uniform_rows_csr(None, 4000, 4000, 16, torch.float32, torch.int32, DEV, seed=2)
    _check_against_oracle(A, 32, torch.float32, expect_window=False)


def test_window_matches_row_tile_kernels_bitwise(monkeypatch):
    """Same accumulation order per row as the row-tile kernels: identical bits with the window path off."""
    import torchsparsegradutils_b200 as tsgu
    from torchsparsegradutils_b200 import _pattern, sparse_mm

    A = W.stencil27_csr(24, torch.float32, torch.int32, DEV, seed=3)
    B = torch.randn(A.shape[1], 32, device=DEV)
    G = torch.randn(A.shape[0], 32, device=DEV)

    def run():
        a = A.detach().requires_grad_(True)
        b = B.detach().requires_grad_(True)
        c = sparse_mm(a, b)
        c.backward(G)
        return c.detach(), a.grad.values(), b.grad

    C1, gA1, gB1 = run()
    monkeypatch.setattr(_pattern, "_WINDOW_ON", False)
    tsgu.clear_pattern_cache()
    C2, gA2, gB2 = run()
    assert torch.equal(C1, C2) and torch.equal(gB1, gB2)
    torch.testing.assert_close(gA1, gA2, rtol=1e-5, atol=1e-5)  # SDDMM: butterfly width differs (8 vs 16 entries)
