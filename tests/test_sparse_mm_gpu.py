"""GPU parity proper: CUDA path vs the CPU oracle on seeded inputs, plus the reference's own test
contract (tests/test_sparse_matmul.py) re-expressed against this implementation."""
import numpy as np
import pytest
import torch

from helpers import TOL, rand_csr
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _np(t):
    return t.detach().to(torch.float64 if t.dtype == torch.bfloat16 else t.dtype).cpu().numpy()


def _oracle(A, B, G):
    """fp64-accumulated oracle on the (upcast) inputs; bf16 is checked against the fp32-upcast oracle
    as SURVEY 8(c) prescribes (the reference's CPU path cannot run bf16 CSR)."""
    odt = np.float64 if A.dtype == torch.float64 else np.float32
    Bn, Gn = _np(B).astype(odt), _np(G).astype(odt)
    if A.layout == torch.sparse_csr:
        return orc.sparse_mm_fwd_bwd("csr", tuple(A.shape), Bn, Gn, crow=_np(A.crow_indices()),
                                     col=_np(A.col_indices()), values=_np(A.values()).astype(odt))
    return orc.sparse_mm_fwd_bwd("coo", tuple(A.shape), Bn, Gn, indices=_np(A._indices()),
                                 values=_np(A._values()).astype(odt))


def _run(A, B, G):
    from torchsparsegradutils_b200 import sparse_mm

    A = A.detach().requires_grad_(True)
    B = B.detach().requires_grad_(True)
    C = sparse_mm(A, B)
    C.backward(G)
    return C.detach(), A.grad, B.grad


def _check(A, B, G, scaled_atol=False):
    """Strict north_star tolerance (fp32: rtol 1e-5 / atol 1e-6) for the reference's own test
    distribution (torch.rand operands, tests/test_sparse_matmul.py:81,99,110: no cancellation).
    `scaled_atol`: for N(0,1) operands (the benchmark distribution) individual outputs are sums with
    heavy cancellation, where no fp32 evaluation order -- the reference's included -- can meet a
    per-element rtol; there atol is scaled by the magnitude of the exact result (max |x|)."""
    C, gA, gB = _run(A, B, G)
    ref = _oracle(A, B, G)
    tol = dict(TOL[A.dtype])
    base_atol = tol["atol"]
    f = lambda t: torch.from_numpy(_np(t).astype(np.float64))  # noqa: E731

    def close(got, want):
        want = torch.from_numpy(want.astype(np.float64))
        if scaled_atol and want.numel():
            tol["atol"] = base_atol * max(1.0, float(want.abs().max()))
        torch.testing.assert_close(f(got).reshape(want.shape), want, **tol)

    close(C, ref["C"])
    close(gB, ref["gradB"])
    close(gA.values() if A.layout == torch.sparse_csr else gA._values(), ref["gradA_values"])
    if A.layout == torch.sparse_coo:
        assert torch.equal(gA._indices().cpu(), torch.from_numpy(ref["gradA_indices"]))


KS = [1, 2, 3, 4, 8, 10, 16, 32, 64, 96, 128, 256, 512, 640, 1024, 1100]


@pytest.mark.parametrize("K", KS)
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16])
def test_csr_vs_oracle_all_K(K, dtype):
    """Every kernel variant (lanes-per-row x vectors-per-lane, scalar and 128-bit paths)."""
    n, m = 193, 161
    A = rand_csr(n, m, 9, dtype=dtype, index_dtype=torch.int32, seed=K, ragged=True)
    B = torch.rand(m, K, device=DEV, dtype=dtype)
    G = torch.rand(n, K, device=DEV, dtype=dtype)
    _check(A, B, G)


@pytest.mark.parametrize("index_dtype", [torch.int32, torch.int64])
@pytest.mark.parametrize("K", [5, 128])
def test_batched_csr_vs_oracle(index_dtype, K):
    A = rand_csr(120, 77, 6, batch=5, index_dtype=index_dtype, seed=3)
    B = torch.rand(5, 77, K, device=DEV)
    G = torch.rand(5, 120, K, device=DEV)
    _check(A, B, G)


@pytest.mark.parametrize("K", [7, 64])
@pytest.mark.parametrize("coalesced", [True, False])
def test_coo_vs_oracle(K, coalesced):
    n, m, nnz = 300, 211, 4000
    g = torch.Generator().manual_seed(K)
    flat = torch.randperm(n * m, generator=g)[:nnz]
    idx = torch.stack([flat // m, flat % m])
    if not coalesced:  # add duplicates and keep the shuffled storage order
        idx = torch.cat([idx, idx[:, :500]], dim=1)
    vals = torch.rand(idx.shape[1], generator=g)
    A = torch.sparse_coo_tensor(idx.to(DEV), vals.to(DEV), (n, m))
    if coalesced:
        A = A.coalesce()
    _check(A, torch.rand(m, K, device=DEV), torch.rand(n, K, device=DEV))


@pytest.mark.parametrize("dups", [False, True])
def test_ragged_batched_coo_vs_oracle(dups):
    b, n, m, K = 4, 50, 40, 32
    g = torch.Generator().manual_seed(11)
    parts = []
    for t, nnz in enumerate([300, 0, 17, 120]):
        flat = torch.randperm(n * m, generator=g)[:nnz]
        parts.append(torch.stack([torch.full((nnz,), t), flat // m, flat % m]))
    idx = torch.cat(parts, dim=1)
    if dups:
        idx = torch.cat([idx, idx[:, 5:60]], dim=1)
    idx = idx[:, torch.randperm(idx.shape[1], generator=g)]
    A = torch.sparse_coo_tensor(idx.to(DEV), torch.rand(idx.shape[1], generator=g).to(DEV), (b, n, m))
    _check(A, torch.rand(b, m, K, device=DEV), torch.rand(b, n, K, device=DEV))


def test_long_rows_and_empty_rows():
    """Rows far longer than a warp batch next to empty rows (row-split corner cases)."""
    n, m, K = 64, 5000, 128
    g = torch.Generator().manual_seed(5)
    cnt = torch.zeros(n, dtype=torch.int64)
    cnt[3], cnt[10], cnt[63] = 4097, 33, 1
    crow = torch.zeros(n + 1, dtype=torch.int64)
    crow[1:] = cnt.cumsum(0)
    col = torch.cat([torch.randperm(m, generator=g)[:c].sort().values for c in cnt.tolist()])
    A = torch.sparse_csr_tensor(crow.to(DEV), col.to(DEV), torch.rand(col.numel(), generator=g).to(DEV), (n, m))
    _check(A, torch.rand(m, K, device=DEV), torch.rand(n, K, device=DEV))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16])
@pytest.mark.parametrize("K", [64, 512])
def test_normal_operands_scaled_tolerance(K, dtype):
    """Benchmark distribution (B, G ~ N(0,1), benchmarks/sparse_mm_rand.py:75)."""
    A = rand_csr(257, 199, 12, dtype=dtype, seed=K)
    _check(A, torch.randn(199, K, device=DEV, dtype=dtype), torch.randn(257, K, device=DEV, dtype=dtype),
           scaled_atol=True)


def test_strided_operands():
    """B and the upstream gradient as transposed / permuted / expanded views
    (distributions/sparse_multivariate_normal.py:93-100 hands sparse_mm exactly these)."""
    from torchsparsegradutils_b200 import sparse_mm

    n, S = 96, 32
    A = rand_csr(n, n, 5, seed=9)
    V = torch.rand(S, n, device=DEV, requires_grad=True)
    out = sparse_mm(A, V.t()).t()  # (S, n): grad arrives transposed as well
    ref = (A.to_dense().double() @ V.detach().double().t()).t()
    torch.testing.assert_close(out.detach().double(), ref, rtol=1e-5, atol=1e-6)
    out.sum().backward()  # expanded (stride-0) upstream gradient
    gref = A.to_dense().double().t() @ torch.ones(n, S, device=DEV, dtype=torch.float64)
    torch.testing.assert_close(V.grad.double(), gref.t(), rtol=1e-5, atol=1e-6)
    Ab = rand_csr(n, n, 5, batch=3, seed=10)
    Vb = torch.rand(S, 3, n, device=DEV)
    outb = sparse_mm(Ab, Vb.permute(1, 2, 0)).permute(2, 0, 1)
    refb = torch.einsum("bij,sbj->sbi", Ab.to_dense().double(), Vb.double())
    torch.testing.assert_close(outb.double(), refb, rtol=1e-5, atol=1e-6)


# ------------------------------------------------- the reference's own test contract, re-targeted
TEST_DATA = [((4, 6), (6, 2), 8), ((8, 16), (16, 10), 32), ((7, 4), (4, 9), 14),
             ((1, 4, 6), (1, 6, 2), 8), ((4, 8, 16), (4, 16, 10), 32), ((11, 7, 4), (11, 4, 9), 14)]


def _rand_sparse(shape, nnz, layout, index_dtype, dtype, seed=0):
    """Output contract of the reference's rand_sparse (unique coords, nnz per item, coalesced / sorted)."""
    g = torch.Generator().manual_seed(seed)
    b = shape[0] if len(shape) == 3 else 1
    n, m = shape[-2:]
    mats = []
    for _ in range(b):
        flat = torch.randperm(n * m, generator=g)[:nnz].sort().values
        mats.append(torch.sparse_coo_tensor(torch.stack([flat // m, flat % m]), torch.rand(nnz, generator=g).to(dtype),
                                            (n, m)).coalesce())
    if layout == torch.sparse_coo:
        A = torch.stack(mats).coalesce() if len(shape) == 3 else mats[0]
        return A.to(DEV)
    csrs = [t.to_sparse_csr() for t in mats]
    crow = torch.stack([c.crow_indices() for c in csrs]) if len(shape) == 3 else csrs[0].crow_indices()
    col = torch.stack([c.col_indices() for c in csrs]) if len(shape) == 3 else csrs[0].col_indices()
    val = torch.stack([c.values() for c in csrs]) if len(shape) == 3 else csrs[0].values()
    return torch.sparse_csr_tensor(crow.to(index_dtype).to(DEV), col.to(index_dtype).to(DEV), val.to(DEV), shape)


@pytest.mark.parametrize("shapes", TEST_DATA, ids=lambda s: "x".join(map(str, s[0])))
@pytest.mark.parametrize("layout", [torch.sparse_coo, torch.sparse_csr], ids=["coo", "csr"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("index_dtype", [torch.int32, torch.int64], ids=["i32", "i64"])
def test_forward_backward_vs_dense(shapes, layout, dtype, index_dtype):
    """tests/test_sparse_matmul.py:78-128 with the reference's tolerances tightened to north_star's."""
    from torchsparsegradutils_b200 import sparse_mm

    A_shape, B_shape, nnz = shapes
    As = _rand_sparse(A_shape, nnz, layout, index_dtype, dtype, seed=nnz).requires_grad_()
    Ad = As.detach().clone().to_dense().requires_grad_()
    B1 = torch.rand(*B_shape, dtype=dtype, device=DEV).requires_grad_()
    B2 = B1.detach().clone().requires_grad_()
    r1, r2 = sparse_mm(As, B1), torch.matmul(Ad, B2)
    tol = TOL[dtype]
    torch.testing.assert_close(r1, r2, **tol)
    go = torch.rand_like(r1)
    r1.backward(go)
    r2.backward(go)
    assert As.grad.layout == layout
    if layout is torch.sparse_csr or len(A_shape) == 2:
        assert As.grad._nnz() == nnz
    else:
        assert As.grad._nnz() == nnz * A_shape[0]
    if layout is torch.sparse_csr:
        assert As.grad.crow_indices().dtype == index_dtype
    mask = As.grad.to_dense() != 0.0
    torch.testing.assert_close(As.grad.to_dense()[mask], Ad.grad[mask], **tol)
    torch.testing.assert_close(B1.grad, B2.grad, **tol)


@pytest.mark.parametrize("layout", [torch.sparse_coo, torch.sparse_csr], ids=["coo", "csr"])
def test_conditional_gradients(layout):
    """tests/test_sparse_matmul.py:134-157."""
    from torchsparsegradutils_b200 import sparse_mm

    A = _rand_sparse((5, 4), 6, layout, torch.int64, torch.float32)
    B = torch.randn(4, 3, device=DEV)
    A1, B1 = A.detach().clone(), B.detach().clone().requires_grad_()
    sparse_mm(A1, B1).sum().backward()
    assert A1.grad is None and B1.grad is not None
    A2, B2 = A.detach().clone().requires_grad_(), B.detach().clone()
    out = sparse_mm(A2, B2)
    assert out.requires_grad
    out.sum().backward()
    assert A2.grad is not None and B2.grad is None
    with torch.no_grad():
        assert not sparse_mm(A2, B2).requires_grad
    assert not sparse_mm(A.detach(), B.detach()).requires_grad


def test_dtype_mismatch_is_runtime_error():
    from torchsparsegradutils_b200 import sparse_mm

    A = _rand_sparse((5, 4), 6, torch.sparse_csr, torch.int64, torch.float32)
    with pytest.raises(RuntimeError, match="same dtype"):
        sparse_mm(A, torch.randn(4, 3, device=DEV, dtype=torch.float64))


@pytest.mark.parametrize("layout", [torch.sparse_coo, torch.sparse_csr], ids=["coo", "csr"])
def test_multi_step_optimisation(layout):
    """tests/test_sparse_matmul.py:295-338: A.grad values drive in-place SGD on A's values for 3 steps."""
    from torchsparsegradutils_b200 import sparse_mm

    A = _rand_sparse((12, 9), 30, layout, torch.int64, torch.float32).requires_grad_()
    B = torch.randn(9, 4, device=DEV)
    tgt = torch.randn(12, 4, device=DEV)
    losses = []
    for _ in range(3):
        loss = ((sparse_mm(A, B) - tgt) ** 2).sum()
        loss.backward()
        losses.append(float(loss))
        with torch.no_grad():
            gv = A.grad._values() if layout == torch.sparse_coo else A.grad.values()
            av = A._values() if layout == torch.sparse_coo else A.values()
            av -= 1e-3 * gv
        A.grad = None
    assert B.grad is None and losses[2] < losses[0]


def test_double_backward_raises():
    """tests/test_sparse_matmul.py:363-376."""
    from torchsparsegradutils_b200 import sparse_mm

    A = _rand_sparse((6, 6), 10, torch.sparse_coo, torch.int64, torch.float32).requires_grad_()
    B = torch.randn(6, 2, device=DEV, requires_grad=True)
    loss = sparse_mm(A, B).sum()
    loss.backward()
    with pytest.raises(RuntimeError, match="second time"):
        loss.backward()


def test_non_leaf_sparse_input_routes_grad_to_values():
    """README.md:145-156: A built from values that require grad."""
    from torchsparsegradutils_b200 import sparse_mm

    idx = torch.tensor([[0, 1, 1], [2, 0, 2]], device=DEV)
    vals = torch.tensor([3.0, 4.0, 5.0], device=DEV, requires_grad=True)
    B = torch.randn(3, 2, device=DEV)
    sparse_mm(torch.sparse_coo_tensor(idx, vals, (2, 3)), B).sum().backward()
    torch.testing.assert_close(vals.grad, B.sum(dim=1)[idx[1]])


def test_quickstart_examples():
    """tests/test_quickstart_guide.py:12-54 and the doctests at sparse_matmul.py:85-111."""
    from torchsparsegradutils_b200 import sparse_mm

    A = torch.tensor([[0, 1.0], [2.0, 0], [0, 3.0]], device=DEV).to_sparse().requires_grad_()
    B = torch.randn(2, 2, device=DEV, requires_grad=True)
    out = sparse_mm(A, B)
    assert out.shape == (3, 2)
    out.sum().backward()
    assert A.grad.is_sparse and A.grad._nnz() == 3
    Ab = torch.stack([A.detach(), A.detach()]).requires_grad_()
    outb = sparse_mm(Ab, torch.randn(2, 2, 2, device=DEV))
    assert outb.shape == (2, 3, 2)
    outb.sum().backward()
    assert Ab.grad.is_sparse and Ab.grad.sparse_dim() == 3
    # known answer, Dockerfile.pip-install:47-52
    K = torch.tensor([[2.0, 0.0], [3.0, 4.0]], device=DEV).to_sparse_coo()
    assert torch.equal(sparse_mm(K, torch.tensor([[5.0], [7.0]], device=DEV)).cpu(), torch.tensor([[10.0], [43.0]]))


def test_pattern_cache_sees_inplace_index_edits():
    from torchsparsegradutils_b200 import sparse_mm

    idx = torch.tensor([[0, 1], [0, 1]], device=DEV)
    A = torch.sparse_coo_tensor(idx, torch.ones(2, device=DEV), (2, 2))
    B = torch.tensor([[1.0, 2.0], [3.0, 4.0]], device=DEV)
    assert torch.equal(sparse_mm(A, B), B)
    A._indices()[1] = torch.tensor([1, 0], device=DEV)  # same storage, new pattern: _version bumps
    assert torch.equal(sparse_mm(A, B), B.flip(0))
    # edits through an unrelated alias of the index storage are invisible to torch's version counters;
    # the documented escape hatch is to drop the cache
    import torchsparsegradutils_b200 as tsgu

    idx[1] = torch.tensor([0, 1], device=DEV)
    tsgu.clear_pattern_cache()
    assert torch.equal(sparse_mm(A, B), B)


def test_memory_no_nnz_by_k_temporaries():
    """tests/test_sparse_matmul.py:217-292 in spirit: fwd+bwd peak stays far below one nnz x K temporary
    (the reference's backward materialises three of them)."""
    from torchsparsegradutils_b200 import sparse_mm

    n, K, per_row = 20000, 512, 16
    A = rand_csr(n, n, per_row, seed=1).requires_grad_()
    B = torch.randn(n, K, device=DEV, requires_grad=True)
    G = torch.randn(n, K, device=DEV)
    sparse_mm(A, B).backward(G)  # warm the pattern cache (transpose build)
    A.grad = B.grad = None
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    sparse_mm(A, B).backward(G)
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    one_temp = n * per_row * K * 4
    assert extra < 0.25 * one_temp, (extra, one_temp)


# ---------------------------------------------------------------- merge-path (nnz-balanced) kernels
def _skewed_csr(n, m, seed, dtype=torch.float32, index_dtype=torch.int32, hub_rows=(0, 7, 300), hub_len=9000):
    """Power-law-ish rows: a few hubs far longer than a tile, many empty rows, short rows in between."""
    g = torch.Generator().manual_seed(seed)
    cnt = torch.randint(0, 4, (n,), generator=g)
    cnt[torch.rand(n, generator=g) < 0.4] = 0
    for r in hub_rows:
        if r < n:
            cnt[r] = min(hub_len, m)
    cnt[n - 1] = min(2500, m)  # long last row: the path ends inside a cut row
    crow = torch.zeros(n + 1, dtype=torch.int64)
    crow[1:] = cnt.cumsum(0)
    col = torch.cat([torch.randperm(m, generator=g)[:c].sort().values for c in cnt.tolist()])
    vals = torch.rand(col.numel(), generator=g, dtype=torch.float64).to(dtype)
    return torch.sparse_csr_tensor(crow.to(index_dtype).to(DEV), col.to(index_dtype).to(DEV), vals.to(DEV), (n, m))


@pytest.mark.parametrize("K", [16, 32, 64, 128, 160, 512, 10])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16])
def test_merge_path_vs_oracle(K, dtype, monkeypatch):
    """Forced merge-path SpMM / SDDMM / transposed SpMM on skewed rows vs the oracle (K = 10 is not vectorisable in
    fp32 / bf16 and must fall back to the row-split kernels)."""
    import torchsparsegradutils_b200 as tsgu

    monkeypatch.setenv("TSGU_B200_ALGO", "merge")
    tsgu.clear_pattern_cache()
    n, m = 1500, 12000
    A = _skewed_csr(n, m, seed=K, dtype=dtype)
    _check(A, torch.rand(m, K, device=DEV, dtype=dtype), torch.rand(n, K, device=DEV, dtype=dtype))
    tsgu.clear_pattern_cache()


@pytest.mark.parametrize("index_dtype", [torch.int32, torch.int64])
def test_merge_path_auto_selected_and_matches_rowsplit(index_dtype, monkeypatch):
    """The skew heuristic picks merge-path by itself, and both kernel families agree bit for bit on
    the integer side (pattern) and to fp32 rounding on values."""
    import torchsparsegradutils_b200 as tsgu
    from torchsparsegradutils_b200 import _native as nat
    from torchsparsegradutils_b200._pattern import csr_pattern

    tsgu.clear_pattern_cache()
    A = _skewed_csr(4000, 20000, seed=1, index_dtype=index_dtype, hub_len=15000)
    assert csr_pattern(A).algo == nat.ALGO_MERGE
    B = torch.rand(20000, 64, device=DEV)
    G = torch.rand(4000, 64, device=DEV)
    C1, gA1, gB1 = _run(A, B, G)
    monkeypatch.setenv("TSGU_B200_ALGO", "rowsplit")
    tsgu.clear_pattern_cache()
    C2, gA2, gB2 = _run(A, B, G)
    tsgu.clear_pattern_cache()
    torch.testing.assert_close(C1, C2, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(gA1.values(), gA2.values(), rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(gB1, gB2, rtol=1e-5, atol=1e-6)


def test_merge_path_coo_unsorted(monkeypatch):
    """COO input (value permutation staged instead of values) through the merge-path kernels."""
    import torchsparsegradutils_b200 as tsgu

    monkeypatch.setenv("TSGU_B200_ALGO", "merge")
    tsgu.clear_pattern_cache()
    Acsr = _skewed_csr(700, 5000, seed=3, index_dtype=torch.int64, hub_len=4000)
    crow, col, vals = Acsr.crow_indices(), Acsr.col_indices(), Acsr.values()
    rows = torch.repeat_interleave(torch.arange(700, device=DEV), crow[1:] - crow[:-1])
    sh = torch.randperm(col.numel(), device=DEV)
    A = torch.sparse_coo_tensor(torch.stack([rows, col])[:, sh], vals[sh], (700, 5000))
    _check(A, torch.rand(5000, 32, device=DEV), torch.rand(700, 32, device=DEV))
    tsgu.clear_pattern_cache()


# ------------------------------------------------------------------ remaining C-ABI entry points
@pytest.mark.parametrize("K", [1, 5, 32, 64, 256, 1100])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16])
def test_sddmm_coo_entry_point(K, dtype):
    """tsgu_sddmm_coo: order-agnostic <G[row], B[col]> on raw int64 COO coordinates (the idiom the
    solve / lstsq backwards share, sparse_solve.py:216-235) vs the oracle."""
    from torchsparsegradutils_b200 import _ops

    n, m, nnz = 150, 90, 2000
    g = torch.Generator().manual_seed(K)
    row = torch.randint(0, n, (nnz,), generator=g).to(DEV)
    col = torch.randint(0, m, (nnz,), generator=g).to(DEV)
    G = torch.rand(n, K, generator=g).to(dtype).to(DEV)
    B = torch.rand(m, K, generator=g).to(dtype).to(DEV)
    out = _ops.sddmm_coo(row, col, G, B)
    odt = np.float64 if dtype == torch.float64 else np.float32
    ref = orc.sddmm(_np(row), _np(col), _np(G).astype(odt), _np(B).astype(odt))
    torch.testing.assert_close(out.double().cpu(), torch.from_numpy(ref.astype(np.float64)), **TOL[dtype])
    # strided operands take the scalar path
    out_t = _ops.sddmm_coo(row, col, G.t().contiguous().t(), B)
    torch.testing.assert_close(out_t, out, **TOL[dtype])


@pytest.mark.parametrize("shape", [(1, 1000, 7), (3, 257, 33), (2, 64, 128), (1, 5, 1)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16])
def test_copy_dense_layouts(shape, dtype):
    """tsgu_pack_dense between every pair of (row-major, column-major, batch-last) layouts."""
    from torchsparsegradutils_b200 import _ops

    x = torch.randn(shape, device=DEV).to(dtype)
    views = [x, x.transpose(1, 2).contiguous().transpose(1, 2), x.permute(1, 2, 0).contiguous().permute(2, 0, 1)]
    for src in views:
        assert torch.equal(_ops.pack_dense(src), x)
        for like in views:
            out = _ops.restride_like(src, src.shape, like.stride())
            assert out.stride() == like.stride() and torch.equal(out, x)


@pytest.mark.parametrize("layout", ["coo", "csr", "bcsr"])
def test_public_sddmm_matches_solve_backward_idiom(layout):
    """sddmm(A, X, Y) == (X.index_select(0,row) * Y.index_select(0,col)).sum(1), the idiom of
    sparse_solve.py:216-235 / sparse_lstsq.py:239-256, on A's storage order."""
    from torchsparsegradutils_b200 import sddmm

    n, m, K = 90, 70, 48
    if layout == "bcsr":
        A = rand_csr(n, m, 6, batch=3, seed=4)
        X, Y = torch.rand(3, n, K, device=DEV), torch.rand(3, m, K, device=DEV)
        out = sddmm(A, X, Y)
        assert out.shape == A.values().shape
        for t in range(3):
            crow, col = A.crow_indices()[t].long(), A.col_indices()[t].long()
            row = torch.repeat_interleave(torch.arange(n, device=DEV), crow[1:] - crow[:-1])
            ref = (X[t].double().index_select(0, row) * Y[t].double().index_select(0, col)).sum(1)
            torch.testing.assert_close(out[t].double(), ref, rtol=1e-5, atol=1e-6)
        return
    Acsr = rand_csr(n, m, 6, seed=5, ragged=True)
    crow, col = Acsr.crow_indices().long(), Acsr.col_indices().long()
    row = torch.repeat_interleave(torch.arange(n, device=DEV), crow[1:] - crow[:-1])
    X, Y = torch.rand(n, K, device=DEV), torch.rand(m, K, device=DEV)
    if layout == "coo":
        sh = torch.randperm(col.numel(), device=DEV)
        row, col = row[sh], col[sh]
        A = torch.sparse_coo_tensor(torch.stack([row, col]), torch.ones(col.numel(), device=DEV), (n, m))
    else:
        A = Acsr
    ref = (X.double().index_select(0, row) * Y.double().index_select(0, col)).sum(1)
    torch.testing.assert_close(sddmm(A, X, Y).double(), ref, rtol=1e-5, atol=1e-6)
    with pytest.raises(ValueError, match="Incompatible shapes"):
        sddmm(A, X, torch.rand(m, K + 1, device=DEV))


# ------------------------------------------ persistent-tile kernels on oracle-sized inputs
@pytest.fixture
def force_tile_kernels(monkeypatch):
    """Small problems normally take the row-split kernels; TSGU_TINY_ROWS=0 sends them through the
    persistent bulk-copy-staged tile kernels so every (lanes-per-row x vectors-per-lane x dtype) variant
    is checked against the oracle."""
    import torchsparsegradutils_b200 as tsgu

    monkeypatch.setenv("TSGU_TINY_ROWS", "0")
    tsgu.clear_pattern_cache()
    yield
    tsgu.clear_pattern_cache()


@pytest.mark.parametrize("K", [4, 8, 16, 24, 32, 64, 96, 128, 192, 256, 512])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64, torch.bfloat16])
def test_tile_kernels_vs_oracle_all_K(K, dtype, force_tile_kernels):
    if K % {torch.float32: 4, torch.float64: 2, torch.bfloat16: 8}[dtype]:
        pytest.skip("K not vectorisable for this dtype: scalar row-split path, covered elsewhere")
    n, m = 700, 450
    A = rand_csr(n, m, 13, dtype=dtype, index_dtype=torch.int32, seed=K, ragged=True)
    _check(A, torch.rand(m, K, device=DEV, dtype=dtype), torch.rand(n, K, device=DEV, dtype=dtype))


@pytest.mark.parametrize("index_dtype", [torch.int32, torch.int64])
def test_tile_kernels_batched_and_long_rows(index_dtype, force_tile_kernels):
    A = rand_csr(300, 200, 9, batch=4, index_dtype=index_dtype, seed=21)
    _check(A, torch.rand(4, 200, 128, device=DEV), torch.rand(4, 300, 128, device=DEV))
    # a row longer than the staging capacity (tile falls back to direct loads) next to empty rows
    n, m = 96, 9000
    g = torch.Generator().manual_seed(5)
    cnt = torch.zeros(n, dtype=torch.int64)
    cnt[2], cnt[40], cnt[95] = 8200, 70, 3
    crow = torch.zeros(n + 1, dtype=torch.int64)
    crow[1:] = cnt.cumsum(0)
    col = torch.cat([torch.randperm(m, generator=g)[:c].sort().values for c in cnt.tolist()])
    A2 = torch.sparse_csr_tensor(crow.to(index_dtype).to(DEV), col.to(index_dtype).to(DEV),
                                 torch.rand(col.numel(), generator=g).to(DEV), (n, m))
    _check(A2, torch.rand(m, 64, device=DEV), torch.rand(n, 64, device=DEV))


def test_tile_kernels_coo_value_permutation(force_tile_kernels):
    """Uncoalesced COO: the tile SpMM stages the value permutation instead of the values, the SDDMM
    scatters through out_index."""
    n, m, nnz = 500, 300, 6000
    g = torch.Generator().manual_seed(2)
    flat = torch.randperm(n * m, generator=g)[:nnz]
    idx = torch.stack([flat // m, flat % m])
    idx = torch.cat([idx, idx[:, :300]], dim=1)  # duplicates, unsorted
    A = torch.sparse_coo_tensor(idx.to(DEV), torch.rand(idx.shape[1], generator=g).to(DEV), (n, m))
    _check(A, torch.rand(m, 32, device=DEV), torch.rand(n, 32, device=DEV))
    Ab = torch.stack([A.coalesce(), A.coalesce()])
    _check(Ab, torch.rand(2, m, 32, device=DEV), torch.rand(2, n, 32, device=DEV))


@pytest.mark.parametrize("layout", ["csr", "coo", "bcsr"])
def test_graphed_step_matches_eager(layout):
    """GraphedSparseMM replays forward+backward from one CUDA graph: same numbers as the eager op, also
    after the values / dense operands change."""
    from torchsparsegradutils_b200 import GraphedSparseMM

    n, m, K = 400, 300, 64
    if layout == "bcsr":
        A = rand_csr(n, m, 7, batch=3, seed=1)
        B, G = torch.rand(3, m, K, device=DEV), torch.rand(3, n, K, device=DEV)
    else:
        A = rand_csr(n, m, 7, seed=1, ragged=True)
        if layout == "coo":
            A = A.to_sparse_coo()
        B, G = torch.rand(m, K, device=DEV), torch.rand(n, K, device=DEV)
    step = GraphedSparseMM(A, B, G)
    vals = A.values() if A.layout == torch.sparse_csr else A._values()
    for trial in range(3):
        v, Bt, Gt = vals * (trial + 1), B + trial, G - 0.5 * trial
        C, gA, gB = step(v, Bt, Gt)
        if A.layout == torch.sparse_csr:
            At = torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(), v, A.shape)
        else:
            At = torch.sparse_coo_tensor(A._indices(), v, A.shape, is_coalesced=A.is_coalesced())
        C2, gA2, gB2 = _run(At, Bt, Gt)
        gA2v = gA2.values() if A.layout == torch.sparse_csr else gA2._values()
        assert torch.equal(C, C2) and torch.equal(gA.reshape(-1), gA2v.reshape(-1)) and torch.equal(gB, gB2)


def test_pattern_cache_key_distinguishes_aliasing_index_views():
    """Two COO tensors whose index tensors are different-length views of ONE buffer at offset 0 (same data pointer,
    same version) must not share a cached pattern (ADVICE r1: the key now carries numel / shape / strides / offset)."""
    import torchsparsegradutils_b200 as tsgu
    from torchsparsegradutils_b200 import sparse_mm

    tsgu.clear_pattern_cache()
    g = torch.Generator().manual_seed(3)
    n = m = 64
    flat = torch.randperm(n * m, generator=g)[:200]
    idx = torch.stack([flat // m, flat % m]).to(DEV)
    v = torch.rand(200, generator=g).to(DEV)
    B = torch.rand(m, 8, generator=g).to(DEV)
    for cnt in (100, 200, 100):
        A = torch.sparse_coo_tensor(idx[:, :cnt], v[:cnt], (n, m))
        assert A._indices().data_ptr() == idx.data_ptr()
        torch.testing.assert_close(sparse_mm(A, B), torch.sparse.mm(A, B), rtol=1e-5, atol=1e-6)
    # CSR: col views of one buffer with different lengths
    crow1 = torch.tensor([0, 2, 3], device=DEV, dtype=torch.int32)
    crow2 = torch.tensor([0, 2, 4], device=DEV, dtype=torch.int32)
    colbuf = torch.tensor([0, 2, 1, 3], device=DEV, dtype=torch.int32)
    vals = torch.tensor([1.0, 2.0, 3.0, 4.0], device=DEV)
    Bs = torch.rand(4, 4, device=DEV)
    A1 = torch.sparse_csr_tensor(crow1, colbuf[:3], vals[:3], (2, 4))
    A2 = torch.sparse_csr_tensor(crow2, colbuf[:4], vals[:4], (2, 4))
    torch.testing.assert_close(sparse_mm(A1, Bs), A1.to_dense() @ Bs)
    torch.testing.assert_close(sparse_mm(A2, Bs), A2.to_dense() @ Bs)
    tsgu.clear_pattern_cache()


def test_graphed_sparse_mm_survives_an_empty_pattern_cache():
    """GraphedSparseMM pins its pattern: capture and replay work with the LRU cache switched off (capacity 0)."""
    import torchsparsegradutils_b200 as tsgu
    from torchsparsegradutils_b200 import GraphedSparseMM, sparse_mm

    tsgu.set_pattern_cache_capacity(0)
    try:
        A = rand_csr(300, 200, 5, seed=11)
        B = torch.rand(200, 16, device=DEV)
        G = torch.rand(300, 16, device=DEV)
        gs = GraphedSparseMM(A, B, G)
        C, gAv, gB = gs(A.values(), B, G)
        C2, gA2, gB2 = _run(A, B, G)
        assert torch.equal(C, C2) and torch.equal(gAv, gA2.values()) and torch.equal(gB, gB2)
    finally:
        tsgu.set_pattern_cache_capacity(16)
        tsgu.clear_pattern_cache()


def test_pattern_cache_byte_cap_evicts():
    import torchsparsegradutils_b200 as tsgu
    from torchsparsegradutils_b200 import _pattern

    tsgu.clear_pattern_cache()
    old = _pattern._CACHE_BYTES
    try:
        mats = [rand_csr(2000, 2000, 8, seed=s) for s in range(4)]
        one = _pattern.pattern_nbytes(_pattern.csr_pattern(mats[0]))
        assert one >= 2000 * 8 * 4
        tsgu.set_pattern_cache_capacity(16, max_bytes=int(2.5 * one))
        for M in mats:
            _pattern.csr_pattern(M)
        assert 1 <= len(_pattern._cache) <= 2
    finally:
        tsgu.set_pattern_cache_capacity(16, max_bytes=old)
        tsgu.clear_pattern_cache()


@pytest.mark.parametrize("mode", ["sampled", "1", "0"])
def test_rewritten_index_memory_under_a_cached_pattern_is_detected(mode, monkeypatch):
    """An in-place rewrite of index memory through an alias is invisible to the cache key; the stored checksum catches
    it on the first reuse (default: re-checked on hits 1, 2, 4, ...; "1": every hit; "0": checks off, stale reuse)."""
    import torchsparsegradutils_b200 as tsgu
    from torchsparsegradutils_b200 import _pattern, sparse_mm

    tsgu.clear_pattern_cache()
    monkeypatch.setattr(_pattern, "_VERIFY", mode)
    idx = torch.tensor([[0, 1], [0, 1]], device=DEV)
    A = torch.sparse_coo_tensor(idx, torch.ones(2, device=DEV), (2, 2))
    B = torch.tensor([[1.0, 2.0], [3.0, 4.0]], device=DEV)
    assert torch.equal(sparse_mm(A, B), B)
    idx[1] = torch.tensor([1, 0], device=DEV)  # alias write: no version bump on A._indices()
    if mode == "0":
        assert torch.equal(sparse_mm(A, B), B)  # the frozen-pattern contract, unchecked: the OLD pattern is used
    elif mode == "1":
        with pytest.raises(RuntimeError, match="rewritten in place"):
            sparse_mm(A, B)
    else:  # checked on the first reuse, reported by the next hit after the check has landed
        with pytest.raises(RuntimeError, match="rewritten in place.*deferred"):
            for _ in range(3):
                sparse_mm(A, B)
                torch.cuda.synchronize()
    tsgu.clear_pattern_cache()
    assert torch.equal(sparse_mm(A, B), B.flip(0))
    # CSR, int32, large enough for the multi-block checksum kernel; a long run of clean hits stays clean
    crow = torch.arange(0, 4 * 3000 + 1, 4, device=DEV, dtype=torch.int32)
    col = (torch.arange(4 * 3000, device=DEV, dtype=torch.int32) * 7) % 3000
    Ac = torch.sparse_csr_tensor(crow, col, torch.ones(4 * 3000, device=DEV), (3000, 3000))
    Bc = torch.randn(3000, 8, device=DEV)
    assert _pattern._fingerprint(crow, col).tolist() == _pattern._fingerprint(crow.cpu(), col.cpu()).tolist()  # kernel == host restatement
    ref = sparse_mm(Ac, Bc)
    for _ in range(9):
        assert torch.equal(sparse_mm(Ac, Bc), ref)
    col[5] = (col[5] + 1) % 3000
    if mode == "1":
        with pytest.raises(RuntimeError, match="rewritten in place"):
            sparse_mm(Ac, Bc)
    elif mode == "sampled":  # hits 10..15 are not checked, hit 16 is -- deferred: a later hit reports it
        with pytest.raises(RuntimeError, match="rewritten in place.*deferred"):
            for _ in range(12):
                sparse_mm(Ac, Bc)
                torch.cuda.synchronize()
    tsgu.clear_pattern_cache()


def test_graph_capture_with_a_deferred_pattern_check_outstanding():
    """The deferred checksum comparison must stay out of a CUDA graph capture: with a check in flight (launched by the
    first reuse of the pattern, not yet collected) a capture of the next call has to succeed -- an event query inside
    the capture would invalidate it, and bench.py would silently fall back to its eager region."""
    import torchsparsegradutils_b200 as tsgu
    from torchsparsegradutils_b200 import sparse_mm
    from torchsparsegradutils_b200._pattern import csr_pattern

    tsgu.clear_pattern_cache()
    A = rand_csr(300, 200, 5, seed=3)
    B = torch.randn(200, 16, device=DEV)
    ref = sparse_mm(A, B)       # miss: pattern built
    sparse_mm(A, B)             # hit 1: deferred check launched
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        sparse_mm(A, B)
    torch.cuda.current_stream().wait_stream(side)
    pat = csr_pattern(A)
    pat.pending_check = (torch.cuda.Event(), torch.zeros(4, dtype=torch.int64))  # a check that has not landed yet
    pat.pending_check[0].record()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = sparse_mm(A, B)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, ref)
    tsgu.clear_pattern_cache()


def test_unsupported_value_dtype_is_a_runtime_error():
    from torchsparsegradutils_b200 import sparse_mm

    A = rand_csr(8, 8, 2, seed=1)
    Ah = torch.sparse_csr_tensor(A.crow_indices(), A.col_indices(), A.values().half(), A.shape)
    with pytest.raises(RuntimeError, match="unsupported value dtype"):
        sparse_mm(Ah, torch.rand(8, 4, device=DEV).half())


def test_misaligned_csr_views_take_the_fast_kernels_and_match():
    """CSR arrays that are views at an odd element offset (a row block cut out of a larger matrix): results equal the
    aligned copy's bit for bit, and the pattern holds aligned copies so that the staged kernels stay eligible."""
    import torchsparsegradutils_b200 as tsgu
    from torchsparsegradutils_b200 import sparse_mm
    from torchsparsegradutils_b200._pattern import csr_pattern

    tsgu.clear_pattern_cache()
    A = rand_csr(30000, 5000, 9, seed=4)
    crow, col, val = A.crow_indices(), A.col_indices(), A.values()
    lo, hi = 7, 30000
    s, e = int(crow[lo]), int(crow[hi])
    assert (s * 4) % 16 != 0
    Av = torch.sparse_csr_tensor((crow[lo:hi + 1] - crow[lo]), col[s:e], val[s:e], (hi - lo, 5000))
    assert Av.col_indices().data_ptr() % 16 != 0
    Ac = torch.sparse_csr_tensor((crow[lo:hi + 1] - crow[lo]).clone(), col[s:e].clone(), val[s:e].clone(), (hi - lo, 5000))
    B = torch.rand(5000, 64, device=DEV)
    G = torch.rand(hi - lo, 64, device=DEV)
    C1, gA1, gB1 = _run(Av, B, G)
    C2, gA2, gB2 = _run(Ac, B, G)
    assert torch.equal(C1, C2) and torch.equal(gA1.values(), gA2.values()) and torch.equal(gB1, gB2)
    p = csr_pattern(Av)
    assert p.colind.data_ptr() % 16 == 0 and p.rowptr.data_ptr() % 16 == 0
    tsgu.clear_pattern_cache()
