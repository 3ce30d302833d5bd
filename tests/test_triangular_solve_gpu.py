"""GPU: ``sparse_triangular_solve`` (csrc/trisolve.cu) against the reference's own solves (x, B.grad and A.grad of
``sparse_triangular_solve`` recorded in tests/golden/solve_grad_cases.npz and solve_batched_cases.npz), against
torch's sparse CSR ``triangular_solve`` over every flag combination, against dense autograd, and at sizes where the
level count matters.  Every solve checks the status word of the bounded waits."""
import os

import numpy as np
import pytest
import torch

import workloads as W

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SG = np.load(os.path.join(GOLDEN_DIR, "solve_grad_cases.npz"))
SB = np.load(os.path.join(GOLDEN_DIR, "solve_batched_cases.npz"))
FIXTURE_CASES = ([("grad", str(c)) for c in SG["__cases__"] if str(c).startswith("tri_")]
                 + [("batched", str(c)) for c in SB["__cases__"] if str(c).startswith("btri_")])


def _solve(A, B, **flags):
    from torchsparsegradutils_b200 import sparse_triangular_solve
    from torchsparsegradutils_b200.triangular_solve import solve_status

    x = sparse_triangular_solve(A, B, **flags)
    assert solve_status(DEV) == 0
    return x


def _backward(x, G):
    from torchsparsegradutils_b200.triangular_solve import solve_status

    x.backward(G)
    assert solve_status(DEV) == 0


def _op(dense, transpose):
    return dense.transpose(-1, -2) if transpose else dense


# ------------------------------------------------------------------------------------ 1. reference fixtures
@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("src,name", FIXTURE_CASES)
def test_reference_parity(src, name, dtype):
    G_ = SG if src == "grad" else SB
    k = lambda s: G_[f"{name}/{s}"]  # noqa: E731
    shape = tuple(int(v) for v in k("shape"))
    upper, transpose = "_upper_" in name, bool(k("transpose"))
    vals = torch.from_numpy(k("values"))
    if str(k("layout")) == "coo":
        A64 = torch.sparse_coo_tensor(torch.from_numpy(k("indices")), vals, shape)
    else:
        A64 = torch.sparse_csr_tensor(torch.from_numpy(k("crow")), torch.from_numpy(k("col")), vals, shape)
    # the fixtures keep x and B.grad but not B or the upstream gradient: rebuild both in fp64
    opA = _op(A64.to_dense(), transpose)
    x_ref, gB_ref = torch.from_numpy(k("x")), torch.from_numpy(k("gradB"))
    B = (opA @ x_ref).to(DEV, dtype).requires_grad_(True)
    G = (opA.transpose(-1, -2) @ gB_ref).to(DEV, dtype)
    A = A64.to(dtype).to(DEV).requires_grad_(True)
    x = _solve(A, B, upper=upper, transpose=transpose)
    _backward(x, G)
    tol = dict(rtol=1e-10, atol=1e-12) if dtype == torch.float64 else dict(rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(x.detach().cpu().double(), x_ref, **tol)
    torch.testing.assert_close(B.grad.cpu().double(), gB_ref, **tol)
    gA = A.grad
    assert gA.layout == A.layout and gA.shape == A.shape
    if A.layout == torch.sparse_csr:
        crow_key, col_key = ("crow", "col") if src == "grad" else ("gradA_crow", "gradA_col")
        assert torch.equal(gA.crow_indices().cpu().long(), torch.from_numpy(k(crow_key)))
        assert torch.equal(gA.col_indices().cpu().long(), torch.from_numpy(k(col_key)))
        got = gA.values()
    else:
        gA = gA.coalesce()
        assert torch.equal(gA.indices().cpu(), torch.from_numpy(k("indices" if src == "grad" else "gradA_indices")))
        got = gA.values()
    torch.testing.assert_close(got.cpu().double().reshape(-1), torch.from_numpy(k("gradA_values")).reshape(-1), **tol)


# ------------------------------------------------------------------------------ 2. torch's CSR solve
def _full_matrix(n, dtype, seed):
    """Entries in both triangles and on the diagonal; every 7th row holds only its diagonal."""
    g = torch.Generator().manual_seed(seed)
    M = torch.rand(n, n, generator=g, dtype=torch.float64) * (torch.rand(n, n, generator=g) < 0.05)
    M = M / 8.0
    M[::7] = 0.0
    M = M + torch.diag(1.0 + torch.rand(n, generator=g, dtype=torch.float64))
    return M.to(dtype)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("K", [1, 6, 32, 129])
@pytest.mark.parametrize("index_dtype", [torch.int32, torch.int64])
@pytest.mark.parametrize("transpose", [False, True])
@pytest.mark.parametrize("unitriangular", [False, True])
@pytest.mark.parametrize("upper", [False, True])
def test_matches_torch_csr_solve(upper, unitriangular, transpose, index_dtype, K, dtype):
    n = 301
    M = _full_matrix(n, dtype, seed=K + 3).to(DEV)
    Mc = M.to_sparse_csr()
    A = torch.sparse_csr_tensor(Mc.crow_indices().to(index_dtype), Mc.col_indices().to(index_dtype), Mc.values(),
                                (n, n))
    Bt = torch.randn(K, n, dtype=dtype, device=DEV)
    B = Bt.t()  # column-major view
    x = _solve(A, B, upper=upper, unitriangular=unitriangular, transpose=transpose)
    want = torch.triangular_solve(B.contiguous(), Mc, upper=upper, transpose=transpose,
                                  unitriangular=unitriangular).solution
    tol = dict(rtol=1e-10, atol=1e-12) if dtype == torch.float64 else dict(rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(x, want, **tol)
    assert x.is_contiguous()


# ------------------------------------------------------------------------------------------ 3. batched
def _batched_tri(b, n, dtype, upper, seed):
    g = torch.Generator().manual_seed(seed)
    mask = torch.rand(n, n, generator=g) < 0.1  # common pattern: batched CSR needs equal nnz per item
    mask = mask.triu(1) if upper else mask.tril(-1)
    off = torch.rand(b, n, n, generator=g, dtype=torch.float64) * mask / 4.0
    return (off + torch.diag_embed(1.0 + torch.rand(b, n, generator=g, dtype=torch.float64))).to(dtype)


@pytest.mark.parametrize("layout", ["csr", "coo"])
@pytest.mark.parametrize("transpose", [False, True])
@pytest.mark.parametrize("upper", [False, True])
def test_batched_against_per_item_torch(layout, upper, transpose):
    b, n, K = 4, 97, 5
    D = _batched_tri(b, n, torch.float64, upper, seed=11).to(DEV)
    A = D.to_sparse_csr() if layout == "csr" else D.to_sparse()
    B = torch.randn(b, n, K, dtype=torch.float64, device=DEV)
    x = _solve(A, B, upper=upper, transpose=transpose)
    for t in range(b):
        want = torch.triangular_solve(B[t], D[t].to_sparse_csr(), upper=upper, transpose=transpose).solution
        torch.testing.assert_close(x[t], want, rtol=1e-10, atol=1e-12)


def _with_duplicates(C, seed):
    """An uncoalesced COO tensor equal to the coalesced C: a third of the entries split in two, storage shuffled."""
    g = torch.Generator().manual_seed(seed)
    idx, v = C.indices().cpu(), C.values().cpu()
    dup = torch.randperm(v.numel(), generator=g)[: v.numel() // 3]
    frac = torch.rand(dup.numel(), generator=g, dtype=v.dtype)
    v2 = v.clone()
    v2[dup] = v[dup] * frac
    idx = torch.cat([idx, idx[:, dup]], dim=1)
    v2 = torch.cat([v2, v[dup] * (1 - frac)])
    sh = torch.randperm(v2.numel(), generator=g)
    return torch.sparse_coo_tensor(idx[:, sh], v2[sh], C.shape).to(DEV)


@pytest.mark.parametrize("batched", [False, True])
def test_uncoalesced_coo_equals_coalesced(batched):
    n, K = 120, 3
    D = _batched_tri(2 if batched else 1, n, torch.float64, False, seed=5).to(DEV)
    D = D if batched else D[0]
    C = D.to_sparse().coalesce()
    U = _with_duplicates(C, seed=9)
    assert not U.is_coalesced()
    B0 = torch.randn(D.shape[:-1] + (K,), dtype=torch.float64, device=DEV)
    G = torch.randn_like(B0)
    outs = []
    for A in (C, U):
        A = A.detach().requires_grad_(True)
        B = B0.clone().requires_grad_(True)
        x = _solve(A, B, upper=False)
        _backward(x, G)
        outs.append((x.detach(), B.grad, A.grad))
    (xc, gbc, gac), (xu, gbu, gau) = outs
    torch.testing.assert_close(xu, xc, rtol=1e-12, atol=1e-13)
    torch.testing.assert_close(gbu, gbc, rtol=1e-12, atol=1e-13)
    # every stored entry of U gets the gradient of its coordinate (duplicates each carry the full value)
    dense_gc = gac.to_dense()
    gau = gau.coalesce() if batched else gau
    ind = gau._indices()
    want = dense_gc[tuple(ind)]
    torch.testing.assert_close(gau._values(), want, rtol=1e-12, atol=1e-13)


@pytest.mark.parametrize("layout", ["csr", "coo"])
@pytest.mark.parametrize("batched", [False, True])
@pytest.mark.parametrize("transpose", [False, True])
@pytest.mark.parametrize("upper", [False, True])
def test_gradients_against_dense_autograd(upper, transpose, batched, layout):
    n, K = 64, 7
    D = _batched_tri(3 if batched else 1, n, torch.float64, upper, seed=21).to(DEV)
    D = D if batched else D[0]
    A = (D.to_sparse_csr() if layout == "csr" else D.to_sparse()).requires_grad_(True)
    B = torch.randn(D.shape[:-1] + (K,), dtype=torch.float64, device=DEV, requires_grad=True)
    G = torch.randn_like(B)
    x = _solve(A, B, upper=upper, transpose=transpose)
    _backward(x, G)

    Dd = D.clone().requires_grad_(True)
    Bd = B.detach().clone().requires_grad_(True)
    xd = torch.linalg.solve_triangular(_op(Dd, transpose), Bd, upper=upper != transpose)
    xd.backward(G)
    torch.testing.assert_close(x.detach(), xd.detach(), rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(B.grad, Bd.grad, rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(A.grad.to_dense(), Dd.grad * (D != 0), rtol=1e-10, atol=1e-12)


def test_only_needed_gradients():
    D = _batched_tri(1, 50, torch.float64, True, seed=2)[0].to(DEV)
    A = D.to_sparse_csr().requires_grad_(True)
    B = torch.randn(50, 2, dtype=torch.float64, device=DEV)
    x = _solve(A, B)
    _backward(x, torch.ones_like(x))
    assert A.grad is not None and B.grad is None


# ------------------------------------------------------------------------------------ 4. size and structure
def test_stencil_level_count():
    from torchsparsegradutils_b200.triangular_solve import solve_plan

    A = W.stencil27_csr(24, torch.float32, torch.int32, DEV, lower=True)
    assert solve_plan(A, upper=False).levels == 162
    assert solve_plan(A, upper=False, transpose=True).levels == 162


def _residual(A, x, B, transpose):
    from torchsparsegradutils_b200 import sparse_mm

    opA = A.to_sparse_coo().t().coalesce() if transpose else A
    r = sparse_mm(opA, x) - B
    return (r.norm() / B.norm()).item()


@pytest.mark.parametrize("transpose", [False, True])
@pytest.mark.parametrize("which", ["stencil48", "random200k"])
def test_large_residual(which, transpose):
    if which == "stencil48":
        A = W.triangular_values(W.stencil27_csr(48, torch.float32, torch.int32, DEV, lower=True), torch.float32)
    else:
        A = W.random_lower_csr(None, 200_000, 16, torch.float32, torch.int32, DEV, seed=13)
    B = torch.randn(A.shape[0], 32, device=DEV)
    x = _solve(A, B, upper=False, transpose=transpose)
    assert _residual(A, x, B, transpose) <= 1e-5
    x2 = _solve(A, B, upper=False, transpose=transpose)
    assert torch.equal(x, x2)  # no value atomics: bit-identical from run to run


@pytest.mark.parametrize("K", [1, 32])
def test_graph_replay_equals_eager(K):
    from torchsparsegradutils_b200 import sparse_triangular_solve
    from torchsparsegradutils_b200.triangular_solve import solve_plan, solve_status

    A = W.random_lower_csr(4, 5000, 16, torch.float32, torch.int32, DEV, seed=17)
    B = torch.randn(4, 5000, K, device=DEV)
    solve_plan(A, upper=False)  # the one-off analysis (one host read) stays outside the capture
    eager = _solve(A, B, upper=False)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            sparse_triangular_solve(A, B, upper=False)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = sparse_triangular_solve(A, B, upper=False)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    assert solve_status(DEV) == 0
    assert torch.equal(out, eager)


def test_bf16_is_rejected():
    from torchsparsegradutils_b200 import sparse_triangular_solve

    A = W.random_lower_csr(None, 100, 4, torch.bfloat16, torch.int32, DEV)
    with pytest.raises(RuntimeError, match="unsupported value dtype"):
        sparse_triangular_solve(A, torch.randn(100, 2, device=DEV, dtype=torch.bfloat16), upper=False)
