"""Sampled dense-dense product on a sparse pattern -- the building block of every sparse gradient.

``sddmm(A, X, Y)[e] = <X[i_e, :], Y[j_e, :]>`` for each stored entry ``(i_e, j_e)`` of ``A``, in A's
storage order.  This is the fused form of the ``index_select x2 -> mul -> sum`` idiom the reference
repeats in ``sparse_matmul.py:201-205`` (grad_A of sparse_mm), ``sparse_solve.py:216-235`` / ``:487-504``
(triangular and generic solves, with a sign flip) and ``sparse_lstsq.py:239-256``; SURVEY.md section 8(f)
rank 1.  No ``nnz x K`` temporary is materialised.  Not differentiable itself (it *is* the backward).
"""
from __future__ import annotations

import torch

from . import _ops
from ._pattern import csr_pattern, pattern_of, sparse_like


def sddmm(A: torch.Tensor, X: torch.Tensor, Y: torch.Tensor) -> torch.Tensor:
    """Values of ``X @ Y^T`` sampled at A's stored entries.

    A : sparse COO (2-D) or CSR (2-D or batched) CUDA tensor, shape ``(n, m)`` / ``(b, n, m)``; only its
        pattern is read.
    X : dense ``(n, K)`` / ``(b, n, K)``;  Y : dense ``(m, K)`` / ``(b, m, K)`` (any strides).
    Returns a dense tensor shaped like ``A.values()`` (CSR) or ``A._values()`` (COO, storage order,
    duplicates each get the full dot product).
    """
    if A.layout not in (torch.sparse_coo, torch.sparse_csr):
        raise ValueError("A should be in either COO or CSR sparse format")
    _check_operands(A, X, Y)
    X, Y = X.detach(), Y.detach()
    if A.layout == torch.sparse_coo:
        if A.dim() != 2 or A.sparse_dim() != 2:
            raise ValueError("COO input to sddmm must be 2-D (use CSR for batched patterns)")
        row, col = A._indices()
        return _ops.sddmm_coo(row, col, X, Y)
    pat = csr_pattern(A)
    out = _ops.sddmm(pat, X, Y, None, pat.nnz_total)
    return out.view(A.values().shape)


def _check_operands(A: torch.Tensor, X: torch.Tensor, Y: torch.Tensor) -> None:
    if not (A.is_cuda and X.is_cuda and Y.is_cuda):
        raise RuntimeError("torchsparsegradutils_b200.sddmm runs on CUDA tensors only; there is no CPU fallback")
    if X.dim() != A.dim() or Y.dim() != A.dim():
        raise ValueError("A, X and Y must all be 2D or all be 3D tensors")
    if X.size(-2) != A.size(-2) or Y.size(-2) != A.size(-1) or X.size(-1) != Y.size(-1):
        raise ValueError(f"Incompatible shapes: A {tuple(A.shape)}, X {tuple(X.shape)}, Y {tuple(Y.shape)}")
    if X.dtype != Y.dtype:
        raise RuntimeError(f"sddmm: X and Y must have the same dtype, got {X.dtype} and {Y.dtype}")


def solve_grad_A(A: torch.Tensor, gradB: torch.Tensor, x: torch.Tensor, transpose: bool = False) -> torch.Tensor:
    """Sparse gradient of a linear solve ``A x = B`` (``A^T x = B`` if ``transpose``) w.r.t. A's stored entries.

    ``gradA[i, j] = -<gradB[i, :], x[j, :]>``; with ``transpose``: ``-<gradB[j, :], x[i, :]>`` -- the step the
    reference evaluates with ``repeat_interleave`` + two ``index_select`` + ``mul`` + ``sum`` in
    ``SparseTriangularSolve.backward`` (``sparse_solve.py:216-235``), ``SparseGenericSolve.backward``
    (``:487-504``) and the first term of ``SparseGenericLstsq.backward`` (``sparse_lstsq.py:239-246``), here one
    fused SDDMM launch with no ``nnz x K`` temporaries.  ``gradB`` is the dense gradient the caller obtained from
    its own (transposed) solve and ``x`` the forward solution, both ``(n, K)`` or ``(n,)``; a batched ``A`` (3-D) takes ``(b, n, K)`` operands and returns
    the gradient in A's batched layout (see :func:`_solve_grad_A_batched`).  (The least-squares
    backward adds a second sampled product: :func:`lstsq_grad_A`.)

    Returns a sparse tensor with A's layout, shape and index tensors (CSR: A's own crow/col; COO: A's indices in
    storage order), like the reference (``sparse_solve.py:237-240``, ``:510-513``).
    """
    if A.layout not in (torch.sparse_coo, torch.sparse_csr):
        raise ValueError("A should be in either COO or CSR sparse format")
    if A.dim() == 3:
        return _solve_grad_A_batched(A, gradB, x, transpose)
    if A.dim() != 2:
        raise ValueError("solve_grad_A expects a 2-D or batched (3-D) sparse matrix")
    if gradB.dim() == 1:
        gradB = gradB.unsqueeze(-1)
    if x.dim() == 1:
        x = x.unsqueeze(-1)
    vals = sddmm(A, x, gradB) if transpose else sddmm(A, gradB, x)
    vals = vals.neg_()
    if vals.dtype != A.dtype:
        vals = vals.to(A.dtype)
    return sparse_like(A, vals)


# ----------------------------------------------------------------- batched plumbing of the solves (SURVEY 8(f) rank 4)
def block_diag_operand(A: torch.Tensor) -> torch.Tensor:
    """The 2-D CSR matrix the reference hands its triangular / generic solver for a BATCHED ``A``:
    ``sparse_block_diag(*A)`` followed, for COO input, by ``convert_coo_to_csr`` (``sparse_solve.py:172-178``).

    The reference assembles it item by item in Python (``utils/utils.py:604-645`` / ``:570-602``, three ``torch.cat``)
    and, for COO, re-sorts the result.  Here: batched CSR -> one index-arithmetic kernel (``tsgu_block_diag_csr``:
    ``crow[t, r] + t*nnz``, ``col + t*m``), values are a zero-copy flat view; batched COO (``sparse_dim == 3``) -> the
    radix-sort COO->CSR builder on the 3-row coordinates (batch-major order IS block-diagonal row order), values gathered
    through its permutation.  The solver itself is out of scope and stays the caller's.
    """
    if A.dim() != 3:
        raise ValueError("block_diag_operand expects a batched (3-D) sparse tensor")
    if not A.is_cuda:
        raise RuntimeError("block_diag_operand runs on CUDA tensors only; there is no CPU fallback")
    b, n, m = A.shape
    if A.layout == torch.sparse_csr:
        crow, col = _ops.block_diag_csr(A.crow_indices(), A.col_indices(), m)
        return torch.sparse_csr_tensor(crow, col, A.values().reshape(-1), (b * n, b * m))
    pat = pattern_of(A)  # COO: flat CSR over b*n rows, item-local columns, duplicates coalesced like the reference (:580)
    csr, vals = pat.csr, pat.values(A)
    if csr.perm is not None:
        vals = _ops.gather_values(vals, csr.perm)
    rows = torch.arange(b * n, device=A.device, dtype=csr.rowptr.dtype)
    item_of_entry = torch.repeat_interleave(rows // n, (csr.rowptr[1:] - csr.rowptr[:-1]).long())
    col = csr.colind.long() + item_of_entry.long() * m
    return torch.sparse_csr_tensor(csr.rowptr.long(), col, vals, (b * n, b * m))


def _solve_grad_A_batched(A: torch.Tensor, gradB: torch.Tensor, x: torch.Tensor, transpose: bool) -> torch.Tensor:
    """Batched form of :func:`solve_grad_A`: ``gradB`` and ``x`` are ``(b, n, K)`` (or the flat ``(b*n, K)`` the solver
    worked on).  Returns the gradient directly in A's batched layout -- batched CSR on A's own crow/col tensors, or a
    batched COO tensor on the coalesced per-item coordinates -- where the reference builds the block-diagonal
    gradient, splits it per item with two host syncs per block and re-stacks it (``sparse_solve.py:242-250``,
    ``utils/utils.py:754-790``, ``:6-88``)."""
    b, n, m = A.shape
    gradB = gradB.reshape(b, n, -1) if gradB.dim() != 3 else gradB
    x = x.reshape(b, m, -1) if x.dim() != 3 else x
    G, Y = (x, gradB) if transpose else (gradB, x)
    _check_operands(A, G, Y)
    pat = pattern_of(A)
    vals = _ops.sddmm(pat.csr, G.detach(), Y.detach(), pat.out_index, pat.nnz_out).neg_()
    return sparse_like(A, vals, pat.grad_indices, is_coalesced=True)


def lstsq_grad_A(A: torch.Tensor, gradB: torch.Tensor, x: torch.Tensor, B: torch.Tensor, Apgb: torch.Tensor) -> torch.Tensor:
    """Sparse gradient of ``x = argmin ||A x - B||`` with respect to A's stored entries -- both sampled products of the
    reference's ``SparseGenericLstsq.backward`` (``sparse_lstsq.py:239-265``), fused:

        gradA[i, j] = -<gradB[i, :], x[j, :]>  +  <(B - A x)[i, :], Apgb[j, :]>

    ``gradB = (A^T)^+ grad`` and ``Apgb = A^+ gradB`` come from the caller's least-squares solver (out of scope here);
    the residual ``B - A x`` is formed with this package's SpMM.  Two SDDMM launches, no ``nnz x K`` temporaries.
    Returns a sparse tensor on A's own index tensors (``:261-265``)."""
    from .sparse_matmul import sparse_mm

    if A.dim() != 2 or A.layout not in (torch.sparse_coo, torch.sparse_csr):
        raise ValueError("lstsq_grad_A expects a 2-D COO or CSR matrix")
    col2 = lambda t: t.unsqueeze(-1) if t.dim() == 1 else t  # noqa: E731
    gradB, x, B, Apgb = col2(gradB), col2(x), col2(B), col2(Apgb)
    with torch.no_grad():
        resid = B - sparse_mm(A.detach(), x.detach())
    vals = sddmm(A, resid, Apgb).sub_(sddmm(A, gradB, x))
    return sparse_like(A, vals)
