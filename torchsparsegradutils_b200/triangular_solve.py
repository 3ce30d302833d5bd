"""``sparse_triangular_solve`` -- drop-in for ``torchsparsegradutils.sparse_triangular_solve`` on B200.

Same signature and autograd contract as the reference (``sparse_solve.py`` ``sparse_triangular_solve`` /
``SparseTriangularSolve``): ``x = op(A)^{-1} B`` with ``op(A) = A`` or ``A^T``, ``B.grad`` from the solve with the
transpose flag negated, ``A.grad`` the sampled product ``-gradB x^T`` on A's pattern.  What changed is underneath:

======================  ===============================================  ==========================================
reference step          reference implementation                         here
======================  ===============================================  ==========================================
forward solve           torch.triangular_solve on CSR (cuSPARSE, its     ``tsgu_trisolve`` over a cached level plan
                        analysis phase inside every call)                (``tsgu_trisolve_levels`` + ``_plan``)
batched layout          sparse_block_diag + convert_coo_to_csr           batch is part of the plan (flat rows)
backward gradB          torch.triangular_solve, transpose negated        ``tsgu_trisolve`` over the other plan
backward gradA          repeat_interleave, 2x index_select, mul, sum     ``solve_grad_A`` (one SDDMM)
======================  ===============================================  ==========================================

Only the strictly off-diagonal entries of the solved triangle and the diagonal are read: entries of the other
triangle are ignored, and so is a stored diagonal when ``unitriangular`` -- what torch's sparse CSR solve does.  A
missing diagonal divides by zero, as the dense solve does.
"""
from __future__ import annotations

from typing import Optional, cast

import torch

from . import _native as nat
from . import _ops
from ._pattern import CsrPattern, TriPlan, _sort_coo, _transpose_csr, pattern_of
from .sddmm import solve_grad_A
from .sparse_matmul import _check_args, _check_runtime


def sparse_triangular_solve(A: torch.Tensor, B: torch.Tensor, upper: bool = True, unitriangular: bool = False,
                            transpose: bool = False) -> torch.Tensor:
    r"""Solve ``op(A) X = B`` for a sparse triangular ``A`` with sparsity-preserving gradients.

    Parameters
    ----------
    A : torch.Tensor
        Sparse COO (2-D, or 3-D with ``sparse_dim == 3``) or CSR (2-D or batched) CUDA tensor of shape ``(n, n)`` or
        ``(b, n, n)``.  Duplicate COO coordinates are summed.
    B : torch.Tensor
        Dense (strided, any strides) CUDA tensor of shape ``(n, K)`` or ``(b, n, K)``, float32 or float64.
    upper : bool
        Solve with A's upper triangle (else the lower one).
    unitriangular : bool
        Take A's diagonal as ones.
    transpose : bool
        Solve ``A^T X = B``.

    Returns
    -------
    torch.Tensor
        Dense contiguous ``(n, K)`` or ``(b, n, K)``.  ``A.grad`` has A's layout and pattern; ``B.grad`` is dense.

    Raises
    ------
    ValueError
        Malformed arguments (same style as :func:`sparse_mm`).
    RuntimeError
        Non-CUDA tensors, mismatching dtypes/devices, a dtype other than float32 / float64, or a kernel failure.
        There is no CPU fallback.
    """
    _check_args(A, B, square=True)
    return cast(torch.Tensor, SparseTriangularSolve.apply(A, B, bool(upper), bool(unitriangular), bool(transpose)))


class SparseTriangularSolve(torch.autograd.Function):
    r"""Autograd node of :func:`sparse_triangular_solve` (mirror of the reference class of the same name)."""

    @staticmethod
    def forward(ctx, A, B, upper, unitriangular, transpose):
        _check_runtime(A, B, "sparse_triangular_solve", float_only=True)
        ctx.batched = B.dim() == 3
        ctx.flags = (upper, unitriangular, transpose)
        A, B = A.detach(), B.detach()
        pat = pattern_of(A, unique=True)  # COO duplicates are summed
        csr, vals = pat.csr, pat.values(A)  # a sort permutation (csr.perm) is folded into the plan's value positions
        x = _solve(csr, vals, B if ctx.batched else B.unsqueeze(0), upper, unitriangular, transpose)
        x = x if ctx.batched else x[0]
        ctx.pattern = csr
        ctx.save_for_backward(A, x, vals)
        return x

    @staticmethod
    def backward(ctx, grad):  # type: ignore[override]
        A, x, vals = ctx.saved_tensors
        upper, unitriangular, transpose = ctx.flags
        if not (ctx.needs_input_grad[0] or ctx.needs_input_grad[1]):
            return None, None, None, None, None
        gradB = _solve(ctx.pattern, vals, grad if ctx.batched else grad.unsqueeze(0), upper, unitriangular,
                       not transpose)
        gradB = gradB if ctx.batched else gradB[0]
        gradA = solve_grad_A(A, gradB, x, transpose) if ctx.needs_input_grad[0] else None
        return gradA, gradB if ctx.needs_input_grad[1] else None, None, None, None


# ------------------------------------------------------------------------------------------ plans
def solve_plan(A: torch.Tensor, upper: bool = True, transpose: bool = False) -> TriPlan:
    """The cached level plan :func:`sparse_triangular_solve` uses for ``A`` with these flags (built on first use).

    Call it ahead of the first solve to take the one-off analysis (one host read) out of the first step, e.g. before a
    ``torch.cuda.graph`` capture; ``.levels`` is the number of dependent steps of the solve."""
    return _plan(pattern_of(A, unique=True).csr, upper, transpose)


def _plan(csr: CsrPattern, upper: bool, transpose: bool) -> TriPlan:
    """Plan of op(A) for the triangle actually solved: A's `upper` triangle, which is the other one of A^T."""
    lower = upper == transpose
    key = ("trisolve", lower, transpose)
    plan = csr.extras.get(key)
    if plan is None:
        plan = csr.extras[key] = _build_plan(csr, lower, transpose)
    return plan


def _build_plan(csr: CsrPattern, lower: bool, transpose: bool) -> TriPlan:
    dev = csr.device
    batch, n = csr.batch, csr.n
    rows = batch * n
    if transpose:
        rowptr, colind, perm, idx = _transpose_csr(csr)
        rbs, nbs = n, 0
    else:
        rowptr, colind, perm, idx = csr.rowptr, csr.colind, csr.perm, csr.idx
        rbs, nbs = csr.rowptr_bstride, csr.nnz_bstride
        if perm is not None and perm.dtype != nat.IDX_TORCH[idx]:
            perm = perm.to(nat.IDX_TORCH[idx])
    idt = nat.IDX_TORCH[idx]
    if rows == 0:
        empty = torch.empty(0, dtype=idt, device=dev)
        return TriPlan(empty, torch.zeros(1, dtype=idt, device=dev), empty, empty, empty, 0, idx)
    L = nat.lib()
    level = torch.empty((2, rows), dtype=torch.int64, device=dev)  # (level, row): the sort keys
    count = torch.empty(rows, dtype=torch.int64, device=dev)
    stats = torch.empty(3, dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        ws = nat.workspace(L.tsgu_trisolve_workspace_bytes(batch, n), dev)
        nat.check(L.tsgu_trisolve_levels(nat.ptr(rowptr), nat.ptr(colind), batch, n, rbs, nbs, idx, int(lower),
                                         level.data_ptr(), count.data_ptr(), stats.data_ptr(), ws.data_ptr(),
                                         ws.numel(), nat.stream_ptr(dev)), "tsgu_trisolve_levels")
        level[1] = torch.arange(rows, device=dev)
        levels, deps, status = nat.host_read(stats)  # the one host read per plan
        if status != 0:
            raise RuntimeError("sparse_triangular_solve: the level analysis timed out waiting on a dependency")
        order, _ = _sort_coo(level, (levels, rows), 1, idx, False)  # stable: rows of a level keep their order
        plan_rowptr = torch.zeros(rows + 1, dtype=idt, device=dev)
        plan_rowptr[1:] = count[order.long()].cumsum(0)
        col = torch.empty(deps, dtype=idt, device=dev)
        pos = torch.empty(deps, dtype=idt, device=dev)
        diag = torch.empty(rows, dtype=idt, device=dev)
        nat.check(L.tsgu_trisolve_plan(nat.ptr(rowptr), nat.ptr(colind), nat.ptr(perm), batch, n, rbs, nbs, idx,
                                       int(lower), order.data_ptr(), plan_rowptr.data_ptr(), col.data_ptr(),
                                       pos.data_ptr(), diag.data_ptr(), nat.stream_ptr(dev)), "tsgu_trisolve_plan")
    return TriPlan(order, plan_rowptr, col, pos, diag, levels, idx)


# ------------------------------------------------------------------------------------------ the solve
_last_status: dict = {}


def solve_status(device: Optional[torch.device] = None) -> int:
    """Status word of the most recent solve on `device` (0: every dependency wait completed).  A solve whose wait
    bound expired writes NaN to the rows concerned and a non-zero status; reading it synchronises with the device."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    st = _last_status.get(dev.index)
    return 0 if st is None else int(nat.host_read(st)[0])


def _solve(csr: CsrPattern, vals: torch.Tensor, B: torch.Tensor, upper: bool, unitriangular: bool,
           transpose: bool) -> torch.Tensor:
    """X (batch, n, K) contiguous from B (batch, n, K), any strides."""
    plan = _plan(csr, upper, transpose)
    batch, n, K = B.shape
    dev = B.device
    X = torch.empty((batch, n, K), dtype=B.dtype, device=dev)
    if X.numel() == 0:
        return X
    L = nat.lib()
    bs, rs, cs = B.stride()
    with _ops._on(dev), _ops._timer("trisolve", dev):
        ws = nat.workspace(L.tsgu_trisolve_workspace_bytes(batch, n), dev)
        nat.check(L.tsgu_trisolve(plan.rowptr.data_ptr(), nat.ptr(plan.col), nat.ptr(plan.pos), plan.diag.data_ptr(),
                                  plan.order.data_ptr(), vals.data_ptr(), B.data_ptr(), X.data_ptr(), batch, n, K,
                                  bs if batch > 1 else 0, rs, cs, int(unitriangular), nat.val_enum(B.dtype), plan.idx,
                                  ws.data_ptr(), ws.numel(), nat.stream_ptr(dev)), "tsgu_trisolve")
    _last_status[dev.index] = ws[8:12].view(torch.int32)
    return X
