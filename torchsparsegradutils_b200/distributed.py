"""Multi-GPU drivers for ``sparse_mm`` on one 8xB200 box (one process per GPU, ``torch.distributed``).

The reference has no distributed code (SURVEY.md section 5); these drivers sit *outside* the
``sparse_mm(A, B)`` signature and only partition work:

* **Batched inputs shard by batch item, with no collective.**  The reference's batched semantics are
  block-diagonal (``sparse_matmul.py:151-153``, ``utils/utils.py:505-513``): item k of C, grad_A and
  grad_B depends only on item k of A, B and the upstream gradient.  Each rank simply calls
  ``sparse_mm`` on its slice (:func:`batch_shard_bounds`, :func:`shard_batched`).
* **One large matrix shards by nnz-balanced row blocks with the dense B replicated.**  Forward and the
  SDDMM are local; grad_B = sum_p A_p^T G_p needs the one exchange step of the path: an all-reduce of
  the (m, K) partials (NCCL over NVLink; gloo in the CPU tests).  :func:`sparse_mm_row_sharded`.

* **Alternative for one large matrix: shard the dense K columns** (:func:`sparse_mm_k_sharded`,
  :func:`k_shard_bounds`).  Row sharding cannot scale: every rank still reads all of the replicated B twice and
  writes a full m x K grad_B partial, then all-reduces it (m x K elements).  Sharding K instead -- rank p owns
  B[:, K_p] and G[:, K_p], the (small) sparse A is replicated -- makes forward and grad_B purely local
  (C[:, K_p] = A B[:, K_p], grad_B[:, K_p] = A^T G[:, K_p]) and leaves one exchange step: grad_A's sampled dot
  products are partial sums over K, so the nnz values are all-reduced (nnz elements instead of m x K: 8 MB vs
  512 MiB on BASELINE config 5).  Every rank does 1/P of the dense traffic.

``local_mm`` lets the tests drive the partition / collective logic on CPU ranks (gloo) with the CPU
oracle as the per-rank operator; the default is the CUDA ``sparse_mm``.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Tuple

import torch
import torch.distributed as dist

import os

from . import _native
from ._pattern import sparse_like, sparse_values
from .sparse_matmul import SparseMatMul, _grad_A, _grad_B, sparse_mm

_OVERLAP_SM_MARGIN = int(os.environ.get("TSGU_B200_OVERLAP_SM_MARGIN", "20"))


# ------------------------------------------------------------------------------ batch sharding
def batch_shard_bounds(batch: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous chunk [lo, hi) of the batch dimension owned by `rank` (sizes differ by at most 1)."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of size {world}")
    base, extra = divmod(batch, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_batched(A: torch.Tensor, world: int, rank: int, *dense: torch.Tensor):
    """Slice a batched CSR / COO tensor and its dense companions down to this rank's batch items."""
    if A.dim() != 3:
        raise ValueError("shard_batched expects a batched (3-D) sparse tensor")
    lo, hi = batch_shard_bounds(A.shape[0], world, rank)
    shape = (hi - lo,) + tuple(A.shape[1:])
    if A.layout == torch.sparse_csr:
        A_loc = torch.sparse_csr_tensor(A.crow_indices()[lo:hi].contiguous(), A.col_indices()[lo:hi].contiguous(),
                                        A.values()[lo:hi].contiguous(), shape)
    elif A.layout == torch.sparse_coo:
        idx, val = A._indices(), A._values()
        keep = (idx[0] >= lo) & (idx[0] < hi)
        sub = idx[:, keep].clone()
        sub[0] -= lo
        A_loc = torch.sparse_coo_tensor(sub, val[keep], shape)
    else:
        raise ValueError("A should be in either COO or CSR sparse format")
    return (A_loc,) + tuple(d[lo:hi].contiguous() for d in dense)


# -------------------------------------------------------------------------------- row sharding
def nnz_balanced_row_blocks(crow: torch.Tensor, world: int) -> List[int]:
    """Row boundaries r_0 = 0 <= r_1 <= ... <= r_world = n such that every block holds ~nnz/world
    stored entries (prefix-sum search on crow; SURVEY.md section 8(e))."""
    n = crow.numel() - 1
    nnz = int(crow[-1])
    targets = torch.tensor([nnz * p // world for p in range(1, world)], dtype=crow.dtype, device=crow.device)
    cuts = torch.searchsorted(crow.contiguous(), targets, right=False).clamp_(0, n).tolist() if world > 1 else []
    bounds = [0] + [int(c) for c in cuts] + [n]
    for i in range(1, len(bounds)):  # monotone even with long empty stretches
        bounds[i] = max(bounds[i], bounds[i - 1])
    return bounds


def shard_rows_csr(A: torch.Tensor, lo: int, hi: int) -> torch.Tensor:
    """Rows [lo, hi) of a 2-D CSR tensor as a CSR tensor of shape (hi - lo, m) (crow rebased to 0)."""
    if A.layout != torch.sparse_csr or A.dim() != 2:
        raise ValueError("shard_rows_csr expects a 2-D CSR tensor")
    crow, col, val = A.crow_indices(), A.col_indices(), A.values()
    s, e = int(crow[lo]), int(crow[hi])
    # clones, not views: a rank keeps only its block alive, and fresh allocations are 16-byte aligned (what the staged
    # kernels need; a view starting at entry s generally is not)
    return torch.sparse_csr_tensor((crow[lo:hi + 1] - crow[lo]).contiguous(), col[s:e].clone(), val[s:e].clone(),
                                   (hi - lo, A.shape[1]))


class _AllReduceGrad(torch.autograd.Function):
    """Identity in forward; sums the gradient over the process group in backward (replicated operand)."""

    @staticmethod
    def forward(ctx, x, group):
        ctx.group = group
        return x.view_as(x)

    @staticmethod
    def backward(ctx, grad):  # type: ignore[override]
        grad = grad.contiguous()
        dist.all_reduce(grad, op=dist.ReduceOp.SUM, group=ctx.group)
        return grad, None


def row_block_bounds(m: int, world: int, rank: int) -> Tuple[int, int]:
    """Rows [lo, hi) of an (m, K) dense gradient that `rank` owns after a reduce-scatter: equal blocks of
    ceil(m / world) rows (NCCL's reduce-scatter needs equal counts; the last block may be short)."""
    per = -(-m // world)
    lo = min(rank * per, m)
    return lo, min(lo + per, m)


def _reduce_grad_b(gradB: torch.Tensor, group, mode: str, wire_dtype: Optional[torch.dtype]):
    """Issue the grad_B collective asynchronously.  Returns (work handles, finish) where finish() runs after the
    handles completed and yields the tensor autograd hands to B.

    mode "all_reduce": every replica of B receives the full sum (NCCL all-reduce; NVLS in-switch reduction where
        NCCL enables it).
    mode "reduce_scatter": every rank receives only ITS block of rows of the sum (row_block_bounds) -- half the wire
        traffic of an all-reduce, for consumers that are themselves sharded (a sharded optimizer).  The returned
        tensor keeps B's full shape (autograd requires it); rows outside the rank's block are zero.
    wire_dtype: optionally send a narrower type (torch.bfloat16 for fp32 gradients halves the bytes on the wire;
        lossy -- opt-in, off by default so that results stay within the fp32 tolerance)."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    send = gradB if wire_dtype is None or wire_dtype == gradB.dtype else gradB.to(wire_dtype)
    if mode == "all_reduce":
        work = dist.all_reduce(send, op=dist.ReduceOp.SUM, group=group, async_op=True)

        def finish():
            return send if send is gradB else send.to(gradB.dtype)

        return [work], finish
    if mode != "reduce_scatter":
        raise ValueError(f"unknown grad_B reduction mode {mode!r}")
    m = gradB.shape[-2]
    K = gradB.shape[-1]
    flat = send.reshape(-1, K)  # (m, K) -- batched operands are not row-sharded
    per = -(-m // world)
    if per * world != m:  # pad to equal blocks
        padded = flat.new_zeros((per * world, K))
        padded[:m] = flat
        flat = padded
    shard = torch.empty((per, K), dtype=flat.dtype, device=flat.device)
    work = dist.reduce_scatter_tensor(shard, flat, op=dist.ReduceOp.SUM, group=group, async_op=True)

    def finish():
        lo, hi = row_block_bounds(m, world, rank)
        out = torch.zeros_like(gradB)
        out.reshape(-1, K)[lo:hi] = shard[: hi - lo].to(gradB.dtype)
        return out

    return [work], finish


class _RowShardedMatMul(torch.autograd.Function):
    """sparse_mm on this rank's row block.  Backward: the local grad_B partial is computed first and its collective is
    issued asynchronously, so it travels over NVLink while the SDDMM (grad_A, purely local) runs (`overlap=False`:
    the SDDMM runs after the collective has finished -- for A/B measurements of the overlap)."""

    @staticmethod
    def forward(ctx, A_local, B, group, mode, wire_dtype, overlap):
        ctx.group, ctx.mode, ctx.wire_dtype, ctx.overlap = group, mode, wire_dtype, overlap
        return SparseMatMul.forward(ctx, A_local, B)

    @staticmethod
    def backward(ctx, grad):  # type: ignore[override]
        gradB = None
        works, finish = [], None
        if ctx.needs_input_grad[1]:
            gradB = _grad_B(ctx, grad).contiguous()
            works, finish = _reduce_grad_b(gradB, ctx.group, ctx.mode, ctx.wire_dtype)
            if not ctx.overlap:
                for w in works:
                    w.wait()
        gradA = None
        if ctx.needs_input_grad[0]:
            # leave a few SMs to NCCL's kernels: a persistent SDDMM grid that owns every SM would make the collective
            # wait until it has drained (measured: no overlap at all, config 5 on 2 GPUs 1.96 ms = kernels + all-reduce)
            with _native.sm_margin(_OVERLAP_SM_MARGIN if (works and ctx.overlap) else 0):
                gradA = _grad_A(ctx, grad)
        if finish is not None:
            for w in works:
                w.wait()
            gradB = finish()
        return gradA, gradB, None, None, None, None


def sparse_mm_row_sharded(A_local: torch.Tensor, B: torch.Tensor, group: Optional[dist.ProcessGroup] = None,
                          local_mm: Callable[[torch.Tensor, torch.Tensor], torch.Tensor] = sparse_mm,
                          grad_b: str = "all_reduce", wire_dtype: Optional[torch.dtype] = None,
                          overlap: bool = True) -> torch.Tensor:
    """C_local = A_local @ B for this rank's row block; B is replicated on every rank.

    grad_A_local and C_local stay local; grad_B = sum_p A_p^T G_p is the one exchange step of the path:
    ``grad_b="all_reduce"`` (default) gives every replica of B the full A^T G; ``grad_b="reduce_scatter"`` gives each
    rank only its block of rows (:func:`row_block_bounds`; the rest of ``B.grad`` is zero) at half the wire traffic.
    """
    distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    if not distributed:
        return local_mm(A_local, B)
    if local_mm is sparse_mm:  # product path: collective overlapped with the SDDMM
        return _RowShardedMatMul.apply(A_local, B, group, grad_b, wire_dtype, overlap)
    if grad_b != "all_reduce":
        raise ValueError("an injected local_mm supports grad_b='all_reduce' only")
    return local_mm(A_local, _AllReduceGrad.apply(B, group))


# ----------------------------------------------------------------------------- K (dense-column) sharding
def k_shard_bounds(K: int, world: int, rank: int, align: int = 1) -> Tuple[int, int]:
    """Contiguous block [lo, hi) of the dense columns owned by `rank`; block edges are multiples of `align`
    (pass the 128-bit vector width, 4 for fp32 / 8 for bf16, so every shard stays on the vectorised kernels)."""
    if not (0 <= rank < world):
        raise ValueError(f"rank {rank} outside world of size {world}")
    units = -(-K // align)
    base, extra = divmod(units, world)
    lo = (rank * base + min(rank, extra)) * align
    hi = lo + (base + (1 if rank < extra else 0)) * align
    return min(lo, K), min(hi, K)


class _AllReduceSparseGrad(torch.autograd.Function):
    """Identity on a sparse operand in forward; sums the gradient's stored values over the group in backward
    (gloo / injected-operator path of :func:`sparse_mm_k_sharded`)."""

    @staticmethod
    def forward(ctx, A, group):
        ctx.group = group
        return A.detach().clone() if A.layout == torch.sparse_coo else torch.sparse_csr_tensor(
            A.crow_indices(), A.col_indices(), A.values().detach().clone(), A.shape)

    @staticmethod
    def backward(ctx, grad):  # type: ignore[override]
        if grad.layout == torch.strided:  # dense gradient from a generic operator: reduce it whole
            g = grad.contiguous()
            dist.all_reduce(g, op=dist.ReduceOp.SUM, group=ctx.group)
            return g, None
        if grad.layout == torch.sparse_coo and not grad.is_coalesced():
            grad = grad.coalesce()
        v = sparse_values(grad).contiguous()
        dist.all_reduce(v, op=dist.ReduceOp.SUM, group=ctx.group)
        return sparse_like(grad, v, is_coalesced=True), None


class _KShardedMatMul(torch.autograd.Function):
    """sparse_mm on this rank's block of dense columns.  Backward: the SDDMM over the local K block gives partial
    grad_A values; their all-reduce is issued asynchronously and travels over NVLink while the (purely local)
    grad_B SpMM runs."""

    @staticmethod
    def forward(ctx, A, B_local, group):
        ctx.group = group
        return SparseMatMul.forward(ctx, A, B_local)

    @staticmethod
    def backward(ctx, grad):  # type: ignore[override]
        gradA = work = None
        if ctx.needs_input_grad[0]:
            gradA = _grad_A(ctx, grad)
            work = dist.all_reduce(sparse_values(gradA), op=dist.ReduceOp.SUM, group=ctx.group, async_op=True)
        gradB = _grad_B(ctx, grad) if ctx.needs_input_grad[1] else None
        if work is not None:
            work.wait()
        return gradA, gradB, None


def sparse_mm_k_sharded(A: torch.Tensor, B_local: torch.Tensor, group: Optional[dist.ProcessGroup] = None,
                        local_mm: Callable[[torch.Tensor, torch.Tensor], torch.Tensor] = sparse_mm) -> torch.Tensor:
    """C[:, K_p] = A @ B[:, K_p] for this rank's block of dense columns; A (sparse) is replicated on every rank.

    C[:, K_p] and grad_B[:, K_p] stay local; grad_A's stored values are all-reduced so every replica of A sees the
    full sampled product (the only collective: nnz elements).  Results equal the single-GPU ones up to the order
    of the K-sum in grad_A (P partial sums are added by the collective)."""
    distributed = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    if not distributed:
        return local_mm(A, B_local)
    if local_mm is sparse_mm:
        return _KShardedMatMul.apply(A, B_local, group)
    return local_mm(_AllReduceSparseGrad.apply(A, group), B_local)
