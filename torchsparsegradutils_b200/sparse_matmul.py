"""``sparse_mm`` -- drop-in for ``torchsparsegradutils.sparse_mm`` on B200.

Host-side mirror of the reference's operator interface (``torchsparsegradutils/sparse_matmul.py``):
same signature, same validation order and messages (``:114-127``), same autograd contract
(``SparseMatMul.forward`` ``:141-163`` / ``.backward`` ``:165-234``).  What changed is everything
underneath: no ``torch.sparse.mm``, no ``index_select`` temporaries, no block-diagonal assembly --
the arithmetic is the sm_100a kernels behind ``include/tsgu_b200.h``.

======================  ===============================================  =====================
reference step          reference implementation                         here
======================  ===============================================  =====================
forward C = A B         torch.sparse.mm (``:155``)                       ``tsgu_spmm_csr``
batched layout          sparse_block_diag + reshape (``:151-153``)       batch strides in-kernel
grad_A (SDDMM)          repeat_interleave, 2x index_select, mul, sum     ``tsgu_sddmm_csr``
                        (``:190-205``), block-diag split (``:213-219``)
grad_B = A^T G          torch.sparse.mm(A.t(), G) (``:229``)             cached ``tsgu_csr_transpose``
                                                                         + ``tsgu_spmm_csr``
======================  ===============================================  =====================
"""
from __future__ import annotations

import os
from typing import cast

import torch

from . import _native, _ops
from ._pattern import pattern_of, sparse_like


def sparse_mm(A: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    r"""Sparse x dense matrix product with sparsity-preserving gradients.

    Parameters
    ----------
    A : torch.Tensor
        Sparse COO (2-D, or 3-D with ``sparse_dim == 3``) or CSR (2-D or batched) CUDA tensor of
        shape ``(n, m)`` or ``(b, n, m)``.
    B : torch.Tensor
        Dense (strided, any strides) CUDA tensor of shape ``(m, p)`` or ``(b, m, p)``.

    Returns
    -------
    torch.Tensor
        Dense contiguous ``(n, p)`` or ``(b, n, p)``.  ``A.grad`` has A's layout and sparsity
        pattern; ``B.grad`` is dense.

    Raises
    ------
    ValueError
        Same conditions and messages as the reference (``sparse_matmul.py:114-127``).
    RuntimeError
        Non-CUDA tensors, mismatching dtypes/devices, unsupported dtype, or a kernel failure.
        There is no CPU fallback.
    """
    _check_args(A, B)
    return cast(torch.Tensor, SparseMatMul.apply(A, B))


def _check_args(A: torch.Tensor, B: torch.Tensor, square: bool = False) -> None:
    """The ValueError checks of sparse_mm (`square`: and of sparse_triangular_solve), in the reference's order."""
    if not isinstance(A, torch.Tensor) or not isinstance(B, torch.Tensor):
        raise ValueError("Both A and B should be instances of torch.Tensor")
    if A.dim() < 2 or B.dim() < 2:
        raise ValueError("Both A and B should be at least 2-dimensional tensors")
    if A.dim() != B.dim() or A.dim() not in (2, 3):
        raise ValueError("A and B must both be 2D or both be 3D tensors")
    if A.layout not in {torch.sparse_coo, torch.sparse_csr}:
        raise ValueError("A should be in either COO or CSR sparse format")
    if B.layout != torch.strided:
        raise ValueError("B must be a dense (strided) tensor")
    if A.dim() == 3 and A.size(0) != B.size(0):
        raise ValueError("If batched, A and B must have the same batch size")
    if square and A.size(-1) != A.size(-2):
        raise ValueError(f"A must be square, got A[..., {A.size(-2)}, {A.size(-1)}]")
    if A.size(-1) != B.size(-2):
        raise ValueError(f"Incompatible inner dimensions: A[..., {A.size(-1)}] vs B[..., {B.size(-2)}]")


def _check_runtime(A: torch.Tensor, B: torch.Tensor, op: str = "sparse_mm", float_only: bool = False) -> None:
    """The RuntimeError checks of `op`; `float_only`: values must be float32 / float64 (no bfloat16)."""
    if not (A.is_cuda and B.is_cuda):
        raise RuntimeError(
            f"torchsparsegradutils_b200.{op} runs on CUDA (sm_100a) tensors only; got "
            f"A on {A.device}, B on {B.device}. There is no CPU fallback.")
    if A.device != B.device:
        raise RuntimeError(f"{op}: A and B must be on the same device, got {A.device} and {B.device}")
    if A.dtype != B.dtype:
        raise RuntimeError(f"{op}: A and B must have the same dtype, got {A.dtype} and {B.dtype}")
    if float_only and B.dtype not in (torch.float32, torch.float64):
        raise RuntimeError(f"{op}: unsupported value dtype {B.dtype}; supported: float32, float64")
    _native.val_enum(B.dtype)  # RuntimeError("unsupported value dtype ...") for float16 / complex / integer operands
    if A.layout == torch.sparse_coo and (A.sparse_dim() != A.dim() or A.dense_dim() != 0):
        raise RuntimeError(f"{op}: COO input must have sparse_dim == ndim and no dense dimensions")


class SparseMatMul(torch.autograd.Function):
    r"""Autograd node of :func:`sparse_mm` (mirror of the reference class of the same name)."""

    @staticmethod
    def forward(ctx, A, B):
        _check_runtime(A, B)
        ctx.batched = B.dim() == 3
        ctx.A_shape = A.size()
        ctx.B_shape = B.size()
        # remember a non-contiguous (but dense) layout of B so grad_B can be handed back in it
        ctx.B_strides = B.stride() if (not B.is_contiguous() and _ops.is_dense_non_overlapping(B)) else None
        A, B = A.detach(), B.detach()
        pat = pattern_of(A)
        vals = pat.values(A)

        # a strided view of B (eps.t(), permute(1,2,0) from _batch_sparse_mv) is packed once here and the
        # packed copy is what backward's SDDMM re-reads -- the reference re-copies it as well (:153)
        Bk = _ops.prepare_dense(B if ctx.batched else B.unsqueeze(0))
        x = _ops.spmm(pat.csr, vals, Bk, tag="spmm_fwd")
        x = x if ctx.batched else x[0]

        ctx.pattern = pat
        ctx.save_for_backward(A, Bk, vals)
        return x

    @staticmethod
    def backward(ctx, grad):  # type: ignore[override]
        if ctx.needs_input_grad[0] and ctx.needs_input_grad[1] and _concurrent_backward_pays(ctx, grad):
            return _backward_two_streams(ctx, grad)
        gradA = _grad_A(ctx, grad) if ctx.needs_input_grad[0] else None
        gradB = _grad_B(ctx, grad) if ctx.needs_input_grad[1] else None
        return gradA, gradB


# grad_A (SDDMM) and grad_B (value gather + transposed SpMM) are independent.  Each is a persistent kernel that owns the
# whole GPU, so for LARGE problems running them concurrently only makes them share the same L2 bandwidth (measured on
# BASELINE config 2: 0.930 -> 0.920 ms, config 3: slower).  A SMALL problem -- one rank's share of a strongly scaled
# batch: 1 M entries, ~45 us per kernel -- spends a third of each kernel ramping up and draining (2 tile waves where
# 1.73 would do); there the second stream fills those holes.  The threshold is the L2->SM gather volume of one pass.
_CONCURRENT_BWD_MAX_GATHER_BYTES = int(os.environ.get("TSGU_B200_CONCURRENT_BWD_BYTES", str(3 << 29)))
_side_streams: dict = {}


def _concurrent_backward_pays(ctx, grad) -> bool:
    return 0 < ctx.pattern.csr.nnz_total * grad.shape[-1] * grad.element_size() <= _CONCURRENT_BWD_MAX_GATHER_BYTES


def _backward_two_streams(ctx, grad):
    dev = grad.device
    main = torch.cuda.current_stream(dev)
    side = _side_streams.get(dev.index)
    if side is None:
        side = _side_streams[dev.index] = torch.cuda.Stream(dev)
    # a transposed structure that must still be built (or get its layout upgrade) is built HERE: tensors a cached
    # pattern owns are allocated -- and the ones it replaces freed -- under the caller's stream, never the side stream
    patT = ctx.pattern.csr.transpose()
    side.wait_stream(main)  # fork (under graph capture: a parallel branch of the graph)
    with torch.cuda.stream(side):
        gradB = _grad_B(ctx, grad, patT)
    gradA = _grad_A(ctx, grad)
    main.wait_stream(side)  # join
    gradB.record_stream(main)
    return gradA, gradB


def _grad_A(ctx, grad):
    """grad_A[e] = <grad[i_e, :], B[j_e, :]> on A's pattern only (reference sparse_matmul.py:173-219)."""
    A, B = ctx.saved_tensors[:2]
    pat = ctx.pattern
    # 2-D COO: per stored entry, in storage order (duplicates each get the full dot product); batched COO: on the
    # sorted unique pattern (reference :213-217)
    v = _ops.sddmm(pat.csr, grad, B, pat.out_index, pat.nnz_out)
    return sparse_like(A, v, pat.grad_indices)


def _grad_B(ctx, grad, patT=None):
    """grad_B = A^T grad through the cached transposed structure (reference sparse_matmul.py:222-232)."""
    vals = ctx.saved_tensors[2]
    want = None
    if ctx.B_strides is not None:  # ask for B's own layout; kernels that can write it directly save the re-stride pass
        want = tuple(ctx.B_strides) if ctx.batched else (ctx.B_shape[0] * ctx.B_shape[1],) + tuple(ctx.B_strides)
    patT = ctx.pattern.csr.transpose() if patT is None else patT
    gradB = _ops.spmm(patT, vals, grad, tag="spmm_gradB", out_strides=want)
    gradB = gradB if ctx.batched else gradB[0]
    if ctx.B_strides is not None and tuple(gradB.stride()) != tuple(ctx.B_strides):
        gradB = _ops.restride_like(gradB, ctx.B_shape, ctx.B_strides)
    return gradB
