"""The affine map of ``SparseMultivariateNormal.rsample`` for the covariance (``scale_tril``) parameterisations --
the immediate caller of ``sparse_mm`` (SURVEY.md 8(f) rank 2; reference
``distributions/sparse_multivariate_normal.py:354-389``):

    LL^T :   x = loc + L eps
    LDL^T:   eta = sqrt(D) * eps;   x = loc + (L eta + eta)

The reference runs ``_batch_sparse_mv(spmm, L, eta)`` -- ``sparse_mm`` on a transposed / permuted *view* of eta, whose
result is transposed / permuted back -- followed by two elementwise adds (``+ eta`` at ``:362``, ``loc +`` at ``:389``)
on strided views.  Here the product is the same ``sparse_mm`` call and everything after it is ONE pass
(``tsgu_pack_dense_add``): the layout change back to eps's layout, ``+ eta`` and ``+ loc`` in a single coalesced kernel.
The precision (``precision_tril``) parameterisations need a triangular solve (``sparse_triangular_solve``); their
``rsample`` / ``log_prob`` are not built here yet.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _native as nat
from .sparse_matmul import sparse_mm


class _TransposeAdd(torch.autograd.Function):
    """out[j, (b,) r] = C[(b,) r, j] + eta[j, (b,) r] + loc[(b,) r]  (eta optional)."""

    @staticmethod
    def forward(ctx, C, eta, loc, out_shape):
        batched = C.dim() == 3
        C3 = C if batched else C.unsqueeze(0)
        b, n, k = C3.shape
        out = torch.empty(out_shape, dtype=C.dtype, device=C.device)
        # view of `out` (and eta) as (batch, rows = n, cols = k): out is (k, [b,] n) contiguous
        o3 = out.reshape(k, b, n).permute(1, 2, 0)
        e3 = None if eta is None else eta.reshape(k, b, n).permute(1, 2, 0)
        if e3 is not None and e3.stride() != o3.stride():
            e3 = eta.contiguous().reshape(k, b, n).permute(1, 2, 0)
        loc2 = loc if loc.dim() == 2 else loc.unsqueeze(0).expand(b, n)
        ctx.shapes = (batched, b, n, k, loc.shape, eta is not None)
        if out.numel():
            C3 = C3.contiguous()
            nat.check(nat.lib().tsgu_pack_dense_add(C3.data_ptr(), nat.ptr(e3), loc2.data_ptr(), out.data_ptr(), b, n, k,
                                                    *C3.stride(), *o3.stride(), loc2.stride(0), loc2.stride(1),
                                                    nat.val_enum(C.dtype), nat.stream_ptr(C.device)), "tsgu_pack_dense_add")
        return out

    @staticmethod
    def backward(ctx, g):  # type: ignore[override]
        batched, b, n, k, loc_shape, has_eta = ctx.shapes
        g3 = g.reshape(k, b, n)
        gC = g3.permute(1, 2, 0)  # a view: sparse_mm's backward reads any strides
        gC = gC if batched else gC[0]
        g_eta = g if has_eta else None
        g_loc = g3.sum(0) if len(loc_shape) == 2 else g3.sum((0, 1))
        return gC, g_eta, g_loc, None


def rsample_transform(scale_tril: torch.Tensor, eps: torch.Tensor, loc: torch.Tensor,
                      diagonal: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``loc + scale_tril @ eps`` (LL^T) or ``loc + scale_tril @ eta + eta`` with ``eta = sqrt(diagonal) * eps`` (LDL^T),
    for ``eps`` of shape ``sample_shape + batch_shape + (n,)`` with at most one sample and one batch dimension -- the
    four rank combinations of the reference's ``_batch_sparse_mv`` (``:16-102``); same ``ValueError`` otherwise.
    Differentiable with respect to the values of ``scale_tril``, ``loc``, ``diagonal`` and ``eps``."""
    eta = eps if diagonal is None else diagonal.sqrt() * eps
    if scale_tril.dim() == 2 and eta.dim() == 1:
        C = sparse_mm(scale_tril, eta.unsqueeze(-1))          # (n, 1)
    elif scale_tril.dim() == 2 and eta.dim() == 2:
        C = sparse_mm(scale_tril, eta.t())                    # (n, k)
    elif scale_tril.dim() == 3 and eta.dim() == 2:
        C = sparse_mm(scale_tril, eta.unsqueeze(-1))          # (B, n, 1)
    elif scale_tril.dim() == 3 and eta.dim() == 3:
        C = sparse_mm(scale_tril, eta.permute(1, 2, 0))       # (B, n, k)
    else:
        raise ValueError("Invalid dimensions for bmat and bvec")
    if loc.dim() == 2 and C.dim() == 2:  # batched loc with an unbatched factor: plain broadcasting, not the fused pass
        x = C.t() if eta.dim() == 2 else C.squeeze(-1)
        return loc + (x + eta if diagonal is not None else x)
    return _TransposeAdd.apply(C, eta if diagonal is not None else None, loc, eta.shape)
