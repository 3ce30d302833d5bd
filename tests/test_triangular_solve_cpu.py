"""Argument validation of ``sparse_triangular_solve`` (raised before any native call, so no GPU is needed)."""
import pytest
import torch

from torchsparsegradutils_b200 import sparse_triangular_solve


def _tri(n=5):
    return (torch.eye(n, dtype=torch.float64) + torch.ones(n, n, dtype=torch.float64).tril(-1)).to_sparse_csr()


@pytest.mark.parametrize("A,B,msg", [
    (lambda: _tri(), lambda: "x", "instances of torch.Tensor"),
    (lambda: _tri(), lambda: torch.ones(5, dtype=torch.float64), "at least 2-dimensional"),
    (lambda: _tri(), lambda: torch.ones(1, 5, 2, dtype=torch.float64), "both be 2D or both be 3D"),
    (lambda: _tri().to_dense(), lambda: torch.ones(5, 2, dtype=torch.float64), "COO or CSR"),
    (lambda: torch.ones(5, 4, dtype=torch.float64).to_sparse_csr(), lambda: torch.ones(4, 2, dtype=torch.float64),
     "square"),
    (lambda: _tri(), lambda: torch.ones(4, 2, dtype=torch.float64), "Incompatible inner dimensions"),
])
def test_value_errors(A, B, msg):
    with pytest.raises(ValueError, match=msg):
        sparse_triangular_solve(A(), B())


def test_cpu_tensors_are_refused():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        sparse_triangular_solve(_tri(), torch.ones(5, 2, dtype=torch.float64), upper=False)
