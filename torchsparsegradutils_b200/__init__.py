"""B200-native drop-in for the ``sparse_mm`` hot path of cai4cai/torchsparsegradutils.

    from torchsparsegradutils_b200 import sparse_mm      # same signature as the reference's

Only the path named by BASELINE.json's north_star lives here: ``sparse_mm`` / ``SparseMatMul`` and the
index/layout helpers it depends on.  The arithmetic is hand-written sm_100a CUDA behind the C ABI in
``include/tsgu_b200.h`` (``libtsgu_b200.so``); there is no CPU or PyTorch fallback.
"""
from . import utils
from .batch_mv import batch_sparse_mv
from ._pattern import clear_pattern_cache, prepare_pattern, set_pattern_cache_capacity
from .graph import GraphedSparseMM
from .rsample import rsample_transform
from .encoders import PairwiseValueAssembler
from .sddmm import block_diag_operand, lstsq_grad_A, sddmm, solve_grad_A
from .sparse_matmul import SparseMatMul, sparse_mm
from .triangular_solve import SparseTriangularSolve, sparse_triangular_solve

__all__ = ["sparse_mm", "SparseMatMul", "sparse_triangular_solve", "SparseTriangularSolve", "sddmm", "solve_grad_A", "lstsq_grad_A", "block_diag_operand", "PairwiseValueAssembler", "batch_sparse_mv", "rsample_transform", "GraphedSparseMM", "utils", "clear_pattern_cache", "prepare_pattern", "set_pattern_cache_capacity"]
__version__ = "0.1.0"
