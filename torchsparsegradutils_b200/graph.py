"""CUDA-graph replay of a ``sparse_mm`` forward + backward for a fixed sparsity pattern.

Enqueueing one eager step costs ~0.3-0.4 ms of host time (Python, ctypes, autograd); a small problem
(BASELINE config 1: three ~10 us kernels) or a strongly scaled batch shard is bound by that, not by the
GPU.  Training loops that keep the pattern and the shapes fixed (``tests/test_sparse_matmul.py:295-338``)
can capture the step once and replay it: config 1 goes from 0.32 ms to 0.031 ms per step.
"""
from __future__ import annotations

from typing import Tuple

import torch

from ._pattern import pattern_of, pin_pattern, sparse_like, sparse_values
from .sparse_matmul import sparse_mm


class GraphedSparseMM:
    """``C, grad_A_values, grad_B = step(values, B, G)`` replayed from one captured CUDA graph.

    Parameters are *templates*: ``A`` fixes the pattern (COO or CSR, unbatched or batched), ``B`` and
    ``G`` fix shapes / dtypes of the dense operand and of the upstream gradient.  Every call copies the
    new data into the graph's static buffers, replays, and returns the graph's static output tensors
    (valid until the next call).
    """

    def __init__(self, A: torch.Tensor, B: torch.Tensor, G: torch.Tensor, warmup: int = 3):
        if not (A.is_cuda and B.is_cuda and G.is_cuda):
            raise RuntimeError("GraphedSparseMM needs CUDA tensors")
        dev = B.device
        with torch.no_grad():
            A_static = sparse_like(A, sparse_values(A).clone(),
                                   is_coalesced=A.is_coalesced() if A.layout == torch.sparse_coo else None)
        self._A = A_static.requires_grad_(True)
        self._B = B.detach().clone().contiguous().requires_grad_(True)
        self._G = G.detach().clone().contiguous()

        def step():
            self._A.grad = None
            self._B.grad = None
            C = sparse_mm(self._A, self._B)
            C.backward(self._G)
            return C

        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            # The pattern builds (sort / transpose, with their host syncs) are not capturable: build the pattern
            # here and PIN it to this object, so the capture below -- and nothing later -- depends on what the
            # LRU pattern cache happens to hold (it may have capacity 0, or evict the entry between steps).
            self._pattern = pattern_of(self._A)
            pin_pattern(self._pattern.cache_key, self._pattern)
            self._pattern.csr.transpose(optimise=True)  # final layout before capture
            for _ in range(max(warmup, 1)):
                step()
        torch.cuda.current_stream(dev).wait_stream(side)
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._C = step()
        self._gA_values = sparse_values(self._A.grad)
        self._gB = self._B.grad

    @torch.no_grad()
    def __call__(self, values: torch.Tensor, B: torch.Tensor, G: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
        A_values = sparse_values(self._A)
        A_values.copy_(values.reshape(A_values.shape))
        self._B.copy_(B)
        self._G.copy_(G)
        self._graph.replay()
        return self._C.detach(), self._gA_values, self._gB
