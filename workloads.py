"""Seeded synthetic inputs for BASELINE.json's five configs (bench + full-size property tests).

Device-agnostic torch code: the same generator feeds the B200 run and the bounded CPU-baseline
sample.  Output contract follows the reference's generators (utils/random_sparse.py: unique
coordinates, exactly nnz per batch item, coalesced COO / sorted CSR); values are U(0,1)
(utils/random_sparse.py:411,534), B and the upstream gradient N(0,1) (benchmarks/sparse_mm_rand.py:75).
The reference's own generator is an O(nnz) Python set rejection sampler (utils/random_sparse.py:246),
unusable at these sizes, hence these vectorised ones.
"""
from __future__ import annotations

import torch


def _gen(device, seed):
    return torch.Generator(device=device).manual_seed(seed)


def distinct_sorted_columns(rows: int, m: int, per_row: int, gen, device) -> torch.Tensor:
    """(rows, per_row) sorted distinct columns, uniform over per_row-subsets of range(m): sorted draws
    from [0, m-per_row] plus 0..per_row-1 (the multiset <-> subset bijection); no rejection loop."""
    x = torch.randint(0, m - per_row + 1, (rows, per_row), generator=gen, device=device)
    return x.sort(dim=1).values + torch.arange(per_row, device=device)


def uniform_rows_csr(batch, n, m, per_row, dtype=torch.float32, index_dtype=torch.int32, device="cuda", seed=2):
    """Configs 2 and 5: every row has exactly `per_row` distinct uniform columns. batch=None -> 2-D CSR."""
    g = _gen(device, seed)
    b = batch or 1
    col = distinct_sorted_columns(b * n, m, per_row, g, device).reshape(b, n * per_row)
    crow = (torch.arange(n + 1, device=device) * per_row).repeat(b, 1)
    vals = torch.rand((b, n * per_row), generator=g, device=device, dtype=torch.float32).to(dtype)
    if batch is None:
        crow, col, vals = crow[0], col[0], vals[0]
    shape = (batch, n, m) if batch is not None else (n, m)
    return torch.sparse_csr_tensor(crow.to(index_dtype), col.to(index_dtype), vals, shape)


def uniform_coo(n, m, nnz, dtype=torch.float32, device="cuda", seed=1):
    """Config 1: nnz unique coordinates uniform without replacement, coalesced COO (int64 indices)."""
    g = _gen(device, seed)
    if n * m <= (1 << 28):
        flat = torch.randperm(n * m, generator=g, device=device)[:nnz].sort().values
    else:  # very sparse, huge index space: draw with replacement, drop the (rare) repeats, keep nnz of them
        flat = torch.unique(torch.randint(0, n * m, (2 * nnz + 16,), generator=g, device=device, dtype=torch.int64))
        flat = flat[torch.randperm(flat.numel(), generator=g, device=device)[:nnz]].sort().values
        assert flat.numel() == nnz
    idx = torch.stack([flat // m, flat % m])
    vals = torch.rand(nnz, generator=g, device=device, dtype=torch.float32).to(dtype)
    return torch.sparse_coo_tensor(idx, vals, (n, m), is_coalesced=True)


def stencil27_csr(D, dtype=torch.float32, index_dtype=torch.int32, device="cuda", seed=3, lower=False):
    """Config 3: 27-point (26-neighbourhood + diagonal) pattern on a D^3 volume, the sparsity
    PairwiseEncoder(radius>=1.74, volume_shape=(1,D,D,D), diag=True) produces
    (encoders/pairwise_encoder.py:383-505); nnz = (3D-2)^3.  `lower`: lower triangle + diagonal only
    (what SparseMultivariateNormal's scale_tril takes)."""
    g = _gen(device, seed)
    n = D ** 3
    v = torch.arange(n, device=device)
    z, y, x = v // (D * D), (v // D) % D, v % D
    cols, masks = [], []
    for dz in (-1, 0, 1):
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                lin = dz * D * D + dy * D + dx
                if lower and lin > 0:
                    continue
                ok = (z + dz >= 0) & (z + dz < D) & (y + dy >= 0) & (y + dy < D) & (x + dx >= 0) & (x + dx < D)
                cols.append(v + lin)
                masks.append(ok)
    cols, masks = torch.stack(cols, dim=1), torch.stack(masks, dim=1)  # offsets ascend => sorted columns
    crow = torch.zeros(n + 1, dtype=torch.int64, device=device)
    crow[1:] = masks.sum(dim=1).cumsum(0)
    col = cols[masks]
    vals = torch.rand(col.numel(), generator=g, device=device, dtype=torch.float32).to(dtype)
    return torch.sparse_csr_tensor(crow.to(index_dtype), col.to(index_dtype), vals, (n, n))


def random_lower_csr(batch, n, per_row, dtype=torch.float32, index_dtype=torch.int32, device="cuda", seed=6):
    """Random lower triangle: row r holds min(r, per_row - 1) distinct uniform columns below the diagonal plus the
    diagonal (sorted).  Every item has the same row lengths, so a batch is a valid batched CSR.  batch=None -> 2-D.
    Values from :func:`triangular_values`."""
    g = _gen(device, seed)
    b, k = batch or 1, per_row - 1
    r = torch.arange(n, device=device)
    span = (r - k + 1).clamp(min=1)  # draws in [0, r - k]: sorted + arange(k) gives k distinct columns below r
    x = (torch.rand((b, n, k), generator=g, device=device) * span[None, :, None]).long().sort(dim=2).values
    x = x + torch.arange(k, device=device)
    cols = torch.cat([x, r.expand(b, n).unsqueeze(-1)], dim=2)
    keep = torch.cat([torch.arange(k, device=device)[None, :] < r.clamp(max=k)[:, None],
                      torch.ones(n, 1, dtype=torch.bool, device=device)], dim=1)  # rows r < k: columns 0..r-1
    col = cols[keep.expand(b, n, k + 1)].reshape(b, -1)
    crow = torch.zeros(n + 1, dtype=torch.int64, device=device)
    crow[1:] = keep.sum(dim=1).cumsum(0)
    crow = crow.repeat(b, 1)
    if batch is None:
        crow, col = crow[0], col[0]
    shape = (batch, n, n) if batch is not None else (n, n)
    A = torch.sparse_csr_tensor(crow.to(index_dtype), col.to(index_dtype), torch.zeros(col.shape, device=device), shape)
    return triangular_values(A, dtype, seed=seed + 1)


def triangular_values(A, dtype=torch.float32, seed=7):
    """A's CSR pattern with well-conditioned triangular-solve values: off-diagonal entries U(0,1) / row length,
    diagonal entries U(1,2)."""
    crow, col = A.crow_indices(), A.col_indices()
    n = A.shape[-1]
    crow2, col2 = crow.reshape(-1, n + 1).long(), col.reshape(crow.numel() // (n + 1), -1).long()
    lens = crow2.diff(dim=1)
    row = torch.repeat_interleave(torch.arange(n, device=col.device).repeat(crow2.shape[0]), lens.reshape(-1),
                                  output_size=col2.numel()).reshape(col2.shape)
    u = torch.rand(col2.shape, generator=_gen(col.device, seed), device=col.device, dtype=torch.float64)
    vals = torch.where(col2 == row, 1.0 + u, u / lens.gather(1, row).clamp(min=1)).to(dtype).reshape(col.shape)
    return torch.sparse_csr_tensor(crow, col, vals, A.shape)


def rmat_csr(scale, edge_factor=16, dtype=torch.bfloat16, index_dtype=torch.int32, device="cuda", seed=4,
             a=0.57, b=0.19, c=0.19):
    """Config 4: Graph500 R-MAT (a,b,c,d = .57,.19,.19,.05), 2^scale vertices, edge_factor*2^scale draws,
    directed, duplicates removed, vertex ids NOT permuted (keeps the hub skew)."""
    g = _gen(device, seed)
    n = 1 << scale
    E = edge_factor * n
    row = torch.zeros(E, dtype=torch.int64, device=device)
    col = torch.zeros(E, dtype=torch.int64, device=device)
    for _ in range(scale):
        r = torch.rand(E, generator=g, device=device)
        row = (row << 1) | (r >= a + b).long()
        col = (col << 1) | (((r >= a) & (r < a + b)) | (r >= a + b + c)).long()
    key = torch.unique(row * n + col)  # sorted, duplicate-free
    row, col = key // n, key % n
    crow = torch.zeros(n + 1, dtype=torch.int64, device=device)
    crow[1:] = torch.bincount(row, minlength=n).cumsum(0)
    vals = torch.rand(key.numel(), generator=g, device=device, dtype=torch.float32).to(dtype)
    return torch.sparse_csr_tensor(crow.to(index_dtype), col.to(index_dtype), vals, (n, n))


def dense_operands(A_shape, K, dtype=torch.float32, device="cuda", seed=100):
    """B (.., m, K) and upstream gradient G (.., n, K), N(0,1)."""
    g = _gen(device, seed)
    lead = tuple(A_shape[:-2])
    n, m = A_shape[-2], A_shape[-1]
    B = torch.randn(lead + (m, K), generator=g, device=device, dtype=torch.float32).to(dtype)
    G = torch.randn(lead + (n, K), generator=g, device=device, dtype=torch.float32).to(dtype)
    return B, G


def algorithmic_bytes(batch, n, m, nnz_item, K, s_v, s_i, coo=False):
    """Compulsory HBM traffic of one fwd+bwd (SURVEY.md section 8(d)); returns dict per kernel + total."""
    idx = 2 * nnz_item * 8 if coo else nnz_item * s_i + (n + 1) * s_i
    idxT = 2 * nnz_item * 8 if coo else nnz_item * s_i + (m + 1) * s_i
    dense = m * K * s_v + n * K * s_v
    fwd = nnz_item * s_v + idx + dense
    sddmm = idx + dense + nnz_item * s_v
    gradb = nnz_item * s_v + idxT + dense
    out = {"spmm_fwd": batch * fwd, "sddmm": batch * sddmm, "spmm_gradB": batch * gradb}
    out["total"] = sum(out.values())
    return out
