"""CPU (`-m "not gpu"`): host logic, error contract and the C-ABI surface -- no compute calls."""
import os
import re
import subprocess

import pytest
import torch

import torchsparsegradutils_b200 as tsgu
from torchsparsegradutils_b200 import _native as nat
from torchsparsegradutils_b200.utils import utils as U

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _coo(shape=(4, 6)):
    return torch.eye(*shape).to_sparse_coo()


# ---- exact validation messages, in the reference's order (tests/test_sparse_matmul.py:162-212) ----
def test_error_not_tensors():
    with pytest.raises(ValueError, match="Both A and B should be instances of torch.Tensor"):
        tsgu.sparse_mm("not a tensor", torch.rand(6, 2))


def test_error_dims():
    with pytest.raises(ValueError, match="Both A and B should be at least 2-dimensional tensors"):
        tsgu.sparse_mm(torch.rand(6).to_sparse(), torch.rand(6, 2))
    with pytest.raises(ValueError, match="A and B must both be 2D or both be 3D tensors"):
        tsgu.sparse_mm(_coo(), torch.rand(1, 6, 2))


def test_error_layouts():
    with pytest.raises(ValueError, match="A should be in either COO or CSR sparse format"):
        tsgu.sparse_mm(_coo().to_sparse_csc(), torch.rand(6, 2))
    with pytest.raises(ValueError, match="A should be in either COO or CSR sparse format"):
        tsgu.sparse_mm(torch.rand(4, 6), torch.rand(6, 2))
    with pytest.raises(ValueError, match=re.escape("B must be a dense (strided) tensor")):
        tsgu.sparse_mm(_coo(), torch.rand(6, 2).to_sparse())


def test_error_batch_and_inner():
    A = torch.stack([_coo(), _coo()])
    with pytest.raises(ValueError, match="If batched, A and B must have the same batch size"):
        tsgu.sparse_mm(A, torch.rand(3, 6, 2))
    with pytest.raises(ValueError, match=re.escape("Incompatible inner dimensions: A[..., 6] vs B[..., 5]")):
        tsgu.sparse_mm(_coo(), torch.rand(5, 2))


def test_cpu_tensors_fail_loudly():
    # north_star: no CPU fallback -- valid CPU inputs are refused, not silently computed
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        tsgu.sparse_mm(_coo(), torch.rand(6, 2))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        U._sort_coo_indices(torch.tensor([[1, 0], [0, 1]]))


def test_utils_validation_messages():
    with pytest.raises(TypeError, match="Expected a list of tensors"):
        U.stack_csr(torch.eye(2).to_sparse_csr())
    with pytest.raises(ValueError, match="Cannot stack empty list of tensors."):
        U.stack_csr([])
    with pytest.raises(ValueError, match="All tensors must have the same shape."):
        U.stack_csr([torch.eye(2).to_sparse_csr(), torch.eye(3).to_sparse_csr()])
    with pytest.raises(ValueError, match="All tensors must be in CSR layout."):
        U.stack_csr([torch.eye(2).to_sparse_coo(), torch.eye(2).to_sparse_coo()])
    with pytest.raises(TypeError, match="row_indices must be a torch.Tensor."):
        U._compress_row_indices([0, 1], 3)
    with pytest.raises(ValueError, match="row_indices must be 1D"):
        U._compress_row_indices(torch.zeros(2, 2, dtype=torch.int64), 3)
    with pytest.raises(TypeError, match="integer dtype"):
        U._compress_row_indices(torch.zeros(2), 3)
    with pytest.raises(ValueError, match="num_rows must be a positive integer."):
        U._compress_row_indices(torch.zeros(2, dtype=torch.int64), 0)
    with pytest.raises(ValueError, match="negative entries"):
        U._compress_row_indices(torch.tensor([-1, 0]), 3)
    with pytest.raises(ValueError, match="entries >= num_rows"):
        U._compress_row_indices(torch.tensor([0, 3]), 3)
    with pytest.raises(ValueError, match="at least 2 rows"):
        U.convert_coo_to_csr_indices_values(torch.zeros(1, 4, dtype=torch.int64), 3)
    with pytest.raises(ValueError, match="at most 3 rows"):
        U.convert_coo_to_csr_indices_values(torch.zeros(4, 4, dtype=torch.int64), 3)
    with pytest.raises(ValueError, match="Row indices must be less than num_rows"):
        U.convert_coo_to_csr_indices_values(torch.tensor([[5, 0], [0, 1]]), 3)
    with pytest.raises(ValueError, match="does not match number of indices"):
        U.convert_coo_to_csr_indices_values(torch.tensor([[1, 0], [0, 1]]), 3, torch.rand(3))
    with pytest.raises(ValueError, match="Unsupported layout"):
        U.convert_coo_to_csr(torch.eye(2).to_sparse_csr())
    with pytest.raises(ValueError, match="either be all sparse_coo or all sparse_csr"):
        U.sparse_block_diag(torch.eye(2).to_sparse_coo(), torch.eye(2).to_sparse_csr())
    with pytest.raises(TypeError, match="not as a list or tuple"):
        U.sparse_block_diag([torch.eye(2).to_sparse_coo()])
    with pytest.raises(ValueError, match="does not match"):
        U.sparse_block_diag_split(torch.eye(4).to_sparse_coo(), (2, 2), (3, 3))


def test_block_diag_roundtrip_host_logic():
    # pure index arithmetic: runs on any device (tests/test_utils.py:137-156, :209-230 semantics)
    for conv in (lambda t: t.to_sparse_coo(), lambda t: t.to_sparse_csr()):
        mats = [torch.rand(4, 6).round(decimals=0) * torch.rand(4, 6), torch.rand(3, 2), torch.rand(5, 5)]
        sp = [conv(m) for m in mats]
        bd = U.sparse_block_diag(*sp)
        assert torch.equal(bd.to_dense(), torch.block_diag(*mats))
        parts = U.sparse_block_diag_split(bd, (4, 6), (3, 2), (5, 5))
        for p, m in zip(parts, mats):
            assert torch.equal(p.to_dense(), m)
    st = U.stack_csr([torch.eye(3).to_sparse_csr(), (2 * torch.eye(3)).to_sparse_csr()])
    assert st.shape == (2, 3, 3) and torch.equal(st.to_dense(), torch.stack([torch.eye(3), 2 * torch.eye(3)]))


# ---- the C ABI: the library loads and exports exactly what include/tsgu_b200.h declares ----
def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "tsgu_b200.h")).read()
    return sorted(set(re.findall(r"TSGU_API[^;]*?\b(tsgu_\w+)\s*\(", text)))


def test_header_binding_and_library_agree():
    declared = _declared_symbols()
    assert declared == sorted(nat.EXPORTED_SYMBOLS), "include/tsgu_b200.h and _native._SIGNATURES drifted apart"
    L = nat.lib()  # sets argtypes for every symbol; AttributeError if one is missing
    for name in declared:
        assert hasattr(L, name)
    assert L.tsgu_version() == 2
    assert L.tsgu_error_string(-3).decode().startswith("tsgu: workspace")
    assert nat.launch_count() >= 0
    out = subprocess.run(["nm", "-D", "--defined-only", nat.LIB_PATH], capture_output=True, text=True).stdout
    exported = sorted(set(re.findall(r" T (tsgu_\w+)", out)))
    assert exported == declared, "only the declared C ABI may be exported"


def test_library_is_sm100a_and_torch_free():
    import shutil

    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    out = ""
    for _ in range(3):  # the tool occasionally returns nothing on a cold page cache
        out = subprocess.run(["cuobjdump", "--list-elf", nat.LIB_PATH], capture_output=True, text=True).stdout
        if "sm_100a" in out:
            break
    assert "sm_100a" in out and not re.search(r"sm_(?!100a)\d+", out)
    ldd = subprocess.run(["ldd", nat.LIB_PATH], capture_output=True, text=True).stdout
    assert "torch" not in ldd and "c10" not in ldd  # plain C ABI: no torch types or libraries behind it


def test_pattern_cache_api():
    tsgu.set_pattern_cache_capacity(4)
    tsgu.clear_pattern_cache()
    tsgu.set_pattern_cache_capacity(16)


def test_batch_sparse_mv_rank_errors():
    """Rank pairs outside the four supported ones raise the reference's message
    (distributions/sparse_multivariate_normal.py:102) before any native call."""
    import pytest
    import torch

    from torchsparsegradutils_b200 import batch_sparse_mv

    A = torch.eye(3).to_sparse_csr()
    with pytest.raises(ValueError, match="Invalid dimensions for bmat and bvec"):
        batch_sparse_mv(A, torch.zeros(2, 3, 3))
    with pytest.raises(ValueError, match="Invalid dimensions for bmat and bvec"):
        batch_sparse_mv(A, torch.tensor(1.0))
    calls = []
    out = batch_sparse_mv(A, torch.ones(5, 3), op=lambda a, b: calls.append(tuple(b.shape)) or torch.zeros(3, 5))
    assert calls == [(3, 5)] and out.shape == (5, 3)  # (k, n) vectors go in as a (n, k) view, come back as (k, n)


def test_uniform_rows_gate_of_k_slicing():
    """`CsrPattern.uniform_rows` (gate of TSGU_ALGO_FLAG_KSLICE): longest row <= 1.25 x mean + 1, for the flat
    layout our builders emit and for torch's batched (b, n+1) crow layout; empty patterns are never 'uniform'."""
    import torch

    from torchsparsegradutils_b200 import _native as nat
    from torchsparsegradutils_b200._pattern import CsrPattern

    def pat(rowptr, batch, n, bstride, nnz_total):
        col = torch.zeros(max(nnz_total, 1), dtype=torch.int32)
        return CsrPattern(rowptr, col, None, batch, n, 8, bstride, 0, nnz_total, nat.I32)

    flat = torch.arange(0, 4 * 6 + 1, 4, dtype=torch.int32)  # 6 rows of exactly 4
    assert pat(flat, 1, 6, 6, 24).uniform_rows
    ragged = torch.tensor([0, 1, 1, 2, 20, 21, 24], dtype=torch.int32)  # one row of 18 among rows of 0-3
    assert not pat(ragged, 1, 6, 6, 24).uniform_rows
    batched = torch.stack([flat[:4], flat[:4]])  # torch batched CSR: (b, n+1) with per-item offsets
    assert pat(batched, 2, 3, 4, 24).uniform_rows
    assert not pat(torch.zeros(7, dtype=torch.int32), 1, 6, 6, 0).uniform_rows


def test_kernel_family_choice(monkeypatch):
    """`choose_algo`: merge-path only for a single matrix whose longest row exceeds both 256 entries and 16 x the mean;
    TSGU_B200_ALGO forces a family, read when a pattern is built (not at import)."""
    from torchsparsegradutils_b200 import _native as nat
    from torchsparsegradutils_b200._pattern import choose_algo

    monkeypatch.delenv("TSGU_B200_ALGO", raising=False)
    assert choose_algo(257, 1, 100, 1000) == nat.ALGO_MERGE  # 257 > 256 and > 16 x 10
    assert choose_algo(256, 1, 100, 1000) == nat.ALGO_AUTO  # not above 256 entries
    assert choose_algo(400, 1, 100, 3000) == nat.ALGO_AUTO  # 400 < 16 x 30
    assert choose_algo(481, 1, 100, 3000) == nat.ALGO_MERGE  # 481 > 16 x 30
    assert choose_algo(480, 1, 100, 3000) == nat.ALGO_AUTO
    assert choose_algo(10**6, 4, 100, 1000) == nat.ALGO_AUTO  # a batch always takes the row-tile kernels
    assert choose_algo(None, 4, 100, 1000) == nat.ALGO_AUTO
    assert choose_algo(0, 1, 100, 0) == nat.ALGO_AUTO and choose_algo(None, 1, 0, 0) == nat.ALGO_AUTO  # empty
    monkeypatch.setenv("TSGU_B200_ALGO", "merge")
    assert choose_algo(1, 1, 100, 100) == nat.ALGO_MERGE and choose_algo(None, 4, 0, 0) == nat.ALGO_MERGE
    monkeypatch.setenv("TSGU_B200_ALGO", "RowSplit")
    assert choose_algo(10**6, 1, 100, 1000) == nat.ALGO_ROWSPLIT


def test_pattern_checksum_schedule_and_host_fingerprint(monkeypatch):
    """Which cache hits re-check a pattern's index checksum (default 1, 2, 4, 8, ...; "1" all; "0" none), the host
    restatement of tsgu_fingerprint (position-weighted sum: order of equal values matters), and the longest-row rule
    that `_analyse` fills `uniform_rows` from."""
    import torch

    from torchsparsegradutils_b200 import _pattern

    monkeypatch.setattr(_pattern, "_VERIFY", "sampled")
    assert [h for h in range(1, 40) if _pattern._verify_due(h)] == [1, 2, 4, 8, 16, 32]
    monkeypatch.setattr(_pattern, "_VERIFY", "1")
    assert all(_pattern._verify_due(h) for h in range(1, 10))
    monkeypatch.setattr(_pattern, "_VERIFY", "0")
    assert not any(_pattern._verify_due(h) for h in range(1, 10))
    a = torch.tensor([3, 1, 2], dtype=torch.int32)
    fa, fb = _pattern._fingerprint(a, a.long()), _pattern._fingerprint(a.flip(0), a.long())
    assert fa.tolist() == [3 * 1 + 1 * 2 + 2 * 3] * 2 and fb[0] != fa[0] and fb[1] == fa[1]
    assert _pattern._uniform_from(None, 4, 16) is None and _pattern._uniform_from(5, 0, 0) is False
    assert _pattern._uniform_from(6, 4, 16) is True and _pattern._uniform_from(7, 4, 16) is False  # 1.25 * 4 + 1 = 6


def test_bench_stdout_carries_only_the_json_line(tmp_path):
    """bench.py's contract: ONE JSON line on stdout.  Anything else written to fd 1 while it runs (NCCL prints its
    version banner there under torchrun) must end up on stderr."""
    import json
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "emit.py"
    script.write_text("\n".join([
        "import os, sys",
        f"sys.path.insert(0, {root!r})",
        "import bench",
        "bench._route_library_chatter_to_stderr()",
        "os.write(1, b'NCCL version banner' + bytes([10]))",
        "print('python-level chatter')",
        "bench.emit_json({'metric': 'm', 'value': 1})",
    ]) + "\n")
    r = subprocess.run([sys.executable, str(script)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0]) == {"metric": "m", "value": 1}
    assert "NCCL version banner" in r.stderr and "python-level chatter" in r.stderr


def test_bench_dump_outputs_is_bounded_and_repeatable(tmp_path):
    """--dump-outputs: float32 / float64 files, whole when small, otherwise the same seeded sample of whole rows (or
    elements of a 1-D output) on every run, within the per-output byte bound."""
    import os
    import sys

    import numpy as np
    import torch

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench

    g = torch.Generator().manual_seed(0)
    outs = {"C": torch.rand(3, 50, 8, generator=g), "grad_A_values": torch.rand(1000, generator=g, dtype=torch.float64),
            "grad_B": torch.rand(4, 6, generator=g).to(torch.bfloat16)}
    for run in ("a", "b"):
        bench.dump_outputs(outs, str(tmp_path / run), max_bytes=1024)
    for name, t in outs.items():
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert np.array_equal(a, b) and a.nbytes <= 1024
        assert a.dtype == (np.float64 if t.dtype == torch.float64 else np.float32)
    assert np.array_equal(np.load(tmp_path / "a" / "grad_B.npy"), outs["grad_B"].float().numpy())  # small: whole
    C = np.load(tmp_path / "a" / "C.npy")
    rows = outs["C"].reshape(-1, 8).numpy()
    assert C.shape == (1024 // 32, 8) and all((rows == r).all(axis=1).any() for r in C)
    gA = np.load(tmp_path / "a" / "grad_A_values.npy")
    assert gA.shape == (128,) and np.isin(gA, outs["grad_A_values"].numpy()).all()


def test_sort_rows_by_length_is_a_row_permutation_with_snake_blocks():
    """Host-side layout optimisation of the cached transpose (pure index arithmetic, runs on any device): rows are
    permuted inside blocks of 64, alternately longest-first / shortest-first, entries of a row stay together and in
    order, and row_map sends every slot back to its original row."""
    import torch

    from torchsparsegradutils_b200 import _pattern as P

    g = torch.Generator().manual_seed(0)
    batch, rows = 2, 200
    lens = torch.randint(0, 9, (batch * rows,), generator=g)
    rowptr = torch.zeros(batch * rows + 1, dtype=torch.int32)
    rowptr[1:] = lens.cumsum(0)
    nnz = int(rowptr[-1])
    col = torch.randint(0, 50, (nnz,), generator=g, dtype=torch.int32)
    perm = torch.randperm(nnz, generator=g).to(torch.int32)
    rp2, col2, perm2, row_map = P._sort_rows_by_length(rowptr, col, perm, batch, rows)
    assert rp2.dtype == rowptr.dtype and int(rp2[-1]) == nnz and row_map.numel() == batch * rows
    new_lens = (rp2[1:] - rp2[:-1]).long()
    for t in range(batch):
        rm = row_map[t * rows:(t + 1) * rows].long()
        assert torch.equal(rm.sort().values, torch.arange(rows))  # a permutation inside every item
        for s in range(rows):
            o = t * rows + int(rm[s])
            a, b = int(rowptr[o]), int(rowptr[o + 1])
            a2, b2 = int(rp2[t * rows + s]), int(rp2[t * rows + s + 1])
            assert torch.equal(col2[a2:b2], col[a:b]) and torch.equal(perm2[a2:b2], perm[a:b])
        blocks = new_lens[t * rows:(t + 1) * rows].split(P._SORT_BLOCK)
        for k, blk in enumerate(blocks):
            d = blk[1:] - blk[:-1]
            assert bool((d <= 0).all()) if k % 2 == 0 else bool((d >= 0).all())
            # block membership is unchanged: a block holds the rows it held before
            lo = k * P._SORT_BLOCK
            assert set(row_map[t * rows + lo: t * rows + lo + blk.numel()].tolist()) == set(range(lo, lo + blk.numel()))


def test_bench_config_is_identical_for_both_arms_and_deterministic():
    import argparse
    import sys, os

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench

    for cid in ("2", "3", "4", "5"):
        for world in (1, 2, 8):
            a = argparse.Namespace(config=cid, scaling="strong", sharding="k", grad_b="all_reduce", no_overlap=False)
            c1 = bench.describe_config(bench.CONFIGS[cid], a, world)
            c2 = bench.describe_config(bench.CONFIGS[cid], a, world)
            assert c1 == c2 and set(c1[0]) == {"workload", "config_id", "K", "l2", "sharding"}
    # strong scaling of the batched config: per-rank footprint shrinks with the ranks, flush policy follows
    a = argparse.Namespace(config="2", scaling="strong", sharding="k", grad_b="all_reduce", no_overlap=False)
    assert bench.describe_config(bench.CONFIGS["2"], a, 1)[3] is False and bench.describe_config(bench.CONFIGS["2"], a, 8)[3] is True


def test_aligned_contiguous_copies_only_misaligned_views():
    import torch

    from torchsparsegradutils_b200._pattern import aligned_contiguous

    base = torch.arange(64, dtype=torch.int32)
    assert aligned_contiguous(base) is base
    v = base[1:33]
    c = aligned_contiguous(v)
    assert c is not v and c.data_ptr() % 16 == 0 and torch.equal(c, v)
