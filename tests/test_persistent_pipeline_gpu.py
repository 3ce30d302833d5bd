"""GPU: the persistent kernels with many tiles per CTA -- row-tile and merge-path SpMM / SDDMM, the column-window pair
and the triangular solve -- on narrow grids, into poisoned outputs, and with NaN probes in the dense operands.

Every persistent kernel walks tiles ``blockIdx.x, blockIdx.x + gridDim.x, ...`` through a two-stage bulk-copy
pipeline (refill of a used stage, parity-1 waits, the window kernels' empty-barrier wait), and the triangular solve
hands rows out by ticket.  At oracle size the grid (148 SMs x resident CTAs) is larger than the tile count, so every
CTA runs at most one tile; here ``_native.sm_margin(147)`` leaves one SM to the grid (at most 8 CTAs at 256 threads)
and every CTA walks many tiles.

Sizing rule.  A row tile holds at most ``TSGU_TILE_ROWS`` = 256 rows, so a launch over at least 24 x 256 rows has at
least 24 tiles, 3 per CTA at margin 147, whatever height ``balance_tile_rows`` picks.  A merge-path tile holds
``TSGU_MERGE_P`` = 3072 path items (rows + stored entries), so a merge launch needs at least 24 x 3072 of them.  A
window tile holds at most 32 rows.

Three checks per case:

1. Narrow grids.  Margins 0, 100 and 147 give bit-identical outputs (per-row / per-entry summation order is fixed,
   merge carries are summed in tile order, the solve has no value atomics), and the margin-0 output matches the fp64
   oracle.  ``g_sm_margin`` is thread-local and autograd runs the backward on a thread of its own, so the operators
   are called directly here (``_ops.spmm`` / ``_ops.sddmm`` on the pattern and its transpose, and the forward solve
   with ``transpose`` flipped instead of its backward).
2. Poisoned outputs.  ``torch.empty`` / ``empty_strided`` of a floating dtype inside ``_ops`` and
   ``triangular_solve`` come back filled with a poison value, and every operator workspace with 0xFF bytes (NaN as a
   float, -1 = "none" as a merge ``carry_row``), so an element a kernel skips cannot pass for a result that happens
   to sit in recycled memory.  Integer outputs (pattern builders) are not poisoned: a missed write there would be
   read back as an index.
3. NaN probes.  Single elements of B and G are NaN (row 0 among them, on a 16-byte vector boundary, in the last
   column and in the last vector of a K the lanes do not fill).  NaN must appear exactly where the structure says --
   a stored entry, explicit zeros included, times NaN is NaN -- and every other element must match the oracle run
   with the probes set to 0.  A kernel that reads a dense row it should not, with weight 0, fails here and nowhere
   else.  The poison is then a finite sentinel, so "never written" and "NaN propagated" stay apart.
"""
import json

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import workloads as W
from helpers import TOL
from oracle import oracle as orc

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
MARGINS = (0, 100, 147)
PROBE_MARGINS = (0, 147)
SENTINEL = -7e37
EPV = {torch.float32: 4, torch.float64: 2, torch.bfloat16: 8}
DTYPES = [torch.float32, torch.float64, torch.bfloat16]
# (non-exact, exact) vectors per dense row for each (lanes per row, vectors per lane) row of with_tile_lanes (tile.cuh)
LANE_ROWS = [(3, 4), (6, 8), (12, 16), (24, 32), (48, 64), (96, 128)]


# ------------------------------------------------------------------------------------------------ fixtures
class _Poisoned:
    """Stands in for a module inside the operators: every attribute is the module's, except the allocators."""

    def __init__(self, module, **overrides):
        self._module = module
        self.__dict__.update(overrides)

    def __getattr__(self, name):
        return getattr(self._module, name)


@pytest.fixture
def poison(monkeypatch):
    """Floating-point outputs of ``_ops`` and ``triangular_solve`` start as ``poison.fill`` (NaN unless a test sets
    it), their workspaces as 0xFF bytes.  The pattern cache is cleared on both sides."""
    import torchsparsegradutils_b200 as tsgu
    from torchsparsegradutils_b200 import _native as nat
    from torchsparsegradutils_b200 import _ops, triangular_solve

    state = _Poisoned(None, fill=float("nan"))

    def _fill(t):
        return t.fill_(state.fill) if t.is_floating_point() else t

    fake_torch = _Poisoned(torch, empty=lambda *a, **k: _fill(torch.empty(*a, **k)),
                           empty_strided=lambda *a, **k: _fill(torch.empty_strided(*a, **k)))
    fake_nat = _Poisoned(nat, workspace=lambda nbytes, device: nat.workspace(nbytes, device).fill_(0xFF))
    for mod in (_ops, triangular_solve):
        monkeypatch.setattr(mod, "torch", fake_torch)
        monkeypatch.setattr(mod, "nat", fake_nat)
    tsgu.clear_pattern_cache()
    yield state
    tsgu.clear_pattern_cache()


@pytest.fixture
def tile_kernels(monkeypatch):
    """Small launches take the row-split kernels unless TSGU_TINY_ROWS says otherwise."""
    monkeypatch.setenv("TSGU_TINY_ROWS", "0")


@pytest.fixture
def windows(monkeypatch):
    """Lift the size gates of the column-window path (as tests/test_window_gpu.py does)."""
    from torchsparsegradutils_b200 import _pattern

    monkeypatch.setattr(_pattern, "_WINDOW_MIN_NNZ", 0)
    monkeypatch.setattr(_pattern, "_WINDOW_MIN_ROWS", 0)


# ------------------------------------------------------------------------------------------------ inputs
class Case:
    """A sparse operand and its stored entries on the host, flat over the batch (row t*n + i, column t*m + j), in the
    order of A's value storage, which is also the order the SDDMM writes."""

    def __init__(self, A, rows, cols, batch, n, m):
        self.A, self.rows, self.cols = A, rows, cols
        self.batch, self.n, self.m = batch, n, m
        self.S = sp.csr_matrix((np.ones(rows.size), (rows, cols)), shape=(batch * n, batch * m))  # the structure


def _values(nnz, dtype, seed):
    return torch.rand(nnz, generator=torch.Generator().manual_seed(seed), dtype=torch.float64).to(dtype)


def _csr_case(rows, cols, n, m, dtype, idx, seed, batch=None):
    """CSR (batched when `batch`: every item holds rows.size // batch entries, rows / cols local to the item)."""
    b = batch or 1
    per = rows.size // b
    crow = np.zeros((b, n + 1), dtype=np.int64)
    for t in range(b):
        crow[t, 1:] = np.cumsum(np.bincount(rows[t * per:(t + 1) * per], minlength=n))
    vals = _values(rows.size, dtype, seed)
    crow_t, col_t = torch.from_numpy(crow), torch.from_numpy(cols.copy())
    if batch is None:
        A = torch.sparse_csr_tensor(crow_t[0].to(idx), col_t.to(idx), vals, (n, m))
    else:
        A = torch.sparse_csr_tensor(crow_t.to(idx), col_t.reshape(b, per).to(idx), vals.reshape(b, per), (b, n, m))
    off = np.repeat(np.arange(b), per)
    return Case(A.to(DEV), rows + off * n, cols + off * m, b, n, m)


def _coo_case(rows, cols, n, m, dtype, seed):
    """Uncoalesced 2-D COO in shuffled storage order (int64 indices: the flat CSR gets a value permutation)."""
    sh = np.random.default_rng(seed).permutation(rows.size)
    r, c = rows[sh], cols[sh]
    A = torch.sparse_coo_tensor(torch.from_numpy(np.stack([r, c])), _values(r.size, dtype, seed), (n, m))
    assert not A.is_coalesced()
    return Case(A.to(DEV), r, c, 1, n, m)


def _random_entries(n, m, nnz, seed):
    """`nnz` distinct uniform coordinates sorted by (row, column)."""
    g = torch.Generator().manual_seed(seed)
    flat = torch.unique(torch.randint(0, n * m, (nnz + nnz // 4 + 16,), generator=g))
    flat = flat[torch.randperm(flat.numel(), generator=g)[:nnz]].sort().values.numpy()
    return flat // m, flat % m


def _entries_from_lengths(cnt, m, seed):
    """Rows of the given lengths with distinct sorted uniform columns."""
    rng = np.random.default_rng(seed)
    cols = [np.sort(rng.choice(m, size=int(c), replace=False)) for c in cnt]
    return np.repeat(np.arange(cnt.size), cnt), np.concatenate(cols).astype(np.int64)


def _layout_case(layout, dtype, idx, seed):
    if layout == "csr":
        return _csr_case(*_random_entries(6200, 6150, 49_000, seed), 6200, 6150, dtype, idx, seed)
    if layout == "coo":
        return _coo_case(*_random_entries(6200, 6150, 49_000, seed), 6200, 6150, dtype, seed)
    b, n, m, per = 3, 2100, 2050, 16_800
    parts = [_random_entries(n, m, per, seed + t) for t in range(b)]
    rows, cols = np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
    return _csr_case(rows, cols, n, m, dtype, idx, seed, batch=b)


def _long_rows_case(dtype, idx, seed):
    """A row longer than any staging capacity every 300 rows, between empty rows; short rows elsewhere: staged and
    unstaged tiles alternate on one CTA."""
    n, m = 6400, 12_000
    rng = np.random.default_rng(seed)
    cnt = rng.integers(1, 12, n)
    for r in range(150, n, 300):
        cnt[r] = 10_000  # > CAP of every stage layout (at most 9216 entries)
        cnt[r - 3:r] = 0
        cnt[r + 1:r + 4] = 0
    return _csr_case(*_entries_from_lengths(cnt, m, seed), n, m, dtype, idx, seed)


def _skewed_case(dtype, idx, seed):
    """Merge-path input: hub rows spanning 3+ merge tiles, many empty rows, a long last row; >= 24 x 3072 path items
    in the matrix and in its transpose."""
    n, m = 30_000, 12_000
    rng = np.random.default_rng(seed)
    cnt = rng.integers(0, 5, n)
    cnt[rng.random(n) < 0.4] = 0
    cnt[[0, 7, 15_001]] = 10_000
    cnt[-1] = 4_000
    return _csr_case(*_entries_from_lengths(cnt, m, seed), n, m, dtype, idx, seed)


def _host_case(A):
    """Case of a CSR tensor built on the device."""
    crow, col = A.crow_indices().cpu().long(), A.col_indices().cpu().long()
    b = A.shape[0] if A.dim() == 3 else 1
    n, m = A.shape[-2], A.shape[-1]
    crow, col = crow.reshape(b, n + 1).numpy(), col.reshape(b, -1).numpy()
    rows = np.concatenate([np.repeat(np.arange(n), np.diff(crow[t])) + t * n for t in range(b)])
    cols = np.concatenate([col[t] + t * m for t in range(b)])
    return Case(A, rows, cols, b, n, m)


def _dense(lead, rows, K, dtype, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(lead + (rows, K), generator=g, dtype=torch.float64).to(dtype).to(DEV)


def _operands(case, K, dtype, seed=5):
    lead = (case.batch,) if case.A.dim() == 3 else ()
    return _dense(lead, case.m, K, dtype, seed), _dense(lead, case.n, K, dtype, seed + 1)


# ------------------------------------------------------------------------------------------------ running
def _transpose(case, padded=False):
    from torchsparsegradutils_b200._pattern import pattern_of

    patT = pattern_of(case.A).csr.transpose(optimise=padded)
    assert (patT.row_map is not None and patT.padded) == padded
    return patT


def _products(case, B, G, algo=None, padded=False, gb_colmajor=False):
    """(C, grad_A values, grad_B) of sparse_mm, each operator called in this thread."""
    from torchsparsegradutils_b200 import _ops
    from torchsparsegradutils_b200._pattern import pattern_of

    pat = pattern_of(case.A)
    vals = pat.values(case.A)
    C = _ops.spmm(pat.csr, vals, B, algo=algo)
    gA = _ops.sddmm(pat.csr, G, B, pat.out_index, pat.nnz_out, algo=algo)
    patT = _transpose(case, padded)
    b, m, K = case.batch, case.m, G.shape[-1]
    gB = _ops.spmm(patT, vals, G, algo=algo, out_strides=(m * K, 1, m) if gb_colmajor else None)
    if gb_colmajor:
        assert gB.stride() == (m * K, 1, m)  # written by the transposing epilogue
    return [C, gA, gB]


def _across_margins(run, margins=MARGINS):
    """Outputs of run() at every margin: bit-identical (a poisoned element never compares equal); returns margin 0's."""
    from torchsparsegradutils_b200 import _native as nat

    outs = []
    for mg in margins:
        with nat.sm_margin(mg):
            outs.append(run())
    torch.cuda.synchronize()
    for mg, other in zip(margins[1:], outs[1:]):
        for k, (a, b) in enumerate(zip(outs[0], other)):
            assert torch.equal(a, b), f"output {k}: margin {mg} differs from margin {margins[0]}"
    return outs[0]


def _h(t):
    return t.detach().double().cpu().numpy()


def _odt(dtype):
    return np.float64 if dtype == torch.float64 else np.float32  # bf16 against the fp32 oracle of its upcast inputs


def _oracle(case, B, G):
    """fp64-accumulated C, grad_A values (A's storage order) and grad_B, flat over the batch."""
    odt = _odt(B.dtype)
    K = B.shape[-1]
    Bf, Gf = _h(B).reshape(-1, K).astype(odt), _h(G).reshape(-1, K).astype(odt)
    vals = _h(case.A.values() if case.A.layout == torch.sparse_csr else case.A._values()).reshape(-1).astype(odt)
    C = orc.spmm_t(case.cols, case.rows, vals, Bf, case.batch * case.n)  # (A^T)^T B
    gA = orc.sddmm(case.rows, case.cols, Gf, Bf)
    gB = orc.spmm_t(case.rows, case.cols, vals, Gf, case.batch * case.m)
    return [C, gA, gB]


def _flat(got, want):
    g = _h(got)
    return g.reshape(want.shape)


def _check_vs_oracle(outs, refs, dtype, names=("C", "grad_A", "grad_B")):
    for got, want, name in zip(outs, refs, names):
        np.testing.assert_allclose(_flat(got, want), want.astype(np.float64), err_msg=name, **TOL[dtype])


def _pipeline(case, K, dtype, **kw):
    """Sections 1 and 2 for one case: margins agree bit for bit, margin 0 matches the oracle."""
    B, G = _operands(case, K, dtype)
    outs = _across_margins(lambda: _products(case, B, G, **kw))
    _check_vs_oracle(outs, _oracle(case, B, G), dtype)


# --------------------------------------------------------------------------------------------- NaN probes
def _probe_columns(K, dtype):
    """A 16-byte vector boundary, the first element of the last vector and the last column."""
    e = EPV[dtype]
    kv = max(K // e, 1)
    return sorted({min(e * (kv // 2), K - 1), e * (kv - 1) if K % e == 0 else K - 1, K - 1})


def _probe_rows(case, rows_per_item):
    """Row 0 of every item, one in the middle, the last one (flat over the batch)."""
    total = case.batch * rows_per_item
    return sorted({t * rows_per_item for t in range(case.batch)} | {total // 2 + 1, total - 1})


def _probed(X, rows, ks, value=float("nan")):
    """X with `value` at (row, k) for every probe row and column, and X with 0 there instead."""
    K = X.shape[-1]
    flat = X.reshape(-1, K).clone()
    zero = flat.clone()
    for r in rows:
        for k in ks:
            flat[r, k] = value
            zero[r, k] = 0
    return flat.reshape(X.shape), zero.reshape(X.shape)


def _probe_masks(case, Bp, Gp):
    """Where NaN must show: C = A B and grad_B = A^T G through the structure, grad_A[e] where row r_e of G or row c_e
    of B holds a probe."""
    K = Bp.shape[-1]
    nb = np.isnan(_h(Bp).reshape(-1, K))
    ng = np.isnan(_h(Gp).reshape(-1, K))
    mC = (case.S @ nb.astype(np.float64)) > 0
    mB = (case.S.T @ ng.astype(np.float64)) > 0
    mA = ng.any(1)[case.rows] | nb.any(1)[case.cols]
    return [mC, mA, mB]


def _check_probes(outs, refs, masks, dtype, names=("C", "grad_A", "grad_B")):
    for got, want, mask, name in zip(outs, refs, masks, names):
        g = _flat(got, want)
        mask = mask.reshape(want.shape)
        assert mask.any(), f"{name}: no probe reaches this output"
        nan = np.isnan(g)
        assert (nan == mask).all(), (f"{name}: {int((nan & ~mask).sum())} unexpected NaN, "
                                     f"{int((mask & ~nan).sum())} missing NaN")
        np.testing.assert_allclose(g[~mask], want[~mask].astype(np.float64), err_msg=name, **TOL[dtype])


def _nan_probes(poison, case, K, dtype, **kw):
    """Section 3 for one case, at the widest and the narrowest grid."""
    from torchsparsegradutils_b200 import _native as nat

    poison.fill = SENTINEL
    B, G = _operands(case, K, dtype, seed=11)
    ks = _probe_columns(K, dtype)
    Bp, B0 = _probed(B, _probe_rows(case, case.m), ks)
    Gp, G0 = _probed(G, _probe_rows(case, case.n), ks)
    refs = _oracle(case, B0, G0)
    masks = _probe_masks(case, Bp, Gp)
    for mg in PROBE_MARGINS:
        with nat.sm_margin(mg):
            outs = _products(case, Bp, Gp, **kw)
        _check_probes(outs, refs, masks, dtype)


# ------------------------------------------------------------------------------- the margin reaches the launch
PERSISTENT_KERNELS = ("spmm_tile_kernel", "sddmm_tile_kernel", "spmm_merge_kernel", "sddmm_merge_kernel",
                      "spmm_window_kernel", "sddmm_window_kernel")


def test_margin_sets_the_persistent_grid(tmp_path, windows):
    """Kernel records of a CUDA-activity trace carry the launch grid: at most 8 CTAs at margin 147 (the grid is
    ctas_per_sm), at least 148 at margin 0, for every persistent SpMM / SDDMM kernel."""
    from torchsparsegradutils_b200 import _native as nat
    from torchsparsegradutils_b200 import _ops
    from torchsparsegradutils_b200._pattern import pattern_of

    rand = W.uniform_rows_csr(None, 200_000, 200_000, 4, torch.float32, torch.int32, DEV, seed=2)
    sten = W.stencil27_csr(20, torch.float32, torch.int32, DEV, seed=3)
    ops = []
    for A, algo in ((rand, nat.ALGO_AUTO), (rand, nat.ALGO_MERGE), (sten, nat.ALGO_AUTO)):
        pat = pattern_of(A).csr
        B, G = _dense((), A.shape[1], 32, torch.float32, 1), _dense((), A.shape[0], 32, torch.float32, 2)
        ops.append(lambda pat=pat, vals=A.values(), B=B, G=G, algo=algo: (_ops.spmm(pat, vals, B, algo=algo),
                                                                          _ops.sddmm(pat, G, B, None, pat.nnz_total,
                                                                                     algo=algo)))
    assert pattern_of(sten).csr.window is not None
    for mg in (147, 0):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            with nat.sm_margin(mg):
                for op in ops:
                    op()
            torch.cuda.synchronize()
        path = tmp_path / f"margin{mg}.json"
        prof.export_chrome_trace(str(path))
        with open(path) as fh:
            events = json.load(fh)["traceEvents"]
        grids = {}
        for e in events:
            if e.get("cat") != "kernel":
                continue
            hit = [k for k in PERSISTENT_KERNELS if k in e.get("name", "")]
            if hit:
                grids.setdefault(hit[0], []).append(int(e["args"]["grid"][0]))
        assert set(grids) == set(PERSISTENT_KERNELS), sorted(grids)
        for name, gs in grids.items():
            assert all(g <= 8 for g in gs) if mg == 147 else all(g >= 148 for g in gs), (mg, name, gs)


# ------------------------------------------------------------------------------------------ row-tile kernels
def _tile_params():
    """One non-exact and one exact K per lane row in int32, the exact one in int64 (COO indices are int64 in torch:
    the width of its flat CSR is the pattern builder's choice, so COO runs once per K)."""
    out = []
    for layout in ("csr", "coo", "bcsr"):
        for dtype in DTYPES:
            for kv_ragged, kv_exact in LANE_ROWS:
                cases = [(kv_ragged, torch.int32), (kv_exact, torch.int32)]
                if layout != "coo":
                    cases.append((kv_exact, torch.int64))
                for kv, idx in cases:
                    K = kv * EPV[dtype]
                    out.append(pytest.param(layout, dtype, K, idx, id=f"{layout}-{str(dtype)[6:]}-K{K}-{str(idx)[6:]}"))
    return out


@pytest.mark.parametrize("layout,dtype,K,idx", _tile_params())
def test_row_tile_many_tiles_per_cta(layout, dtype, K, idx, poison, tile_kernels):
    """Row-tile SpMM (values staged, or the COO value permutation staged), SDDMM and the transposed SpMM."""
    from torchsparsegradutils_b200 import _native as nat

    case = _layout_case(layout, dtype, idx, seed=K)
    _pipeline(case, K, dtype, algo=nat.ALGO_AUTO)


@pytest.mark.parametrize("dtype,K", [(d, kv * EPV[d]) for d in DTYPES for kv in (6, 32)])
@pytest.mark.parametrize("idx", [torch.int32, torch.int64])
def test_row_tile_staged_and_unstaged_tiles(dtype, K, idx, poison, tile_kernels):
    """Tiles over a row longer than the staging capacity read global memory, their neighbours are staged."""
    from torchsparsegradutils_b200 import _native as nat

    case = _long_rows_case(dtype, idx, seed=K)
    _pipeline(case, K, dtype, algo=nat.ALGO_AUTO)
    _nan_probes(poison, case, K, dtype, algo=nat.ALGO_AUTO)


# ----------------------------------------------------------------------- row-mapped padded transpose, K slices
@pytest.fixture
def padded_transpose(monkeypatch):
    """Every transpose gets the length-sorted, padded layout (conftest already applies it from the first use)."""
    from torchsparsegradutils_b200 import _pattern

    monkeypatch.setattr(_pattern, "_PAD_MIN_NNZ", 0)


@pytest.mark.parametrize("dtype,K", [(d, kv * EPV[d]) for d in DTYPES for kv in (3, 12, 32, 96)])
def test_padded_transpose_rowmap(dtype, K, poison, tile_kernels, padded_transpose):
    """grad_B through tsgu_spmm_csr_rowmap: rows sorted by length, padded with explicit zeros."""
    from torchsparsegradutils_b200 import _native as nat

    case = _layout_case("csr", dtype, torch.int32, seed=K + 1)
    _pipeline(case, K, dtype, algo=nat.ALGO_AUTO, padded=True)
    _nan_probes(poison, case, K, dtype, algo=nat.ALGO_AUTO, padded=True)


@pytest.mark.xfail(strict=True, reason="DESIGN.md section 7 item 8: a padded slot multiplies its explicit 0 with the "
                                       "row's last dense row, so an inf there gives NaN instead of inf")
def test_padded_transpose_inf_is_inf(poison, tile_kernels, padded_transpose):
    from torchsparsegradutils_b200 import _native as nat
    from torchsparsegradutils_b200 import _ops
    from torchsparsegradutils_b200._pattern import pattern_of

    case = _layout_case("csr", torch.float32, torch.int32, seed=3)
    A, K = case.A, 32
    T = case.S.T.tocsr()  # rows of A^T: the columns of A, their entries in ascending row order
    lens = np.diff(T.indptr)
    j = int(np.flatnonzero(lens % 4)[0])  # a transposed row with padding
    r = int(T.indices[T.indptr[j + 1] - 1])  # its last real column: the dense row the padding repeats
    _, G = _operands(case, K, torch.float32)
    Gi, _ = _probed(G, [r], [5], value=float("inf"))
    gB = _ops.spmm(_transpose(case, padded=True), pattern_of(A).values(A), Gi, algo=nat.ALGO_AUTO)[0]
    readers = T.indices[T.indptr[j]:T.indptr[j + 1]]
    assert r in readers
    # every A value is positive: a column of A that stores row r gets +inf in grad_B[:, 5]
    want = np.flatnonzero(np.asarray(case.S[r].todense()).ravel())
    assert torch.isposinf(gB[torch.from_numpy(want).to(DEV), 5]).all()


def test_k_sliced_forward(poison, tile_kernels):
    """Uniform rows whose dense operand exceeds 60 % of L2 (400 000 x 64 fp32 = 102 MB): the forward SpMM runs as
    two K = 32 slices (TSGU_ALGO_FLAG_KSLICE), each a persistent launch over the whole pattern."""
    from torchsparsegradutils_b200 import _native as nat
    from torchsparsegradutils_b200 import _ops
    from torchsparsegradutils_b200._pattern import pattern_of

    n = m = 400_000
    K, dtype = 64, torch.float32
    A = W.uniform_rows_csr(None, n, m, 4, dtype, torch.int32, DEV, seed=9)
    case = _host_case(A)
    pat = pattern_of(A).csr
    assert pat.uniform_rows and pat.window is None

    def forward(B):
        before = nat.launch_count()
        C = _ops.spmm(pat, A.values(), B)
        assert nat.launch_count() - before == 2  # one launch per K slice
        return [C]

    B, _ = _operands(case, K, dtype)
    outs = _across_margins(lambda: forward(B), margins=(0, 120))  # 28 SMs: 1.6 M entries, still many tiles per CTA
    _check_vs_oracle(outs, _oracle(case, B, B[:n])[:1], dtype, names=("C",))
    poison.fill = SENTINEL
    ks = [0, 31, 32, 63]  # either side of the slice boundary
    Bp, B0 = _probed(B, [0, m // 2 + 1, m - 1], ks)
    refs = _oracle(case, B0, B0[:n])[:1]
    masks = _probe_masks(case, Bp, Bp[:n])[:1]
    for mg in (0, 120):
        with nat.sm_margin(mg):
            outs = forward(Bp)
        _check_probes(outs, refs, masks, dtype, names=("C",))


# ------------------------------------------------------------------------------------------- merge-path kernels
@pytest.mark.parametrize("dtype,K", [(d, kv * EPV[d]) for d in DTYPES for kv in (6, 32)])
@pytest.mark.parametrize("idx", [torch.int32, torch.int64])
def test_merge_path_many_tiles_per_cta(dtype, K, idx, poison, monkeypatch):
    from torchsparsegradutils_b200 import _native as nat
    from torchsparsegradutils_b200._pattern import pattern_of

    monkeypatch.setenv("TSGU_B200_ALGO", "merge")
    case = _skewed_case(dtype, idx, seed=K)
    assert pattern_of(case.A).csr.algo == nat.ALGO_MERGE and _transpose(case).algo == nat.ALGO_MERGE
    _pipeline(case, K, dtype)
    _nan_probes(poison, case, K, dtype)


# ------------------------------------------------------------------------------------------ column-window kernels
def _banded(n, m, offsets, seed):
    r = np.arange(n)[:, None]
    c = r + np.array(sorted(offsets))[None, :]
    ok = (c >= 0) & (c < m)
    rows, cols = np.broadcast_to(r, c.shape)[ok], c[ok]
    return rows.astype(np.int64), cols.astype(np.int64)


def _window_case(kind, dtype):
    if kind == "stencil":
        return _host_case(W.stencil27_csr(20, dtype, torch.int32, DEV, seed=3))
    if kind == "banded":
        offs = [-120, -119, -61, -60, -59, -1, 0, 1, 2, 59, 60, 61, 119, 120, 121]
        return _csr_case(*_banded(3000, 2800, offs, 5), 3000, 2800, dtype, torch.int32, seed=5)
    As = [W.stencil27_csr(14, dtype, torch.int32, DEV, seed=s) for s in (1, 2)]
    A = torch.sparse_csr_tensor(torch.stack([a.crow_indices() for a in As]), torch.stack([a.col_indices() for a in As]),
                                torch.stack([a.values() for a in As]), (2,) + tuple(As[0].shape))
    return _host_case(A)


@pytest.mark.parametrize("K,dtype", [(16, torch.float32), (32, torch.float32), (64, torch.float32),
                                     (32, torch.bfloat16), (64, torch.bfloat16), (128, torch.bfloat16)])
@pytest.mark.parametrize("kind", ["stencil", "banded", "batched"])
def test_window_many_tiles_per_cta(kind, K, dtype, poison, windows):
    """Window SpMM / SDDMM / transposed SpMM, grad_B written column-major by the transposing epilogue."""
    from torchsparsegradutils_b200._pattern import pattern_of

    case = _window_case(kind, dtype)
    assert pattern_of(case.A).csr.window is not None and _transpose(case).window is not None

    def run(B, G):
        C, gA, gB = _products(case, B, G)
        return [C, gA, gB, _products(case, B, G, gb_colmajor=True)[2]]

    B, G = _operands(case, K, dtype)
    outs = _across_margins(lambda: run(B, G))
    refs = _oracle(case, B, G)
    _check_vs_oracle(outs, refs + refs[2:], dtype, names=("C", "grad_A", "grad_B", "grad_B column-major"))
    assert torch.equal(outs[2], outs[3])
    _nan_probes(poison, case, K, dtype)
    _nan_probes(poison, case, K, dtype, gb_colmajor=True)


# ------------------------------------------------------------------------------------------- triangular solve
TRI_FLAGS = [pytest.param(False, False, id="lower"), pytest.param(True, False, id="upper"),
             pytest.param(False, True, id="lower-transposed")]


@pytest.mark.parametrize("idx", [torch.int32, torch.int64])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("upper,transpose", TRI_FLAGS)
def test_triangular_solve_many_rows_per_warp(upper, transpose, dtype, idx, poison):
    """Levels + plan + solve at every margin: equal level counts, bit-identical x, status 0, and agreement with an
    fp64 dense solve.  K = 1, 4: entry mode; 6, 129: scalar; 8: vector; 260 (fp32) / 130 (fp64): vector mode in
    several k0 passes with a partial last one."""
    from torchsparsegradutils_b200 import sparse_triangular_solve
    from torchsparsegradutils_b200._pattern import pattern_of
    from torchsparsegradutils_b200.triangular_solve import solve_plan, solve_status

    n = 20_000
    L = W.random_lower_csr(None, n, 6, torch.float64, idx, DEV, seed=6)
    if upper:
        U = sp.csr_matrix((_h(L.values()), L.col_indices().cpu().numpy(), L.crow_indices().cpu().numpy()),
                          shape=(n, n)).T.tocsr()
        U.sort_indices()
        A64 = torch.sparse_csr_tensor(torch.from_numpy(U.indptr.astype(np.int64)).to(idx),
                                      torch.from_numpy(U.indices.astype(np.int64)).to(idx),
                                      torch.from_numpy(U.data), (n, n)).to(DEV)
    else:
        A64 = L
    A = torch.sparse_csr_tensor(A64.crow_indices(), A64.col_indices(), A64.values().to(dtype), (n, n))
    opA = A.to(torch.float64).to_dense()
    opA = opA.t() if transpose else opA
    solves_upper = upper != transpose
    Ks = [1, 4, 6, 8, 129, 260 if dtype == torch.float32 else 130]
    Bs = [_dense((), n, K, dtype, 20 + K) for K in Ks]
    ref = torch.linalg.solve_triangular(opA, torch.cat(Bs, 1).double(), upper=solves_upper).cpu()
    del opA
    csr = pattern_of(A, unique=True).csr
    tol = dict(rtol=1e-10, atol=1e-12) if dtype == torch.float64 else dict(rtol=1e-4, atol=1e-5)

    def run():
        csr.extras.clear()  # a fresh level analysis and plan under this margin
        xs = [sparse_triangular_solve(A, B, upper=upper, transpose=transpose) for B in Bs]
        assert solve_status(DEV) == 0
        return [torch.tensor(solve_plan(A, upper, transpose).levels)] + xs

    outs = _across_margins(run)
    assert int(outs[0]) > 1
    torch.testing.assert_close(torch.cat(outs[1:], 1).double().cpu(), ref, **tol)
