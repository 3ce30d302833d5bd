"""GPU: what ``_pattern.pattern_of`` gives an operator for each layout of A -- the host reads a new pattern costs, and
A's values in the order the kernels index them."""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
N = 50


def _operands():
    """Small integer-valued matrices (sums of duplicates are exact), well below the column-window size thresholds."""
    g = torch.Generator().manual_seed(0)
    mask = (torch.rand(N, N, generator=g) < 0.1) | torch.eye(N, dtype=torch.bool)  # one pattern: batched CSR needs it
    D = mask * torch.randint(1, 5, (3, N, N), generator=g).double()

    def uncoalesced(ind, extra, shape):
        """`ind` plus `extra` duplicated coordinates, shuffled; values 1, 2, 3, ..."""
        ind = torch.cat([ind, ind[:, :extra]], 1)[:, torch.randperm(ind.shape[1] + extra, generator=g)]
        vals = torch.arange(1, ind.shape[1] + 1, dtype=torch.float64)
        return torch.sparse_coo_tensor(ind.to(DEV), vals.to(DEV), shape)

    return {
        "csr": D[0].to_sparse_csr().to(DEV),
        "csr_batched": D.to_sparse_csr().to(DEV),
        "coo_coalesced": D[0].to_sparse().to(DEV),
        "coo_uncoalesced": uncoalesced(D[0].to_sparse()._indices(), 7, (N, N)),
        "coo_batched_dups": uncoalesced(D.to_sparse()._indices(), 5, (3, N, N)),
        "coo_batched_shuffled": uncoalesced(D.to_sparse()._indices(), 0, (3, N, N)),
    }


@pytest.fixture
def host_reads(monkeypatch):
    from torchsparsegradutils_b200 import _native as nat

    calls = [0]
    orig = nat.host_read

    def counting(t):
        calls[0] += 1
        return orig(t)

    monkeypatch.setattr(nat, "host_read", counting)
    return calls


# one read (longest row + window verdict) per new single-matrix pattern; none for a small batch, whose kernel family
# does not depend on its rows; one more for the duplicate check of uncoalesced COO that coalesces
@pytest.mark.parametrize("name,unique,reads", [
    ("csr", False, 1), ("csr_batched", False, 0), ("coo_coalesced", False, 1), ("coo_uncoalesced", False, 1),
    ("coo_uncoalesced", True, 2), ("coo_batched_dups", False, 1), ("coo_batched_shuffled", False, 1),
])
def test_host_reads_of_a_new_pattern(name, unique, reads, host_reads):
    from torchsparsegradutils_b200 import clear_pattern_cache
    from torchsparsegradutils_b200._pattern import pattern_of

    A = _operands()[name]
    clear_pattern_cache()
    host_reads[0] = 0
    pattern_of(A, unique)
    assert host_reads[0] == reads
    pattern_of(A, unique)
    assert host_reads[0] == reads  # a cache hit reads nothing
    clear_pattern_cache()


def test_host_reads_of_a_transpose_and_a_solve_plan(host_reads):
    from torchsparsegradutils_b200 import clear_pattern_cache
    from torchsparsegradutils_b200._pattern import csr_pattern
    from torchsparsegradutils_b200.triangular_solve import solve_plan

    A = _operands()["csr"]
    clear_pattern_cache()
    pat = csr_pattern(A)
    for build, reads in ((pat.transpose, 1), (lambda: solve_plan(A, upper=False), 1),
                         (lambda: solve_plan(A, upper=False, transpose=True), 1)):
        host_reads[0] = 0
        build()
        assert host_reads[0] == reads
    clear_pattern_cache()


@pytest.mark.parametrize("name,unique", [
    ("csr", False), ("csr_batched", False), ("coo_coalesced", False), ("coo_uncoalesced", False),
    ("coo_uncoalesced", True), ("coo_batched_dups", False), ("coo_batched_shuffled", False),
])
def test_operand_values_in_kernel_order(name, unique):
    from torchsparsegradutils_b200 import clear_pattern_cache
    from torchsparsegradutils_b200._pattern import pattern_of, sparse_values

    A = _operands()[name]
    clear_pattern_cache()
    pat = pattern_of(A, unique)
    vals = pat.values(A)
    assert vals.is_contiguous() and vals.data_ptr() % 16 == 0
    summed = getattr(pat, "seg", None) is not None
    assert summed == (name == "coo_batched_dups" or unique)
    # duplicates summed onto the unique pattern, else A's storage order (read through csr.perm where there is one)
    want = A.coalesce()._values() if summed else sparse_values(A)
    assert torch.equal(vals.reshape(-1), want.reshape(-1))
    assert (pat.csr.perm is not None) == (name in ("coo_uncoalesced", "coo_batched_shuffled") and not unique)
    csr = pat.csr
    if csr.rowptr.dim() == 1:  # the flat CSR our builders emit: the kernels' view of A is A itself
        lens = (csr.rowptr[1:] - csr.rowptr[:-1]).long()
        rows = torch.repeat_interleave(torch.arange(csr.batch * csr.n, device=DEV), lens)
        v = vals.reshape(-1) if csr.perm is None else vals.reshape(-1)[csr.perm.long()]
        dense = torch.zeros(csr.batch * csr.n, csr.m, dtype=vals.dtype, device=DEV)
        dense.index_put_((rows, csr.colind.long()), v, accumulate=True)
        assert torch.equal(dense.reshape(A.shape), A.to_dense())
    clear_pattern_cache()
