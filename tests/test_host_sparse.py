"""Host side of the sparse-observation path (pyvb_b200/sparse.py), on the CPU: input normalisation and validation, the
row-blocked column-major layout of the statistics kernel and the X-only cache.  No GPU is needed."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from pyvb_b200 import sparse as S


def _rand_sparse(N, D, density, seed=0, dyadic=False):
    rng = np.random.RandomState(seed)
    A = sp.random(N, D, density=density, format="coo", random_state=rng)
    if dyadic:                              # multiples of 1/8 below 2^10: every sum of them is exact in FP64
        A.data = np.round(rng.randn(A.nnz) * 64.0) / 8.0
    else:
        A.data = rng.randn(A.nnz)
    return A


def _triples(csr):
    indptr = csr.indptr.numpy()
    rows = np.repeat(np.arange(csr.N), np.diff(indptr))
    return rows, csr.indices.numpy().astype(np.int64), csr.values.numpy()


def _check_csr_against(csr, A):
    """csr holds exactly the stored entries of A, row-major with sorted columns."""
    A = sp.coo_matrix(A)
    assert csr.N == A.shape[0] and csr.D == A.shape[1]
    assert csr.indptr.dtype == torch.int64 and csr.indices.dtype == torch.int32 and csr.values.dtype == torch.float64
    r, c, v = _triples(csr)
    key = r * csr.D + c
    assert np.all(np.diff(key) > 0)                              # sorted, no duplicates
    order = np.lexsort((A.col, A.row))
    np.testing.assert_array_equal(r, A.row[order])
    np.testing.assert_array_equal(c, A.col[order])
    np.testing.assert_array_equal(v, A.data[order])


@pytest.mark.parametrize("fmt", ["csr", "csc", "coo", "lil", "dok", "bsr"])
def test_scipy_formats(fmt):
    A = _rand_sparse(37, 23, 0.2, seed=1)
    csr = S.to_csr(A.asformat(fmt))
    _check_csr_against(csr, A)


def test_scipy_sparse_array_and_torch_csr():
    A = _rand_sparse(50, 31, 0.1, seed=2)
    _check_csr_against(S.to_csr(sp.csr_array(A)), A)
    t = torch.sparse_csr_tensor(torch.as_tensor(A.tocsr().indptr, dtype=torch.int64),
                                torch.as_tensor(A.tocsr().indices, dtype=torch.int64),
                                torch.as_tensor(A.tocsr().data), size=A.shape)
    _check_csr_against(S.to_csr(t), A)
    assert S.is_sparse(t) and S.is_sparse(A) and not S.is_sparse(A.toarray()) and not S.is_sparse(torch.zeros(2, 2))


def test_unsorted_columns_within_rows():
    # a CSR whose column indices are not sorted within a row (allowed by scipy and torch)
    indptr = np.array([0, 3, 3, 5])
    indices = np.array([4, 0, 2, 3, 1])
    data = np.array([1.0, 2.0, 3.0, 4.0, 5.0])
    A = sp.csr_matrix((data, indices, indptr), shape=(3, 5))
    csr = S.to_csr(A)
    np.testing.assert_array_equal(csr.indptr.numpy(), [0, 3, 3, 5])
    np.testing.assert_array_equal(csr.indices.numpy(), [0, 2, 4, 1, 3])
    np.testing.assert_array_equal(csr.values.numpy(), [2.0, 3.0, 1.0, 5.0, 4.0])


def test_stored_zeros_are_observations():
    A = sp.csr_matrix((np.array([0.0, 1.5, 0.0]), np.array([0, 2, 1]), np.array([0, 2, 2, 3])), shape=(3, 3))
    csr = S.to_csr(A)
    assert csr.values.numel() == 3
    X = S.densify(csr)
    assert X[0, 0] == 0.0 and X[2, 1] == 0.0 and np.isnan(X[1]).all()
    xc = S.x_cache(csr).numpy()
    np.testing.assert_array_equal(xc[:3], [1.0, 1.0, 1.0])       # cnt counts the stored zeros
    assert xc[-1] == 3.0


def test_rejects_duplicates():
    coo = sp.coo_matrix((np.array([1.0, 2.0]), (np.array([1, 1]), np.array([3, 3]))), shape=(4, 5))
    with pytest.raises(ValueError, match="duplicate"):
        S.to_csr(coo)
    csr = sp.csr_matrix((np.array([1.0, 2.0]), np.array([2, 2]), np.array([0, 2])), shape=(1, 4))
    with pytest.raises(ValueError, match="duplicate"):
        S.to_csr(csr)
    t = torch.sparse_csr_tensor(torch.tensor([0, 2]), torch.tensor([1, 1]), torch.tensor([1.0, 2.0], dtype=torch.float64),
                                size=(1, 3))
    with pytest.raises(ValueError, match="duplicate"):
        S.to_csr(t)


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
def test_rejects_non_finite(bad):
    A = sp.csr_matrix((np.array([1.0, bad]), np.array([0, 1]), np.array([0, 1, 2])), shape=(2, 2))
    with pytest.raises(ValueError, match="NaN or Inf"):
        S.to_csr(A)


def test_rejects_out_of_range_columns():
    t = torch.sparse_csr_tensor(torch.tensor([0, 1]), torch.tensor([7]), torch.tensor([1.0], dtype=torch.float64),
                                size=(1, 8), check_invariants=False)
    t2 = torch.sparse_csr_tensor(torch.tensor([0, 1]), torch.tensor([8]), torch.tensor([1.0], dtype=torch.float64),
                                 size=(1, 8), check_invariants=False)
    assert S.to_csr(t).indices.tolist() == [7]
    with pytest.raises(ValueError, match="outside"):
        S.to_csr(t2)
    t3 = torch.sparse_csr_tensor(torch.tensor([0, 1]), torch.tensor([-1]), torch.tensor([1.0], dtype=torch.float64),
                                 size=(1, 8), check_invariants=False)
    with pytest.raises(ValueError, match="outside"):
        S.to_csr(t3)


def test_rejects_other_torch_layouts():
    with pytest.raises(ValueError, match="CSR"):
        S.to_csr(torch.eye(3, dtype=torch.float64).to_sparse())


def test_empty_rows_columns_and_single_row():
    A = sp.csr_matrix((np.array([2.0, -1.0]), np.array([1, 4]), np.array([0, 0, 2, 2])), shape=(3, 6))
    csr = S.to_csr(A)
    np.testing.assert_array_equal(csr.indptr.numpy(), [0, 0, 2, 2])
    X = S.densify(csr)
    assert np.isnan(X[0]).all() and np.isnan(X[2]).all() and np.isnan(X[:, 0]).all()
    one = S.to_csr(sp.csr_matrix(np.array([[0.0, 3.0, 0.0]])))      # N = 1 (scipy stores no zeros here)
    assert one.N == 1 and one.indices.tolist() == [1]
    empty = S.to_csr(sp.csr_matrix((4, 3)))
    assert empty.values.numel() == 0 and empty.indptr.tolist() == [0] * 5
    b = S.block_csc(empty, 2)
    assert b.nblk == 2 and b.colptr.numel() == 2 * 3 + 1 and int(b.colptr.max()) == 0
    np.testing.assert_array_equal(S.x_cache(empty).numpy(), np.zeros(2 * 3 + 2))


def _check_blocked(csr, b):
    """Every (row, column, value) of csr appears exactly once in the blocked layout, in its block and column, rows
    increasing within a column."""
    N, D = csr.N, csr.D
    R = b.rows_per_block
    assert b.nblk == max(1, -(-N // R))
    cp = b.colptr.numpy()
    assert cp.shape == (b.nblk * D + 1,) and cp[0] == 0 and cp[-1] == csr.values.numel() and np.all(np.diff(cp) >= 0)
    rows, vals = b.rows.numpy().astype(np.int64), b.vals.numpy()
    got = []
    for item in range(b.nblk * D):
        blk, d = divmod(item, D)
        rr = rows[cp[item]:cp[item + 1]]
        assert np.all(np.diff(rr) > 0)
        assert np.all(rr // R == blk)
        got += [(int(r), d, float(v)) for r, v in zip(rr, vals[cp[item]:cp[item + 1]])]
    r, c, v = _triples(csr)
    assert sorted(got) == sorted(zip(r.tolist(), c.tolist(), v.tolist()))


@pytest.mark.parametrize("N,D,density,R", [(40, 7, 0.3, 40), (40, 7, 0.3, 1000), (40, 7, 0.3, 9), (41, 13, 0.1, 4),
                                           (1, 5, 0.6, 1), (64, 3, 0.02, 8)])
def test_blocked_csc_reproduces_entries(N, D, density, R):
    csr = S.to_csr(_rand_sparse(N, D, density, seed=N + D))
    b = S.block_csc(csr, R)
    _check_blocked(csr, b)


def test_blocked_csc_with_empty_blocks():
    # rows 0..3 and 12..15 hold entries, rows 4..11 none: with 4 rows per block, blocks 1 and 2 are empty
    dense = np.zeros((16, 5))
    dense[:4] = np.arange(20).reshape(4, 5) + 1.0
    dense[12:] = -(np.arange(20).reshape(4, 5) + 1.0)
    csr = S.to_csr(sp.csr_matrix(dense))
    b = S.block_csc(csr, 4)
    assert b.nblk == 4
    cp = b.colptr.numpy()
    assert cp[1 * 5] == cp[3 * 5]                                 # nothing in blocks 1 and 2
    _check_blocked(csr, b)


@pytest.mark.parametrize("N,D,density", [(200, 37, 0.1), (1, 9, 0.7), (300, 64, 0.6)])
def test_x_cache_matches_densified(N, D, density):
    csr = S.to_csr(_rand_sparse(N, D, density, seed=5, dyadic=True))
    X = S.densify(csr)
    O = ~np.isnan(X)
    X0 = np.where(O, X, 0.0)
    xc = S.x_cache(csr).numpy()
    assert xc.shape == (2 * D + 2,)
    np.testing.assert_array_equal(xc[:D], O.sum(0))
    np.testing.assert_array_equal(xc[D:2 * D], X0.sum(0))         # exact: dyadic values, every partial sum representable
    assert xc[2 * D] == (X0 ** 2).sum()
    assert xc[2 * D + 1] == O.sum()


def test_x_cache_is_reproducible_on_real_values():
    csr = S.to_csr(_rand_sparse(500, 50, 0.2, seed=9))
    a, b = S.x_cache(csr).numpy(), S.x_cache(csr).numpy()
    assert a.tobytes() == b.tobytes()
    X = S.densify(csr)
    X0 = np.where(np.isnan(X), 0.0, X)
    np.testing.assert_allclose(a[50:100], X0.sum(0), rtol=1e-13, atol=1e-13)
