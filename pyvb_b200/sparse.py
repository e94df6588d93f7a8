"""Host side of the sparse-observation path: input normalisation and the layouts the CSR kernels read.

A sparse input matrix means: every STORED entry is an observation (a stored zero is an observed 0.0), everything not
stored is missing.  This module turns scipy.sparse matrices / arrays (any format) and torch sparse CSR tensors into

    CSR       indptr int64 [N + 1], indices int32 (sorted within a row), values float64        (the Z step, K1-csr)
    blocked   colptr int64 [nblk * D + 1], rows int32, vals float64: the same entries column-major within each block of
    CSC       `rows_per_block` consecutive rows, blocks one after the other                     (the statistics, K3-csc)
    xcache    float64 [cnt (D) | colsumX (D) | sum x^2 | number of stored entries]              (stats_reduce's X-only sums)

Per-entry observation weights (PlateEngine(..., weights=...)) travel with the values: one float64 per stored entry, in CSR order
and through the same permutation into the blocked CSC (`wts`); the X-only sums then become [sum s | sum s x | sum s x^2 | number
of entries with s > 0].

(include/pyvb_b200.h, "sparse observations").  Everything here is construction-time plumbing on torch / numpy: it runs
without a GPU (on the CPU, or on the device where the input already lives) and is not on the per-sweep path.
"""
import collections
import math

import numpy as np
import torch

CSR = collections.namedtuple("CSR", "indptr indices values N D")
BlockedCSC = collections.namedtuple("BlockedCSC", "colptr rows vals nblk rows_per_block wts", defaults=(None,))


def is_sparse(X):
    """True for a scipy.sparse matrix / array or a torch tensor with a sparse layout."""
    if isinstance(X, torch.Tensor):
        return X.layout != torch.strided
    try:
        import scipy.sparse as sp
    except ImportError:  # pragma: no cover
        return False
    return sp.issparse(X)


def _coo_of(X, device):
    """(row int64, col int64, values float64, N, D) of the stored entries, in stored order, duplicates kept."""
    if isinstance(X, torch.Tensor):
        if X.layout != torch.sparse_csr:
            raise ValueError("sparse torch input must have the sparse CSR layout (tensor.to_sparse_csr()); got %s" % X.layout)
        if X.dim() != 2:
            raise ValueError("sparse input must be a matrix, got %d dimensions" % X.dim())
        if X.is_complex():
            raise ValueError("sparse input must be real")
        dev = X.device if device is None else torch.device(device)
        N, D = int(X.shape[0]), int(X.shape[1])
        crow = X.crow_indices().to(device=dev, dtype=torch.int64)
        col = X.col_indices().to(device=dev, dtype=torch.int64)
        val = X.values().to(device=dev, dtype=torch.float64)
        row = torch.repeat_interleave(torch.arange(N, device=dev, dtype=torch.int64), crow[1:] - crow[:-1])
        return row, col, val, N, D
    import scipy.sparse as sp
    if not sp.issparse(X):
        raise ValueError("not a sparse matrix")
    if X.ndim != 2:
        raise ValueError("sparse input must be a matrix")
    if np.iscomplexobj(X.dtype.type(0)):
        raise ValueError("sparse input must be real")
    # .tocoo() keeps duplicates and stored zeros (.tocsr() of a COO matrix would silently sum duplicates)
    coo = X.tocoo()
    N, D = int(X.shape[0]), int(X.shape[1])
    dev = torch.device("cpu") if device is None else torch.device(device)
    row = torch.as_tensor(np.asarray(coo.row, dtype=np.int64)).to(dev)
    col = torch.as_tensor(np.asarray(coo.col, dtype=np.int64)).to(dev)
    val = torch.as_tensor(np.asarray(coo.data, dtype=np.float64)).to(dev)
    return row, col, val, N, D


def to_csr(X, device=None):
    """Normalise and validate a sparse input into a CSR (row-sorted, column indices sorted within each row).

    Raises ValueError for a NaN / Inf stored value, a duplicate (row, column) entry and a column index outside [0, D).
    device: where the arrays are built and returned (default: the tensor's device, or the CPU for scipy input)."""
    row, col, val, N, D = _coo_of(X, device)
    if D < 1 or N < 0:
        raise ValueError("sparse input needs at least one column")
    if D >= 2 ** 31 or N >= 2 ** 31:
        raise ValueError("sparse input: N and D must be below 2^31 (int32 indices)")
    nnz = int(val.numel())
    if nnz:
        if not bool(torch.isfinite(val).all()):
            raise ValueError("sparse input has a NaN or Inf stored value (a missing entry is one that is not stored)")
        if bool(((col < 0) | (col >= D)).any()):
            raise ValueError("sparse input has a column index outside [0, %d)" % D)
        if bool(((row < 0) | (row >= N)).any()):
            raise ValueError("sparse input has a row index outside [0, %d)" % N)
        key = row * D + col
        if nnz > 1 and not bool((key[1:] >= key[:-1]).all()):
            key, perm = torch.sort(key, stable=True)
            row, col, val = row[perm], col[perm], val[perm]
        if nnz > 1 and bool((key[1:] == key[:-1]).any()):
            raise ValueError("sparse input has a duplicate (row, column) entry")
    counts = torch.bincount(row, minlength=N) if nnz else torch.zeros(N, dtype=torch.int64, device=row.device)
    indptr = torch.zeros(N + 1, dtype=torch.int64, device=row.device)
    if N:
        indptr[1:] = torch.cumsum(counts, 0)
    return CSR(indptr.contiguous(), col.to(torch.int32).contiguous(), val.contiguous(), N, D)


def weights_csr(W, csr):
    """The per-entry weights of the sparse observations `csr` as a float64 array in CSR order.  W: a sparse matrix / tensor
    (any format to_csr accepts) whose stored pattern is exactly that of the observations.  Raises ValueError for a different
    shape or pattern and for a negative or non-finite weight."""
    if not is_sparse(W):
        raise ValueError("weights of sparse observations must be a sparse matrix with the observations' stored pattern")
    row, col, val, N, D = _coo_of(W, csr.indptr.device)
    if (N, D) != (csr.N, csr.D):
        raise ValueError("weights have shape %s, the observations %s" % ((N, D), (csr.N, csr.D)))
    if val.numel() and not bool(torch.isfinite(val).all()):
        raise ValueError("weights must be finite on the observed entries")
    w = to_csr(W, device=csr.indptr.device)
    if not (torch.equal(w.indptr, csr.indptr) and torch.equal(w.indices, csr.indices)):
        raise ValueError("weights must store exactly the entries the observations store (same sparse pattern)")
    if w.values.numel() and bool((w.values < 0).any()):
        raise ValueError("weights must be >= 0 on the observed entries")
    return w.values


def block_csc(csr, rows_per_block, weights=None):
    """The row-blocked column-major copy of `csr`: rows cut into blocks of `rows_per_block` (the last may hold fewer);
    within block b the entries of column d are colptr[b*D + d] .. colptr[b*D + d + 1], rows increasing.  weights (optional,
    CSR order): carried through the same permutation into `wts`."""
    N, D = csr.N, csr.D
    R = max(1, int(rows_per_block))
    nblk = max(1, (N + R - 1) // R)
    dev = csr.indptr.device
    nnz = int(csr.values.numel())
    if nnz == 0:
        empty = torch.zeros(0, dtype=torch.float64, device=dev)
        return BlockedCSC(torch.zeros(nblk * D + 1, dtype=torch.int64, device=dev),
                          torch.zeros(0, dtype=torch.int32, device=dev), empty, nblk, R,
                          None if weights is None else empty)
    row = torch.repeat_interleave(torch.arange(N, device=dev, dtype=torch.int64), csr.indptr[1:] - csr.indptr[:-1])
    key = (row // R) * D + csr.indices.to(torch.int64)
    # the CSR order is (row, column): a stable sort on (block, column) keeps the rows increasing within a column
    key, perm = torch.sort(key, stable=True)
    counts = torch.bincount(key, minlength=nblk * D)
    colptr = torch.zeros(nblk * D + 1, dtype=torch.int64, device=dev)
    colptr[1:] = torch.cumsum(counts, 0)
    return BlockedCSC(colptr, row[perm].to(torch.int32).contiguous(), csr.values[perm].contiguous(), nblk, R,
                      None if weights is None else weights[perm].contiguous())


def column_sums(csr, weights=None):
    """Per column: stored entries, their sum and their sum of squares (float64 numpy arrays of length D); with weights (CSR
    order) the weighted sums sum s, sum s x, sum s x^2.  Sequential sums in stored order (numpy bincount): the same input
    always gives the same bits."""
    D = csr.D
    col = csr.indices.cpu().numpy().astype(np.int64, copy=False)
    val = csr.values.cpu().numpy()
    if weights is None:
        cnt = np.bincount(col, minlength=D).astype(np.float64)
        sv = val
    else:
        s = weights.cpu().numpy()
        cnt = np.bincount(col, weights=s, minlength=D)
        sv = s * val
    colx = np.bincount(col, weights=sv, minlength=D)
    colxx = np.bincount(col, weights=sv * val, minlength=D)
    return cnt, colx, colxx


def x_cache(csr, weights=None):
    """[cnt (D) | colsumX (D) | sum x^2 | entries] as a float64 CPU tensor, from column_sums; sum x^2 exactly rounded over its
    per-column parts.  entries: the stored entries, or with weights those of positive weight."""
    cnt, colx, colxx = column_sums(csr, weights)
    n = csr.values.numel() if weights is None else int((weights > 0).sum())
    out = np.concatenate([cnt, colx, [math.fsum(colxx.tolist()), float(n)]])
    return torch.as_tensor(out, dtype=torch.float64)


def densify(csr):
    """Dense float64 numpy copy with NaN where nothing is stored (tests, and the dense side of comparisons)."""
    out = np.full((csr.N, csr.D), np.nan)
    indptr = csr.indptr.cpu().numpy()
    rows = np.repeat(np.arange(csr.N), np.diff(indptr))
    out[rows, csr.indices.cpu().numpy().astype(np.int64)] = csr.values.cpu().numpy()
    return out
