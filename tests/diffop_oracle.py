"""NumPy restatement of the differential operator (pygsp/graphs/difference.py, graph.py:962-1029)
and of the exact operation order of its products, in the input's dtype.

  edge_list   : get_edge_list() of a CSR adjacency.
  diffop      : the CSC arrays of D, each value computed in float64 by the reference's operation
                sequence and rounded once to the requested dtype.
  exact_spmm  : y = A x for CSR arrays (A, x in one dtype): every output starts at +0.0 and adds
                the products in stored order, multiply and add rounded separately -- SciPy's
                csr_matvec(s) order.  grad is exact_spmm over D's CSC arrays (the CSR of D^T),
                div over D.tocsr() (edge ids ascending in a row, csc_matvec(s)'s order).
"""
import numpy as np
from scipy import sparse


def edge_list(W, directed):
    """(sources, targets, weights): all stored entries of W row-major if directed, else the
    upper triangle (diagonal included)."""
    W = sparse.csr_matrix(W)
    rows = np.repeat(np.arange(W.shape[0], dtype=np.int32), np.diff(W.indptr))
    keep = np.ones(W.nnz, bool) if directed else W.indices >= rows
    return rows[keep], W.indices[keep].astype(np.int32), W.data[keep]


def diffop(n, sources, targets, weights, dw, lap_type, directed, dtype=np.float64):
    """CSC arrays (indptr, indices, data) of the N x Ne differential operator."""
    s = np.asarray(sources, np.int64)
    t = np.asarray(targets, np.int64)
    w = np.asarray(weights, np.float64)
    dw = np.asarray(dw, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        if lap_type == "combinatorial":
            vt = np.sqrt(w)
            vs = -vt
        elif lap_type == "normalized":
            vs = -np.sqrt(w / dw[s])
            vt = np.sqrt(w / dw[t])
        else:
            raise ValueError(lap_type)
        if directed:
            vs = vs / np.sqrt(2)
            vt = vt / np.sqrt(2)
    keep = s != t                                   # a self-loop's entries cancel exactly
    counts = np.where(keep, 2, 0)
    indptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    s_first = s < t
    first_idx = np.where(s_first, s, t)[keep]
    second_idx = np.where(s_first, t, s)[keep]
    first_val = np.where(s_first, vs, vt)[keep].astype(dtype)
    second_val = np.where(s_first, vt, vs)[keep].astype(dtype)
    indices = np.stack([first_idx, second_idx], axis=1).ravel().astype(np.int32)
    data = np.stack([first_val, second_val], axis=1).ravel()
    return indptr, indices, data


def exact_spmm(indptr, indices, data, x):
    """A x in A's dtype, in stored order from +0.0 without contraction.  Vectorised by incidence
    rank: pass r adds the r-th entry of every row that has one."""
    indptr = np.asarray(indptr, np.int64)
    dt = data.dtype
    x = np.asarray(x, dt)
    X = x.reshape(x.shape[0], int(np.prod(x.shape[1:], dtype=np.int64)))
    n = indptr.size - 1
    out = np.zeros((n, X.shape[1]), dt)
    lengths = np.diff(indptr)
    for r in range(int(lengths.max()) if n else 0):
        rows = np.flatnonzero(lengths > r)
        k = indptr[rows] + r
        prod = data[k][:, None] * X[indices[k]]
        out[rows] = out[rows] + prod
    return out.reshape((n,) + x.shape[1:])


def grad(D_csc, x):
    """D^T x on the CSC arrays of D."""
    return exact_spmm(D_csc.indptr, D_csc.indices, D_csc.data, x)


def div(D_csc, y):
    """D y: the product over D as CSR, edge ids ascending in a row."""
    Dr = D_csc.tocsr()
    Dr.sort_indices()
    return exact_spmm(Dr.indptr, Dr.indices, Dr.data, y)
