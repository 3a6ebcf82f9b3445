"""The differential-operator oracle (tests/diffop_oracle.py) against the reference's results
(tests/golden/diffop.npz) and against SciPy's products on the same D, bit for bit."""
import os

import numpy as np
import pytest
from scipy import sparse

import diffop_oracle as dorc
from oracle import pygsp_oracle as orc


def _case(golden, case):
    g = golden("diffop")
    return {k[len(case) + 2:]: v for k, v in g.items() if k.startswith(case + "__")}


def _W(c):
    return sparse.csr_matrix((c["W_data"], c["W_indices"], c["W_indptr"]),
                             shape=tuple(int(v) for v in c["W_shape"]))


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype == np.float32 else np.uint64)


def _assert_same_bits(a, b):
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    np.testing.assert_array_equal(_bits(a), _bits(b))


CASES = [str(c) for c in np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                               "golden", "diffop.npz"))["cases"]]


@pytest.mark.parametrize("case", CASES)
def test_edge_list_and_D_match_the_reference(golden, case):
    c = _case(golden, case)
    lap_type = case.split("__")[1]
    W = _W(c)
    directed = bool(c["directed"])
    assert directed == orc.is_directed(W)
    s, t, w = dorc.edge_list(W, directed)
    np.testing.assert_array_equal(s, c["sources"])
    np.testing.assert_array_equal(t, c["targets"])
    _assert_same_bits(w.astype(np.float64), c["weights"])
    indptr, indices, data = dorc.diffop(W.shape[0], s, t, w, c["dw"], lap_type, directed)
    np.testing.assert_array_equal(indptr, c["D_indptr"])
    np.testing.assert_array_equal(indices, c["D_indices"])
    _assert_same_bits(data, c["D_data"])
    # L = D D^T
    D = sparse.csc_matrix((data, indices, indptr), shape=(W.shape[0], s.size))
    L = orc.laplacian(W, lap_type)
    assert np.abs((D @ D.T - L).toarray()).max() <= 1e-12


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("case", CASES)
def test_exact_products_equal_scipy(golden, case, dtype):
    c = _case(golden, case)
    D = sparse.csc_matrix((c["D_data"].astype(dtype), c["D_indices"], c["D_indptr"]),
                          shape=(int(c["W_shape"][0]), c["sources"].size))
    for x in (c["x"], c["X"]):
        x = x.astype(dtype)
        _assert_same_bits(dorc.grad(D, x), D.T.dot(x))
    for y in (c["y"], c["Y"]):
        y = y.astype(dtype)
        _assert_same_bits(dorc.div(D, y), D.dot(y))
    if dtype == np.float64:                 # the reference's own float64 results
        _assert_same_bits(dorc.grad(D, c["x"]), c["grad_x"])
        _assert_same_bits(dorc.grad(D, c["X"]), c["grad_X"])
        _assert_same_bits(dorc.div(D, c["y"]), c["div_y"])
        _assert_same_bits(dorc.div(D, c["Y"]), c["div_Y"])


def test_exact_spmm_order_canary():
    """A row whose products cancel: +0.0 start, no FMA, stored order all matter."""
    data = np.array([1.0, -1.0, 2.0 ** -30], np.float32)
    indptr = np.array([0, 3])
    indices = np.array([0, 1, 2])
    x = np.array([1.0 + 2.0 ** -23, 1.0, 1.0], np.float32)
    y = dorc.exact_spmm(indptr, indices, data, x)
    assert y[0] == np.float32(2.0 ** -23 + 2.0 ** -30)
    neg = dorc.exact_spmm(np.array([0, 1]), np.array([0]), np.array([-1.0], np.float32),
                          np.array([0.0], np.float32))
    assert neg[0] == 0 and not np.signbit(neg[0])           # +0.0 + (-0.0) = +0.0
    empty = dorc.exact_spmm(np.array([0, 0]), np.array([], np.int32), np.array([], np.float32),
                            np.zeros(1, np.float32))
    assert empty[0] == 0 and not np.signbit(empty[0])
