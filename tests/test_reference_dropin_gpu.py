"""Drop-in evidence: stock PyGSP 0.6.1 filtering through `patch_pygsp()`.

`patch_pygsp()` rebinds `pygsp.filters.approximations.cheby_op`, which the reference's
`Filter.filter` looks up at call time (filter.py:309,319), so stock graphs -- SciPy `L`,
`lmax`, `N` -- have every Chebyshev recurrence served by the CUDA engine.  The stock package
is stood in for by that one module, its `cheby_op` the SciPy recurrence (the oracle's
restatement, pinned to the reference by test_oracle_golden.py).  What the reference computed
is stored under tests/golden/ (dropin.npz, refsuite.npz; tests/golden/make_golden_dropin.py):
(1) stock Logo objects filtered through `patch_pygsp()` equal the stock SciPy results;
(2) the `cheby_op` calls the reference's OWN test file `pygsp/tests/test_filters.py` makes
give, on the CUDA engine in float64, the stock results of those calls."""
import sys
import types

import numpy as np
import pytest

from conftest import csr_from, relerr_cols
from oracle import pygsp_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture
def stock_pygsp(monkeypatch):
    """The module `patch_pygsp()` rebinds, as a stock installation has it."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import pygsp_b200
    from pygsp_b200.filters import approximations as ours
    stock = orc.cheby_op
    apx = types.ModuleType("pygsp.filters.approximations")
    apx.cheby_op = lambda G, c, signal, **kwargs: stock(G.L, G.lmax, c, signal)
    filters = types.ModuleType("pygsp.filters")
    filters.approximations = apx
    pkg = types.ModuleType("pygsp")
    pkg.filters = filters
    for name, mod in (("pygsp", pkg), ("pygsp.filters", filters),
                      ("pygsp.filters.approximations", apx)):
        monkeypatch.setitem(sys.modules, name, mod)
    monkeypatch.setattr(ours, "PATCH_DEFAULT_DTYPE", ours.PATCH_DEFAULT_DTYPE)
    yield apx
    pygsp_b200.unpatch_pygsp()


def _stock_graph(L, lmax):
    return types.SimpleNamespace(L=L, lmax=float(lmax), N=L.shape[0])


def _stock_filter(apx, G, kernels, s, order):
    """Filter.filter(s, method='chebyshev', order) (filter.py:280-328) for an (N,) / (N, Nsig)
    signal (analysis) or an (N, Nsig, Nf) one (synthesis)."""
    c = orc.cheby_coeff(kernels, G.lmax, order)
    s = s.reshape(G.N, -1, 1) if s.ndim < 3 else s
    if s.shape[2] == 1:
        r = apx.cheby_op(G, c, s[:, :, 0])
        return r.reshape(len(kernels), G.N, -1).transpose(1, 2, 0).squeeze()
    return sum(apx.cheby_op(G, c[i], s[:, :, i]) for i in range(len(kernels)))


def test_patched_reference_objects(stock_pygsp, golden):
    import torch
    import pygsp_b200
    logo, gold = golden("logo"), golden("dropin")
    G = _stock_graph(csr_from(logo, "logo_Lc"), gold["lmax"])
    s = gold["signal"]                                        # README.rst:68-89
    block = np.random.default_rng(0).standard_normal((G.N, 7))
    rows = gold["rows"]
    heat = orc.heat_kernels(G.lmax, 50)
    bank = orc.mexican_hat_kernels(G.lmax, Nf=5)
    want = [gold["heat50"], gold["mh5_analysis40"], gold["mh5_synthesis25"]]
    stock = stock_pygsp.cheby_op
    for dtype, tol in ((torch.float32, 1e-5), (torch.float64, 1e-10)):
        assert pygsp_b200.patch_pygsp(dtype=dtype) is stock
        assert stock_pygsp.cheby_op is not stock
        if hasattr(G, "_gspb200_L"):
            del G._gspb200_L
        got = [_stock_filter(stock_pygsp, G, heat, s, 30),
               _stock_filter(stock_pygsp, G, bank, block, 40)[rows],
               _stock_filter(stock_pygsp, G, bank, _stock_filter(stock_pygsp, G, bank, block, 30),
                             25)[rows]]
        pygsp_b200.unpatch_pygsp()
        assert stock_pygsp.cheby_op is stock
        for a, b in zip(got, want):
            assert a.shape == b.shape and a.dtype == np.float64
            assert np.abs(a - b).max() / np.abs(b).max() <= tol
    # this engine's own Graph against the reference's Graph on the same adjacency
    H = pygsp_b200.graphs.Graph(csr_from(logo, "W"), dtype=np.float64)
    Lr = G.L
    Lo = H.L.to_scipy()
    np.testing.assert_array_equal(Lo.indptr, Lr.indptr)
    np.testing.assert_array_equal(Lo.indices, Lr.indices)
    np.testing.assert_allclose(Lo.data, Lr.data, rtol=1e-13)
    assert H.n_edges == int(logo["logo_n_edges"])
    assert abs(H._get_upper_bound() - float(logo["logo_bound_c"])) < 1e-9
    H.estimate_lmax()
    assert abs(H.lmax - G.lmax) / G.lmax < 2e-4              # ARPACK's own run-to-run spread is 1e-5


def test_reference_test_suite_on_cuda_engine(stock_pygsp, golden):
    """pygsp/tests/test_filters.py's cheby_op calls (every kind of call it makes) with
    approximations.cheby_op -> CUDA (float64), as that suite runs them."""
    import torch
    import pygsp_b200
    gold = golden("refsuite")
    n_calls = int(gold["n_calls"])
    assert n_calls > 20
    G = _stock_graph(csr_from(gold, "L"), 0.0)
    pygsp_b200.patch_pygsp(dtype=torch.float64)
    for i in range(n_calls):
        G.lmax = float(gold["lmax%03d" % i])
        want = gold["y%03d" % i]
        got = stock_pygsp.cheby_op(G, gold["c%03d" % i], gold["x%03d" % i])
        assert got.shape == want.shape and got.dtype == np.float64, i
        assert relerr_cols(got, want) <= 1e-10, i
