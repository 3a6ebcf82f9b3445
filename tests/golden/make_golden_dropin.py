"""Golden fixtures of the drop-in tests (tests/test_reference_dropin_gpu.py), from the REAL
reference (PyGSP 0.6.1 importable as `pygsp`, its test-suite included):

    PYTHONPATH=<reference checkout> python tests/golden/make_golden_dropin.py

  dropin.npz   : stock `pygsp.graphs.Logo()` filtered by stock `Heat(G, 50)` and
                 `MexicanHat(G, Nf=5)` (analysis at order 40, analysis + synthesis at order 25)
                 of seven seeded signals; the bank's results on a seeded sample of ROWS
                 vertices.  lmax is the one the reference estimated for these results (its
                 ARPACK start vector is unseeded).
  refsuite.npz : `approximations.cheby_op` calls the reference's own
                 `pygsp/tests/test_filters.py` makes (graph Laplacian, lmax, coefficients,
                 signal, stock SciPy result): a seeded sample of PER_KIND distinct calls for
                 every (coefficient shape, signal shape) the suite uses.  Signals wider than
                 MAX_COLS columns keep a seeded sample of MAX_COLS columns (the recurrence
                 treats columns independently).
"""
import hashlib
import logging
import os

import numpy as np
import pytest
from scipy import sparse

import pygsp
from pygsp import filters, graphs
from pygsp.filters import approximations

logging.disable(logging.CRITICAL)
HERE = os.path.dirname(os.path.abspath(__file__))
MAX_COLS = 2
PER_KIND = 2
ROWS = 128


def dropin():
    G = graphs.Logo()
    G.estimate_lmax()
    s = np.zeros(G.N)
    s[[20, 30, 1090]] = 1                                  # README.rst:68-89
    bank = filters.MexicanHat(G, Nf=5)
    heat = filters.Heat(G, scale=50)
    block = np.random.default_rng(0).standard_normal((G.N, 7))
    rows = np.sort(np.random.default_rng(1).choice(G.N, ROWS, replace=False))
    np.savez_compressed(os.path.join(HERE, "dropin.npz"), lmax=np.float64(G.lmax), signal=s,
                        heat50=heat.filter(s), rows=rows,
                        mh5_analysis40=bank.filter(block, order=40)[rows],
                        mh5_synthesis25=bank.filter(bank.filter(block), order=25)[rows])


class Recorder:
    """pytest plugin: wraps approximations.cheby_op, which Filter.filter looks up at call time."""

    def __init__(self):
        self.calls, self.seen = [], set()

    def pytest_configure(self, config):
        stock = approximations.cheby_op

        def recorded(G, c, signal, **kwargs):
            out = stock(G, c, signal, **kwargs)
            c, x = np.atleast_2d(np.asarray(c, dtype=np.float64)), np.asarray(signal)
            key = hashlib.sha1(c.tobytes() + x.tobytes() + repr(x.shape).encode()).digest()
            if key not in self.seen:
                self.seen.add(key)
                self.calls.append((sparse.csr_matrix(G.L), float(G.lmax), c, x, np.asarray(out)))
            return out
        approximations.cheby_op = recorded


def refsuite():
    rec = Recorder()
    suite = os.path.join(os.path.dirname(pygsp.__file__), "tests", "test_filters.py")
    assert pytest.main(["-q", "-p", "no:cacheprovider", suite], plugins=[rec]) == 0
    L = rec.calls[0][0]
    out = {"L_indptr": L.indptr.astype(np.int32), "L_indices": L.indices.astype(np.int32),
           "L_data": L.data.astype(np.float64), "L_shape": np.array(L.shape, dtype=np.int64)}
    kinds = {}
    for i, (Li, lmax, c, x, y) in enumerate(rec.calls):
        assert (Li != L).nnz == 0, "the suite filters on one graph"
        kinds.setdefault((c.shape, x.shape), []).append(i)
    keep = []
    for k, (kind, idx) in enumerate(sorted(kinds.items())):
        keep += list(np.random.default_rng(k).permutation(idx)[:PER_KIND])
    out["n_calls"] = np.int64(len(keep))
    for i, j in enumerate(sorted(keep)):
        _, lmax, c, x, y = rec.calls[j]
        n = x.shape[0]
        x2 = x.reshape(n, -1)
        y2 = y.reshape(c.shape[0], n, x2.shape[1])
        if x2.shape[1] > MAX_COLS:
            cols = np.sort(np.random.default_rng(i).choice(x2.shape[1], MAX_COLS, replace=False))
            x2, y2 = x2[:, cols], y2[:, :, cols]
        out["c%03d" % i] = c
        out["lmax%03d" % i] = np.float64(lmax)
        out["x%03d" % i] = x2 if x.ndim == 2 else x2[:, 0]
        out["y%03d" % i] = y2.reshape(c.shape[0] * n, -1) if x.ndim == 2 else y2.reshape(-1)
    np.savez_compressed(os.path.join(HERE, "refsuite.npz"), **out)


if __name__ == "__main__":
    print("pygsp", pygsp.__version__)
    dropin()
    refsuite()
    for f in ("dropin.npz", "refsuite.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)))
