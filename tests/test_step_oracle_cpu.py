"""The exact step oracle (oracle/cheby_oracle.c: cheby_step_exact_f32 / _f64), on the CPU.

It restates gsp_cheby_step_* bit for bit (tests/test_tiled_step_gpu.py compares the kernels
with it at zero tolerance), so these tests pin what it computes: single rounding of every
fma (the canary), the step's value (against a float64 NumPy step), and the recurrence it
builds (against the float64 oracle of approximations.cheby_op)."""
import numpy as np
import pytest
from scipy import sparse

from oracle import build_oracle
from oracle import pygsp_oracle as orc


def _graph(n=300, seed=0):
    W = sparse.random(n, n, 0.03, random_state=seed, format="csr")
    W = W + W.T
    W.setdiag(0)
    W.eliminate_zeros()
    return orc.laplacian(W)


def _numpy_step(L, first, x_cur, x_old, r, ck, c0, alpha, beta, gamma, add_source=False):
    """float64 step of the gsp_cheby_step contract (include/gspb200.h)."""
    x_new = alpha * L.dot(x_cur) + beta * x_cur
    if not first:
        x_new = x_new + gamma * x_old
    r = r.copy()
    if add_source:
        for i in range(len(ck)):
            x_new = x_new + ck[i] * r[i]
        return x_new, r
    for i in range(len(ck)):
        r[i] = (0.5 * c0[i] * x_cur if first else r[i]) + ck[i] * x_new
    return x_new, r


def test_fmaf_canary_single_rounding():
    """r = fmaf(a, a, -(1 + 2^-11)) with a = 1 + 2^-12 is 2^-24 exactly; rounding a*a first
    to float32 gives 0."""
    a = 1.0 + 2.0 ** -12
    x = np.ones((1, 1), np.float32)
    x_new = np.zeros((1, 1), np.float32)
    r = np.zeros((1, 1, 1), np.float32)
    build_oracle.cheby_step_exact(True, 0, 1, [0, 0], np.zeros(0, np.int32), np.zeros(0, np.float32),
                                  x, None, x_new, r, 1, 1, [a], [-(2.0 + 2.0 ** -10)], 0.75, a, 0.0)
    assert x_new[0, 0] == np.float32(a)
    assert r[0, 0, 0] == np.float32(2.0 ** -24)
    separately = np.float32(np.float32(a) * np.float32(a)) - np.float32(1.0 + 2.0 ** -11)
    assert separately == 0.0


@pytest.mark.parametrize("first,nscales,add_source",
                         [(f, ns, False) for f in (True, False) for ns in (0, 1, 3)] + [(False, 2, True)])
def test_exact_f32_step_against_float64(first, nscales, add_source):
    L = _graph()
    n, nsig = L.shape[0], 5
    rng = np.random.default_rng(nscales * 2 + first)
    x_cur = rng.standard_normal((n, nsig))
    x_old = rng.standard_normal((n, nsig))
    r = rng.standard_normal((nscales, n, nsig))
    ck, c0 = rng.standard_normal(nscales), rng.standard_normal(nscales)
    alpha, beta, gamma = 4.0 / 7.3, -2.0, -1.0
    want_x, want_r = _numpy_step(L, first, x_cur, x_old, r, ck, c0, alpha, beta, gamma, add_source)
    f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
    xc, xo, r32 = f32(x_cur), f32(x_old), f32(r)
    x_new = xo if not first else np.zeros((n, nsig), np.float32)        # x_new aliases x_old
    build_oracle.cheby_step_exact(first, 0, n, L.indptr, L.indices, f32(L.data), xc, xo, x_new,
                                  r32, n, nscales, ck, c0, alpha, beta, gamma, add_source=add_source)
    scale = np.abs(want_x).max()
    assert np.abs(x_new - want_x).max() <= 2e-6 * scale
    if nscales:
        assert np.abs(r32 - want_r).max() <= 2e-6 * np.abs(want_r).max()
    if add_source:
        assert np.array_equal(r32, f32(r))                          # sources are read only


def test_exact_f32_rows_outside_the_range_are_untouched():
    L = _graph(64, seed=3)
    n, nsig = 64, 4
    rng = np.random.default_rng(1)
    xc = rng.standard_normal((n, nsig)).astype(np.float32)
    x_new = np.full((n, nsig), 7.0, np.float32)
    r = np.full((2, n + 4, nsig), 9.0, np.float32)
    build_oracle.cheby_step_exact(True, 10, 33, L.indptr, L.indices, L.data.astype(np.float32),
                                  xc, None, x_new, r, n + 4, 2, [1.0, 2.0], [0.5, 0.25], 0.3, -1.0, 0.0)
    assert (x_new[:10] == 7).all() and (x_new[33:] == 7).all() and not (x_new[10:33] == 7).all()
    assert (r[:, :10] == 9).all() and (r[:, 33:] == 9).all()


def test_exact_f64_steps_against_the_oracle():
    """First and second recurrence steps == approximations.cheby_op of order 1 and 2."""
    L = _graph(500, seed=5)
    n, nsig, lmax = L.shape[0], 3, orc.lambda_max_exact(L) * 1.01
    rng = np.random.default_rng(2)
    x = rng.standard_normal((n, nsig))
    c = rng.standard_normal((2, 3))
    t1 = np.empty((n, nsig))
    r = np.empty((2, n, nsig))
    build_oracle.cheby_step_exact(True, 0, n, L.indptr, L.indices, L.data, x, None, t1, r, n, 2,
                                  c[:, 1], c[:, 0], 2.0 / lmax, -1.0, 0.0)
    ref1 = orc.cheby_op(L, lmax, c[:, :2], x).reshape(2, n, nsig)
    assert np.abs(r - ref1).max() <= 1e-13 * np.abs(ref1).max()
    t2 = x.copy()                                                  # T_2 written over T_0
    build_oracle.cheby_step_exact(False, 0, n, L.indptr, L.indices, L.data, t1, t2, t2, r, n, 2,
                                  c[:, 2], c[:, 0], 4.0 / lmax, -2.0, -1.0)
    ref2 = orc.cheby_op(L, lmax, c, x).reshape(2, n, nsig)
    assert np.abs(r - ref2).max() <= 1e-13 * np.abs(ref2).max()
