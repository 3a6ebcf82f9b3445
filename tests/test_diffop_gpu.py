"""Differential operator on the B200: get_edge_list, G.D, grad, div and dirichlet_energy.

  * structure: the edge list and D's CSC indptr / indices equal the reference's exactly; D's
    values equal the oracle fed the engine's own dw and weights bit for bit, and the
    reference's to 1e-15 (float64) / 1e-6 (float32) relative;
  * kernels: G.grad(x) / G.div(y) are bit-identical to SciPy's D.T.dot(x) / D.dot(y) on the
    engine's D, in the graph's dtype (bit patterns compared, so -0.0 for +0.0 fails);
  * against the reference: grad / div / dirichlet_energy per column to 1e-12 (float64) and
    1e-5 (float32);
  * a 1e6-vertex sensor graph with 64 signals.
"""
import os

import numpy as np
import pytest
from scipy import sparse

import diffop_oracle as dorc
from conftest import relerr_cols

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = [str(c) for c in np.load(os.path.join(HERE, "golden", "diffop.npz"))["cases"]]
NSIGS = [None, 1, 2, 3, 8, 63, 64, 128]          # None: a 1-D signal
DTYPES = [np.float32, np.float64]
TOL = {np.float32: 1e-5, np.float64: 1e-12}


@pytest.fixture(scope="module")
def gsp():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import pygsp_b200
    return pygsp_b200


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


def _signal(rng, rows, nsig, dtype):
    """Seeded signal with exact zeros (whole rows and scattered entries) and a few -0.0."""
    shape = (rows,) if nsig is None else (rows, nsig)
    x = rng.standard_normal(shape).astype(dtype)
    x[::5] = 0
    x.reshape(-1)[3::11] = 0
    x.reshape(-1)[7::13] = -0.0
    return x


def _graph(gsp, c, lap_type, dtype):
    return gsp.graphs.Graph(_W(c), lap_type=lap_type, dtype=dtype)


def _isolated_graph(directed, seed=7):
    """300 vertices, a third of them isolated, some self-loops."""
    rng = np.random.default_rng(seed)
    n = 300
    A = sparse.random(200, 200, density=0.03, random_state=seed, format="csr")
    A.data = rng.uniform(0.1, 2.0, A.nnz)
    if not directed:
        A = sparse.triu(A, k=1)
        A = (A + A.T).tocsr()
    A = A + sparse.diags(np.where(rng.uniform(size=200) < 0.1, 0.7, 0.0))
    W = sparse.block_diag([A, sparse.csr_matrix((100, 100))]).tocsr()
    perm = rng.permutation(n)
    W = W[perm][:, perm].tocsr()
    W.eliminate_zeros()
    W.sort_indices()
    return W


# ------------------------------------------------------------------------ structure
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", CASES)
def test_edge_list_and_D_structure(gsp, golden, case, dtype):
    c = _case(golden, case)
    lap_type = case.split("__")[1]
    G = _graph(gsp, c, lap_type, dtype)
    assert G.is_directed() == bool(c["directed"])
    s, t, w = G.get_edge_list()
    assert s.dtype == np.int32 and t.dtype == np.int32 and w.dtype == dtype
    np.testing.assert_array_equal(s, c["sources"])
    np.testing.assert_array_equal(t, c["targets"])
    _assert_same_bits(w, c["weights"].astype(dtype))
    G.compute_differential_operator()
    assert G.D.shape == (G.N, G.Ne) and G.D.T.shape == (G.Ne, G.N)
    D = G.D.to_scipy()
    assert isinstance(D, sparse.csc_matrix) and D.dtype == dtype and G.D.nnz == D.nnz
    np.testing.assert_array_equal(D.indptr, c["D_indptr"])
    np.testing.assert_array_equal(D.indices, c["D_indices"])
    _, _, own = dorc.diffop(G.N, s, t, w, G.dw, lap_type, G.is_directed(), dtype)
    _assert_same_bits(D.data, own)
    np.testing.assert_allclose(D.data, c["D_data"], rtol=1e-15 if dtype == np.float64 else 1e-6,
                               atol=0)
    np.testing.assert_array_equal(G.D.toarray(), D.toarray())


# ------------------------------------------------------------------ kernels, exact
def _check_products(G, rng, nsigs, tensor=False):
    import torch
    D = G.D.to_scipy()
    dtype = D.dtype.type
    for nsig in nsigs:
        x = _signal(rng, G.N, nsig, dtype)
        y = _signal(rng, G.Ne, nsig, dtype)
        gx, dy = G.grad(x), G.div(y)
        assert isinstance(gx, np.ndarray) and isinstance(dy, np.ndarray)
        _assert_same_bits(gx, D.T.dot(x))
        _assert_same_bits(dy, D.dot(y))
        _assert_same_bits(G.D.T.dot(x), gx)
        _assert_same_bits(G.D.dot(y), dy)
        if tensor:
            xt, yt = torch.from_numpy(x).to(G.device), torch.from_numpy(y).to(G.device)
            gt, dt = G.grad(xt), G.div(yt)
            assert torch.is_tensor(gt) and gt.is_cuda and torch.is_tensor(dt) and dt.is_cuda
            _assert_same_bits(gt.cpu().numpy(), gx)
            _assert_same_bits(dt.cpu().numpy(), dy)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", CASES)
def test_grad_div_bit_identical_to_scipy(gsp, golden, case, dtype):
    c = _case(golden, case)
    G = _graph(gsp, c, case.split("__")[1], dtype)
    G.compute_differential_operator()
    _check_products(G, np.random.default_rng(len(case)), NSIGS, tensor=True)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("lap_type", ["combinatorial", "normalized"])
@pytest.mark.parametrize("directed", [False, True])
def test_grad_div_with_isolated_vertices_and_loops(gsp, directed, lap_type, dtype):
    W = _isolated_graph(directed)
    G = gsp.graphs.Graph(W, lap_type=lap_type, dtype=dtype)
    assert G.is_directed() == directed and G.has_loops()
    G.compute_differential_operator()
    s, t, w = G.get_edge_list()
    ref = dorc.edge_list(W, directed)
    np.testing.assert_array_equal(s, ref[0])
    np.testing.assert_array_equal(t, ref[1])
    assert G.Ne == s.size and G.D.nnz == 2 * int((s != t).sum())
    D = G.D.to_scipy()
    assert np.all(np.diff(D.indptr)[s == t] == 0)
    L = G.L.to_scipy().astype(np.float64)
    assert abs(D.astype(np.float64) @ D.T.astype(np.float64) - L).max() <= TOL[dtype] * 10
    _check_products(G, np.random.default_rng(3), NSIGS)


@pytest.mark.parametrize("dtype", DTYPES)
def test_loops_only_and_no_edges(gsp, dtype):
    n = 37
    for adjacency, ne in ((np.identity(n), n), (np.zeros((n, n)), 0)):
        for lap_type in ("combinatorial", "normalized"):
            G = gsp.graphs.Graph(adjacency, lap_type=lap_type, dtype=dtype)
            G.compute_differential_operator()
            assert G.Ne == ne and G.D.shape == (n, ne) and G.D.nnz == 0
            s, t, w = G.get_edge_list()
            assert len(s) == len(t) == len(w) == ne
            for nsig in NSIGS:
                x = _signal(np.random.default_rng(0), n, nsig, dtype)
                y = _signal(np.random.default_rng(1), ne, nsig, dtype)
                gx, dy = G.grad(x), G.div(y)
                _assert_same_bits(gx, np.zeros_like(gx))          # +0.0 everywhere
                _assert_same_bits(dy, np.zeros_like(dy))
                assert gx.shape[0] == ne and dy.shape[0] == n
            assert G.dirichlet_energy(np.ones(n)) == 0


# ------------------------------------------------------------- against the reference
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("case", CASES)
def test_matches_the_reference(gsp, golden, case, dtype):
    c = _case(golden, case)
    G = _graph(gsp, c, case.split("__")[1], dtype)
    G.compute_differential_operator()
    tol = TOL[dtype]
    for key, fn, arg in (("grad_x", G.grad, "x"), ("grad_X", G.grad, "X"),
                         ("div_y", G.div, "y"), ("div_Y", G.div, "Y")):
        ref = c[key]
        got = fn(c[arg].astype(dtype))
        assert got.shape == ref.shape
        if ref.size:
            assert relerr_cols(got, ref) <= tol, key
    e = G.dirichlet_energy(c["x"].astype(dtype))
    assert np.ndim(e) == 0
    assert abs(float(e) - float(c["energy_x"])) <= tol * max(abs(float(c["energy_x"])), 1e-300)
    E = G.dirichlet_energy(c["X"].astype(dtype))
    assert E.shape == (3, 3)
    assert relerr_cols(E, c["energy_X"]) <= tol


def test_path_doctests(gsp):
    """The values printed by the reference's doctests (graph.py dirichlet_energy,
    difference.py grad / div)."""
    G = gsp.graphs.Graph(sparse.diags([1.0] * 4, 1, shape=(5, 5)) +
                         sparse.diags([1.0] * 4, -1, shape=(5, 5)), dtype=np.float64)
    assert G.dirichlet_energy([0, 2, 2, 4, 4]) == 8.0
    G.compute_differential_operator()
    np.testing.assert_array_equal(G.grad([0, 2, 2, 4, 4]), [2.0, 0.0, 2.0, 0.0])
    Gd = gsp.graphs.Graph(sparse.diags([1.0] * 4, 1, shape=(5, 5)), dtype=np.float64)
    assert Gd.dirichlet_energy([0, 2, 2, 4, 4]) == 4.0
    Gd.compute_differential_operator()
    np.testing.assert_allclose(Gd.grad([0, 2, 2, 4, 4]), [2 ** 0.5, 0, 2 ** 0.5, 0], rtol=1e-15)
    G3 = gsp.graphs.Graph([[0, 2, 0], [2, 0, 1], [0, 1, 0]], dtype=np.float64)
    G3.compute_differential_operator()
    np.testing.assert_allclose(G3.D.toarray(), [[-1.41421356, 0], [1.41421356, -1], [0, 1]],
                               atol=1e-8)


# ------------------------------------------------------------------------ behaviour
def test_errors_warning_and_recompute(gsp, caplog):
    import torch
    G = gsp.graphs.Graph(_isolated_graph(False), dtype=np.float64)
    with caplog.at_level("WARNING"):
        G.grad(np.zeros(G.N))
    assert any("The differential operator G.D is not available" in r.getMessage()
               for r in caplog.records)
    caplog.clear()
    with caplog.at_level("WARNING"):
        G.D
    assert not caplog.records
    with pytest.raises(ValueError, match="First dimension must be the number of vertices"):
        G.grad(np.zeros(G.N + 1))
    with pytest.raises(ValueError, match="First dimension must be the number of edges "
                                         "G.Ne = %d" % G.Ne):
        G.div(np.zeros(G.Ne - 1))
    with pytest.raises(ValueError, match="number of edges"):
        G.div(torch.zeros(G.Ne + 1, device=G.device, dtype=torch.float64))
    with pytest.raises(ValueError, match="First dimension must be the number of vertices"):
        G.dirichlet_energy(np.zeros((G.N - 1, 2)))

    D_comb = G.D.to_scipy()
    G.compute_laplacian("combinatorial")             # same type: D is kept
    assert G.D.to_scipy() is not None and not caplog.records
    G.compute_laplacian("normalized")
    with caplog.at_level("WARNING"):
        D_norm = G.D.to_scipy()
    assert any("G.D is not available" in r.getMessage() for r in caplog.records)
    s, t, w = G.get_edge_list()
    _, _, own = dorc.diffop(G.N, s, t, w, G.dw, "normalized", False, np.float64)
    _assert_same_bits(D_norm.data, own)
    assert not np.array_equal(D_norm.data, D_comb.data)
    L = G.L.to_scipy()
    assert abs(D_norm @ D_norm.T - L).max() <= 1e-12


def test_dirichlet_energy_tensor(gsp):
    import torch
    G = gsp.graphs.Graph(_isolated_graph(True), dtype=np.float64)
    x = np.random.default_rng(5).standard_normal((G.N, 4))
    xt = torch.from_numpy(x).to(G.device)
    E = G.dirichlet_energy(xt)
    assert torch.is_tensor(E) and E.is_cuda and tuple(E.shape) == (4, 4)
    np.testing.assert_allclose(E.cpu().numpy(), G.dirichlet_energy(x), rtol=1e-12)
    e = G.dirichlet_energy(xt[:, 0])
    assert torch.is_tensor(e) and e.ndim == 0
    g = G.grad(x)
    np.testing.assert_allclose(np.diag(E.cpu().numpy()), (g ** 2).sum(axis=0), rtol=1e-12)


# ------------------------------------------------------------------------ full size
def test_full_size_sensor(gsp):
    import torch
    G = gsp.graphs.Sensor(1_000_000, k=10, seed=0, order="morton")
    G.compute_differential_operator()
    assert G.D.shape == (G.N, G.Ne) and G.Ne > G.N
    x = torch.from_numpy(np.random.default_rng(0).standard_normal((G.N, 64)).astype(np.float32)
                         ).to(G.device)
    g = G.grad(x)
    z = G.div(g)
    L = G.L.to_scipy().astype(np.float64)
    xh = x.cpu().numpy().astype(np.float64)
    assert relerr_cols(z.cpu().numpy(), L @ xh) <= 1e-5
    E = G.dirichlet_energy(x)
    gn = (g.double() ** 2).sum(dim=0)
    assert float(((torch.diagonal(E).double() - gn).abs() / gn).max()) <= 1e-5
    del G, g, z, E

    G64 = gsp.graphs.Sensor(1_000_000, k=10, seed=0, order="morton", dtype=np.float64)
    G64.compute_differential_operator()
    x1 = xh[:, 5].copy()
    _assert_same_bits(G64.grad(x1), G64.D.to_scipy().T.dot(x1))
