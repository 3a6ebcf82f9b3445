"""Golden fixture of the differential-operator tests (tests/test_oracle_diffop.py,
tests/test_diffop_gpu.py), from the REAL reference (PyGSP 0.6.1 importable as `pygsp`):

    PYTHONPATH=<reference checkout> python tests/golden/make_golden_diffop.py

  diffop.npz : for every graph below and both Laplacian types, with key prefix "<case>__":
    W_indptr / W_indices / W_data / W_shape  the adjacency (tests rebuild the graph from it)
    directed, dw                             G.is_directed(), G.dw
    sources / targets / weights              G.get_edge_list()
    D_indptr / D_indices / D_data            CSC arrays of G.D
    x (N,), X (N, 3), y (Ne,), Y (Ne, 3)     seeded vertex and edge signals
    grad_x, grad_X, div_y, div_Y             G.grad / G.div of them
    energy_x, energy_X                       G.dirichlet_energy(x), G.dirichlet_energy(X)
  and "cases", the case names.
"""
import logging
import os

import numpy as np

from pygsp import graphs

logging.disable(logging.CRITICAL)
HERE = os.path.dirname(os.path.abspath(__file__))
N = 98


def cases():
    """The graphs of the reference's test_differential_operator, the Path(5) doctests,
    the graph of test_dirichlet_energy (seeded) and a sensor network."""
    return [
        ("zeros", lambda: graphs.Graph(np.zeros((N, N)))),
        ("identity", lambda: graphs.Graph(np.identity(N))),
        ("pair", lambda: graphs.Graph([[0, 0.8], [0.8, 0]])),
        ("pair_loops", lambda: graphs.Graph([[1.3, 0], [0.4, 0.5]])),
        ("er_undirected", lambda: graphs.ErdosRenyi(N, directed=False, seed=42)),
        ("er_directed", lambda: graphs.ErdosRenyi(N, directed=True, seed=42)),
        ("path5_undirected", lambda: graphs.Path(5, directed=False)),
        ("path5_directed", lambda: graphs.Path(5, directed=True)),
        ("barabasi_albert", lambda: graphs.BarabasiAlbert(100, seed=42)),
        ("sensor", lambda: graphs.Sensor(200, seed=42)),
    ]


def main():
    out = {}
    names = []
    for i, (name, make) in enumerate(cases()):
        for lap_type in ["combinatorial", "normalized"]:
            G = make()
            G.compute_laplacian(lap_type)
            G.compute_differential_operator()
            case = "%s__%s" % (name, lap_type)
            names.append(case)
            rng = np.random.default_rng(1000 + i)
            W = G.W.tocsr()
            D = G.D.tocsc()
            assert D.has_canonical_format
            s, t, w = G.get_edge_list()
            x = rng.standard_normal(G.N)
            X = rng.standard_normal((G.N, 3))
            y = rng.standard_normal(G.Ne)
            Y = rng.standard_normal((G.Ne, 3))
            rec = {
                "W_indptr": W.indptr.astype(np.int32), "W_indices": W.indices.astype(np.int32),
                "W_data": W.data.astype(np.float64), "W_shape": np.array(W.shape),
                "directed": np.array(G.is_directed()), "dw": np.asarray(G.dw, np.float64),
                "sources": s.astype(np.int32), "targets": t.astype(np.int32),
                "weights": w.astype(np.float64),
                "D_indptr": D.indptr.astype(np.int32), "D_indices": D.indices.astype(np.int32),
                "D_data": D.data.astype(np.float64),
                "x": x, "X": X, "y": y, "Y": Y,
                "grad_x": G.grad(x), "grad_X": G.grad(X), "div_y": G.div(y), "div_Y": G.div(Y),
                "energy_x": np.array(G.dirichlet_energy(x)),
                "energy_X": np.asarray(G.dirichlet_energy(X)),
            }
            for k, v in rec.items():
                out[case + "__" + k] = v
    out["cases"] = np.array(names)
    path = os.path.join(HERE, "diffop.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, len(names), "cases")


if __name__ == "__main__":
    main()
