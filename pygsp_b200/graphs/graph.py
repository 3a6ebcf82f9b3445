"""``Graph``: the reference's graph object with its sparse algebra in HBM.

Mirror of the part of ``pygsp.graphs.Graph`` that the Chebyshev filtering path
uses (pygsp/graphs/graph.py:98-176 constructor, :510-630 compute_laplacian,
:632-640 _check_signal, :729-838 d / dw, :840-960 lmax / estimate_lmax /
_get_upper_bound, :368-405 is_directed) and of its vertex calculus
(graph.py:642-704 dirichlet_energy, :962-1029 get_edge_list, difference.py
D / compute_differential_operator / grad / div).  Same constructor signature,
same attributes, same exceptions and log messages; the adjacency, the
Laplacian, the differential operator and every vector derived from them live
on the GPU and are produced by the kernels of ``libgspb200`` (csrc/graph.cu,
csrc/lanczos.cu, csrc/diffop.cu).  Out of scope here, as in SURVEY.md
section 2: Fourier basis, plotting, IO.
"""
import numpy as np
from scipy import sparse

from .. import _native as nat
from .. import utils
from .csr import DeviceCSR, DifferentialOperator

_LAP = {"combinatorial": 0, "normalized": 1}


class Graph:
    r"""Graph defined by a (weighted) adjacency matrix.

    Parameters
    ----------
    adjacency : sparse matrix, array_like, DeviceCSR or (indptr, indices, data)
        Square adjacency.  Host inputs are converted to CSR (duplicates summed,
        columns sorted) and uploaded; a ``DeviceCSR`` / tensor triple is used
        in place (it must be canonical CSR).
    lap_type : {'combinatorial', 'normalized'}
    coords : array_like, optional
    plotting : dict, optional (kept for signature compatibility)
    dtype : numpy/torch floating dtype, keyword only
        Arithmetic type of the engine: float32 (default) or float64.  The
        reference computes in float64; float64 here reproduces its results to
        round-off, float32 to 1e-5 (normwise).
    device : torch device, keyword only (default: current CUDA device)
    """

    def __init__(self, adjacency, lap_type="combinatorial", coords=None, plotting={},
                 *, dtype=None, device=None):
        torch = nat.require_cuda()
        self.logger = utils.build_logger(__name__)
        self.device = torch.device(device if device is not None
                                   else "cuda:%d" % torch.cuda.current_device())
        self.dtype = _torch_dtype(torch, dtype)
        self._sfx = nat.suffix(self.dtype)

        if isinstance(adjacency, DeviceCSR):
            W = adjacency
        elif isinstance(adjacency, tuple) and len(adjacency) == 3 and torch.is_tensor(adjacency[2]):
            indptr, indices, data = adjacency
            n = indptr.numel() - 1
            W = DeviceCSR(indptr, indices, data, (n, n))
        else:
            if not sparse.issparse(adjacency):
                adjacency = np.asanyarray(adjacency)
            if adjacency.ndim != 2 or adjacency.shape[0] != adjacency.shape[1]:
                raise ValueError("Adjacency: must be a square matrix.")
            host = sparse.csr_matrix(adjacency)          # format conversion only
            if not host.has_canonical_format:
                host = host.copy()
                host.sum_duplicates()
            W = DeviceCSR.from_scipy(host, self.dtype, self.device)
        if W.shape[0] != W.shape[1]:
            raise ValueError("Adjacency: must be a square matrix.")
        if W.data.dtype != self.dtype:
            W = DeviceCSR(W.indptr, W.indices, W.data.to(self.dtype), W.shape)
        W = DeviceCSR(W.indptr.to(self.device, torch.int32).contiguous(),
                      W.indices.to(self.device, torch.int32).contiguous(),
                      W.data.to(self.device).contiguous(), W.shape)
        self.n_vertices = W.shape[0]

        stats = self._inspect(W)
        if stats[5] or stats[6]:
            raise ValueError("Adjacency: CSR columns must be sorted, unique and in range.")
        if stats[0]:
            raise ValueError("Adjacency: there is a Not a Number (NaN).")
        if stats[1]:
            raise ValueError("Adjacency: there is an infinite value.")
        if stats[3]:
            self.logger.warning("Adjacency: there are self-loops (non-zeros on the diagonal). "
                                "The Laplacian will not see them.")
        if stats[2]:
            self.logger.warning("Adjacency: there are negative edge weights.")
        if stats[4]:                                     # graph.py:128 eliminate_zeros()
            W = self._compact(W)
        self._adjacency = W
        self._n_loops = int(stats[3])

        self._directed = None
        self._connected = None
        if self.is_directed():
            self.n_edges = W.nnz
        else:
            self.n_edges = (W.nnz - self._n_loops) // 2 + self._n_loops

        if coords is not None:
            self.coords = np.asanyarray(coords)
        self.plotting = dict(plotting)
        self.signals = dict()

        self._d = None
        self._dw = None
        self._dw_dev = None
        self._d_dev = None
        self._Wt = None
        self._Ws = None
        self._lmax = None
        self._lmax_method = None
        self._lanczos_steps = None
        self._edges = None
        self._D = None

        self.lap_type = lap_type
        self.compute_laplacian(lap_type)
        self.Ne = self.n_edges

    @classmethod
    def from_coo(cls, rows, cols, vals, n_vertices, lap_type="combinatorial", **kwargs):
        """Graph from COO triplets already in HBM (int32 rows / cols, float values).

        What ``sparse.csr_matrix(coo)`` does at graph.py:109 -- sort by (row, col), sum
        duplicates -- runs on the device (``gsp_coo_to_csr_*``); no host matrix exists.
        """
        import ctypes
        torch = nat.require_cuda()
        dev = vals.device
        dt = _torch_dtype(torch, kwargs.get("dtype", vals.dtype if vals.dtype in
                                            (torch.float32, torch.float64) else None))
        rows = rows.to(dev, torch.int32).contiguous()
        cols = cols.to(dev, torch.int32).contiguous()
        vals = vals.to(dev, dt).contiguous()
        nnz = int(vals.numel())
        indptr = torch.empty(n_vertices + 1, dtype=torch.int32, device=dev)
        indices = torch.empty(nnz, dtype=torch.int32, device=dev)
        data = torch.empty(nnz, dtype=dt, device=dev)
        uniq = ctypes.c_int64(0)
        with torch.cuda.device(dev):
            nat.call("gsp_coo_to_csr_" + nat.suffix(dt), nat.i64(n_vertices), nat.i64(nnz), rows,
                     cols, vals, indptr, indices, data, ctypes.byref(uniq), nat.stream_ptr(dev))
        m = int(uniq.value)
        W = DeviceCSR(indptr, indices[:m].contiguous(), data[:m].contiguous(),
                      (n_vertices, n_vertices))
        kwargs.setdefault("dtype", dt)
        kwargs.setdefault("device", dev)
        return cls(W, lap_type=lap_type, **kwargs)

    # ------------------------------------------------------------------ basics
    @property
    def N(self):
        return self.n_vertices

    def __repr__(self):
        return "{}(n_vertices={}, n_edges={})".format(type(self).__name__, self.n_vertices,
                                                      self.n_edges)

    @property
    def W(self):
        r"""Weighted adjacency matrix (a :class:`DeviceCSR`)."""
        return self._adjacency

    @W.setter
    def W(self, value):
        raise AttributeError("In-place modification of the graph is not supported. "
                             "Create another Graph object.")

    def _stream(self):
        return nat.stream_ptr(self.device)

    def _call(self, name, *args):
        torch = nat.require_cuda()
        with torch.cuda.device(self.device):
            nat.call(name + "_" + self._sfx, *args, self._stream())

    def _inspect(self, W):
        torch = nat.require_cuda()
        stats = torch.zeros(8, dtype=torch.int64, device=self.device)
        self._call("gsp_csr_inspect", nat.i64(W.shape[0]), W.indptr, W.indices, W.data, stats)
        return stats.cpu().numpy()

    def _compact(self, W):
        torch = nat.require_cuda()
        n = W.shape[0]
        indptr = torch.empty(n + 1, dtype=torch.int32, device=self.device)
        self._call("gsp_csr_compact_count", nat.i64(n), W.indptr, W.data, indptr)
        nnz = int(indptr[-1].item()) if n else 0
        indices = torch.empty(nnz, dtype=torch.int32, device=self.device)
        data = torch.empty(nnz, dtype=self.dtype, device=self.device)
        self._call("gsp_csr_compact_fill", nat.i64(n), W.indptr, W.indices, W.data, indptr,
                   indices, data)
        return DeviceCSR(indptr, indices, data, W.shape)

    def has_loops(self):
        return self._n_loops > 0

    def is_directed(self):
        r"""True iff W differs from its transpose (cached; graph.py:368-405)."""
        if self._directed is None:
            torch = nat.require_cuda()
            W = self._adjacency
            count = torch.zeros(1, dtype=torch.int64, device=self.device)
            self._call("gsp_csr_asymmetry", nat.i64(self.n_vertices), W.indptr, W.indices,
                       W.data, count)
            self._directed = bool(count.item() != 0)
        return self._directed

    # ---------------------------------------------------- symmetric part, degree
    def _transpose(self):
        if self._Wt is None:
            torch = nat.require_cuda()
            W, n = self._adjacency, self.n_vertices
            tp = torch.empty(n + 1, dtype=torch.int32, device=self.device)
            ti = torch.empty(W.nnz, dtype=torch.int32, device=self.device)
            td = torch.empty(W.nnz, dtype=self.dtype, device=self.device)
            self._call("gsp_csr_transpose", nat.i64(n), nat.i64(W.nnz), W.indptr, W.indices,
                       W.data, tp, ti, td)
            self._Wt = DeviceCSR(tp, ti, td, W.shape)
        return self._Wt

    def _symmetric_adjacency(self):
        """W for an undirected graph, (W + W^T)/2 otherwise (graph.py:613-616)."""
        if not self.is_directed():
            return self._adjacency
        if self._Ws is None:
            torch = nat.require_cuda()
            W, Wt, n = self._adjacency, self._transpose(), self.n_vertices
            sp = torch.empty(n + 1, dtype=torch.int32, device=self.device)
            self._call("gsp_csr_average_count", nat.i64(n), W.indptr, W.indices, W.data,
                       Wt.indptr, Wt.indices, Wt.data, sp)
            nnz = int(sp[-1].item()) if n else 0
            si = torch.empty(nnz, dtype=torch.int32, device=self.device)
            sd = torch.empty(nnz, dtype=self.dtype, device=self.device)
            self._call("gsp_csr_average_fill", nat.i64(n), W.indptr, W.indices, W.data,
                       Wt.indptr, Wt.indices, Wt.data, sp, si, sd)
            self._Ws = DeviceCSR(sp, si, sd, W.shape)
        return self._Ws

    def _degrees(self):
        if self._dw_dev is None:
            torch = nat.require_cuda()
            W, n = self._adjacency, self.n_vertices
            dw = torch.empty(n, dtype=torch.float64, device=self.device)
            d = torch.empty(n, dtype=torch.float64, device=self.device)
            if self.is_directed():
                Wt = self._transpose()
                self._call("gsp_degree", nat.i64(n), W.indptr, W.data, Wt.indptr, Wt.data, dw, d)
            else:
                self._call("gsp_degree", nat.i64(n), W.indptr, W.data, None, None, dw, d)
            self._dw_dev, self._d_dev = dw, d
        return self._dw_dev, self._d_dev

    @property
    def dw(self):
        r"""Weighted degree (graph.py:783-838): sum_j W[j,i], or (in+out)/2 if directed."""
        if self._dw is None:
            self._dw = self._degrees()[0].cpu().numpy()
        return self._dw

    @property
    def d(self):
        r"""Number of neighbours (graph.py:729-781); (in+out)/2 if directed."""
        if self._d is None:
            d = self._degrees()[1].cpu().numpy()
            self._d = d if self.is_directed() else d.astype(np.int32)
        return self._d

    # ------------------------------------------------------------------ Laplacian
    def compute_laplacian(self, lap_type="combinatorial"):
        r"""Build the graph Laplacian ``self.L`` on the device (graph.py:510-630).

        combinatorial: L = D - W;  normalized: L = I - D^-1/2 W D^-1/2, where a
        directed W is first replaced by (W + W^T)/2.  ``L.indptr`` /
        ``L.indices`` equal SciPy's bit for bit: sorted rows, the diagonal
        merged in place, exact zeros (isolated vertices) not stored.
        """
        if lap_type not in _LAP:
            raise ValueError("Unknown Laplacian type {}".format(lap_type))
        if lap_type != self.lap_type:
            # the reference forgets _lmax_method here, so that G.lmax then returns
            # None (SURVEY.md 3.5); both are reset in this implementation.
            self._lmax = None
            self._lmax_method = None
            self._D = None
        self.lap_type = lap_type

        torch = nat.require_cuda()
        Ws, n = self._symmetric_adjacency(), self.n_vertices
        dw = self._degrees()[0]
        lp = torch.empty(n + 1, dtype=torch.int32, device=self.device)
        self._call("gsp_laplacian_count", nat.i64(n), Ws.indptr, Ws.indices, Ws.data, dw,
                   nat.i32(_LAP[lap_type]), lp)
        nnz = int(lp[-1].item()) if n else 0
        li = torch.empty(nnz, dtype=torch.int32, device=self.device)
        ld = torch.empty(nnz, dtype=self.dtype, device=self.device)
        self._call("gsp_laplacian_fill", nat.i64(n), Ws.indptr, Ws.indices, Ws.data, dw,
                   nat.i32(_LAP[lap_type]), lp, li, ld)
        self.L = DeviceCSR(lp, li, ld, (n, n))

    def _check_signal(self, s):
        r"""Validate a signal's first dimension (graph.py:632-640)."""
        torch = nat.require_cuda()
        if not torch.is_tensor(s):
            s = np.asanyarray(s)
        if s.shape[0] != self.n_vertices:
            raise ValueError("First dimension must be the number of vertices "
                             "G.N = {}, got {}.".format(self.N, tuple(s.shape)))
        return s

    def dirichlet_energy(self, x):
        r"""Dirichlet energy x^T L x of a vertex signal (graph.py:642-704).

        L x runs on the SpMV / SpMM kernel.  A vector gives a scalar, an (N, nsig) block the
        (nsig, nsig) matrix x^T L x; NumPy in gives NumPy out, a CUDA tensor gives a tensor.
        """
        torch = nat.require_cuda()
        x = self._check_signal(x)
        Lx = self.L.dot(x)
        if torch.is_tensor(Lx):
            x = x.to(device=self.device, dtype=self.dtype)
            return torch.dot(x, Lx) if x.ndim == 1 else x.T @ Lx
        return np.asarray(x, dtype=Lx.dtype).T.dot(Lx)

    # ------------------------------------------------------- differential operator
    def _edge_list(self):
        """Device (sources, targets, weights) of get_edge_list (cached: W is immutable)."""
        if self._edges is None:
            torch = nat.require_cuda()
            W, n = self._adjacency, self.n_vertices
            directed = nat.i32(self.is_directed())
            ptr = torch.empty(n + 1, dtype=torch.int32, device=self.device)
            with torch.cuda.device(self.device):
                nat.call("gsp_edge_list_count", nat.i64(n), W.indptr, W.indices, directed, ptr,
                         self._stream())
            ne = int(ptr[-1].item())
            sources = torch.empty(ne, dtype=torch.int32, device=self.device)
            targets = torch.empty(ne, dtype=torch.int32, device=self.device)
            weights = torch.empty(ne, dtype=self.dtype, device=self.device)
            self._call("gsp_edge_list_fill", nat.i64(n), W.indptr, W.indices, W.data, directed,
                       ptr, sources, targets, weights)
            self._edges = (sources, targets, weights)
        return self._edges

    def get_edge_list(self):
        r"""Edge list (sources, targets, weights) of W (graph.py:962-1029).

        A directed graph gives every stored entry of W in row-major order, an undirected one
        the upper triangle (diagonal included), so that sources <= targets.  Sources and
        targets are int32 NumPy arrays, weights are in the graph's dtype.
        """
        sources, targets, weights = self._edge_list()
        assert self.n_edges == sources.numel() == targets.numel() == weights.numel()
        return sources.cpu().numpy(), targets.cpu().numpy(), weights.cpu().numpy()

    @property
    def D(self):
        r"""Differential operator (a :class:`DifferentialOperator`, computed lazily)."""
        if self._D is None:
            self.logger.warning("The differential operator G.D is not available, we need to "
                                "compute it. Explicitly call "
                                "G.compute_differential_operator() once beforehand to "
                                "suppress the warning.")
            self.compute_differential_operator()
        return self._D

    def compute_differential_operator(self):
        r"""Compute the differential operator D, L = D D^T (difference.py; cached as G.D).

        Column k of the N x Ne matrix D (edge k = (s, t) of :meth:`get_edge_list`) holds
        -sqrt(W[s, t]) at s and +sqrt(W[s, t]) at t (combinatorial), or -sqrt(W[s, t] / dw[s])
        and +sqrt(W[s, t] / dw[t]) (normalized), both divided by sqrt(2) for a directed graph;
        a self-loop's column is empty.
        """
        torch = nat.require_cuda()
        sources, targets, weights = self._edge_list()
        n, ne = self.n_vertices, self.n_edges
        d_indptr = torch.empty(ne + 1, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            nat.call("gsp_diffop_count", nat.i64(ne), sources, targets, d_indptr, self._stream())
        nnz = int(d_indptr[-1].item())
        d_indices = torch.empty(nnz, dtype=torch.int32, device=self.device)
        d_data = torch.empty(nnz, dtype=self.dtype, device=self.device)
        v_indptr = torch.empty(n + 1, dtype=torch.int32, device=self.device)
        v_indices = torch.empty(nnz, dtype=torch.int32, device=self.device)
        v_data = torch.empty(nnz, dtype=self.dtype, device=self.device)
        self._call("gsp_diffop_fill", nat.i64(n), nat.i64(ne), nat.i64(nnz), sources, targets,
                   weights, self._degrees()[0], nat.i32(_LAP[self.lap_type]),
                   nat.i32(self.is_directed()), d_indptr, d_indices, d_data, v_indptr, v_indices,
                   v_data)
        self._D = DifferentialOperator((n, ne), d_indptr, d_indices, d_data, v_indptr,
                                       v_indices, v_data)

    def grad(self, x):
        r"""Gradient D^T x of a vertex signal (difference.py grad).

        x is (N,) or (N, nsig); the result is (Ne,) or (Ne, nsig) in the graph's dtype, equal
        bit for bit to SciPy's ``G.D.to_scipy().T.dot(x)``.  NumPy in gives NumPy out, a CUDA
        tensor gives a tensor.
        """
        x = self._check_signal(x)
        return self.D.T.dot(x)

    def div(self, y):
        r"""Divergence D y of an edge signal (difference.py div).

        y is (Ne,) or (Ne, nsig); the result is (N,) or (N, nsig) in the graph's dtype, equal
        bit for bit to SciPy's ``G.D.to_scipy().dot(y)``.  NumPy in gives NumPy out, a CUDA
        tensor gives a tensor.
        """
        torch = nat.require_cuda()
        if not torch.is_tensor(y):
            y = np.asanyarray(y)
        if y.shape[0] != self.Ne:
            raise ValueError("First dimension must be the number of edges "
                             "G.Ne = {}, got {}.".format(self.Ne, tuple(y.shape)))
        return self.D.dot(y)

    # ------------------------------------------------------------------------ lmax
    @property
    def lmax(self):
        r"""Largest eigenvalue of the Laplacian (estimated lazily, with a warning)."""
        if self._lmax is None:
            self.logger.warning("The largest eigenvalue G.lmax is not available, we need to "
                                "estimate it. Explicitly call G.estimate_lmax() or "
                                "G.compute_fourier_basis() once beforehand to suppress the "
                                "warning.")
            self.estimate_lmax()
        return self._lmax

    def estimate_lmax(self, method="lanczos", *, seed=0):
        r"""Estimate the largest eigenvalue of L (cached per method; graph.py:858-931).

        'lanczos' runs a device Lanczos recurrence on the SpMV kernel until the
        Ritz residual is below 5e-3 |theta| (the reference's ARPACK tolerance)
        and returns 1.01 * theta; 'bounds' returns the algebraic upper bound.
        Unlike the reference (unseeded ARPACK start vector) the result is
        reproducible: the start vector is a counter-based function of ``seed``.
        """
        if method == self._lmax_method:
            return
        if method == "lanczos":
            theta = self._lanczos(tol=5e-3, seed=seed)
            bound = self._get_upper_bound()
            slack = 1e-12 if self.dtype == nat.require_cuda().float64 else 1e-5 * abs(bound)
            assert not theta > bound + slack, (theta, bound)
            self._lmax = theta * 1.01
        elif method == "bounds":
            self._lmax = self._get_upper_bound()
        else:
            raise ValueError("Unknown method {}".format(method))
        self._lmax_method = method

    def _lanczos(self, tol, seed, max_steps=400, polish_steps=60):
        """Largest Ritz value of L.

        Stopping rule of the reference (ARPACK, graph.py:911-917): Ritz residual
        |beta_m s_m| <= tol |theta|.  ARPACK checks it only every ncv-1 = 9 products
        and therefore usually overshoots it by far (its Logo estimates agree to
        1e-5); to be as tight, and reproducible to the digits the reference's
        doctest prints, iterations continue -- products are cheap here -- until the
        eigenvalue error estimate resid^2 / (theta_1 - theta_2) is below 1e-5 |theta|
        or ``polish_steps`` products have been spent.
        """
        torch = nat.require_cuda()
        n, L = self.n_vertices, self.L
        if n == 0 or L.nnz == 0:
            return 0.0
        cap = int(min(n, max_steps))
        V = torch.empty(3 * n, dtype=self.dtype, device=self.device)
        scal = torch.zeros(2 * cap + 1 + 4096, dtype=torch.float64, device=self.device)
        done = 0
        theta = None
        converged = False
        while done < cap:
            nxt = min(cap, done + (10 if done == 0 else 5))     # ncv = min(N, 10) first
            self._call("gsp_lanczos", nat.i64(n), nat.i64(L.nnz), L.indptr, L.indices, L.data, V,
                       nat.i32(done), nat.i32(nxt), nat.i32(cap), nat.u64(seed), scal)
            done = nxt
            host = scal.cpu().numpy()
            theta, m, stop, ref_rule = ritz_check(host[:done], host[cap + 1:cap + 1 + done], tol,
                                                  self._sfx == "f32", done >= polish_steps)
            self._lanczos_steps = m
            converged = converged or ref_rule
            if stop:
                return theta
        if converged or cap == n:   # cap == n: the Krylov space is the whole space
            return theta
        raise ValueError("The Lanczos method did not converge. Try to use bounds.")

    def _get_upper_bound(self):
        r"""Algebraic upper bound on the spectrum of L (graph.py:933-960)."""
        if self.lap_type == "normalized":
            return 2
        if self.lap_type != "combinatorial":
            raise ValueError("Unknown Laplacian type {}".format(self.lap_type))
        torch = nat.require_cuda()
        W, Ws, n = self._adjacency, self._symmetric_adjacency(), self.n_vertices
        dw = self._degrees()[0]
        out = torch.empty(5, dtype=torch.float64, device=self.device)
        self._call("gsp_spectral_bounds", nat.i64(n), W.indptr, W.indices, W.data, Ws.indptr,
                   Ws.indices, Ws.data, dw, out)
        max_w, max_dw, max_edge, merris, n_nan = out.cpu().numpy()
        if W.nnz < n * n:                       # np.max of a sparse matrix sees the zeros
            max_w = max(max_w, 0.0)
        bounds = [n * max_w, 2 * max_dw]
        if self.n_edges > 0:
            bounds.append(max_edge)
        bounds.append(float("nan") if n_nan else merris)
        # Python's min() skips a NaN that is not first: with an isolated vertex the
        # reference silently drops the last bound.  Same here.
        return float(min(bounds))

    # -------------------------------------------------- documented non-features
    def compute_fourier_basis(self, *args, **kwargs):
        raise NotImplementedError(
            "The dense eigendecomposition (pygsp/graphs/fourier.py) is outside the Chebyshev "
            "filtering path this engine implements; use estimate_lmax().")


def ritz_check(alpha, beta, tol, single_precision, polish_done):
    """Largest Ritz value of the Lanczos tridiagonal matrix and whether to stop.

    alpha[0..m), beta[0..m): recurrence coefficients so far (beta[j] couples v_j, v_j+1).
    Returns (theta, steps_used, stop).  Stop rule: the reference's (|beta_m s_m| <=
    tol |theta|, graph.py:911-917) and then either the eigenvalue error estimate
    resid^2 / (theta_1 - theta_2) <= 1e-5 |theta| or ``polish_done``; an (almost) zero
    beta_j means an invariant subspace (T_{j+1} exact) and stops at once.
    """
    from scipy.linalg import eigh_tridiagonal
    done = len(alpha)
    scale = max(np.abs(alpha).max(), np.abs(beta).max(), 1e-300)
    floor = (1e-5 if single_precision else 1e-12) * scale
    tiny = np.flatnonzero(beta <= floor)
    m = int(tiny[0]) + 1 if tiny.size else done
    if m == 1:
        theta, second, last = float(alpha[0]), None, 1.0
    else:
        w, v = eigh_tridiagonal(alpha[:m], beta[:m - 1])
        theta, second, last = float(w[-1]), float(w[-2]), abs(float(v[-1, -1]))
    resid = float(beta[m - 1]) * last
    ref_rule = resid <= tol * max(abs(theta), np.finfo(float).eps ** (2.0 / 3))
    gap = max(theta - second, resid) if second is not None else resid
    tight = resid == 0 or resid * resid / max(gap, 1e-300) <= 1e-5 * abs(theta)
    return theta, m, bool(tiny.size or (ref_rule and (tight or polish_done))), ref_rule


def symmetrize_average_device(W):
    """(W + W^T)/2 of a DeviceCSR, on the device (utils.py:247-248)."""
    torch = nat.require_cuda()
    n, dev, sfx = W.shape[0], W.device, nat.suffix(W.dtype)

    def call(name, *args):
        with torch.cuda.device(dev):
            nat.call(name + "_" + sfx, *args, nat.stream_ptr(dev))
    tp = torch.empty(n + 1, dtype=torch.int32, device=dev)
    ti = torch.empty(W.nnz, dtype=torch.int32, device=dev)
    td = torch.empty(W.nnz, dtype=W.dtype, device=dev)
    call("gsp_csr_transpose", nat.i64(n), nat.i64(W.nnz), W.indptr, W.indices, W.data, tp, ti, td)
    sp = torch.empty(n + 1, dtype=torch.int32, device=dev)
    call("gsp_csr_average_count", nat.i64(n), W.indptr, W.indices, W.data, tp, ti, td, sp)
    nnz = int(sp[-1].item()) if n else 0
    si = torch.empty(nnz, dtype=torch.int32, device=dev)
    sd = torch.empty(nnz, dtype=W.dtype, device=dev)
    call("gsp_csr_average_fill", nat.i64(n), W.indptr, W.indices, W.data, tp, ti, td, sp, si, sd)
    return DeviceCSR(sp, si, sd, W.shape)


def _torch_dtype(torch, dtype):
    if dtype is None:
        return torch.float32
    if isinstance(dtype, torch.dtype):
        out = dtype
    else:
        out = {np.dtype("float32"): torch.float32, np.dtype("float64"): torch.float64}.get(
            np.dtype(dtype))
    if out not in (torch.float32, torch.float64):
        raise TypeError("dtype must be float32 or float64")
    return out
