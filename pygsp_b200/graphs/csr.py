"""CSR matrix resident in HBM: int32 indptr / indices + float32|float64 data.

This is what ``Graph.W`` and ``Graph.L`` are in this engine (the reference
holds ``scipy.sparse.csr_matrix`` objects, graph.py:109,620).  It offers the
small read-only surface the filtering path and its callers use: ``shape``,
``nnz``, ``dot``, ``toarray``, ``diagonal``, plus ``to_scipy`` to leave the
device.  ``DifferentialOperator`` holds ``Graph.D`` (the reference's CSC
matrix, difference.py) in the two layouts its gradient and divergence walk.
"""
import numpy as np

from .. import _native as nat


class DeviceCSR:
    def __init__(self, indptr, indices, data, shape):
        self.indptr = indptr
        self.indices = indices
        self.data = data
        self.shape = (int(shape[0]), int(shape[1]))
        self._plans = {}

    def tile_plan(self, nsig, nscales):
        """Tiling of the float32 TMA path for this matrix (cached; None = row-group kernel)."""
        torch = nat.require_cuda()
        if self.data.dtype != torch.float32:
            return None
        key = (int(nsig), int(nscales))
        if key not in self._plans:
            plan = nat.TilePlan()
            with torch.cuda.device(self.device):
                nat.call("gsp_cheby_tile_plan", nat.i64(self.shape[0]), self.indptr,
                         nat.i64(nsig), nat.i32(nscales), plan, nat.stream_ptr(self.device))
            self._plans[key] = plan if plan.rows_per_tile > 0 else None
        return self._plans[key]

    # -- construction ---------------------------------------------------------
    @classmethod
    def from_scipy(cls, M, dtype, device):
        torch = nat.require_cuda()
        M = M.tocsr()
        if M.nnz >= 2 ** 31:
            raise ValueError("nnz must fit int32 indices")
        indptr = torch.from_numpy(np.ascontiguousarray(M.indptr, dtype=np.int32)).to(device)
        indices = torch.from_numpy(np.ascontiguousarray(M.indices, dtype=np.int32)).to(device)
        data = torch.from_numpy(np.ascontiguousarray(M.data)).to(device=device, dtype=dtype)
        return cls(indptr, indices, data, M.shape)

    # -- introspection --------------------------------------------------------
    @property
    def nnz(self):
        return int(self.indices.numel())

    @property
    def dtype(self):
        return self.data.dtype

    @property
    def device(self):
        return self.data.device

    def __repr__(self):
        return "<DeviceCSR {}x{}, nnz={}, {}, {}>".format(
            self.shape[0], self.shape[1], self.nnz, self.data.dtype, self.data.device)

    # -- leaving the device -----------------------------------------------------
    def to_scipy(self):
        from scipy import sparse
        return sparse.csr_matrix((self.data.cpu().numpy(), self.indices.cpu().numpy(),
                                  self.indptr.cpu().numpy()), shape=self.shape)

    def toarray(self):
        return self.to_scipy().toarray()

    def diagonal(self):
        return self.to_scipy().diagonal()

    # -- product: scipy's csr_matrix.dot on the device SpMM kernel ------------------
    def dot(self, x):
        """``A @ x`` for a vector or an (n, nsig) block; numpy in -> numpy out."""
        torch = nat.require_cuda()
        host = not torch.is_tensor(x)
        xt = torch.as_tensor(np.asarray(x) if host else x).to(device=self.device, dtype=self.dtype)
        if xt.shape[0] != self.shape[1]:
            raise ValueError("dimension mismatch")
        flat = xt.reshape(xt.shape[0], -1).contiguous()
        y = torch.empty((self.shape[0], flat.shape[1]), dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            if flat.shape[1] == 1:                      # one vector: the sub-warp SpMV
                nat.call("gsp_spmv_" + nat.suffix(self.dtype), nat.i64(self.shape[0]),
                         nat.i64(self.nnz), self.indptr, self.indices, self.data, flat, y,
                         nat.stream_ptr(self.device))
            else:
                nat.call("gsp_spmm_" + nat.suffix(self.dtype), nat.i64(self.shape[0]),
                         self.indptr, self.indices, self.data, flat, nat.i64(flat.shape[1]), y,
                         nat.stream_ptr(self.device))
        y = y.reshape((self.shape[0],) + tuple(xt.shape[1:]))
        return y.cpu().numpy() if host else y

    __matmul__ = dot


class DifferentialOperator:
    """The N x Ne differential operator ``G.D`` (difference.py), held in HBM in two layouts.

    The edge-major layout is SciPy's CSC arrays of D (``d_indptr`` over edges, vertex indices,
    values), which is what ``grad`` walks; the vertex-major layout is D as CSR (edge ids
    ascending in a row), which is what ``div`` walks.  ``to_scipy()`` returns the reference's
    ``csc_matrix``; ``dot(y)`` is ``div`` and ``T.dot(x)`` is ``grad``, both on the exact-order
    kernels of csrc/diffop.cu (results equal SciPy's on the same D bit for bit).  Not a
    :class:`DeviceCSR`: D is rectangular and Ne < N happens.
    """

    def __init__(self, shape, d_indptr, d_indices, d_data, v_indptr, v_indices, v_data):
        self.shape = (int(shape[0]), int(shape[1]))
        self.d_indptr, self.d_indices, self.d_data = d_indptr, d_indices, d_data
        self.v_indptr, self.v_indices, self.v_data = v_indptr, v_indices, v_data
        self.T = _TransposedOperator(self)

    @property
    def nnz(self):
        return int(self.d_indices.numel())

    @property
    def dtype(self):
        return self.d_data.dtype

    @property
    def device(self):
        return self.d_data.device

    def __repr__(self):
        return "<DifferentialOperator {}x{}, nnz={}, {}, {}>".format(
            self.shape[0], self.shape[1], self.nnz, self.dtype, self.device)

    def to_scipy(self):
        from scipy import sparse
        return sparse.csc_matrix((self.d_data.cpu().numpy(), self.d_indices.cpu().numpy(),
                                  self.d_indptr.cpu().numpy()), shape=self.shape)

    def toarray(self):
        return self.to_scipy().toarray()

    def dot(self, y):
        """``D @ y`` (the divergence) for an edge vector or an (Ne, nsig) block."""
        return self._product("gsp_div_", self.shape[1], self.shape[0], self.v_indptr,
                             self.v_indices, self.v_data, y)

    __matmul__ = dot

    def _product(self, fn, n_in, n_out, indptr, indices, data, x):
        torch = nat.require_cuda()
        host = not torch.is_tensor(x)
        xt = torch.as_tensor(np.asarray(x) if host else x).to(device=self.device, dtype=self.dtype)
        if xt.ndim == 0 or xt.shape[0] != n_in:
            raise ValueError("dimension mismatch")
        nsig = int(np.prod(xt.shape[1:], dtype=np.int64))
        flat = xt.reshape(n_in, nsig).contiguous()
        out = torch.empty((n_out, nsig), dtype=self.dtype, device=self.device)
        if out.numel():
            with torch.cuda.device(self.device):
                nat.call(fn + nat.suffix(self.dtype), nat.i64(n_out), indptr, indices, data, flat,
                         nat.i64(nsig), out, nat.stream_ptr(self.device))
        out = out.reshape((n_out,) + tuple(xt.shape[1:]))
        return out.cpu().numpy() if host else out


class _TransposedOperator:
    """``D.T``: its ``dot(x)`` is the gradient (D^T x), over the edge-major layout."""

    def __init__(self, D):
        self._D = D

    @property
    def shape(self):
        return (self._D.shape[1], self._D.shape[0])

    def dot(self, x):
        D = self._D
        return D._product("gsp_grad_", D.shape[0], D.shape[1], D.d_indptr, D.d_indices,
                          D.d_data, x)

    __matmul__ = dot
