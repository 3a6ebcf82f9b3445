"""Compiles oracle/cheby_oracle.c with gcc into oracle/_build/libcheby_oracle.so
(test infrastructure; building the checker is not using it)."""
import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_build")
LIB = os.path.join(OUT, "libcheby_oracle.so")
_lib = None


def build(force=False):
    os.makedirs(OUT, exist_ok=True)
    src = os.path.join(HERE, "cheby_oracle.c")
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(src):
        # -ffp-contract=off: the exact step oracles round every product separately, as
        # the kernels do (gcc would otherwise fuse a*b + c on aarch64 hosts)
        subprocess.check_call(["gcc", "-O3", "-fopenmp", "-fPIC", "-shared", "-ffp-contract=off",
                               src, "-o", LIB, "-lm"])
    return LIB


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


def cheby_op(L, lmax, c, signal):
    """float64 C oracle of approximations.cheby_op; L is a scipy CSR matrix."""
    c = np.ascontiguousarray(np.atleast_2d(np.asarray(c, dtype=np.float64)))
    x = np.ascontiguousarray(np.asarray(signal, dtype=np.float64))
    n = L.shape[0]
    x2 = x.reshape(n, -1)
    nsig = x2.shape[1]
    r = np.empty((c.shape[0] * n, nsig))
    Ap = np.ascontiguousarray(L.indptr, dtype=np.int32)
    Aj = np.ascontiguousarray(L.indices, dtype=np.int32)
    Ax = np.ascontiguousarray(L.data, dtype=np.float64)
    P = ctypes.c_void_p
    rc = lib().cheby_op(ctypes.c_int64(n), P(Ap.ctypes.data), P(Aj.ctypes.data), P(Ax.ctypes.data),
                        ctypes.c_double(lmax), P(c.ctypes.data), ctypes.c_int64(c.shape[0]),
                        ctypes.c_int64(c.shape[1]), P(x2.ctypes.data), ctypes.c_int64(nsig),
                        P(r.ctypes.data))
    if rc == -1:
        raise TypeError("The coefficients have an invalid shape")
    if rc != 0:
        raise MemoryError("cheby_oracle")
    return r.reshape((c.shape[0] * n,) + x.shape[1:])


def cheby_step_exact(first, row_begin, row_end, indptr, indices, data, x_cur, x_old, x_new, r,
                     r_rows, nscales, ck, c0, alpha, beta, gamma, add_source=False):
    """Bit-exact host restatement of ``gsp_cheby_step_*`` (include/gspb200.h) in the dtype of
    ``data`` (float32 or float64): rows [row_begin, row_end) of ``x_new`` (n, nsig) and of
    ``r`` (>= nscales, r_rows, nsig) are written in place.  ``x_old`` may be ``x_new`` and is
    ignored (may be None) on the first step.  ``add_source``: Clenshaw form,
    x_new += sum_i ck_i r_i and r is only read (not part of the C ABI)."""
    data = np.asarray(data)
    if data.dtype == np.float32:
        fn, dt = lib().cheby_step_exact_f32, np.float32
    elif data.dtype == np.float64:
        fn, dt = lib().cheby_step_exact_f64, np.float64
    else:
        raise TypeError("float32 / float64 only")
    fn.restype = None
    arrays = [x_cur, x_new] + ([x_old] if x_old is not None else []) + ([r] if r is not None else [])
    for a in arrays:
        if a.dtype != dt or not a.flags.c_contiguous:
            raise TypeError("contiguous %s arrays expected" % np.dtype(dt).name)
    if not x_new.flags.writeable or (r is not None and not r.flags.writeable):
        raise ValueError("x_new / r must be writeable")
    nsig = x_cur.shape[1] if x_cur.ndim == 2 else 1
    Ap = np.ascontiguousarray(indptr, dtype=np.int32)
    Aj = np.ascontiguousarray(indices, dtype=np.int32)
    Ax = np.ascontiguousarray(data, dtype=dt)
    ck = np.ascontiguousarray(np.asarray(ck, dtype=np.float64).reshape(-1))
    c0 = np.ascontiguousarray(np.asarray(c0, dtype=np.float64).reshape(-1))
    if ck.size < nscales or c0.size < nscales:
        raise ValueError("one ck / c0 per scale")
    if r is not None and r.size < nscales * r_rows * nsig:
        raise ValueError("r is too small")
    if not (0 <= row_begin <= row_end <= len(Ap) - 1 <= x_new.shape[0]):
        raise ValueError("row range outside the matrix")
    P = ctypes.c_void_p
    ptr = lambda a: P(a.ctypes.data) if a is not None and a.size else P(0)
    fn(ctypes.c_int(int(bool(first))), ctypes.c_int(int(bool(add_source))),
       ctypes.c_int64(row_begin), ctypes.c_int64(row_end), ptr(Ap), ptr(Aj), ptr(Ax),
       ptr(x_cur), ptr(x_old), ptr(x_new), ptr(r), ctypes.c_int64(r_rows), ctypes.c_int64(nsig),
       ctypes.c_int64(nscales), ptr(ck), ptr(c0), ctypes.c_double(alpha), ctypes.c_double(beta),
       ctypes.c_double(gamma))


if __name__ == "__main__":
    print(build(force=True))
