"""ctypes front-ends for the two CPU checkers.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
import this module.  Nothing under rcppsparse_b200/ does (tests/test_boundary.py greps
for that).

  Port  -> oracle/liboracle_port.so     plain-C restatement (oracle_port.c)
  Ref   -> oracle/_ref/liboracle_ref.so the reference header + example.cpp compiled
                                         unmodified against oracle/stub (ref_shim.cpp)

Both take/return numpy arrays in the dgCMatrix layout of reference RcppSparse.h:29-30:
x float64[nnz], i int32[nnz], p int32[ncol+1], Dim = (nrow, ncol).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_SO = os.path.join(HERE, "liboracle_port.so")
REF_SO = os.path.join(HERE, "_ref", "liboracle_ref.so")

_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")


def build(ref: bool = True) -> None:
    """Compile the checkers (the reference one only where /root/reference exists)."""
    targets = ["port"] + (["ref"] if ref else [])
    subprocess.run(["make", "-s", "-C", HERE] + targets, check=True)


def _prep(i, p, x):
    return (np.ascontiguousarray(i, np.int32), np.ascontiguousarray(p, np.int32),
            np.ascontiguousarray(x, np.float64))


class Port:
    """Plain-C restatement; function names follow the reference's."""

    kind = "port"

    def __init__(self):
        if not os.path.exists(PORT_SO):
            build(ref=False)
        L = C.CDLL(PORT_SO)
        L.oport_colSums.argtypes = [_i32p, _f64p, C.c_int, _f64p]
        L.oport_columnSums.argtypes = [_i32p, _f64p, C.c_int, _f64p]
        L.oport_rowSums.argtypes = [_i32p, _i32p, _f64p, C.c_int, C.c_int, _f64p]
        L.oport_colMeans.argtypes = [_i32p, _f64p, C.c_int, C.c_int, _f64p]
        L.oport_rowMeans.argtypes = [_i32p, _i32p, _f64p, C.c_int, C.c_int, _f64p]
        L.oport_transpose.argtypes = [_i32p, _i32p, _f64p, C.c_int, C.c_int, _i32p, _i32p, _f64p]
        L.oport_transpose.restype = C.c_int
        L.oport_spmv.argtypes = [_i32p, _i32p, _f64p, C.c_int, C.c_int, _f64p, _f64p]
        L.oport_spmv_t.argtypes = [_i32p, _i32p, _f64p, C.c_int, _f64p, _f64p]
        L.oport_abs_colSums.argtypes = [_i32p, _f64p, C.c_int, _f64p]
        L.oport_crossprod.argtypes = [_i32p, _i32p, _f64p, C.c_int, _f64p]
        L.oport_crossprod.restype = None
        for f in ("oport_colSums", "oport_columnSums", "oport_rowSums", "oport_colMeans", "oport_rowMeans",
                  "oport_spmv", "oport_spmv_t", "oport_abs_colSums"):
            getattr(L, f).restype = None
        self.L = L

    def colSums(self, i, p, x, nrow, ncol):
        i, p, x = _prep(i, p, x)
        out = np.empty(ncol, np.float64)
        self.L.oport_colSums(p, x, ncol, out)
        return out

    def crossprod(self, i, p, x, nrow, ncol):
        """Dense A^T A as an (ncol, ncol) array (symmetric, so memory order does not matter)."""
        i, p, x = _prep(i, p, x)
        out = np.empty((ncol, ncol), np.float64)
        self.L.oport_crossprod(i, p, x, ncol, out.reshape(-1))
        return out

    def columnSums(self, i, p, x, nrow, ncol):
        i, p, x = _prep(i, p, x)
        out = np.empty(ncol, np.float64)
        self.L.oport_columnSums(p, x, ncol, out)
        return out

    def rowSums(self, i, p, x, nrow, ncol):
        i, p, x = _prep(i, p, x)
        out = np.empty(nrow, np.float64)
        self.L.oport_rowSums(i, p, x, nrow, ncol, out)
        return out

    def colMeans(self, i, p, x, nrow, ncol):
        i, p, x = _prep(i, p, x)
        out = np.empty(ncol, np.float64)
        self.L.oport_colMeans(p, x, nrow, ncol, out)
        return out

    def rowMeans(self, i, p, x, nrow, ncol):
        i, p, x = _prep(i, p, x)
        out = np.empty(nrow, np.float64)
        self.L.oport_rowMeans(i, p, x, nrow, ncol, out)
        return out

    def transpose(self, i, p, x, nrow, ncol):
        i, p, x = _prep(i, p, x)
        nnz = int(p[ncol])
        po = np.empty(nrow + 1, np.int32)
        io = np.empty(nnz, np.int32)
        xo = np.empty(nnz, np.float64)
        if self.L.oport_transpose(i, p, x, nrow, ncol, po, io, xo) != 0:
            raise MemoryError("oport_transpose")
        return io, po, xo

    def spmv(self, i, p, x, nrow, ncol, v):
        i, p, x = _prep(i, p, x)
        out = np.empty(nrow, np.float64)
        self.L.oport_spmv(i, p, x, nrow, ncol, np.ascontiguousarray(v, np.float64), out)
        return out

    def spmv_t(self, i, p, x, nrow, ncol, v):
        i, p, x = _prep(i, p, x)
        out = np.empty(ncol, np.float64)
        self.L.oport_spmv_t(i, p, x, ncol, np.ascontiguousarray(v, np.float64), out)
        return out

    # tolerance denominators (north_star: |delta| <= 1e-12 * sum |a_ij| feeding the output)
    def abs_colSums(self, i, p, x, nrow, ncol):
        i, p, x = _prep(i, p, x)
        out = np.empty(ncol, np.float64)
        self.L.oport_abs_colSums(p, x, ncol, out)
        return out


class Ref:
    """The reference's own compiled code (present when built in the container from /root/reference)."""

    kind = "reference"

    @staticmethod
    def available() -> bool:
        return os.path.exists(REF_SO)

    def __init__(self):
        if not os.path.exists(REF_SO):
            raise FileNotFoundError(REF_SO + " (run `make -C oracle ref` where /root/reference exists)")
        L = C.CDLL(REF_SO)
        common = [_i32p, _i32p, _f64p, C.c_int, C.c_int, C.c_int64]
        for f in ("oref_columnSums", "oref_colSums", "oref_rowSums", "oref_colMeans", "oref_rowMeans"):
            getattr(L, f).argtypes = common + [_f64p]
            getattr(L, f).restype = C.c_int
        L.oref_transpose.argtypes = common + [_i32p, _i32p, _f64p, _i32p]
        L.oref_transpose.restype = C.c_int
        L.oref_spmv.argtypes = common + [_f64p, _f64p]
        L.oref_spmv.restype = C.c_int
        L.oref_spmv_t.argtypes = common + [_f64p, _f64p]
        L.oref_spmv_t.restype = C.c_int
        L.oref_last_error.restype = C.c_char_p
        if hasattr(L, "oref_crossprod"):
            L.oref_crossprod.argtypes = common + [_f64p]
            L.oref_crossprod.restype = C.c_int
        self.L = L

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(self.L.oref_last_error().decode())

    def _vec(self, fn, i, p, x, nrow, ncol, n_out):
        i, p, x = _prep(i, p, x)
        out = np.empty(n_out, np.float64)
        self._check(fn(i, p, x, nrow, ncol, x.shape[0], out))
        return out

    def columnSums(self, i, p, x, nrow, ncol):
        return self._vec(self.L.oref_columnSums, i, p, x, nrow, ncol, ncol)

    def colSums(self, i, p, x, nrow, ncol):
        return self._vec(self.L.oref_colSums, i, p, x, nrow, ncol, ncol)

    def crossprod(self, i, p, x, nrow, ncol):
        i, p, x = _prep(i, p, x)
        ipad = np.concatenate([i, np.array([nrow], np.int32)])  # the reference reads i[] one past a column's end
        out = np.empty((ncol, ncol), np.float64)
        self._check(self.L.oref_crossprod(ipad, p, x, nrow, ncol, x.shape[0], out.reshape(-1)))
        return out

    def rowSums(self, i, p, x, nrow, ncol):
        return self._vec(self.L.oref_rowSums, i, p, x, nrow, ncol, nrow)

    def colMeans(self, i, p, x, nrow, ncol):
        return self._vec(self.L.oref_colMeans, i, p, x, nrow, ncol, ncol)

    def rowMeans(self, i, p, x, nrow, ncol):
        return self._vec(self.L.oref_rowMeans, i, p, x, nrow, ncol, nrow)

    def transpose(self, i, p, x, nrow, ncol):
        i, p, x = _prep(i, p, x)
        nnz = x.shape[0]
        po = np.empty(nrow + 1, np.int32)
        io = np.empty(nnz, np.int32)
        xo = np.empty(nnz, np.float64)
        dim = np.empty(2, np.int32)
        self._check(self.L.oref_transpose(i, p, x, nrow, ncol, nnz, po, io, xo, dim))
        assert dim[0] == ncol and dim[1] == nrow
        return io, po, xo

    def spmv(self, i, p, x, nrow, ncol, v):
        i, p, x = _prep(i, p, x)
        out = np.empty(nrow, np.float64)
        self._check(self.L.oref_spmv(i, p, x, nrow, ncol, x.shape[0], np.ascontiguousarray(v, np.float64), out))
        return out

    def spmv_t(self, i, p, x, nrow, ncol, v):
        i, p, x = _prep(i, p, x)
        out = np.empty(ncol, np.float64)
        self._check(self.L.oref_spmv_t(i, p, x, nrow, ncol, x.shape[0], np.ascontiguousarray(v, np.float64), out))
        return out


def best() -> "Port | Ref":
    """The strongest checker present: the compiled reference where oracle/_ref has been built from a reference
    tree, else the port.  The port needs nothing outside this repository; tests/test_oracle.py holds it bit for
    bit to the committed golden vectors, which the compiled reference produced (and its crossprod, which they do
    not cover, to scipy and a known answer)."""
    return Ref() if Ref.available() else Port()


# ------------------------------------------------------------------------------------------
# tolerance helpers shared by the parity tests (north_star criterion, SURVEY.md 8c)
# ------------------------------------------------------------------------------------------
TOL = 1e-12


def abs_feed(op: str, i, p, x, nrow, ncol, v=None) -> np.ndarray:
    """sum of |terms| feeding each output entry of `op` (terms = a_ij, or a_ij*v_j for SpMV)."""
    i, p, x = _prep(i, p, x)
    ax = np.abs(x)
    col_of = np.repeat(np.arange(ncol), np.diff(p))
    if op in ("colSums", "columnSums"):
        return np.bincount(col_of, weights=ax, minlength=ncol)
    if op == "colMeans":
        return np.bincount(col_of, weights=ax, minlength=ncol) / nrow
    if op == "rowSums":
        return np.bincount(i, weights=ax, minlength=nrow)
    if op == "rowMeans":
        return np.bincount(i, weights=ax, minlength=nrow) / ncol
    if op == "spmv":
        return np.bincount(i, weights=ax * np.abs(np.asarray(v)[col_of]), minlength=nrow)
    if op == "spmv_t":
        return np.bincount(col_of, weights=ax * np.abs(np.asarray(v)[i]), minlength=ncol)
    if op == "crossprod":  # |A|^T |A|, dense (small n only)
        dense = np.zeros((nrow, ncol))
        dense[i, col_of] = ax
        return dense.T @ dense
    raise KeyError(op)


def assert_within(op: str, got, want, i, p, x, nrow, ncol, v=None, tol: float = TOL) -> float:
    """Assert |got-want| <= tol * sum|terms| per entry (NaN/Inf must match exactly); return worst ratio."""
    got = np.asarray(got)
    want = np.asarray(want)
    assert got.shape == want.shape, (got.shape, want.shape)
    fin = np.isfinite(want)
    assert np.array_equal(np.isnan(got), np.isnan(want)), "NaN pattern differs"
    assert np.array_equal(got[~fin & ~np.isnan(want)], want[~fin & ~np.isnan(want)]), "Inf pattern differs"
    feed = abs_feed(op, i, p, x, nrow, ncol, v)
    err = np.abs(got[fin] - want[fin])
    bound = tol * feed[fin]
    bad = err > bound
    assert not bad.any(), f"{op}: {bad.sum()} entries outside {tol}*sum|a|; worst err {err.max():.3e}"
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(feed[fin] > 0, err / feed[fin], 0.0)
    return float(r.max()) if r.size else 0.0
