"""Host-side mirror of the reference's interface for the hot path, over the C ABI.

R and Rcpp are not installed in this image, so the reference-facing surface that tests and
benchmarks drive is this Python mirror of ``RcppSparse::Matrix`` (reference
inst/include/RcppSparse.h:25-395) and of the exported ``columnSums`` (src/example.cpp:26-32,
R/RcppExports.R:26-28).  Names, argument meaning and error behaviour follow the reference; the
C++ drop-in header ``include/RcppSparse.h`` is the same thing for real R/Rcpp builds and calls
the same ``sb200_*`` entry points.

Two layers:
  * ``DeviceMatrix`` — thin owner of one ``sb200_matrix*`` (one dgCMatrix or one column shard
    resident in HBM); device-pointer methods used by the sharding layer and bench.py.
  * ``Matrix`` — the reference-shaped class: public ``x, i, p, Dim`` numpy members that ALIAS
    the caller's arrays (zero-copy view, README.md:7-9), host-array results.

Nothing here computes on the CPU: every sweep is a kernel launch behind the C ABI, and
importing this module without the built library raises.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import SparseB200Error, check


def _ptr(a) -> C.c_void_p:
    """Raw address of a numpy array, a torch tensor (data_ptr), an int, or None."""
    if a is None:
        return C.c_void_p(0)
    if isinstance(a, int):
        return C.c_void_p(a)
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    raise TypeError(f"cannot take the address of {type(a)}")


class DeviceMatrix:
    """Owner of one device-resident mirror (``sb200_matrix*``)."""

    def __init__(self, handle: int, keepalive=None):
        self._h = C.c_void_p(handle)
        self._keep = keepalive  # tensors whose memory the handle borrows (adopt)
        nrow, ncol, nnz = C.c_int32(), C.c_int32(), C.c_int64()
        check(_lib.lib().sb200_matrix_dims(self._h, C.byref(nrow), C.byref(ncol), C.byref(nnz)))
        self.nrow, self.ncol, self.nnz = nrow.value, ncol.value, nnz.value

    # ---- construction ---------------------------------------------------------------------------
    @classmethod
    def from_host(cls, i, p, x, nrow: int, ncol: int, device: int = 0, pin: bool = False,
                  validate: bool = True, lazy_rows: bool = False) -> "DeviceMatrix":
        """Upload host i/p/x (numpy or pinned torch CPU tensors). reference: Exporter::get(), RcppSparse.h:417-419.
        lazy_rows (SB200_LAZY_ROWS): `i` goes up only when an op reads it — colSums / colMeans never do (the reference's
        loops do not either, RcppSparse.h:133-135); the array is kept alive by the object and must not change meanwhile."""
        nnz = int(x.shape[0])
        if isinstance(i, np.ndarray):
            if i.dtype != np.int32 or p.dtype != np.int32 or x.dtype != np.float64:
                raise TypeError("dgCMatrix slots are int32 i/p and float64 x (reference RcppSparse.h:29-30)")
            if not (i.flags.c_contiguous and p.flags.c_contiguous and x.flags.c_contiguous):
                raise ValueError("slot arrays must be contiguous")
        if int(p.shape[0]) != ncol + 1:
            raise ValueError("p must have ncol + 1 entries")
        flags = (_lib.PIN_HOST if pin else 0) | (0 if validate else _lib.NO_VALIDATE) | (_lib.LAZY_ROWS if lazy_rows else 0)
        out = C.c_void_p()
        check(_lib.lib().sb200_matrix_create(_ptr(i), _ptr(p), _ptr(x), nrow, ncol, nnz, device, flags, C.byref(out)))
        obj = cls(out.value)
        if lazy_rows:
            obj._lazy_i = i  # the library reads it on the first row-indexed call
        return obj

    @classmethod
    def adopt(cls, d_i, d_p, d_x, nrow: int, ncol: int, device: int = 0, validate: bool = False) -> "DeviceMatrix":
        """Wrap CUDA tensors (int32, int32, float64) without copying; they are kept alive by the object."""
        nnz = int(d_x.shape[0])
        out = C.c_void_p()
        flags = 0 if validate else _lib.NO_VALIDATE
        check(_lib.lib().sb200_matrix_adopt_device(_ptr(d_i), _ptr(d_p), _ptr(d_x), nrow, ncol, nnz, device, flags,
                                                   C.byref(out)))
        return cls(out.value, keepalive=(d_i, d_p, d_x))

    @classmethod
    def synth(cls, spec, col_begin: int = 0, col_end: int | None = None, device: int = 0) -> "DeviceMatrix":
        """Generate columns [col_begin, col_end) of a synth.SynthSpec directly in HBM."""
        if col_end is None:
            col_end = spec.ncol
        out = C.c_void_p()
        check(_lib.lib().sb200_synth_create(
            spec.nrow, col_begin, col_end, spec.seed, _ptr(spec.len_table), spec.empty_permille, spec.n_bands,
            _ptr(spec.band_lo), _ptr(spec.band_hi), _ptr(spec.band_w), device, C.byref(out)))
        return cls(out.value)

    # ---- lifetime ---------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            _lib.lib().sb200_matrix_destroy(self._h)
            self._h = C.c_void_p(0)
            self._keep = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- plumbing ------------------------------------------------------------------------------------
    def set_stream(self, cuda_stream: int) -> None:
        check(_lib.lib().sb200_matrix_set_stream(self._h, C.c_void_p(cuda_stream)))

    def sync(self) -> None:
        check(_lib.lib().sb200_matrix_sync(self._h))

    def device_arrays(self):
        a, b, c = C.c_void_p(), C.c_void_p(), C.c_void_p()
        check(_lib.lib().sb200_matrix_device_arrays(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def algorithmic_bytes(self, op: str) -> int:
        n = C.c_int64()
        check(_lib.lib().sb200_algorithmic_bytes(self._h, op.encode(), C.byref(n)))
        return n.value

    def row_path(self) -> str:
        """'banded' or 'l2-atomics': which kernel serves rowSums / rowMeans / A v for this matrix;
        'row-companion' once rowSums / rowMeans / A v run on the row-ordered copy."""
        b = C.c_int()
        check(_lib.lib().sb200_matrix_row_path(self._h, C.byref(b)))
        return ("l2-atomics", "banded", "row-companion")[b.value]

    def row_companion(self, action: int = 1) -> None:
        """1 build the row-ordered copy now, 0 drop it, -1 drop and never build (sparse_b200.h)."""
        check(_lib.lib().sb200_matrix_row_companion(self._h, int(action)))

    def band_companion(self, which: int = 0, action: int = 1) -> None:
        """Band-major companion (sparse_b200.h): which 0 = the layout A^T v runs on, 1 = the layout A v runs on
        (builds the row-ordered copy too); action 1 build now, 0 drop, -1 drop and never build."""
        check(_lib.lib().sb200_matrix_band_companion(self._h, int(which), int(action)))

    def layouts(self) -> int:
        """Bit mask: 1 row-ordered copy, 2 band-major companion (A^T v), 4 the copy's companion (A v), 8 transpose plan."""
        m = C.c_int()
        check(_lib.lib().sb200_matrix_layouts(self._h, C.byref(m)))
        return m.value

    def layout_bytes(self) -> int:
        """HBM the cached layouts occupy beside i/p/x (row-ordered copy + band-major companions)."""
        n = C.c_int64()
        check(_lib.lib().sb200_matrix_layout_bytes(self._h, C.byref(n)))
        return n.value

    def refresh_values(self, x) -> None:
        check(_lib.lib().sb200_matrix_refresh_values(self._h, _ptr(x)))

    def download_columns(self, c0: int = 0, c1: int | None = None):
        if c1 is None:
            c1 = self.ncol
        n = C.c_int64()
        check(_lib.lib().sb200_matrix_download_columns(self._h, c0, c1, None, None, None, C.byref(n)))
        i = np.empty(n.value, np.int32)
        p = np.empty(c1 - c0 + 1, np.int32)
        x = np.empty(n.value, np.float64)
        check(_lib.lib().sb200_matrix_download_columns(self._h, c0, c1, _ptr(i), _ptr(p), _ptr(x), C.byref(n)))
        return i, p, x

    # ---- host-buffer sweeps (what the C++ header calls) --------------------------------------------------
    def _host_vec(self, fn, n, out=None):
        """out: optional caller-owned result buffer (float64 numpy array or pinned torch CPU tensor of n entries),
        as in the C ABI; a fresh numpy array otherwise."""
        if out is None:
            out = np.empty(n, np.float64)
        elif int(out.shape[0]) != n or (isinstance(out, np.ndarray) and (out.dtype != np.float64 or not out.flags.c_contiguous)):
            raise ValueError(f"out must be a contiguous float64 buffer of {n} entries")
        check(fn(self._h, _ptr(out)))
        return out

    def col_sums(self, out=None):
        return self._host_vec(_lib.lib().sb200_col_sums, self.ncol, out)

    def row_sums(self, out=None):
        return self._host_vec(_lib.lib().sb200_row_sums, self.nrow, out)

    def col_means(self, out=None):
        return self._host_vec(_lib.lib().sb200_col_means, self.ncol, out)

    def row_means(self, out=None):
        return self._host_vec(_lib.lib().sb200_row_means, self.nrow, out)

    def col_vars(self, out=None):
        """Sample variance of every column, implicit zeros included, over nrow - 1 (R's var(A[, c])); two passes around
        the col_means result (sparse_b200.h sb200_col_vars).  NaN everywhere when nrow < 2."""
        return self._host_vec(_lib.lib().sb200_col_vars, self.ncol, out)

    def row_vars(self, out=None):
        """Sample variance of every row over ncol - 1 (R's var(A[r, ])), around the row_means result."""
        return self._host_vec(_lib.lib().sb200_row_vars, self.nrow, out)

    def crossprod(self):
        """Dense A^T A, (ncol, ncol), exactly symmetric (reference Matrix::crossprod(), RcppSparse.h:158-194)."""
        out = np.empty((self.ncol, self.ncol), np.float64)
        check(_lib.lib().sb200_crossprod(self._h, _ptr(out)))
        return out

    def crossprod_dev(self, d_out) -> None:
        check(_lib.lib().sb200_crossprod_dev(self._h, _ptr(d_out)))

    def spmv(self, v):
        v = np.ascontiguousarray(v, np.float64)
        if v.shape[0] != self.ncol:
            raise ValueError("A v: v must have ncol entries")
        y = np.empty(self.nrow, np.float64)
        check(_lib.lib().sb200_spmv(self._h, _ptr(v), _ptr(y)))
        return y

    def spmv_t(self, v):
        v = np.ascontiguousarray(v, np.float64)
        if v.shape[0] != self.nrow:
            raise ValueError("A^T v: v must have nrow entries")
        y = np.empty(self.ncol, np.float64)
        check(_lib.lib().sb200_spmv_t(self._h, _ptr(v), _ptr(y)))
        return y

    # ---- sparse x dense block: k right-hand sides in one sweep (sparse_b200.h sb200_spmm) ---------------------------
    def _spmm(self, fn, B, rows: int, out_rows: int, what: str):
        B = np.asarray(B)
        if B.ndim != 2 or B.shape[0] != rows:
            raise ValueError(f"{what}: B must be a 2-D array with {rows} rows")
        B = np.asfortranarray(B, np.float64)
        k = int(B.shape[1])
        Y = np.empty((out_rows, k), np.float64, order="F")
        check(fn(self._h, _ptr(B), k, _ptr(Y)))
        return Y

    def spmm(self, B):
        """A B for a dense (ncol, k) block, as a Fortran-ordered (nrow, k) array: k products A v in one sweep."""
        return self._spmm(_lib.lib().sb200_spmm, B, self.ncol, self.nrow, "A B")

    def spmm_t(self, B):
        """A^T B for a dense (nrow, k) block, as a Fortran-ordered (ncol, k) array: k products A^T v in one sweep."""
        return self._spmm(_lib.lib().sb200_spmm_t, B, self.nrow, self.ncol, "A^T B")

    # ---- range cursors and dense extraction as batched device ops (SURVEY.md 8f N4) --------------------------------
    def col_sums_in_rows(self, rows, negate: bool = False):
        """Per column, the sum over the entries whose row is (negate: is not) in ``rows`` — every column's
        InnerIteratorInRange / InnerIteratorNotInRange sweep at once (reference RcppSparse.h:238-321)."""
        rows = np.ascontiguousarray(rows, np.int32)
        out = np.empty(self.ncol, np.float64)
        check(_lib.lib().sb200_col_sums_in_rows(self._h, _ptr(rows), int(rows.shape[0]), 1 if negate else 0, _ptr(out)))
        return out

    def gather_block(self, rows=None, cols=None):
        """Dense A[rows, cols] (reference :76-128 operator()(IntegerVector, IntegerVector), col(...), row(...));
        None = every row / column."""
        r = None if rows is None else np.ascontiguousarray(rows, np.int32)
        c = None if cols is None else np.ascontiguousarray(cols, np.int32)
        nr = self.nrow if r is None else int(r.shape[0])
        nc = self.ncol if c is None else int(c.shape[0])
        out = np.empty((nc, nr), np.float64)  # column-major nr x nc
        check(_lib.lib().sb200_gather_block(self._h, _ptr(r), nr, _ptr(c), nc, _ptr(out)))
        return out.T

    def transpose_host(self):
        p = np.empty(self.nrow + 1, np.int32)
        i = np.empty(self.nnz, np.int32)
        x = np.empty(self.nnz, np.float64)
        check(_lib.lib().sb200_transpose(self._h, _ptr(p), _ptr(i), _ptr(x)))
        return i, p, x

    # ---- device-buffer sweeps (asynchronous on the handle's stream) -----------------------------------------
    def col_sums_dev(self, d_out, divisor: float = 0.0) -> None:
        check(_lib.lib().sb200_col_sums_dev(self._h, divisor, _ptr(d_out)))

    def row_sums_dev(self, d_out, divisor: float = 0.0) -> None:
        check(_lib.lib().sb200_row_sums_dev(self._h, divisor, _ptr(d_out)))

    def col_vars_dev(self, d_out) -> None:
        check(_lib.lib().sb200_col_vars_dev(self._h, _ptr(d_out)))

    def row_vars_dev(self, d_out) -> None:
        check(_lib.lib().sb200_row_vars_dev(self._h, _ptr(d_out)))

    def spmv_dev(self, d_v, d_y) -> None:
        check(_lib.lib().sb200_spmv_dev(self._h, _ptr(d_v), _ptr(d_y)))

    def spmv_t_dev(self, d_v, d_y) -> None:
        check(_lib.lib().sb200_spmv_t_dev(self._h, _ptr(d_v), _ptr(d_y)))

    def spmm_dev(self, d_B, k: int, d_Y) -> None:
        """d_Y (nrow x k) = A d_B (ncol x k), both column-major device buffers (e.g. torch tensors whose transpose is
        contiguous)."""
        check(_lib.lib().sb200_spmm_dev(self._h, _ptr(d_B), int(k), _ptr(d_Y)))

    def spmm_t_dev(self, d_B, k: int, d_Y) -> None:
        """d_Y (ncol x k) = A^T d_B (nrow x k), both column-major device buffers."""
        check(_lib.lib().sb200_spmm_t_dev(self._h, _ptr(d_B), int(k), _ptr(d_Y)))

    def vec_div_dev(self, d, n: int, divisor: float) -> None:
        check(_lib.lib().sb200_vec_div_dev(self._h, _ptr(d), n, divisor))

    def transpose_dev(self) -> "DeviceMatrix":
        out = C.c_void_p()
        check(_lib.lib().sb200_transpose_dev(self._h, C.byref(out)))
        return DeviceMatrix(out.value)

    def transpose_into(self, t: "DeviceMatrix") -> None:
        """The transpose again, into a result of `transpose_dev` of this structure: no allocation (sparse_b200.h)."""
        check(_lib.lib().sb200_transpose_into(self._h, t._h))

    def synth_vector_dev(self, seed: int, begin: int, n: int, d_out) -> None:
        check(_lib.lib().sb200_synth_vector_dev(self._h, seed, begin, n, _ptr(d_out)))


class ShardedHostMatrix:
    """One process, several GPUs: owner of one ``sb200_sharded*`` (sparse_b200.h) — the dgCMatrix cut into nnz-balanced
    column blocks, one per device, behind the same host-vector entry points as a single-GPU mirror."""

    def __init__(self, i, p, x, nrow: int, ncol: int, n_gpus: int, devices=None, validate: bool = True):
        if isinstance(i, np.ndarray) and (i.dtype != np.int32 or p.dtype != np.int32 or x.dtype != np.float64):
            raise TypeError("dgCMatrix slots are int32 i/p and float64 x (reference RcppSparse.h:29-30)")
        if int(p.shape[0]) != ncol + 1:
            raise ValueError("p must have ncol + 1 entries")
        dev = None if devices is None else np.ascontiguousarray(devices, np.int32)
        out = C.c_void_p()
        check(_lib.lib().sb200_sharded_create(_ptr(i), _ptr(p), _ptr(x), nrow, ncol, int(x.shape[0]), int(n_gpus), _ptr(dev),
                                              0 if validate else _lib.NO_VALIDATE, C.byref(out)))
        self._h = out
        self.nrow, self.ncol, self.nnz, self.n_gpus = nrow, ncol, int(x.shape[0]), int(n_gpus)

    def bounds(self):
        b = np.zeros(self.n_gpus + 1, np.int64)
        n = C.c_int()
        check(_lib.lib().sb200_sharded_info(self._h, C.byref(n), _ptr(b)))
        return b.tolist()

    def block(self, k: int) -> "DeviceMatrix":
        """Block k's mirror, borrowed (tuning: cached layouts); do not close it."""
        h = C.c_void_p()
        check(_lib.lib().sb200_sharded_block(self._h, k, C.byref(h)))
        d = DeviceMatrix.__new__(DeviceMatrix)
        d._h, d._keep = h, self
        nrow, ncol, nnz = C.c_int32(), C.c_int32(), C.c_int64()
        check(_lib.lib().sb200_matrix_dims(h, C.byref(nrow), C.byref(ncol), C.byref(nnz)))
        d.nrow, d.ncol, d.nnz = nrow.value, ncol.value, nnz.value
        d.close = lambda: None
        return d

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            _lib.lib().sb200_sharded_destroy(self._h)
            self._h = C.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _vec(self, fn, n, *args):
        out = np.empty(n, np.float64)
        check(fn(self._h, *args, _ptr(out)))
        return out

    def col_sums(self):
        return self._vec(_lib.lib().sb200_sharded_col_sums, self.ncol)

    def row_sums(self):
        return self._vec(_lib.lib().sb200_sharded_row_sums, self.nrow)

    def col_means(self):
        return self._vec(_lib.lib().sb200_sharded_col_means, self.ncol)

    def row_means(self):
        return self._vec(_lib.lib().sb200_sharded_row_means, self.nrow)

    def col_vars(self):
        """Column variances on every GPU of the handle (sparse_b200.h sb200_sharded_col_vars)."""
        return self._vec(_lib.lib().sb200_sharded_col_vars, self.ncol)

    def row_vars(self):
        """Row variances on every GPU of the handle: per-block sums of squares and counts, reduced in block order."""
        return self._vec(_lib.lib().sb200_sharded_row_vars, self.nrow)

    def spmv(self, v):
        v = np.ascontiguousarray(v, np.float64)
        if v.shape[0] != self.ncol:
            raise ValueError("A v: v must have ncol entries")
        return self._vec(_lib.lib().sb200_sharded_spmv, self.nrow, _ptr(v))

    def spmv_t(self, v):
        v = np.ascontiguousarray(v, np.float64)
        if v.shape[0] != self.nrow:
            raise ValueError("A^T v: v must have nrow entries")
        return self._vec(_lib.lib().sb200_sharded_spmv_t, self.ncol, _ptr(v))

    # the same argument checks and column-major handling as the one-GPU block products
    _spmm = DeviceMatrix._spmm

    def spmm(self, B):
        """A B for a dense (ncol, k) block on every GPU of the handle, as a Fortran-ordered (nrow, k) array
        (sparse_b200.h sb200_sharded_spmm)."""
        return self._spmm(_lib.lib().sb200_sharded_spmm, B, self.ncol, self.nrow, "A B")

    def spmm_t(self, B):
        """A^T B for a dense (nrow, k) block on every GPU of the handle, as a Fortran-ordered (ncol, k) array."""
        return self._spmm(_lib.lib().sb200_sharded_spmm_t, B, self.nrow, self.ncol, "A^T B")

    def transpose_host(self):
        """CSC(A^T) of the whole matrix: local transposes on every GPU, row pieces exchanged over peer memory, every
        GPU copies its rows home (sparse_b200.h sb200_sharded_transpose; reference RcppSparse.h:375-385)."""
        p = np.empty(self.nrow + 1, np.int32)
        i = np.empty(self.nnz, np.int32)
        x = np.empty(self.nnz, np.float64)
        check(_lib.lib().sb200_sharded_transpose(self._h, _ptr(p), _ptr(i), _ptr(x)))
        return i, p, x

    def crossprod(self):
        """Dense A^T A, (ncol, ncol), on every GPU of the handle: the reference's result bit for bit, exactly symmetric
        (sparse_b200.h sb200_sharded_crossprod; reference RcppSparse.h:158-194)."""
        out = np.empty((self.ncol, self.ncol), np.float64)
        check(_lib.lib().sb200_sharded_crossprod(self._h, _ptr(out)))
        return out


class Matrix:
    """Python mirror of ``RcppSparse::Matrix`` (reference RcppSparse.h:25-395), hot-path members.

    Public members ``x, i, p, Dim`` alias the arrays passed in (no copy), like the Rcpp handles
    of RcppSparse.h:29-30.  The reference's methods read those vectors LIVE on every call and its vignette
    edits them in place (vignettes/Documentation.Rmd:325-347), so by default nothing outlives a call here either:
    every method uploads the slots as they are now, runs, and drops the device mirror — what a fresh Matrix per
    ``.Call`` pays anyway (src/RcppExports.cpp:20).  ``resident=True`` (or ``resident()``) keeps the mirror, and
    the layouts the library caches on it, between calls; it is tied to THIS object (SURVEY.md H4: never cached
    by host address), rebuilt when a member is re-pointed, and after an in-place edit of ``x`` it needs
    ``refresh()`` (of ``i``/``p``: ``release()``).  ``gpus > 1`` (default: SB200_GPUS) runs every op on that many
    GPUs of this process (sb200_sharded_*).
    """

    def __init__(self, x=None, i=None, p=None, Dim=None, device: int = 0, pin: bool = False, resident: bool = False,
                 gpus: int | None = None):
        # RcppSparse.h:33 (four vectors) and :42 (default)
        self.x = np.zeros(0, np.float64) if x is None else x
        self.i = np.zeros(0, np.int32) if i is None else i
        self.p = np.zeros(1, np.int32) if p is None else p
        self.Dim = np.zeros(2, np.int32) if Dim is None else np.asarray(Dim, dtype=np.int32)
        self._device = device
        self._pin = pin
        self._resident = bool(resident)
        import os as _os
        self._gpus = max(1, int(gpus if gpus is not None else _os.environ.get("SB200_GPUS", "1")))
        self._dev: DeviceMatrix | None = None
        self._sharded: ShardedHostMatrix | None = None
        self._src = None

    @classmethod
    def from_S4(cls, s, **kw) -> "Matrix":
        """RcppSparse.h:34-41: any object with x/i/p/Dim slots; throws like the reference if one is missing.
        scipy.sparse CSC matrices (data/indices/indptr/shape) are accepted as the dgCMatrix of this host language."""
        if all(hasattr(s, a) for a in ("data", "indices", "indptr", "shape")) and not hasattr(s, "Dim"):
            if getattr(s, "format", "csc") != "csc":
                raise ValueError("Cannot construct RcppSparse::Matrix from this S4 object")
            return cls(np.ascontiguousarray(s.data, np.float64), np.ascontiguousarray(s.indices, np.int32),
                       np.ascontiguousarray(s.indptr, np.int32), np.array(s.shape, np.int32), **kw)
        if not all(hasattr(s, a) for a in ("x", "p", "i", "Dim")):
            raise ValueError("Cannot construct RcppSparse::Matrix from this S4 object")  # std::invalid_argument, :36
        return cls(s.x, s.i, s.p, s.Dim, **kw)

    # ---- accessors, RcppSparse.h:44-51,357-359 ---------------------------------------------------------------
    def rows(self) -> int:
        return int(self.Dim[0])

    def cols(self) -> int:
        return int(self.Dim[1])

    nrow = rows
    ncol = cols

    def n_nonzero(self) -> int:
        return int(self.x.shape[0])

    def nonzeros(self):
        return self.x

    def innerIndexPtr(self):
        return self.i

    def outerIndexPtr(self):
        return self.p

    def InnerNNZs(self, col: int) -> int:
        return int(self.p[col + 1] - self.p[col])

    def clone(self) -> "Matrix":
        """Deep copy of the four vectors (RcppSparse.h:54-60)."""
        return Matrix(self.x.copy(), self.i.copy(), self.p.copy(), self.Dim.copy(), self._device, self._pin, self._resident, self._gpus)

    def wrap(self):
        """RcppSparse.h:387-394: back to the host language's dgCMatrix (scipy CSC sharing the arrays)."""
        import scipy.sparse as sp

        return sp.csc_matrix((self.x, self.i, self.p), shape=(self.rows(), self.cols()), copy=False)

    class InnerIterator:
        """RcppSparse.h:218-233 — unchanged host-side cursor over one column."""

        def __init__(self, ptr: "Matrix", col: int):
            self.ptr, self._col = ptr, col
            self.index, self.max_index = int(ptr.p[col]), int(ptr.p[col + 1])

        def __bool__(self):
            return self.index < self.max_index

        def next(self):
            self.index += 1
            return self

        def value(self) -> float:
            return float(self.ptr.x[self.index])

        def row(self) -> int:
            return int(self.ptr.i[self.index])

        def col(self) -> int:
            return self._col

    # ---- device mirror -------------------------------------------------------------------------------------------
    def _slots(self):
        i = np.ascontiguousarray(self.i, np.int32)
        p = np.ascontiguousarray(self.p, np.int32)
        x = np.ascontiguousarray(self.x, np.float64)
        if p.shape[0] != self.cols() + 1 or i.shape[0] != x.shape[0]:
            raise SparseB200Error(_lib.E_STRUCTURE, "slot lengths inconsistent with Dim")
        return i, p, x

    def _lease(self, multi: bool):
        """The device handle for one call (a ShardedHostMatrix when the op has a several-GPU form and gpus > 1):
        uploaded from the slots as they are now unless this Matrix is resident and its members were not re-pointed."""
        src = (id(self.x), id(self.i), id(self.p), int(self.Dim[0]), int(self.Dim[1]))
        if not self._resident or src != self._src:
            self.release()
        self._src = src
        if multi and self._gpus > 1:
            if self._sharded is None:
                i, p, x = self._slots()
                self._sharded = ShardedHostMatrix(i, p, x, self.rows(), self.cols(), self._gpus)
            return self._sharded
        if self._dev is None:
            i, p, x = self._slots()
            self._dev = DeviceMatrix.from_host(i, p, x, self.rows(), self.cols(), self._device, self._pin,
                                               lazy_rows=not self._resident)  # a per-call mirror: the slots outlive it
        return self._dev

    def _call(self, multi: bool, fn):
        try:
            return fn(self._lease(multi))
        finally:
            if not self._resident:
                self.release()

    def _mirror(self) -> DeviceMatrix:
        """The single-GPU mirror of a RESIDENT matrix (tests and tools that drive the device layer directly)."""
        self._resident = True
        return self._lease(False)

    def resident(self, on: bool = True) -> "Matrix":
        self._resident = bool(on)
        if not on:
            self.release()
        return self

    def refresh(self) -> None:
        """Re-upload x into a resident mirror after an in-place change of the aliased host array (a no-op otherwise:
        non-resident calls read x live)."""
        x = np.ascontiguousarray(self.x, np.float64)
        if self._dev is not None:
            self._dev.refresh_values(x)
        if self._sharded is not None:
            b = self._sharded.bounds()
            for k in range(self._sharded.n_gpus):
                self._sharded.block(k).refresh_values(x[int(self.p[b[k]]):])

    def release(self) -> None:
        if self._dev is not None:
            self._dev.close()
            self._dev = None
        if self._sharded is not None:
            self._sharded.close()
            self._sharded = None

    # ---- the sweeps, RcppSparse.h:131-156 -----------------------------------------------------------------------------
    def colSums(self):
        return self._call(True, lambda m: m.col_sums())

    def rowSums(self):
        return self._call(True, lambda m: m.row_sums())

    def colMeans(self):
        return self._call(True, lambda m: m.col_means())

    def rowMeans(self):
        return self._call(True, lambda m: m.row_means())

    def crossprod(self):
        return self._call(True, lambda m: m.crossprod())

    # ---- sample variances of the columns / rows (sparseMatrixStats::colVars / rowVars): additions -------------------------
    def colVars(self):
        return self._call(True, lambda m: m.col_vars())

    def rowVars(self):
        return self._call(True, lambda m: m.row_vars())

    # ---- A v and A^T v: additions (the reference has only the iterator idiom, SURVEY.md D1) -----------------------------
    def spmv(self, v):
        return self._call(True, lambda m: m.spmv(v))

    def spmv_t(self, v):
        return self._call(True, lambda m: m.spmv_t(v))

    # ---- A B and A^T B for a dense block of k right-hand sides: additions ---------------------------------------------------
    def spmm(self, B):
        return self._call(True, lambda m: m.spmm(B))

    def spmm_t(self, B):
        return self._call(True, lambda m: m.spmm_t(B))

    # ---- RcppSparse.h:375-385 ---------------------------------------------------------------------------------------------
    def transpose(self) -> "Matrix":
        ti, tp, tx = self._call(True, lambda m: m.transpose_host())
        return Matrix(tx, ti, tp, np.array([self.cols(), self.rows()], np.int32), self._device, self._pin)

    t = transpose  # the vignette lists .t() (Documentation.Rmd:250); the header defines transpose()


def columnSums(A) -> np.ndarray:
    """The package's one exported function (reference NAMESPACE:4, src/example.cpp:26-32):
    column sums of a dgCMatrix, as a plain numeric vector of length ncol."""
    m = A if isinstance(A, Matrix) else Matrix.from_S4(A)
    try:
        return m.colSums()
    finally:
        if m is not A:
            m.release()  # a fresh Matrix per call, like the Exporter per .Call (src/RcppExports.cpp:20)
