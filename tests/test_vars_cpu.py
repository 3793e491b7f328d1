"""colVars / rowVars without a GPU: the exact reference the GPU tests hold them to, the accuracy bar, and the error.

colVars()[c] is the sample variance of the nrow values of column c (its stored entries and nrow - nnz_c implicit zeros)
over nrow - 1, rowVars()[r] the same over the ncol values of row r (R's var()).  The reference here is exact: every
finite double is an integer times a power of two, so the sums of x and x^2 are Python integers, and the variance
(n sum x^2 - (sum x)^2) / (n (n - 1)) is a rational number, rounded once to the nearest double.  The bar is

    |got - exact| <= 1e-12 * exact + 2 * spacing(mean)^2

where the second term covers the one rounding of the mean the two passes use.  It must be able to tell a two-pass
result from the one-pass sum(x^2)/n - mean^2: on a nearly constant column (2^30 + small integers) the latter is off
by about a hundred, far outside it.

These helpers are imported by tests/test_vars_gpu.py and tests/test_sharded_vars_gpu.py.
"""
from __future__ import annotations

import ctypes as C
import os
from fractions import Fraction

import numpy as np
import pytest
import scipy.sparse as sp

from rcppsparse_b200 import Matrix, SparseB200Error, _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
_i32 = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_f64 = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")


# ---- exact reference -----------------------------------------------------------------------------------------------------
def _as_scaled_ints(x):
    """(X, s): x[k] == X[k] / 2**s exactly, X integers (non-finite entries give 0): an int64 array where every |X| is
    below 2^31, a list of Python integers otherwise."""
    x = np.where(np.isfinite(x), x, 0.0)
    m, e = np.frexp(x)
    M = (m * 2.0**53).astype(np.int64)  # x = M * 2**(e - 53), exactly
    E = e.astype(np.int64) - 53
    nz = M != 0
    s = 0
    if nz.any():
        # the lowest set bit of every M decides how far x must be scaled to become an integer
        low = np.zeros(len(M), np.int64)
        low[nz] = np.log2((M[nz] & -M[nz]).astype(np.float64)).astype(np.int64)
        s = int(max(0, -(E[nz] + low[nz]).min()))
    scaled = x * 2.0**s
    if not nz.any() or np.abs(scaled).max() < 2.0**31:
        return scaled.astype(np.int64), s
    # b + s < 0 only drops low bits that are zero
    return [(a << (b + s)) if b + s >= 0 else (a >> -(b + s)) for a, b in zip(M.tolist(), E.tolist())], s


def exact_vars(i, p, x, nrow, ncol, axis):
    """Exact colVars (axis 0) / rowVars (axis 1) rounded to doubles, and the exact means rounded to doubles.
    NaN where the dimension is below 2 or a stored entry of the column / row is NaN or +-Inf."""
    i, p, x = np.asarray(i), np.asarray(p, np.int64), np.asarray(x, np.float64)
    n, m = (nrow, ncol) if axis == 0 else (ncol, nrow)  # values per output, outputs
    group = np.repeat(np.arange(ncol), np.diff(p)) if axis == 0 else np.asarray(i, np.int64)
    X, s = _as_scaled_ints(x)
    bad = np.zeros(m, bool)
    np.logical_or.at(bad, group, ~np.isfinite(x))
    terms = np.bincount(group, minlength=m).max(initial=0) if m else 0
    if isinstance(X, np.ndarray) and float(np.abs(X).max(initial=0)) ** 2 * terms < 2.0**62:
        sx, sxx = np.zeros(m, np.int64), np.zeros(m, np.int64)  # no int64 sum can overflow
        np.add.at(sx, group, X)
        np.add.at(sxx, group, X * X)
        sx, sxx = sx.tolist(), sxx.tolist()
    else:
        sx, sxx = [0] * m, [0] * m
        for g, v in zip(group.tolist(), list(X)):
            if v:
                sx[g] += int(v)
                sxx[g] += int(v) * int(v)
    var = np.full(m, np.nan)
    mean = np.full(m, np.nan)
    if n >= 1:
        mean = np.array([float(Fraction(a, n << s)) for a in sx]) if m else np.zeros(0)
    if n >= 2:
        den = n * (n - 1) << (2 * s)
        var = np.array([(n * b - a * a) / den for a, b in zip(sx, sxx)]) if m else np.zeros(0)
    var[bad] = np.nan
    mean[bad] = np.nan
    return var, mean


def bar(exact, mean):
    return 1e-12 * np.abs(exact) + 2.0 * np.spacing(np.abs(mean)) ** 2


def assert_within_bar(got, exact, mean, what=""):
    """NaN exactly where the reference has NaN; everywhere else within the bar."""
    got = np.asarray(got, np.float64)
    assert got.shape == exact.shape, what
    nan = np.isnan(exact)
    assert np.array_equal(np.isnan(got), nan), f"{what}: NaN positions differ ({np.flatnonzero(np.isnan(got) != nan)[:8]})"
    err = np.abs(got[~nan] - exact[~nan])
    lim = bar(exact[~nan], mean[~nan])
    worst = int(np.argmax(err - lim)) if err.size else 0
    assert np.all(err <= lim), f"{what}: outside the bar at output {np.flatnonzero(~nan)[worst]}: {got[~nan][worst]!r} vs {exact[~nan][worst]!r}"


def assert_same_bits(got, want, what=""):
    got, want = np.ascontiguousarray(got, np.float64), np.ascontiguousarray(want, np.float64)
    assert got.shape == want.shape, what
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), f"{what}: NaN positions differ"
    diff = np.flatnonzero(got[~nan].view(np.uint64) != want[~nan].view(np.uint64))
    assert diff.size == 0, f"{what}: {diff.size} outputs differ, first {np.flatnonzero(~nan)[diff[0]]}: {got[~nan][diff[0]]!r} vs {want[~nan][diff[0]]!r}"


# ---- fixtures ----------------------------------------------------------------------------------------------------------------
def golden(name):
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    return g["i"].astype(np.int32), g["p"].astype(np.int32), g["x"].astype(np.float64), int(g["dim"][0]), int(g["dim"][1])


def csc(A):
    A = sp.csc_matrix(A)
    A.sort_indices()
    return A.indices.astype(np.int32), A.indptr.astype(np.int32), A.data.astype(np.float64), A.shape[0], A.shape[1]


def nearly_constant(n=1000, seed=7):
    """A dense column and a dense row of 2^30 + small integers (mean ~1e9, variance ~4), next to sparse ones."""
    rng = np.random.default_rng(seed)
    D = np.zeros((n, n // 4))
    D[rng.random(D.shape) < 0.02] = rng.integers(1, 50)
    D[:, 0] = 2.0**30 + rng.integers(-3, 4, n)
    D[1, :] = 2.0**30 + rng.integers(-3, 4, n // 4)
    return csc(D)


def edge_cases():
    """Small fixtures of the semantics: empty and dense columns and rows, explicit zeros, NaN / Inf, tiny dimensions."""
    rng = np.random.default_rng(11)
    out = {}
    D = np.zeros((9, 7))
    D[:, 2] = rng.standard_normal(9)  # fully dense column
    D[4, :] = rng.standard_normal(7)  # fully dense row
    D[1, 5] = 3.5
    out["empty_and_dense"] = csc(D)  # column 0, 1, 3, 4, 6 and most rows: empty apart from the dense ones
    i, p, x, nrow, ncol = csc(D)
    x = x.copy()
    x[[0, 3]] = 0.0  # explicit zeros count as values
    out["explicit_zeros"] = (i, p, x, nrow, ncol)
    S = np.zeros((10, 8))
    S[rng.random(S.shape) < 0.5] = 1.0
    S[S != 0] = rng.standard_normal(int((S != 0).sum()))
    S[2, 1], S[5, 4], S[7, 4], S[0, 6] = np.nan, np.inf, -np.inf, np.inf
    out["nan_inf"] = csc(S)
    for shape in ((0, 3), (3, 0), (0, 0), (1, 4), (4, 1), (2, 3), (3, 2), (1, 1), (2, 2)):
        M = np.zeros(shape)
        M[rng.random(shape) < 0.6] = rng.integers(1, 9)
        out[f"dims_{shape[0]}x{shape[1]}"] = csc(M)
    return out


# ---- the reference itself ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["vignette_5x5", "all_dense_17x13", "specials_12x9", "one_row_1x9", "nrow0_0x3", "ncol0_5x0",
                                  "synth_uniform_2000x300"])
def test_exact_reference_agrees_with_numpy(name):
    i, p, x, nrow, ncol = golden(name)
    dense = sp.csc_matrix((x, i, p), shape=(nrow, ncol)).toarray()
    with np.errstate(all="ignore"):
        for axis in (0, 1):
            var, mean = exact_vars(i, p, x, nrow, ncol, axis)
            n = dense.shape[axis]
            want = np.var(dense, axis=axis, ddof=1) if n >= 2 else np.full(dense.shape[1 - axis], np.nan)
            assert var.shape == want.shape
            assert np.array_equal(np.isnan(var), np.isnan(want)), (name, axis)
            ok = ~np.isnan(want)
            assert np.allclose(var[ok], want[ok], rtol=1e-12, atol=0), (name, axis)
            if n >= 1:
                assert np.allclose(mean[ok], dense.mean(axis=axis)[ok], rtol=1e-12, atol=1e-14)


@pytest.mark.parametrize("name", sorted(edge_cases()))
def test_exact_reference_semantics(name):
    i, p, x, nrow, ncol = edge_cases()[name]
    dense = sp.csc_matrix((x, i, p), shape=(nrow, ncol)).toarray()
    for axis in (0, 1):
        var, _ = exact_vars(i, p, x, nrow, ncol, axis)
        n = dense.shape[axis]
        assert var.shape == (dense.shape[1 - axis],)
        if n < 2:
            assert np.all(np.isnan(var))
            continue
        for g in range(var.size):
            vals = dense[:, g] if axis == 0 else dense[g, :]
            if not np.all(np.isfinite(vals)):
                assert np.isnan(var[g])
            else:
                assert var[g] == float(sum((Fraction(v) - Fraction(sum(map(Fraction, vals)), n)) ** 2 for v in vals) / (n - 1))
                if not np.any(vals):
                    assert var[g] == 0.0 and not np.signbit(var[g])


def test_one_pass_formula_fails_the_bar_on_nearly_constant_data():
    """The fixture tells two passes from one: sum(x^2)/n - mean^2 in float64 misses by far more than the bar allows,
    while the two-pass formula around the rounded mean stays inside it."""
    i, p, x, nrow, ncol = nearly_constant()
    dense = sp.csc_matrix((x, i, p), shape=(nrow, ncol)).toarray()
    for axis, g in ((0, 0), (1, 1)):
        var, mean = exact_vars(i, p, x, nrow, ncol, axis)
        vals = dense[:, g] if axis == 0 else dense[g, :]
        n = vals.size
        m = np.sum(vals) / n
        one_pass = (np.sum(vals * vals) / n - m * m) * n / (n - 1)
        two_pass = np.sum((vals - m) ** 2) / (n - 1)
        assert 1.0 < var[g] < 10.0
        assert abs(one_pass - var[g]) > 1e3 * bar(var[g], mean[g]), "the fixture cannot tell the formulas apart"
        assert abs(two_pass - var[g]) <= bar(var[g], mean[g])


# ---- no device: an error, never a CPU path --------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    """tests/dropin/vars_shim.cpp against the drop-in header, built into a temporary directory."""
    import shutil
    import subprocess

    from rcppsparse_b200 import build

    lib = build.build_library()
    out = str(tmp_path_factory.mktemp("vars_shim") / "libvars_shim.so")
    pkg = os.path.dirname(lib)
    cmd = [shutil.which("g++") or "g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-I" + os.path.join(ROOT, "include"),
           "-I" + os.path.join(ROOT, "oracle", "stub"), os.path.join(ROOT, "tests", "dropin", "vars_shim.cpp"), "-o", out,
           "-L" + pkg, "-lsparse_b200", "-Wl,-rpath," + pkg]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    L = C.CDLL(out)
    L.vars_shim_last_error.restype = C.c_char_p
    L.vars_shim.argtypes = [C.c_int, _i32, _i32, _f64, C.c_int, C.c_int, C.c_int64, _f64]
    return L


def test_without_gpu_vars_are_an_error(shim):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    i, p, x, nrow, ncol = golden("vignette_5x5")
    A = Matrix(x, i, p, np.array([nrow, ncol], np.int32))
    for fn in (A.colVars, A.rowVars):
        with pytest.raises(SparseB200Error) as e:
            fn()
        assert e.value.code == _lib.E_NODEVICE
    for rows in (0, 1):
        assert shim.vars_shim(rows, i, p, x, nrow, ncol, len(x), np.empty(max(nrow, ncol))) == 2
        assert b"no CUDA device" in shim.vars_shim_last_error()
