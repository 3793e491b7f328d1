"""colVars / rowVars on one GPU (sparse_b200.h sb200_col_vars / sb200_row_vars), on every path they take.

Every result is held to the exact reference of tests/test_vars_cpu.py: within |got - exact| <= 1e-12 exact +
2 spacing(mean)^2, NaN exactly where a stored NaN / Inf touches the output or the dimension is below 2, +0.0 for
empty columns and rows.  Where the divisor dimension n is a power of two (<= 4096) and the values are integers with
|x| <= 127, every intermediate of the two passes is exact: the mean is an integer over 2^12, a deviation needs 19 bits,
its square 38, and all the squares of an output with the (n - cnt) m^2 term sum to n times a variance of at most
127^2, a multiple of 2^-24 below 2^26.  The one IEEE division then rounds the exact value, so those results must equal
the exact reference bit for bit whatever order the atomics add in; a term dropped or counted twice cannot hide.

Paths: colVars at every sweep geometry of tests/test_exact_paths_gpu.py (SB200_SWEEP_CFG, read on every call); rowVars
on the L2 kernel (SB200_ROW_PLAN=0), the row bands (SB200_ROW_PLAN=1), the row-ordered copy, a non-resident Matrix (a
per-call mirror whose row indices go up lazily) and adopted device arrays.  row_path() confirms which served a call.
"""
from __future__ import annotations

import zlib

import numpy as np
import pytest
import scipy.sparse as sp

from rcppsparse_b200 import DeviceMatrix, Matrix, _lib
from test_exact_paths_gpu import SWEEP_CFGS, _repeat_columns, structure
from test_parity_gpu import LENGTH_REGIMES, _columns_of_lengths
from test_vars_cpu import assert_same_bits, assert_within_bar, csc, edge_cases, exact_vars, golden, nearly_constant

gpu = pytest.mark.gpu
N_EXACT = 4096
MIN_ITEMS = 2_500_000  # merge items of a repeated regime, as in tests/test_exact_paths_gpu.py


# ---- data ---------------------------------------------------------------------------------------------------------------------
def dyadic(n, seed):
    """Values +-k / 64, k in 1 .. 4096: every sum of them, and of their squares, is exact in the reference."""
    rng = np.random.default_rng(seed)
    return rng.integers(1, 4097, n) * rng.choice([-1.0, 1.0], n) / 64.0


def small_ints(n, seed):
    """Integers in [-127, 127], explicit zeros included."""
    return np.random.default_rng(seed).integers(-127, 128, n).astype(np.float64)


def with_specials(x, seed):
    x = x.copy()
    pos = np.random.default_rng(seed).choice(len(x), 6, replace=False)
    x[pos] = [np.nan, np.inf, -np.inf, np.inf, np.nan, -np.inf]
    return x


def exact_col_structure(regime):
    """A length regime repeated to >= MIN_ITEMS merge items at nrow = 4096 (colVars divides by a power of two)."""
    lengths = LENGTH_REGIMES[regime]
    i, p, _ = _columns_of_lengths(lengths, N_EXACT, zlib.crc32(regime.encode()))
    reps = -(-MIN_ITEMS // (len(lengths) + len(i)))
    i, p = _repeat_columns(i, p, reps)
    return i, p, N_EXACT, len(p) - 1


def transposed(i, p, x, nrow, ncol):
    return csc(sp.csc_matrix((x, i, p), shape=(nrow, ncol)).T)


EXACT_REGIMES = ["sawtooth", "const_3", "const_938_939_940", "const_2815_2816_2817"]
BAR_SHAPES = ["regime/sawtooth", "regime/const_0_1_2", "regime/long_then_dust", "few_huge_columns", "tiny_columns",
              "powerlaw_hot_rows", "tall_short_columns"]


def bar_case(shape, specials=False):
    i, p, nrow, ncol = structure(shape)
    x = dyadic(len(i), zlib.crc32(shape.encode()))
    if specials:
        x = with_specials(x, 5)
    return i, p, x, nrow, ncol


def small_cases():
    out = {n: golden(n) for n in ("vignette_5x5", "specials_12x9", "all_empty_7x4", "all_dense_17x13", "one_row_1x9", "nrow0_0x3",
                                  "ncol0_5x0", "one_dense_column_64x1", "max_column_between_empties_300x11", "synth_wide_50x4000")}
    out.update(edge_cases())
    out["nearly_constant"] = nearly_constant()
    return out


def check_vars(got, A, axis, what):
    i, p, x, nrow, ncol = A
    var, mean = exact_vars(i, p, x, nrow, ncol, axis)
    assert_within_bar(got, var, mean, what)
    zero = var == 0.0
    assert not np.any(np.signbit(np.asarray(got)[zero])), f"{what}: a zero variance must be +0.0"


def row_paths(A, monkeypatch):
    """(label, rowVars result) on every row path: L2 kernel, row bands (1, 4 and 64 column splits), row-ordered copy
    (twice), non-resident Matrix, adopted device arrays."""
    import torch

    i, p, x, nrow, ncol = A
    out = []
    for plan, label, splits in (("0", "l2-atomics", "4"), ("1", "banded", "1"), ("1", "banded", "4"), ("1", "banded", "64")):
        monkeypatch.setenv("SB200_ROW_PLAN", plan)
        monkeypatch.setenv("SB200_SCATTER_SPLITS", splits)  # 1: one store per row; more: FP64 reductions of the splits
        with DeviceMatrix.from_host(i, p, x, nrow, ncol) as D:
            D.row_companion(-1)
            got = D.row_vars()
            if len(x) and nrow and ncol:
                assert D.row_path() == label
            out.append((f"{label}, {splits} splits", got))
    monkeypatch.delenv("SB200_ROW_PLAN")
    monkeypatch.delenv("SB200_SCATTER_SPLITS")
    with DeviceMatrix.from_host(i, p, x, nrow, ncol) as D:
        if len(x) and nrow:
            D.row_companion(1)
            assert D.row_path() == "row-companion"
        a, b = D.row_vars(), D.row_vars()
        if len(x) and nrow:
            assert_same_bits(b, a, "rowVars on the row-ordered copy, run to run")
        out.append(("row-companion", a))
    out.append(("per-call mirror", Matrix(x, i, p, np.array([nrow, ncol], np.int32)).rowVars()))
    di, dp, dx = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (i, p, x))
    with DeviceMatrix.adopt(di, dp, dx, nrow, ncol) as D:
        out.append(("adopted", D.row_vars()))
    return out


# ---- small fixtures: the semantics on every path -----------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", sorted(small_cases()))
def test_small_fixtures(name, monkeypatch):
    A = small_cases()[name]
    i, p, x, nrow, ncol = A
    with DeviceMatrix.from_host(i, p, x, nrow, ncol) as D:
        c = D.col_vars()
        assert c.shape == (ncol,)
        check_vars(c, A, 0, f"colVars on {name}")
        assert_same_bits(D.col_vars(), c, f"colVars on {name}, run to run")
    assert_same_bits(Matrix(x, i, p, np.array([nrow, ncol], np.int32)).colVars(), c, f"colVars of a per-call mirror on {name}")
    for label, r in row_paths(A, monkeypatch):
        assert r.shape == (nrow,)
        check_vars(r, A, 1, f"rowVars [{label}] on {name}")


# ---- bit-exact cases ----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("regime", EXACT_REGIMES)
def test_col_vars_bit_exact_every_sweep_geometry(regime, monkeypatch):
    i, p, nrow, ncol = exact_col_structure(regime)
    x = small_ints(len(i), zlib.crc32(regime.encode()) + 1)
    want, _ = exact_vars(i, p, x, nrow, ncol, 0)
    with DeviceMatrix.from_host(i, p, x, nrow, ncol) as D:
        for cfg in SWEEP_CFGS:
            monkeypatch.setenv("SB200_SWEEP_CFG", cfg)
            a = D.col_vars()
            assert_same_bits(a, want, f"colVars at {cfg} on {regime}")
            assert_same_bits(D.col_vars(), a, f"colVars at {cfg} on {regime}, run to run")


@gpu
@pytest.mark.parametrize("regime", EXACT_REGIMES)
def test_row_vars_bit_exact_every_path(regime, monkeypatch):
    i, p, nrow, ncol = exact_col_structure(regime)
    x = small_ints(len(i), zlib.crc32(regime.encode()) + 2)
    A = transposed(i, p, x, nrow, ncol)  # ncol = 4096: rowVars divides by a power of two
    want, _ = exact_vars(*A, 1)
    for label, got in row_paths(A, monkeypatch):
        assert_same_bits(got, want, f"rowVars [{label}] on {regime}")


# ---- synthetic shapes at the sweep's CTA geometries, within the bar --------------------------------------------------------------
@gpu
@pytest.mark.parametrize("specials", [False, True], ids=["finite", "specials"])
@pytest.mark.parametrize("shape", BAR_SHAPES)
def test_synthetic_shapes_within_bar(shape, specials, monkeypatch):
    if specials and shape not in ("regime/sawtooth", "powerlaw_hot_rows"):
        pytest.skip("NaN / Inf on two shapes")
    A = bar_case(shape, specials)
    i, p, x, nrow, ncol = A
    with DeviceMatrix.from_host(i, p, x, nrow, ncol) as D:
        first = None
        for cfg in SWEEP_CFGS:
            monkeypatch.setenv("SB200_SWEEP_CFG", cfg)
            c = D.col_vars()
            check_vars(c, A, 0, f"colVars at {cfg} on {shape}")
            assert_same_bits(D.col_vars(), c, f"colVars at {cfg} on {shape}, run to run")
            first = c if first is None else first
        monkeypatch.delenv("SB200_SWEEP_CFG")
    for label, r in row_paths(A, monkeypatch):
        check_vars(r, A, 1, f"rowVars [{label}] on {shape}")


# ---- device forms, arguments ---------------------------------------------------------------------------------------------------
@gpu
def test_device_forms_match_the_host_forms():
    import torch

    A = bar_case("regime/sawtooth")
    i, p, x, nrow, ncol = A
    with DeviceMatrix.from_host(i, p, x, nrow, ncol) as D:
        D.row_companion(1)  # rowVars bit-stable: the two forms can be compared bit for bit
        c = torch.empty(ncol, dtype=torch.float64, device="cuda")
        r = torch.empty(nrow, dtype=torch.float64, device="cuda")
        D.col_vars_dev(c)
        D.row_vars_dev(r)
        D.sync()
        assert_same_bits(c.cpu().numpy(), D.col_vars(), "colVars device form")
        assert_same_bits(r.cpu().numpy(), D.row_vars(), "rowVars device form")
        assert D.algorithmic_bytes("col_vars") == D.algorithmic_bytes("col_sums")
        assert D.algorithmic_bytes("row_vars") == D.algorithmic_bytes("row_sums")


@gpu
def test_arguments():
    i, p, x, nrow, ncol = golden("vignette_5x5")
    L = _lib.lib()
    with DeviceMatrix.from_host(i, p, x, nrow, ncol) as D:
        for fn in (L.sb200_col_vars, L.sb200_row_vars, L.sb200_col_vars_dev, L.sb200_row_vars_dev):
            assert fn(D._h, None) == _lib.E_INVALID
        assert np.all(np.isfinite(D.col_vars()))  # still usable
    assert L.sb200_col_vars(None, None) == _lib.E_INVALID
