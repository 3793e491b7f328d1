"""colVars / rowVars on every GPU of the process (sparse_b200.h sb200_sharded_col_vars / sb200_sharded_row_vars).

colVars runs the one-GPU two-pass sweep on every column block, so it is bit-stable and, with one block, bit-identical to
the one-GPU result.  rowVars takes the global row means as sb200_sharded_row_means computes them, sums every block's
squared deviations and entry counts, and reduces them in block order over peer memory.  Both are held to the exact
reference and bar of tests/test_vars_cpu.py, and to the exact bits on the power-of-two shapes of tests/test_vars_gpu.py.

The reduce is ordered by CUDA events only, so a handle whose `devices` list repeats one GPU (devices=[0] * W) runs every
multi-block code path on a one-GPU machine, empty blocks included.  Matrix(gpus=2) and the drop-in header under
SB200_GPUS=2 need two GPUs and skip otherwise."""
from __future__ import annotations

import zlib

import numpy as np
import pytest

from rcppsparse_b200 import DeviceMatrix, Matrix, ShardedHostMatrix, _lib
from test_vars_cpu import assert_same_bits, exact_vars, shim  # noqa: F401 (shim: the drop-in harness fixture)
from test_vars_gpu import EXACT_REGIMES, bar_case, check_vars, exact_col_structure, small_cases, small_ints, transposed

gpu = pytest.mark.gpu
WORLDS = [1, 2, 3]
SMALL = ["vignette_5x5", "specials_12x9", "all_empty_7x4", "nrow0_0x3", "ncol0_5x0", "one_dense_column_64x1", "nan_inf",
         "dims_4x1", "dims_1x4", "dims_2x3", "explicit_zeros", "nearly_constant"]
BAR = ["regime/sawtooth", "powerlaw_hot_rows", "tall_short_columns"]


def sharded(A, W):
    i, p, x, nrow, ncol = A
    return ShardedHostMatrix(i, p, x, nrow, ncol, W, devices=[0] * W)


def case(name):
    if name in small_cases():
        return small_cases()[name]
    return bar_case(name)


@gpu
@pytest.mark.parametrize("W", WORLDS)
@pytest.mark.parametrize("name", SMALL + BAR)
def test_within_bar(name, W):
    A = case(name)
    i, p, x, nrow, ncol = A
    with sharded(A, W) as S:
        c, r = S.col_vars(), S.row_vars()
        assert c.shape == (ncol,) and r.shape == (nrow,)
        check_vars(c, A, 0, f"sharded colVars W={W} on {name}")
        check_vars(r, A, 1, f"sharded rowVars W={W} on {name}")
        assert_same_bits(S.col_vars(), c, f"sharded colVars W={W} on {name}, run to run")
    if W == 1:
        with DeviceMatrix.from_host(i, p, x, nrow, ncol) as D:
            assert_same_bits(c, D.col_vars(), f"sharded colVars W=1 against one GPU on {name}")


@gpu
@pytest.mark.parametrize("W", WORLDS)
@pytest.mark.parametrize("regime", EXACT_REGIMES[:2])
def test_bit_exact(regime, W):
    i, p, nrow, ncol = exact_col_structure(regime)
    x = small_ints(len(i), zlib.crc32(regime.encode()) + 1)
    A = (i, p, x, nrow, ncol)  # nrow = 4096: colVars exact
    with sharded(A, W) as S:
        assert_same_bits(S.col_vars(), exact_vars(*A, 0)[0], f"sharded colVars W={W} on {regime}")
    T = transposed(*A)  # ncol = 4096: rowVars exact
    with sharded(T, W) as S:
        want = exact_vars(*T, 1)[0]
        for k in range(W):  # the row-ordered copy on every block: the other row paths
            S.block(k).row_companion(1 if k % 2 else -1)
        assert_same_bits(S.row_vars(), want, f"sharded rowVars W={W} on {regime}")


@gpu
def test_row_ordered_copies_built_on_their_own():
    """rowVars counts toward every block's row-ordered copy like rowMeans; once the blocks sweep their copies the result
    is still within the bar, and bit-stable."""
    A = bar_case("regime/sawtooth")
    with sharded(A, 2) as S:
        check_vars(S.row_vars(), A, 1, "sharded rowVars on the CSC arrays")
        for _ in range(10):  # past SB200_ROW_COMPANION_AFTER
            S.row_vars()
        assert S.block(0).row_path() == "row-companion" and S.block(1).row_path() == "row-companion"
        again = S.row_vars()
        check_vars(again, A, 1, "sharded rowVars on the row-ordered copies")
        assert_same_bits(S.row_vars(), again, "sharded rowVars on the row-ordered copies, run to run")


@gpu
def test_two_gpus_through_matrix_and_the_header(shim, monkeypatch):
    if _lib.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    A = bar_case("powerlaw_hot_rows")
    i, p, x, nrow, ncol = A
    M = Matrix(x, i, p, np.array([nrow, ncol], np.int32), gpus=2)
    check_vars(M.colVars(), A, 0, "Matrix(gpus=2).colVars")
    check_vars(M.rowVars(), A, 1, "Matrix(gpus=2).rowVars")
    monkeypatch.setenv("SB200_GPUS", "2")
    for rows in (0, 1):
        out = np.empty(max(nrow, ncol))
        assert shim.vars_shim(rows, i, p, x, nrow, ncol, len(x), out) == 0, shim.vars_shim_last_error()
        check_vars(out[: (nrow if rows else ncol)], A, rows, f"drop-in {'rowVars' if rows else 'colVars'} under SB200_GPUS=2")


@gpu
def test_arguments():
    A = small_cases()["vignette_5x5"]
    with sharded(A, 2) as S:
        assert _lib.lib().sb200_sharded_col_vars(S._h, None) == _lib.E_INVALID
        assert _lib.lib().sb200_sharded_row_vars(S._h, None) == _lib.E_INVALID
        assert np.all(np.isfinite(S.row_vars()))  # still usable
    assert _lib.lib().sb200_sharded_row_vars(None, None) == _lib.E_INVALID
