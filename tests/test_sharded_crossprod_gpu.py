"""crossprod() on every GPU of the process (sparse_b200.h sb200_sharded_crossprod).

Block w computes the result columns of its column block from the row-ordered copy of the whole matrix, adding every
entry in ascending row order like the reference (RcppSparse.h:158-194).  So the result must be the reference's bit for
bit (NaN positions equal, every other bit equal), exactly symmetric, and the same for every placement and every call.

The devices are ordered by CUDA events and host synchronisation only, so a handle whose `devices` list repeats one GPU
(devices=[0] * W) runs every multi-block code path on a one-GPU machine: the all-gather of the rows, empty blocks, the
slabs and their copies home.  The same cases run on W distinct GPUs where the machine has them."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import oracle
from rcppsparse_b200 import Matrix, ShardedHostMatrix, SparseB200Error, _lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
gpu = pytest.mark.gpu
_i32 = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_f64 = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")

# (placement, W): W blocks on GPU 0, or on GPUs 0 .. W-1
PLACEMENTS = [("one-gpu", 1), ("one-gpu", 2), ("one-gpu", 3), ("distinct", 2), ("distinct", 4), ("distinct", 8)]
PLACEMENT_IDS = [f"{p}-W{w}" for p, w in PLACEMENTS]


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def assert_same_bits(got, want, what=""):
    """NaN positions equal, every other entry bit for bit equal (NaN payloads may differ)."""
    assert got.shape == want.shape, what
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), f"{what}: NaN positions differ"
    diff = bits(got)[~nan] != bits(want)[~nan]
    assert not diff.any(), f"{what}: {int(diff.sum())} entries differ from the reference"


def sharded(args, placement, W):
    """A ShardedHostMatrix of W blocks on one GPU or on W distinct GPUs (skips where there are fewer)."""
    i, p, x, nrow, ncol = args
    if placement == "distinct":
        if _lib.device_count() < W:
            pytest.skip(f"needs {W} GPUs")
        return ShardedHostMatrix(i, p, x, nrow, ncol, W)
    return ShardedHostMatrix(i, p, x, nrow, ncol, W, devices=[0] * W)


def load_golden(name):
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    return g["i"].astype(np.int32), g["p"].astype(np.int32), g["x"].astype(np.float64), int(g["dim"][0]), int(g["dim"][1])


GOLDEN = sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.endswith(".npz"))
SYNTH = {
    "uniform": lambda: synth.uniform_spec(20_000, 300, 0.05, 61),
    "powerlaw": lambda: synth.powerlaw_spec(6_000, 2_500, 25.0, 62),
    "banded": lambda: synth.powerlaw_spec(5_000, 1_500, 40.0, 63, row_levels=5),
}


def synth_args(name):
    spec = SYNTH[name]()
    return synth.generate_host(spec) + (spec.nrow, spec.ncol)


def two_columns():
    """7 x 2: fewer columns than blocks at W >= 3."""
    A = sp.random(7, 2, density=0.6, random_state=5, format="csc")
    A.data[:] = np.round(A.data * 10 - 5, 2)
    return A.indices.astype(np.int32), A.indptr.astype(np.int32), A.data.astype(np.float64), 7, 2


def long_rows():
    """300 x 2000 with three rows of 1500-1999 entries: rows longer than the one-GPU kernel's 480-entry piece."""
    A = sp.random(300, 2000, density=0.01, random_state=9, format="lil")
    rng = np.random.default_rng(9)
    for r, n in ((0, 2000), (150, 1500), (299, 1777)):
        cols = np.sort(rng.choice(2000, n, replace=False))
        A[r, cols] = np.round(rng.standard_normal(n), 3) + 0.001
    A = A.tocsc()
    A.sort_indices()
    return A.indices.astype(np.int32), A.indptr.astype(np.int32), A.data.astype(np.float64), 300, 2000


def ascending_row_crossprod(i, p, x, nrow, ncol):
    """The reference's sum for every entry, written as rows: from +0.0, row r's products x_ra * x_rb added in ascending r."""
    R = np.zeros((ncol, ncol))
    if ncol == 0 or len(x) == 0:
        return R
    T = sp.csc_matrix((x, i, p), shape=(nrow, ncol)).tocsr()
    T.sort_indices()
    for r in range(nrow):
        c, v = T.indices[T.indptr[r]:T.indptr[r + 1]], T.data[T.indptr[r]:T.indptr[r + 1]]
        if len(c):
            R[np.ix_(c, c)] += np.multiply.outer(v, v)
    return R


_WANT = {}


def reference(name, args):
    """oracle.best().crossprod, once per shape."""
    if name not in _WANT:
        _WANT[name] = oracle.best().crossprod(*args)
    return _WANT[name]


def shape_args(name):
    if name in SYNTH:
        return synth_args(name)
    return {"two_columns": two_columns, "long_rows": long_rows}[name]()


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    """tests/dropin/dropin_shim.cpp against the drop-in header, built into a temporary directory."""
    import shutil
    import subprocess

    from rcppsparse_b200 import build

    lib = build.build_library()
    out = str(tmp_path_factory.mktemp("sharded_crossprod_shim") / "libdropin_shim.so")
    pkg = os.path.dirname(lib)
    cmd = [shutil.which("g++") or "g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-I" + os.path.join(ROOT, "include"),
           "-I" + os.path.join(ROOT, "oracle", "stub"), os.path.join(ROOT, "tests", "dropin", "dropin_shim.cpp"), "-o", out,
           "-L" + pkg, "-lsparse_b200", "-Wl,-rpath," + pkg]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    L = C.CDLL(out)
    L.dropin_last_error.restype = C.c_char_p
    L.dropin_crossprod.argtypes = [_i32, _i32, _f64, C.c_int, C.c_int, C.c_int64, _f64]
    return L


# ---- 0. no GPU needed --------------------------------------------------------------------------------------------------
def test_binding_declares_and_resolves_the_sharded_crossprod():
    header = open(os.path.join(ROOT, "include", "sparse_b200.h")).read()
    assert re.search(r"\bint sb200_sharded_crossprod\(sb200_sharded\* s, double\* out\b", header)
    assert "sb200_sharded_crossprod" in _lib.SYMBOLS
    fn = _lib.lib().sb200_sharded_crossprod
    assert fn.restype is C.c_int and fn.argtypes == [C.c_void_p, C.c_void_p]


@pytest.mark.parametrize("name", GOLDEN)
def test_ascending_row_order_is_the_reference_bit_for_bit(name):
    """The order this test's reference adds in is the order of the port of the reference's merges."""
    args = load_golden(name)
    assert_same_bits(ascending_row_crossprod(*args), oracle.Port().crossprod(*args), name)


# ---- 1. parity with the reference, bit for bit; symmetry; independence of the placement; stability ---------------------
@gpu
@pytest.mark.parametrize("placement,W", PLACEMENTS, ids=PLACEMENT_IDS)
@pytest.mark.parametrize("name", GOLDEN)
def test_golden_fixtures(name, placement, W):
    args = load_golden(name)
    with sharded(args, placement, W) as S:
        R = S.crossprod()
        assert_same_bits(R, reference(name, args), name)
        assert_same_bits(R, R.T, f"{name}: symmetry")
        assert np.array_equal(bits(S.crossprod()), bits(R)), "two calls give the same bits"


@gpu
@pytest.mark.parametrize("placement,W", PLACEMENTS, ids=PLACEMENT_IDS)
@pytest.mark.parametrize("name", sorted(SYNTH) + ["two_columns", "long_rows"])
def test_synthetic_shapes(name, placement, W):
    args = shape_args(name)
    with sharded(args, placement, W) as S:
        R = S.crossprod()
        assert_same_bits(R, reference(name, args), name)
        assert np.array_equal(bits(R), bits(R.T)), "exactly symmetric"
        assert np.array_equal(bits(S.crossprod()), bits(R)), "two calls give the same bits"
    with ShardedHostMatrix(*args, 1, devices=[0]) as S1:
        assert np.array_equal(bits(S1.crossprod()), bits(R)), "every placement gives the bits of W = 1"


# ---- 2. exact integer data, 10k x 10k: checked fully against scipy; the 800 MB result at W = 2 goes home through the
#         pinned-chunk copies (pageable slabs of 400 MB) ------------------------------------------------------------------
@pytest.fixture(scope="module")
def exact_data():
    """x = +-{1..7}, about one entry in 64 scaled by 2^16: every sum |x_ra x_rb| stays far below 2^52, so every order of
    the additions gives the same exact integers."""
    A = sp.random(10_000, 10_000, density=0.01, random_state=17, format="csc")
    A.sort_indices()
    rng = np.random.default_rng(17)
    n = A.nnz
    x = rng.integers(1, 8, n) * np.where(rng.random(n) < 0.5, -1.0, 1.0) * 2.0 ** (16 * (rng.random(n) < 1.0 / 64))
    A = sp.csc_matrix((x, A.indices, A.indptr), shape=A.shape)
    want = (A.T @ A).toarray()
    assert np.abs(want).max() < 2.0**52
    return (A.indices.astype(np.int32), A.indptr.astype(np.int32), x, 10_000, 10_000), want


@gpu
@pytest.mark.parametrize("placement,W", [("one-gpu", 1), ("one-gpu", 2), ("distinct", 2), ("distinct", 4)],
                         ids=["one-gpu-W1", "one-gpu-W2", "distinct-W2", "distinct-W4"])
def test_exact_integer_data(exact_data, placement, W):
    args, want = exact_data
    with sharded(args, placement, W) as S:
        got = S.crossprod()
    assert np.array_equal(got, want), f"{int((got != want).sum())} entries differ from scipy's exact A^T A"


# ---- 3. edge cases -----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("W", [1, 2, 3])
def test_empty_shapes(W):
    for nrow, ncol, nnz in ((5, 0, 0), (7, 4, 0), (0, 3, 0)):
        i, p, x = np.zeros(nnz, np.int32), np.zeros(ncol + 1, np.int32), np.zeros(nnz)
        with ShardedHostMatrix(i, p, x, nrow, ncol, W, devices=[0] * W) as S:
            R = S.crossprod()
            assert R.shape == (ncol, ncol) and not R.any() and not np.signbit(R).any()


@gpu
@pytest.mark.parametrize("placement,W", [("one-gpu", 1), ("one-gpu", 3), ("distinct", 2)],
                         ids=["one-gpu-W1", "one-gpu-W3", "distinct-W2"])
def test_refresh_after_an_in_place_change(placement, W):
    i, p, x, nrow, ncol = synth_args("powerlaw")
    x = x.copy()
    with sharded((i, p, x, nrow, ncol), placement, W) as S:
        R0 = S.crossprod()
        assert all(S.block(w).layouts() & 1 for w in range(W) if S.block(w).nnz), "blocks keep their row-ordered copies"
        x *= -2.0
        b = S.bounds()
        for w in range(W):
            S.block(w).refresh_values(x[int(p[b[w]]):])
        R1 = S.crossprod()
    assert_same_bits(R1, oracle.best().crossprod(i, p, x, nrow, ncol), "after refresh")
    assert np.array_equal(R1, 4.0 * R0)


# ---- 4. errors ---------------------------------------------------------------------------------------------------------
@gpu
def test_arguments():
    args = synth_args("banded")
    L = _lib.lib()
    S = sharded(args, "one-gpu", 2)
    buf = np.zeros(args[4] * args[4])
    assert L.sb200_sharded_crossprod(None, buf.ctypes.data) == _lib.E_INVALID
    assert L.sb200_sharded_crossprod(S._h, None) == _lib.E_INVALID
    S.close()
    with pytest.raises(SparseB200Error) as e:
        S.crossprod()
    assert e.value.code == _lib.E_INVALID


@gpu
def test_result_that_does_not_fit_is_refused_and_the_handle_stays_usable():
    """200 000 columns, two blocks on one GPU: 2 x 160 GB of slabs.  Refused before `out` is touched (a small buffer
    stands in for it)."""
    nrow, ncol = 1000, 200_000
    cols = np.array([3, 77_777, 150_000, 199_999])
    p = np.zeros(ncol + 1, np.int32)
    p[cols + 1] = 2
    p = np.cumsum(p).astype(np.int32)
    i = np.tile(np.array([10, 500], np.int32), len(cols))
    x = np.arange(1.0, 2 * len(cols) + 1)
    with ShardedHostMatrix(i, p, x, nrow, ncol, 2, devices=[0, 0]) as S:
        small = np.zeros(16)
        assert _lib.lib().sb200_sharded_crossprod(S._h, small.ctypes.data) == _lib.E_NOMEM
        assert not small.any(), "nothing is written"
        cs = S.col_sums()
    want = np.zeros(ncol)
    want[cols] = x[0::2] + x[1::2]
    assert np.array_equal(cs, want)


# ---- 5. 64-bit indices: ncol^2 > 2^31 ----------------------------------------------------------------------------------
@gpu
def test_index_width_past_two_to_the_31():
    import torch

    ncol, nrow = 48_000, 60_000
    assert ncol * ncol > 2**31
    if torch.cuda.mem_get_info()[0] < 40 << 30:
        pytest.skip("needs 40 GB of free device memory")
    if os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_AVPHYS_PAGES") < 64 << 30:
        pytest.skip("needs 64 GB of free host memory for the 18 GB result")
    # row r holds columns r mod ncol and (7 r + 3) mod ncol (one entry when they coincide), values small integers
    r = np.arange(nrow)
    c1, c2 = r % ncol, (7 * r + 3) % ncol
    rows = np.concatenate([r, r[c1 != c2]])
    cols = np.concatenate([c1, c2[c1 != c2]])
    vals = (1 + (rows * 5 + cols) % 7).astype(np.float64)
    A = sp.csc_matrix((vals, (rows, cols)), shape=(nrow, ncol))
    A.sort_indices()
    want = (A.T @ A).tocoo()
    with ShardedHostMatrix(A.indices.astype(np.int32), A.indptr.astype(np.int32), A.data, nrow, ncol, 1, devices=[0]) as S:
        got = S.crossprod()
    assert np.array_equal(got[want.row, want.col], want.data), "the nonzero entries"
    assert np.count_nonzero(got) == want.nnz, "every other entry is zero"


# ---- 6. routing: the Python drop-in and the C++ header under SB200_GPUS = 2 ---------------------------------------------
@gpu
def test_matrix_routes_crossprod_to_the_sharded_handle():
    if _lib.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    i, p, x, nrow, ncol = args = synth_args("banded")
    x = x.copy()
    A = Matrix(x, i, p, np.array([nrow, ncol], np.int32), gpus=2, resident=True)
    assert_same_bits(A.crossprod(), reference("banded", args), "gpus = 2")
    assert A._sharded is not None and A._dev is None, "gpus = 2 runs crossprod on the sharded handle, no one-GPU mirror"
    x *= -2.0
    A.refresh()
    assert_same_bits(A.crossprod(), oracle.best().crossprod(i, p, x, nrow, ncol), "after refresh")
    A.release()


@gpu
def test_dropin_header_under_SB200_GPUS(shim, monkeypatch, capfd):
    if _lib.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    monkeypatch.setenv("SB200_GPUS", "2")
    monkeypatch.setenv("SB200_TRACE", "1")  # the sharded entry points name themselves on stderr
    i, p, x, nrow, ncol = args = synth_args("powerlaw")
    R = np.empty((ncol, ncol))
    capfd.readouterr()
    assert shim.dropin_crossprod(i, p, x, nrow, ncol, len(x), R.reshape(-1)) == 0, shim.dropin_last_error()
    assert "sharded crossprod" in capfd.readouterr().err
    assert_same_bits(R, reference("powerlaw", args), "the header under SB200_GPUS=2")
