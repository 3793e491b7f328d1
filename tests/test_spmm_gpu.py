"""Sparse x dense block (sparse_b200.h sb200_spmm / sb200_spmm_t): Y = A B and Y = A^T B for k right-hand sides.

Column j of Y must be what spmv / spmv_t gives for column j of B, within |delta| <= 1e-12 * sum |a b| per entry,
with NaN and Inf in B reaching exactly the outputs they touch; B and Y are column-major at every boundary."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import oracle
from rcppsparse_b200 import DeviceMatrix, Matrix, SparseB200Error, _lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
_i32 = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_f64 = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def operand(seed, rows, k, specials=False):
    B = np.round(np.random.default_rng(seed).standard_normal((rows, k)), 3)
    if specials and rows > 2 and k > 0:
        j = min(1, k - 1)
        B[0, j], B[rows // 2, j] = np.nan, np.inf
    return np.asfortranarray(B)


def assert_columns(op, Y, B, args, chk):
    """Every column of Y against the checker's spmv / spmv_t of that column of B."""
    nrow, ncol = args[3], args[4]
    assert Y.shape == ((nrow if op == "spmv" else ncol), B.shape[1])
    for j in range(B.shape[1]):
        v = np.ascontiguousarray(B[:, j])
        oracle.assert_within(op, Y[:, j], getattr(chk, op)(*args, v), *args, v=v)


@pytest.fixture(scope="module")
def chk():
    return oracle.best()


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    """tests/dropin/spmm_shim.cpp against the drop-in header, built into a temporary directory."""
    import shutil
    import subprocess

    from rcppsparse_b200 import build

    lib = build.build_library()
    out = str(tmp_path_factory.mktemp("spmm_shim") / "libspmm_shim.so")
    pkg = os.path.dirname(lib)
    cmd = [shutil.which("g++") or "g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wall", "-I" + os.path.join(ROOT, "include"),
           "-I" + os.path.join(ROOT, "oracle", "stub"), os.path.join(ROOT, "tests", "dropin", "spmm_shim.cpp"), "-o", out,
           "-L" + pkg, "-lsparse_b200", "-Wl,-rpath," + pkg]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    L = C.CDLL(out)
    L.spmm_shim_last_error.restype = C.c_char_p
    L.spmm_shim.argtypes = [C.c_int, _i32, _i32, _f64, C.c_int, C.c_int, C.c_int64, _f64, C.c_int64, C.c_int64, _f64]
    return L


# ---- 1. golden fixtures ----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k", [1, 3, 8, 33])
def test_golden_fixtures(golden, k, chk):
    g = golden
    args = (g["i"], g["p"], g["x"], g["nrow"], g["ncol"])
    specials = g["name"].startswith("specials")
    with DeviceMatrix.from_host(g["i"], g["p"], g["x"], g["nrow"], g["ncol"]) as M:
        B = operand(k, g["ncol"], k, specials)
        assert_columns("spmv", M.spmm(B), B, args, chk)
        Bt = operand(k + 100, g["nrow"], k, specials)
        assert_columns("spmv_t", M.spmm_t(Bt), Bt, args, chk)


# ---- 2. synthetic shapes: every slab width, the tail slab, columns spanning many tiles ------------------------------------
SHAPES = {
    "uniform": lambda: synth.uniform_spec(20_000, 300, 0.05, 61),  # ~1000 entries per column: columns span tiles
    "powerlaw": lambda: synth.powerlaw_spec(6_000, 2_500, 25.0, 62),
    "banded": lambda: synth.powerlaw_spec(5_000, 1_500, 40.0, 63, row_levels=5),
}


@pytest.fixture(scope="module", params=sorted(SHAPES))
def shape(request):
    spec = SHAPES[request.param]()
    i, p, x = synth.generate_host(spec)
    return spec, (i, p, x, spec.nrow, spec.ncol)


@gpu
@pytest.mark.parametrize("k", [2, 7, 16, 32, 64, 100, 257])
def test_synthetic_shapes(shape, k, chk):
    spec, args = shape
    with DeviceMatrix.from_host(*args) as M:
        B = operand(k, spec.ncol, k)
        assert_columns("spmv", M.spmm(B), B, args, chk)
        Bt = operand(k + 1, spec.nrow, k)
        assert_columns("spmv_t", M.spmm_t(Bt), Bt, args, chk)


# ---- 3. regimes and determinism ----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k", [5, 40])
def test_regimes_and_bit_stability(shape, k, chk):
    spec, args = shape
    B, Bt = operand(7, spec.ncol, k), operand(8, spec.nrow, k)
    with DeviceMatrix.from_host(*args) as M:
        M.row_companion(-1)  # A B on the CSC arrays: L2 reductions
        assert_columns("spmv", M.spmm(B), B, args, chk)
        y1, y2 = M.spmm_t(Bt), M.spmm_t(Bt)
        assert_columns("spmv_t", y1, Bt, args, chk)
        assert np.array_equal(bits(y1), bits(y2)), "A^T B on the CSC arrays must be bit-stable"
        M.row_companion(0)
        M.row_companion(1)  # A B on the row-ordered copy: gather-only
        assert M.row_path() == "row-companion"
        y1, y2 = M.spmm(B), M.spmm(B)
        assert_columns("spmv", y1, B, args, chk)
        assert np.array_equal(bits(y1), bits(y2)), "A B on the row-ordered copy must be bit-stable"


@gpu
def test_block_products_count_once_toward_the_row_ordered_copy():
    spec = SHAPES["powerlaw"]()
    args = synth.generate_host(spec) + (spec.nrow, spec.ncol)
    B = operand(3, spec.ncol, 4)
    with DeviceMatrix.from_host(*args) as M:
        for _ in range(8):  # SB200_ROW_COMPANION_AFTER defaults to 8 row-indexed calls
            M.spmm(B)
        assert M.row_path() != "row-companion"
        M.spmm(B)
        assert M.row_path() == "row-companion"


# ---- 4. column independence and k = 1 -------------------------------------------------------------------------------------
@gpu
def test_columns_match_the_device_spmv(shape):
    spec, args = shape
    with DeviceMatrix.from_host(*args) as M:
        M.band_companion(0, -1)
        M.row_companion(-1)
        B, Bt = operand(11, spec.ncol, 9), operand(12, spec.nrow, 9)
        Y, Yt = M.spmm(B), M.spmm_t(Bt)
        for j in range(9):
            oracle.assert_within("spmv", Y[:, j], M.spmv(B[:, j]), *args, v=B[:, j])
            oracle.assert_within("spmv_t", Yt[:, j], M.spmv_t(Bt[:, j]), *args, v=Bt[:, j])
        # k = 1 is the single-vector sweep: bitwise where that sweep is deterministic
        assert np.array_equal(bits(M.spmm_t(Bt[:, :1])[:, 0]), bits(M.spmv_t(Bt[:, 0])))
        oracle.assert_within("spmv", M.spmm(B[:, :1])[:, 0], M.spmv(B[:, 0]), *args, v=B[:, 0])
        M.row_companion(0)
        M.row_companion(1)
        assert np.array_equal(bits(M.spmm(B[:, :1])[:, 0]), bits(M.spmv(B[:, 0])))


# ---- 5. lazily uploaded row indices --------------------------------------------------------------------------------------
@gpu
def test_lazy_rows(chk):
    spec = SHAPES["banded"]()
    i, p, x = synth.generate_host(spec)
    args = (i, p, x, spec.nrow, spec.ncol)
    B, Bt = operand(21, spec.ncol, 6), operand(22, spec.nrow, 6)
    with DeviceMatrix.from_host(i, p, x, spec.nrow, spec.ncol, lazy_rows=True) as M:
        assert_columns("spmv_t", M.spmm_t(Bt), Bt, args, chk)
    with DeviceMatrix.from_host(i, p, x, spec.nrow, spec.ncol, lazy_rows=True) as M:
        assert_columns("spmv", M.spmm(B), B, args, chk)
    bad = i.copy()
    bad[len(bad) // 3] = spec.nrow + 9
    with DeviceMatrix.from_host(bad, p, x, spec.nrow, spec.ncol, lazy_rows=True) as M:
        for f, b in ((M.spmm, B), (M.spmm_t, Bt)):
            with pytest.raises(SparseB200Error) as e:
                f(b)
            assert e.value.code == _lib.E_STRUCTURE
    A = Matrix(x, i, p, np.array([spec.nrow, spec.ncol], np.int32))  # a per-call mirror of the Python drop-in
    assert_columns("spmv", A.spmm(B), B, args, chk)
    assert_columns("spmv_t", A.spmm_t(Bt), Bt, args, chk)


# ---- 6. arguments ------------------------------------------------------------------------------------------------------
@gpu
def test_arguments():
    import torch

    spec = SHAPES["powerlaw"]()
    args = synth.generate_host(spec) + (spec.nrow, spec.ncol)
    L = _lib.lib()
    with DeviceMatrix.from_host(*args) as M:
        before = L.sb200_launch_count()
        Y, Yt = M.spmm(np.zeros((spec.ncol, 0))), M.spmm_t(np.zeros((spec.nrow, 0)))
        assert Y.shape == (spec.nrow, 0) and Yt.shape == (spec.ncol, 0)
        assert L.sb200_launch_count() == before, "k = 0 launches nothing"
        buf = np.zeros(max(spec.nrow, spec.ncol) * 2)
        for fn in (L.sb200_spmm, L.sb200_spmm_t, L.sb200_spmm_dev, L.sb200_spmm_t_dev):
            assert fn(M._h, buf.ctypes.data, -1, buf.ctypes.data) == _lib.E_INVALID
            assert fn(M._h, None, 2, buf.ctypes.data) == _lib.E_INVALID
            assert fn(M._h, buf.ctypes.data, 2, None) == _lib.E_INVALID
        for bad in (np.zeros((spec.ncol + 1, 2)), np.zeros(spec.ncol), np.zeros((spec.ncol, 2, 1))):
            with pytest.raises(ValueError):
                M.spmm(bad)
        with pytest.raises(ValueError):
            M.spmm_t(np.zeros((spec.ncol, 2)))
        # device form on torch tensors: a column-major (rows, k) block is a contiguous (k, rows) tensor
        k = 19
        Bt = operand(31, spec.nrow, k)
        d_B = torch.from_numpy(np.ascontiguousarray(Bt.T)).cuda()
        d_Y = torch.full((k, spec.ncol), np.nan, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        M.spmm_t_dev(d_B, k, d_Y)
        M.sync()
        assert np.array_equal(bits(d_Y.cpu().numpy().T), bits(M.spmm_t(Bt)))
        B = operand(32, spec.ncol, k)
        d_B = torch.from_numpy(np.ascontiguousarray(B.T)).cuda()
        d_Y = torch.full((k, spec.nrow), np.nan, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        M.spmm_dev(d_B, k, d_Y)
        M.sync()
        oracle.assert_within("spmv", d_Y.cpu().numpy()[3], M.spmm(B)[:, 3], *args, v=B[:, 3])


# ---- 7. 64-bit sizes: nrow * k > 2^31 ----------------------------------------------------------------------------------
@gpu
def test_index_width_past_two_to_the_31():
    import scipy.sparse as sp
    import torch

    nrow, k = 1 << 25, 65
    assert nrow * k > 2**31
    if torch.cuda.mem_get_info()[0] < 64 << 30:
        pytest.skip("needs 64 GB of free device memory")
    spec = synth.uniform_spec(nrow, 48, 1e-4, 71)
    i, p, x = synth.generate_host(spec)
    A = sp.csc_matrix((x, i, p), shape=(nrow, spec.ncol))
    rows = np.unique(np.concatenate([i[:: max(1, len(i) // 300)], [0, nrow - 1], i[-5:]]))
    with DeviceMatrix.from_host(i, p, x, nrow, spec.ncol) as M:
        B = operand(41, spec.ncol, k)
        d_B = torch.from_numpy(np.ascontiguousarray(B.T)).cuda()
        d_Y = torch.empty((k, nrow), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        M.spmm_dev(d_B, k, d_Y)
        M.sync()
        got = d_Y[:, torch.from_numpy(rows).cuda()].cpu().numpy().T
        del d_Y
        want = A[rows] @ B
        assert np.all(np.abs(got - want) <= 1e-12 * (abs(A[rows]) @ np.abs(B)))
        # A^T B with an operand of nrow * k entries, B[r, j] = ((131 r + 7 j) mod 1000) / 100 - 5
        d_B = torch.empty((k, nrow), dtype=torch.float64, device="cuda")
        r = torch.arange(nrow, dtype=torch.int64, device="cuda")
        for j in range(k):
            d_B[j] = ((131 * r + 7 * j) % 1000).double() / 100.0 - 5.0
        del r
        d_Yt = torch.empty((k, spec.ncol), dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        M.spmm_t_dev(d_B, k, d_Yt)
        M.sync()
        got = d_Yt.cpu().numpy().T
        del d_B
    col_of = np.repeat(np.arange(spec.ncol), np.diff(p))
    Bv = ((131 * i.astype(np.int64)[:, None] + 7 * np.arange(k)[None, :]) % 1000) / 100.0 - 5.0
    want = np.zeros((spec.ncol, k))
    feed = np.zeros((spec.ncol, k))
    np.add.at(want, col_of, x[:, None] * Bv)
    np.add.at(feed, col_of, np.abs(x[:, None] * Bv))
    assert np.all(np.abs(got - want) <= 1e-12 * feed)


# ---- 8. the drop-in C++ header -----------------------------------------------------------------------------------------
@gpu
def test_dropin_header(shim, golden, chk):
    g = golden
    i, p, x, nrow, ncol = g["i"], g["p"], g["x"], g["nrow"], g["ncol"]
    args = (i, p, x, nrow, ncol)
    for transposed, rows, out_rows, op in ((0, ncol, nrow, "spmv"), (1, nrow, ncol, "spmv_t")):
        B = operand(5 + transposed, rows, 4)
        Y = np.empty((4, out_rows))  # column-major out_rows x 4
        assert shim.spmm_shim(transposed, i, p, x, nrow, ncol, len(x), np.ascontiguousarray(B.T).reshape(-1), rows, 4,
                                Y.reshape(-1)) == 0, shim.spmm_shim_last_error()
        assert_columns(op, Y.T, B, args, chk)
        wrong = np.zeros((rows + 1) * 4)
        assert shim.spmm_shim(transposed, i, p, x, nrow, ncol, len(x), wrong, rows + 1, 4, np.empty(max(out_rows, 1) * 4)) == 1
        assert b"invalid_argument" in shim.spmm_shim_last_error()


# ---- 9. no device: an error, never a CPU path ------------------------------------------------------------------------------
def test_without_gpu_spmm_is_an_error(shim):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "vignette_5x5.npz")))
    g["nrow"], g["ncol"] = int(g["dim"][0]), int(g["dim"][1])
    A = Matrix(g["x"], g["i"], g["p"], g["dim"])
    with pytest.raises(SparseB200Error) as e:
        A.spmm(np.ones((g["ncol"], 3)))
    assert e.value.code == _lib.E_NODEVICE
    B = np.ones(g["ncol"] * 3)
    assert shim.spmm_shim(0, g["i"], g["p"], g["x"], g["nrow"], g["ncol"], len(g["x"]), B, g["ncol"], 3,
                            np.empty(g["nrow"] * 3)) == 2
    assert b"no CUDA device" in shim.spmm_shim_last_error()
