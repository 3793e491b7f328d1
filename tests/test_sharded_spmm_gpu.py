"""Block products on every GPU of the process (sparse_b200.h sb200_sharded_spmm / sb200_sharded_spmm_t).

Column j of Y must be what spmv / spmv_t gives for column j of B, within |delta| <= 1e-12 * sum |a b| per entry, with
NaN and Inf in B reaching exactly the outputs they touch.  A B sums the blocks' partials across devices with a new
rank-ordered reduce; A^T B copies every block's rows of Y straight home.

Both are ordered across devices by CUDA events only, so a handle whose `devices` list repeats one GPU
(ShardedHostMatrix(..., n_gpus=W, devices=[0] * W)) runs every multi-block code path on a one-GPU machine: the column
split of B, empty blocks, the rank-ordered reduce and the strided copies.  On such handles only spmm / spmm_t are
called: rowSums, rowMeans and spmv exchange through a kernel with an in-kernel barrier, which needs the blocks' kernels
to be resident at once.  The same cases run on W distinct GPUs where the machine has them."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import oracle
from rcppsparse_b200 import DeviceMatrix, Matrix, ShardedHostMatrix, SparseB200Error, _lib, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
gpu = pytest.mark.gpu
_i32 = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_f64 = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")

# (placement, W): W blocks on GPU 0, or on GPUs 0 .. W-1
PLACEMENTS = [("one-gpu", 1), ("one-gpu", 2), ("one-gpu", 3), ("distinct", 2), ("distinct", 4), ("distinct", 8)]
PLACEMENT_IDS = [f"{p}-W{w}" for p, w in PLACEMENTS]
KS = [1, 2, 3, 8, 33, 65]


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def operand(seed, rows, k, specials=False):
    B = np.round(np.random.default_rng(seed).standard_normal((rows, k)), 3)
    if specials and rows > 2 and k > 0:
        j = min(1, k - 1)
        B[0, j], B[rows // 2, j], B[rows - 1, k - 1] = np.nan, np.inf, -np.inf
    return np.asfortranarray(B)


def assert_columns(op, Y, B, args, chk, what=""):
    """Every column of Y against the checker's spmv / spmv_t of that column of B."""
    nrow, ncol = args[3], args[4]
    assert Y.shape == ((nrow if op == "spmv" else ncol), B.shape[1]), what
    for j in range(B.shape[1]):
        v = np.ascontiguousarray(B[:, j])
        oracle.assert_within(op, Y[:, j], getattr(chk, op)(*args, v), *args, v=v)


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
    "uniform": lambda: synth.uniform_spec(20_000, 300, 0.05, 61),  # ~1000 entries per column: columns span tiles
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
    out = str(tmp_path_factory.mktemp("sharded_spmm_shim") / "libspmm_shim.so")
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


# ---- 0. the binding, no GPU needed -------------------------------------------------------------------------------------
def test_binding_declares_and_resolves_the_sharded_block_products():
    header = open(os.path.join(ROOT, "include", "sparse_b200.h")).read()
    L = _lib.lib()
    for name in ("sb200_sharded_spmm", "sb200_sharded_spmm_t"):
        assert name in _lib.SYMBOLS
        assert re.search(r"\bint " + name + r"\(sb200_sharded\* s, const double\* B", header), name
        fn = getattr(L, name)
        assert fn.restype is C.c_int and len(fn.argtypes) == 4 and fn.argtypes[2] is C.c_int64


# ---- 1. parity with the checker's spmv / spmv_t, every column ----------------------------------------------------------
@gpu
@pytest.mark.parametrize("placement,W", PLACEMENTS, ids=PLACEMENT_IDS)
def test_creation_with_repeated_or_distinct_devices(placement, W):
    args = load_golden("vignette_5x5")
    with sharded(args, placement, W) as S:
        b = S.bounds()
        assert len(b) == W + 1 and b[0] == 0 and b[-1] == args[4]


@gpu
@pytest.mark.parametrize("placement,W", PLACEMENTS, ids=PLACEMENT_IDS)
@pytest.mark.parametrize("name", GOLDEN)
def test_golden_fixtures(name, placement, W, chk):
    args = load_golden(name)
    nrow, ncol = args[3], args[4]
    with sharded(args, placement, W) as S:
        for k in KS:
            specials = k in (3, 33) or name.startswith("specials")
            B = operand(k, ncol, k, specials)
            assert_columns("spmv", S.spmm(B), B, args, chk)
            Bt = operand(k + 100, nrow, k, specials)
            assert_columns("spmv_t", S.spmm_t(Bt), Bt, args, chk)


@gpu
@pytest.mark.parametrize("placement,W", PLACEMENTS, ids=PLACEMENT_IDS)
@pytest.mark.parametrize("name", sorted(SYNTH) + ["two_columns"])
def test_synthetic_shapes(name, placement, W, chk):
    args = two_columns() if name == "two_columns" else synth_args(name)
    nrow, ncol = args[3], args[4]
    with sharded(args, placement, W) as S:
        for k in KS:
            B = operand(k, ncol, k, specials=k == 8)
            assert_columns("spmv", S.spmm(B), B, args, chk)
            Bt = operand(k + 1, nrow, k, specials=k == 8)
            assert_columns("spmv_t", S.spmm_t(Bt), Bt, args, chk)


# ---- 2. exact: integer data, every output bit for bit ------------------------------------------------------------------
EXACT_MAX = 2.0**52


def exact_case(i, p, nrow, ncol, transposed, K, seed):
    """x = +-{1..7}, about one entry in 64 scaled by 2^E; B = +-{1..7}, about one in 64 scaled by 2^10; E the largest
    with sum |terms| <= 2^52 for every output, so every partial sum is an exact integer and any order gives the same
    bits.  Returns x, B (Fortran) and the exact Y."""
    rng = np.random.default_rng(seed)
    nnz = len(i)
    col_of = np.repeat(np.arange(ncol), np.diff(p))
    out, opi, n_out, n_op = (col_of, i, ncol, nrow) if transposed else (i, col_of, nrow, ncol)
    mag = rng.integers(1, 8, nnz).astype(np.float64)
    sgn = np.where(rng.random(nnz) < 0.5, -1.0, 1.0)
    big = rng.random(nnz) < 1.0 / 64
    w = rng.integers(1, 8, (n_op, K)).astype(np.float64) * 2.0 ** (10 * (rng.random((n_op, K)) < 1.0 / 64))
    small = np.asarray(sp.csr_matrix((mag * ~big, (out, opi)), shape=(n_out, n_op)) @ w)
    large = np.asarray(sp.csr_matrix((mag * big, (out, opi)), shape=(n_out, n_op)) @ w)
    E = next(e for e in range(52, -1, -1) if (small + large * 2.0**e).max() <= EXACT_MAX)
    x = sgn * mag * 2.0 ** (E * big)
    B = np.asfortranarray(np.where(rng.random((n_op, K)) < 0.5, -1.0, 1.0) * w)
    Y = np.asarray(sp.csr_matrix((x, (out, opi)), shape=(n_out, n_op)) @ B)
    return x, B, Y


@pytest.fixture(scope="module")
def exact_data():
    """~9 M stored entries over 60 000 columns: at least 2.5 M merge items per block at W <= 3, so tiles, carries and
    the sweeps' CTA rings wrap inside every block there.  The distinct W = 4 and W = 8 placements split the same matrix
    into smaller blocks: they check the reduce and the copies exactly, not the wrapping.  Exact data for A^T B (True)
    and A B (False), 33 columns of B."""
    spec = synth.uniform_spec(50_000, 60_000, 0.003, 81)
    i, p, _ = synth.generate_host(spec)
    assert (len(i) + spec.ncol) // 3 >= 2_500_000
    return i, p, spec.nrow, spec.ncol, {t: exact_case(i, p, spec.nrow, spec.ncol, t, 33, 90 + t) for t in (True, False)}


@gpu
@pytest.mark.parametrize("placement,W", PLACEMENTS, ids=PLACEMENT_IDS)
def test_exact(exact_data, placement, W):
    i, p, nrow, ncol, cases = exact_data
    for transposed in (True, False):
        x, B, want = cases[transposed]
        with sharded((i, p, x, nrow, ncol), placement, W) as S:
            f = S.spmm_t if transposed else S.spmm
            for k in (2, 8, 33):
                got = f(B[:, :k])
                assert np.array_equal(got, want[:, :k]), f"{'A^T B' if transposed else 'A B'} k = {k}: " \
                    f"{int((got != want[:, :k]).sum())} outputs differ from the exact reference"
            if not transposed:  # A B once more, every block on its row-ordered copy
                for w in range(W):
                    S.block(w).row_companion(1)
                assert np.array_equal(f(B), want), "A B on the row-ordered copies"


# ---- 3. one block: bit for bit the one-GPU path ------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", sorted(SYNTH))
def test_world_one_equals_one_gpu(name):
    args = synth_args(name)
    with ShardedHostMatrix(*args, 1) as S, DeviceMatrix.from_host(*args) as M:
        for k in (1, 5, 40):
            Bt = operand(k, args[3], k)
            assert np.array_equal(bits(S.spmm_t(Bt)), bits(M.spmm_t(Bt))), f"A^T B, k = {k}"
        S.block(0).row_companion(1)
        M.row_companion(1)
        for k in (1, 5, 40):
            B = operand(k + 50, args[4], k)
            assert np.array_equal(bits(S.spmm(B)), bits(M.spmm(B))), f"A B on the row-ordered copy, k = {k}"


# ---- 4. run-to-run bit stability ---------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("placement,W", PLACEMENTS, ids=PLACEMENT_IDS)
def test_bit_stability(placement, W, chk):
    args = synth_args("powerlaw")
    with sharded(args, placement, W) as S:
        for k in (4, 40):
            Bt = operand(k, args[3], k)
            assert np.array_equal(bits(S.spmm_t(Bt)), bits(S.spmm_t(Bt))), f"A^T B, k = {k}"
        for w in range(W):
            S.block(w).row_companion(1)
        for k in (1, 4, 40):
            B = operand(k + 7, args[4], k)
            y1, y2 = S.spmm(B), S.spmm(B)
            assert np.array_equal(bits(y1), bits(y2)), f"A B on the row-ordered copies, k = {k}"
            assert_columns("spmv", y1, B, args, chk)


# ---- 5. ski rental: a k-wide call counts once per block toward its row-ordered copy ------------------------------------
@gpu
@pytest.mark.parametrize("placement,W", [("one-gpu", 3), ("distinct", 2)], ids=["one-gpu-W3", "distinct-W2"])
def test_row_ordered_copies_built_after_repeated_calls(placement, W, chk):
    args = synth_args("powerlaw")
    B = operand(3, args[4], 4)
    with sharded(args, placement, W) as S:
        for _ in range(8):  # SB200_ROW_COMPANION_AFTER defaults to 8 row-indexed calls
            y = S.spmm(B)
        assert not any(S.block(w).layouts() & 1 for w in range(W))
        assert_columns("spmv", y, B, args, chk)
        y = S.spmm(B)
        assert all(S.block(w).layouts() & 1 for w in range(W)), "every block keeps its row-ordered copy"
        assert_columns("spmv", y, B, args, chk)
        assert np.array_equal(bits(S.spmm(B)), bits(y))


# ---- 6. k = 0 and k = 1 ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("placement,W", PLACEMENTS, ids=PLACEMENT_IDS)
def test_k_zero_launches_nothing(placement, W):
    args = synth_args("banded")
    L = _lib.lib()
    with sharded(args, placement, W) as S:
        before = L.sb200_launch_count()
        Y, Yt = S.spmm(np.zeros((args[4], 0))), S.spmm_t(np.zeros((args[3], 0)))
        assert Y.shape == (args[3], 0) and Yt.shape == (args[4], 0)
        assert L.sb200_launch_count() == before, "k = 0 launches nothing"


@gpu
@pytest.mark.parametrize("W", [2, 4, 8])
def test_k_one_agrees_with_the_sharded_spmv(W):
    args = synth_args("uniform")
    with sharded(args, "distinct", W) as S:
        B, Bt = operand(1, args[4], 1), operand(2, args[3], 1)
        assert np.array_equal(bits(S.spmm_t(Bt)[:, 0]), bits(S.spmv_t(Bt[:, 0]))), "A^T v: the same sweeps"
        oracle.assert_within("spmv", S.spmm(B)[:, 0], S.spmv(B[:, 0]), *args, v=B[:, 0])


# ---- 7. arguments ------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("placement,W", [("one-gpu", 2), ("distinct", 2)], ids=["one-gpu-W2", "distinct-W2"])
def test_arguments(placement, W, chk):
    args = synth_args("powerlaw")
    nrow, ncol = args[3], args[4]
    L = _lib.lib()
    S = sharded(args, placement, W)
    buf = np.zeros(max(nrow, ncol) * 2)
    for fn in (L.sb200_sharded_spmm, L.sb200_sharded_spmm_t):
        assert fn(S._h, buf.ctypes.data, -1, buf.ctypes.data) == _lib.E_INVALID
        assert fn(S._h, None, 2, buf.ctypes.data) == _lib.E_INVALID
        assert fn(S._h, buf.ctypes.data, 2, None) == _lib.E_INVALID
        assert fn(None, buf.ctypes.data, 2, buf.ctypes.data) == _lib.E_INVALID
        # scratch that cannot fit: SB200_E_NOMEM before anything is read, and the handle stays usable
        assert fn(S._h, buf.ctypes.data, 1 << 40, buf.ctypes.data) == _lib.E_NOMEM
    for bad in (np.zeros((ncol + 1, 2)), np.zeros(ncol), np.zeros((ncol, 2, 1))):
        with pytest.raises(ValueError):
            S.spmm(bad)
    with pytest.raises(ValueError):
        S.spmm_t(np.zeros((ncol, 2)))
    B = operand(5, ncol, 6)
    assert_columns("spmv", S.spmm(B), B, args, chk)
    S.close()
    for f, b in ((S.spmm, B), (S.spmm_t, operand(6, nrow, 6))):
        with pytest.raises(SparseB200Error) as e:
            f(b)
        assert e.value.code == _lib.E_INVALID


# ---- 8. 64-bit sizes: nrow * k > 2^31 ----------------------------------------------------------------------------------
@gpu
def test_index_width_past_two_to_the_31():
    import torch

    nrow, k, W = (1 << 25) + 3, 65, 2
    assert nrow * k > 2**31
    if torch.cuda.mem_get_info()[0] < 80 << 30:
        pytest.skip("needs 80 GB of free device memory")
    if os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_AVPHYS_PAGES") < 48 << 30:
        pytest.skip("needs 48 GB of free host memory for the 17 GB result")
    spec = synth.uniform_spec(nrow, 48, 1e-4, 71)
    i, p, x = synth.generate_host(spec)
    A = sp.csc_matrix((x, i, p), shape=(nrow, spec.ncol))
    rows = np.unique(np.concatenate([i[:: max(1, len(i) // 300)], [0, nrow - 1, nrow // 2, nrow // 2 - 1], i[-5:]]))
    B = operand(41, spec.ncol, k)
    placement = "distinct" if _lib.device_count() >= W else "one-gpu"
    with sharded((i, p, x, nrow, spec.ncol), placement, W) as S:
        Y = S.spmm(B)
    got = Y[rows]
    del Y
    want = A[rows] @ B
    assert np.all(np.abs(got - want) <= 1e-12 * (abs(A[rows]) @ np.abs(B)))


# ---- 8b. pageable operands and results above the staging threshold: the strided pinned-chunk copies, both ways -----------
@gpu
def test_large_pageable_operands_go_through_the_strided_staged_copies():
    """1.2 M x 1.2 M, k = 33 at W = 2 on one GPU: every block's slice of B (A B: ncol/2 rows of a column-major B) and
    every piece of Y is ~160 MB of pageable memory, over the 32 MB from which the library stages host copies through
    its pinned-chunk workers.  A^T B uploads all of B (317 MB) to every block.  Every output is checked."""
    n, k = 1_200_000, 33
    spec = synth.uniform_spec(n, n, 4e-6, 83)
    i, p, x = synth.generate_host(spec)
    A = sp.csc_matrix((x, i, p), shape=(n, n))
    absA = abs(A)
    pattern = sp.csc_matrix((np.ones_like(x), i, p), shape=(n, n))
    assert n // 2 * k * 8 >= 32 << 20
    with sharded((i, p, x, n, n), "one-gpu", 2) as S:
        for op, f, M, Ma, Mp in (("A B", S.spmm, A, absA, pattern), ("A^T B", S.spmm_t, A.T.tocsr(), absA.T.tocsr(), pattern.T.tocsr())):
            B = operand(17, n, k, specials=True)
            Y = f(B)
            want = M @ np.nan_to_num(B, nan=0.0, posinf=0.0, neginf=0.0)
            feed = Ma @ np.abs(np.nan_to_num(B, nan=0.0, posinf=0.0, neginf=0.0))
            special = (Mp @ (~np.isfinite(B)).astype(np.float64)) > 0  # outputs a NaN or Inf of B reaches
            assert np.all(np.abs(Y[~special] - want[~special]) <= 1e-12 * feed[~special]), op
            assert not np.isfinite(Y[special]).any(), f"{op}: a NaN or Inf of B must reach every output it touches"


# ---- 9. routing: the Python drop-in and the C++ header under SB200_GPUS = 2 ---------------------------------------------
@gpu
def test_matrix_routes_block_products_to_the_sharded_handle(chk):
    if _lib.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    i, p, x, nrow, ncol = synth_args("banded")
    x = x.copy()
    A = Matrix(x, i, p, np.array([nrow, ncol], np.int32), gpus=2, resident=True)
    B, Bt = operand(1, ncol, 5), operand(2, nrow, 5)
    assert_columns("spmv", A.spmm(B), B, (i, p, x, nrow, ncol), chk)
    assert_columns("spmv_t", A.spmm_t(Bt), Bt, (i, p, x, nrow, ncol), chk)
    assert A._sharded is not None and A._dev is None, "gpus = 2 runs the block products on the sharded handle"
    x *= -2.0  # in place: the resident mirror sees it after refresh()
    A.refresh()
    assert_columns("spmv", A.spmm(B), B, (i, p, x, nrow, ncol), chk)
    assert_columns("spmv_t", A.spmm_t(Bt), Bt, (i, p, x, nrow, ncol), chk)
    A.release()
    per_call = Matrix(x, i, p, np.array([nrow, ncol], np.int32), gpus=2)
    assert_columns("spmv", per_call.spmm(B), B, (i, p, x, nrow, ncol), chk)


@gpu
def test_dropin_header_under_SB200_GPUS(shim, chk, monkeypatch, capfd):
    if _lib.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    monkeypatch.setenv("SB200_GPUS", "2")
    monkeypatch.setenv("SB200_TRACE", "1")  # the sharded entry points name themselves on stderr
    i, p, x, nrow, ncol = args = synth_args("powerlaw")
    for transposed, rows, out_rows, op in ((0, ncol, nrow, "spmv"), (1, nrow, ncol, "spmv_t")):
        B = operand(5 + transposed, rows, 4)
        Y = np.empty((4, out_rows))  # column-major out_rows x 4
        capfd.readouterr()
        assert shim.spmm_shim(transposed, i, p, x, nrow, ncol, len(x), np.ascontiguousarray(B.T).reshape(-1), rows, 4,
                              Y.reshape(-1)) == 0, shim.spmm_shim_last_error()
        assert ("sharded spmm_t" if transposed else "sharded spmm:") in capfd.readouterr().err
        assert_columns(op, Y.T, B, args, chk)
