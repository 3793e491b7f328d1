"""GPU parity tests: the CUDA path, called through the C ABI (host-buffer entry points, the same
ones include/RcppSparse.h calls), against the oracle on identical inputs.

Bar (BASELINE.json north_star): transpose structure p/i and the permuted values bit-exact;
FP64 reductions within |delta| <= 1e-12 * sum|a_ij| (|a_ij * v_j| for SpMV) per output entry.
"""
import os

import numpy as np
import pytest

from oracle import oracle
from rcppsparse_b200 import DeviceMatrix, Matrix, SparseB200Error, _lib, columnSums, synth

pytestmark = pytest.mark.gpu

TOL = 1e-12  # north_star tolerance


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def zlib_seed(name):
    import zlib

    return zlib.crc32(name.encode())


@pytest.fixture(scope="module")
def checker():
    return oracle.best()  # the compiled reference when it travelled to this box, else the C port


def as_matrix(g):
    return Matrix(g["x"], g["i"], g["p"], g["dim"])


# ---------------------------------------------------------------------------------------------------
# committed golden vectors (produced by the reference's own compiled code, tests/golden/make_golden.py)
# ---------------------------------------------------------------------------------------------------
def test_golden_reductions(golden):
    g = golden
    A = as_matrix(g)
    args = (g["i"], g["p"], g["x"], g["nrow"], g["ncol"])
    for op, got in (("colSums", A.colSums()), ("rowSums", A.rowSums()), ("colMeans", A.colMeans()),
                    ("rowMeans", A.rowMeans()), ("columnSums", columnSums(A))):
        oracle.assert_within(op, got, g[op], *args, tol=TOL)
    A.release()


def test_golden_spmv(golden):
    g = golden
    A = as_matrix(g)
    args = (g["i"], g["p"], g["x"], g["nrow"], g["ncol"])
    oracle.assert_within("spmv", A.spmv(g["v_col"]), g["spmv"], *args, v=g["v_col"], tol=TOL)
    oracle.assert_within("spmv_t", A.spmv_t(g["v_row"]), g["spmv_t"], *args, v=g["v_row"], tol=TOL)
    A.release()


def test_golden_transpose_bit_exact(golden):
    g = golden
    A = as_matrix(g)
    T = A.transpose()
    assert T.Dim.tolist() == [g["ncol"], g["nrow"]]
    assert np.array_equal(T.p, g["t_p"]), "p' differs"
    assert np.array_equal(T.i, g["t_i"]), "i' differs (order inside a column must be ascending)"
    assert np.array_equal(bits(T.x), bits(g["t_x"])), "x' must be a bit-exact permutation"
    assert A.t().p.tolist() == g["t_p"].tolist()  # the vignette's .t() alias
    A.release()


def test_vignette_known_answers_on_gpu():
    """The only literal matrix in the reference tree (vignettes/Documentation.Rmd:213-216)."""
    A = Matrix(np.array([0.41, 0.35, 0.84, 0.37, 0.26]), np.array([0, 2, 0, 1, 1], np.int32),
               np.array([0, 0, 1, 2, 4, 5], np.int32), np.array([5, 5], np.int32))
    assert A.colSums().tolist() == [0.0, 0.41, 0.35, 1.21, 0.26]
    assert A.rowSums().tolist() == [1.25, 0.63, 0.35, 0.0, 0.0]
    assert A.colMeans().tolist() == [0.0, 0.08199999999999999, 0.069999999999999993, 0.24199999999999999,
                                     0.052000000000000005]
    T = A.transpose()
    assert T.p.tolist() == [0, 2, 4, 5, 5, 5] and T.i.tolist() == [1, 3, 3, 4, 2]
    assert T.x.tolist() == [0.41, 0.84, 0.37, 0.26, 0.35]


# ---------------------------------------------------------------------------------------------------
# seeded synthetic matrices at sizes the oracle finishes in seconds
# ---------------------------------------------------------------------------------------------------
SYNTH_CASES = {
    "C1_full": lambda: synth.config("C1"),                      # 10k x 10k, 1e6 nnz — BASELINE configs[0]
    "C2_scaled": lambda: synth.config("C2", 0.05),              # 1M x 5k, 5e6 nnz
    "C3_scaled": lambda: synth.config("C3", 0.004),             # 30k x 4k, ~6e6 nnz, banded row popularity
    "C4_scaled": lambda: synth.config("C4", 0.003),             # 2^20 x 6k power-law columns
    "many_tiny_columns": lambda: synth.powerlaw_spec(5000, 300_000, 2.0, 77, empty_permille=400),
    "few_huge_columns": lambda: synth.uniform_spec(400_000, 7, 0.9, 78),
    "tall_sparse": lambda: synth.uniform_spec(3_000_000, 64, 0.01, 79),
}


@pytest.fixture(scope="module", params=sorted(SYNTH_CASES))
def synth_case(request):
    spec = SYNTH_CASES[request.param]()
    i, p, x = synth.generate_host(spec)
    return request.param, spec, i, p, x


def test_synth_device_generator_matches_host_bitwise(synth_case):
    name, spec, i, p, x = synth_case
    with DeviceMatrix.synth(spec) as D:
        di, dp, dx = D.download_columns()
    assert np.array_equal(dp, p) and np.array_equal(di, i) and np.array_equal(bits(dx), bits(x)), name


def test_synth_reductions_and_spmv(synth_case, checker):
    name, spec, i, p, x = synth_case
    nrow, ncol = spec.nrow, spec.ncol
    A = Matrix(x, i, p, np.array([nrow, ncol], np.int32))
    args = (i, p, x, nrow, ncol)
    worst = {}
    for op in ("colSums", "rowSums", "colMeans", "rowMeans"):
        worst[op] = oracle.assert_within(op, getattr(A, op)(), getattr(checker, op)(*args), *args, tol=TOL)
    v_col, v_row = synth.dense_vector(spec.seed, ncol), synth.dense_vector(spec.seed + 7, nrow)
    worst["spmv"] = oracle.assert_within("spmv", A.spmv(v_col), checker.spmv(*args, v_col), *args, v=v_col, tol=TOL)
    worst["spmv_t"] = oracle.assert_within("spmv_t", A.spmv_t(v_row), checker.spmv_t(*args, v_row), *args, v=v_row,
                                           tol=TOL)
    print(name, {k: f"{v:.2e}" for k, v in worst.items()})
    A.release()


def test_synth_transpose_bit_exact(synth_case, checker):
    name, spec, i, p, x = synth_case
    nrow, ncol = spec.nrow, spec.ncol
    A = Matrix(x, i, p, np.array([nrow, ncol], np.int32))
    T = A.transpose()
    ti, tp, tx = checker.transpose(i, p, x, nrow, ncol)
    assert np.array_equal(T.p, tp), name
    assert np.array_equal(T.i, ti), name
    assert np.array_equal(bits(T.x), bits(tx)), name
    A.release()


@pytest.mark.parametrize("rank", ["bitmap", "match"])
@pytest.mark.parametrize("cfg", ["256x2048:1", "256x2048:3", "256x4096:4", "512x3072:2", "256x1024:1", "256x1024:2", "512x2048:1",
                                 "256x1024:1:nocarry", "256x2048:2:nocarry"])
def test_transpose_chunk_sort_placement_on_every_shape(synth_case, cfg, rank, monkeypatch, checker):
    """The chunk-sorting placement kernel (transpose.cu) forced on every synthetic shape — also the tall ones the
    library would give to the banded two-pass kernel — in both block geometries and with 1, 2 and 4 columns per
    thread and chunk: bit-exact whatever the geometry."""
    name, spec, i, p, x = synth_case
    geom, kcols = cfg.split(":")[:2]
    # bitmap ranks place a window in full rounds and carry the rest into the next window; nocarry = whole windows
    monkeypatch.setenv("SB200_TRANSPOSE_CARRY", "0" if cfg.endswith(":nocarry") else "1")
    monkeypatch.setenv("SB200_TRANSPOSE_PATH", "place")
    monkeypatch.setenv("SB200_TRANSPOSE_RANK", rank)  # bitmap ranks (default) or per-warp counters + match.any
    monkeypatch.setenv("SB200_TRANSPOSE_CFG", geom)
    monkeypatch.setenv("SB200_TRANSPOSE_KCOLS", kcols)
    with DeviceMatrix.from_host(i, p, x, spec.nrow, spec.ncol) as D:
        for _ in range(2):  # the second call reuses the plan kept on the handle
            ti, tp, tx = D.transpose_host()
            wi, wp, wx = checker.transpose(i, p, x, spec.nrow, spec.ncol)
            assert np.array_equal(tp, wp) and np.array_equal(ti, wi) and np.array_equal(bits(tx), bits(wx)), (name, cfg)
        assert D.layouts() & 8


@pytest.mark.parametrize("kcols", ["1", "4"])
@pytest.mark.parametrize("bands", ["3", "40"])
def test_transpose_chunks_larger_than_the_image(bands, kcols, monkeypatch, checker):
    """Half-dense matrix, few wide bands: a chunk's runs hold many times the 4096 entries of the shared-memory image,
    so every chunk is placed in several rounds; the forced banded path must give the same bits."""
    spec = synth.uniform_spec(1000, 2000, 0.5, 93)
    i, p, x = synth.generate_host(spec)
    want = checker.transpose(i, p, x, spec.nrow, spec.ncol)
    monkeypatch.setenv("SB200_TRANSPOSE_BANDS", bands)
    monkeypatch.setenv("SB200_TRANSPOSE_KCOLS", kcols)
    for path in ("place", "place-match", "banded"):
        monkeypatch.setenv("SB200_TRANSPOSE_RANK", "match" if path == "place-match" else "bitmap")
        path = "place" if path.startswith("place") else path
        monkeypatch.setenv("SB200_TRANSPOSE_PATH", path)
        with DeviceMatrix.from_host(i, p, x, spec.nrow, spec.ncol) as D:
            ti, tp, tx = D.transpose_host()
        assert np.array_equal(tp, want[1]) and np.array_equal(ti, want[0]) and np.array_equal(bits(tx), bits(want[2])), path


@pytest.mark.parametrize("shift", [None, "2", "7", "11"])
def test_transpose_two_stream_splits_on_every_shape(synth_case, shift, monkeypatch, checker):
    """The two-split transpose of tall matrices (transpose_split.cu) forced on every synthetic shape, with the band
    width the library would pick and with forced ones (4, 128 and 2048 rows per band; where the key table holds fewer
    bands than that gives, the narrowest band it allows): bit-exact whatever the band width; the second call reuses
    the plan kept on the handle."""
    name, spec, i, p, x = synth_case
    monkeypatch.setenv("SB200_TRANSPOSE_PATH", "split")
    if shift is not None:
        sh = int(shift)
        while (spec.nrow >> sh) >= 3072:  # at most 3072 bands (SP_MAX_KEYS)
            sh += 1
        monkeypatch.setenv("SB200_SPLIT_SHIFT", str(sh))
    wi, wp, wx = checker.transpose(i, p, x, spec.nrow, spec.ncol)
    with DeviceMatrix.from_host(i, p, x, spec.nrow, spec.ncol) as D:
        launches = []
        for _ in range(2):
            n0 = _lib.lib().sb200_launch_count()
            ti, tp, tx = D.transpose_host()
            launches.append(_lib.lib().sb200_launch_count() - n0)
            assert np.array_equal(tp, wp) and np.array_equal(ti, wi) and np.array_equal(bits(tx), bits(wx)), (name, shift)
        if len(x):
            assert D.layouts() & 8 and launches[1] == 2, launches  # the two passes, nothing else, on a cached plan


def test_transpose_two_stream_splits_hot_rows_and_short_columns(monkeypatch, checker):
    """What the stable split must not trip over: a few rows holding most of the entries (thousands of equal keys in
    one chunk), columns of length 0 and 1 between long ones (the column walk), a last tile of one entry."""
    rng = np.random.default_rng(77)
    nrow = 70_000
    hot = np.array([5, 6, 40_000, 69_999])
    lengths = list(rng.choice([0, 1, 2, 40, 3000], 5_000, p=[0.3, 0.3, 0.2, 0.15, 0.05]))
    cols = []
    for n in lengths:
        rows = rng.choice(nrow, n, replace=False)
        if n >= 2:
            rows[:min(4, n)] = hot[:min(4, n)]
        cols.append(np.unique(rows))
    while (sum(len(c) for c in cols) % 4096) != 1:  # single-entry columns until the last tile holds one entry
        cols.append(rng.integers(0, nrow, 1))
    ncol = len(cols)
    p = np.zeros(ncol + 1, np.int32)
    p[1:] = np.cumsum([len(c) for c in cols])
    i = np.concatenate(cols).astype(np.int32)
    x = rng.standard_normal(len(i))
    monkeypatch.setenv("SB200_TRANSPOSE_PATH", "split")
    wi, wp, wx = checker.transpose(i, p, x, nrow, ncol)
    with DeviceMatrix.from_host(i, p, x, nrow, ncol) as D:
        ti, tp, tx = D.transpose_host()
    assert np.array_equal(tp, wp) and np.array_equal(ti, wi) and np.array_equal(bits(tx), bits(wx))


def test_transpose_five_million_rows(checker, monkeypatch):
    """Beyond 2^22 rows the two-split transpose runs with 2048 rows a band and more bands than rows per band (2442 here):
    the widest key tables it supports.  (Forced: the library keeps matrices this small on the banded kernel.)"""
    monkeypatch.setenv("SB200_TRANSPOSE_PATH", "split")
    spec = synth.uniform_spec(5_000_000, 48, 0.003, 81)
    i, p, x = synth.generate_host(spec)
    wi, wp, wx = checker.transpose(i, p, x, spec.nrow, spec.ncol)
    with DeviceMatrix.from_host(i, p, x, spec.nrow, spec.ncol) as D:
        ti, tp, tx = D.transpose_host()
        assert D.layouts() & 8
    assert np.array_equal(tp, wp) and np.array_equal(ti, wi) and np.array_equal(bits(tx), bits(wx))


def test_transpose_fuzz_every_path(monkeypatch):
    """tools/transpose_fuzz.py: random shapes (1 .. 4e6 rows, 1 .. 5e4 columns, uniform and power-law, empty columns,
    row popularity levels) through the two-split path (library's and a random band width), the chunk sort, the banded
    kernel and the library's own choice, twice each (second call on the cached plan), bit for bit against the oracle."""
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "transpose_fuzz.py"), "16", "5"], capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0 and "bit-exact" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("path", ["place", "split", "banded"])
def test_transpose_into_an_existing_result(path, monkeypatch, checker):
    """sb200_transpose_into: the transpose again into a result of the same structure (new values), nothing allocated; the
    target's cached layouts go, its tile plans stay valid (sums on it are checked); wrong shapes are refused."""
    monkeypatch.setenv("SB200_TRANSPOSE_PATH", path)
    spec = synth.powerlaw_spec(20_000, 3_000, 40.0, 55, row_levels=3)
    i, p, x = synth.generate_host(spec)
    x2 = np.random.default_rng(3).standard_normal(len(x))
    with DeviceMatrix.from_host(i, p, x, spec.nrow, spec.ncol) as D, D.transpose_dev() as T:
        T.row_companion(1)
        D.refresh_values(x2)
        n0 = _lib.lib().sb200_launch_count()
        D.transpose_into(T)
        assert _lib.lib().sb200_launch_count() - n0 <= 2 and not (T.layouts() & 1)
        ti, tp, tx = T.download_columns()
        wi, wp, wx = checker.transpose(i, p, x2, spec.nrow, spec.ncol)
        assert np.array_equal(tp, wp) and np.array_equal(ti, wi) and np.array_equal(bits(tx), bits(wx))
        args = (wi, wp, wx, spec.ncol, spec.nrow)
        oracle.assert_within("colSums", T.col_sums(), checker.colSums(*args), *args, tol=TOL)
        oracle.assert_within("rowSums", T.row_sums(), checker.rowSums(*args), *args, tol=TOL)
        with pytest.raises(SparseB200Error):
            D.transpose_into(D)
        with DeviceMatrix.from_host(i[:p[5]], p[:6], x[:p[5]], spec.nrow, 5) as other, pytest.raises(SparseB200Error):
            other.transpose_into(T)


def test_transpose_golden_edges_on_both_paths(golden, monkeypatch):
    g = golden
    for path in ("place", "banded", "split"):
        monkeypatch.setenv("SB200_TRANSPOSE_PATH", path)
        with DeviceMatrix.from_host(g["i"], g["p"], g["x"], g["nrow"], g["ncol"]) as D:
            ti, tp, tx = D.transpose_host()
        assert np.array_equal(tp, g["t_p"]) and np.array_equal(ti, g["t_i"]) and np.array_equal(bits(tx), bits(g["t_x"])), path


def _columns_of_lengths(lengths, nrow, seed):
    rng = np.random.default_rng(seed)
    p = np.zeros(len(lengths) + 1, np.int64)
    p[1:] = np.cumsum(lengths)
    i = np.empty(int(p[-1]), np.int32)
    for c, n in enumerate(lengths):
        if n:
            start = int(rng.integers(0, nrow - n + 1))
            gaps = np.sort(rng.choice(nrow - start, n, replace=False)) if n < (nrow - start) // 2 else np.arange(n)
            i[p[c]:p[c + 1]] = start + gaps
    x = rng.standard_normal(int(p[-1])) * np.exp(rng.uniform(-3, 3, int(p[-1])))
    return i, p.astype(np.int32), x


# column-length regimes of the sweep kernel (sweep.cu): tiles of 2816 (sums) / 1792 (A^T v) items take the
# per-thread walk with 0-1 column ends, a warp per column with 2-7, 8 lanes per column with 8-512, the walk again
# beyond; every boundary, constant and mixed, including empty columns between long ones
LENGTH_REGIMES = {
    "const_0_1_2": [0] * 700 + [1] * 3000 + [2] * 3000,
    "const_3": [3] * 9000, "const_4": [4] * 7000, "const_5": [5] * 6000, "const_6": [6] * 5000,
    "const_10": [10] * 4000, "const_44": [44] * 900, "const_100": [100] * 500,
    "const_223_224_225": [223] * 90 + [224] * 90 + [225] * 90,
    "const_351_352_353": [351] * 60 + [352] * 60 + [353] * 60,
    "const_402_403": [402] * 60 + [403] * 60,
    "const_938_939_940": [938] * 30 + [939] * 30 + [940] * 30,
    "const_1407_1408": [1407] * 25 + [1408] * 25,
    "const_2815_2816_2817": [2815] * 12 + [2816] * 12 + [2817] * 12,
    "long_then_dust": [5600] * 3 + [1] * 4000 + [5600] * 2 + [0] * 3000 + [7] * 2000 + [5000],
    "sawtooth": [n for k in range(120) for n in (2900, 0, 3, 350, 9, 1, 1500, 0, 0, 60)],
}


@pytest.mark.parametrize("regime", sorted(LENGTH_REGIMES))
def test_sweep_column_length_regimes(regime, checker):
    lengths = LENGTH_REGIMES[regime]
    nrow = 6000
    i, p, x = _columns_of_lengths(lengths, nrow, zlib_seed(regime))
    ncol = len(lengths)
    args = (i, p, x, nrow, ncol)
    v_row = synth.dense_vector(5, nrow)
    with DeviceMatrix.from_host(*args) as D:
        oracle.assert_within("colSums", D.col_sums(), checker.colSums(*args), *args, tol=TOL)
        oracle.assert_within("colMeans", D.col_means(), checker.colMeans(*args), *args, tol=TOL)
        oracle.assert_within("spmv_t", D.spmv_t(v_row), checker.spmv_t(*args, v_row), *args, v=v_row, tol=TOL)
        a, b = D.col_sums(), D.col_sums()
        assert np.array_equal(bits(a), bits(b)), "column sums must be bit-stable run to run"
        D.row_companion(1)  # the row-ordered copy is swept by the same kernel, with its own length regime
        oracle.assert_within("rowSums", D.row_sums(), checker.rowSums(*args), *args, tol=TOL)
        oracle.assert_within("rowMeans", D.row_means(), checker.rowMeans(*args), *args, tol=TOL)


@pytest.mark.parametrize("case", ["C1_full", "C2_scaled", "C3_scaled", "C4_scaled", "many_tiny_columns", "few_huge_columns"])
def test_banded_gather_opt_in_parity(case, checker, monkeypatch):
    """A^T v with v's band slice in shared memory (bands.cu, band_gather_kernel; opt-in, SB200_GATHER_PLAN=1):
    lane groups of 2 / 8 / 32 per column and the whole-warp path for outlier runs, against the reference."""
    monkeypatch.setenv("SB200_GATHER_PLAN", "1")
    spec = SYNTH_CASES[case]()
    i, p, x = synth.generate_host(spec)
    args = (i, p, x, spec.nrow, spec.ncol)
    v_row = synth.dense_vector(spec.seed + 7, spec.nrow)
    with DeviceMatrix.from_host(*args) as D:
        for _ in range(2):
            oracle.assert_within("spmv_t", D.spmv_t(v_row), checker.spmv_t(*args, v_row), *args, v=v_row, tol=TOL)


@pytest.mark.parametrize("row_plan", ["0", "1"])
@pytest.mark.parametrize("case", ["C2_scaled", "C3_scaled", "many_tiny_columns"])
def test_row_indexed_ops_on_both_paths(row_plan, case, monkeypatch, checker):
    """rowSums / rowMeans / A v have a plan-free L2-atomic kernel and a banded shared-memory kernel;
    the library picks by shape.  Both must meet the parity bar on every shape."""
    monkeypatch.setenv("SB200_ROW_PLAN", row_plan)
    spec = SYNTH_CASES[case]()
    i, p, x = synth.generate_host(spec)
    nrow, ncol = spec.nrow, spec.ncol
    args = (i, p, x, nrow, ncol)
    A = Matrix(x, i, p, np.array([nrow, ncol], np.int32))
    oracle.assert_within("rowSums", A.rowSums(), checker.rowSums(*args), *args, tol=TOL)
    oracle.assert_within("rowMeans", A.rowMeans(), checker.rowMeans(*args), *args, tol=TOL)
    v = synth.dense_vector(spec.seed, ncol)
    oracle.assert_within("spmv", A.spmv(v), checker.spmv(*args, v), *args, v=v, tol=TOL)
    A.release()


@pytest.mark.parametrize("path", ["banded", "place"])
@pytest.mark.parametrize("bands", [1, 2, 7, 64, 300])
def test_transpose_is_independent_of_band_count(bands, path, monkeypatch, checker):
    """The band decomposition is an implementation detail: any band count gives the same bits, with either
    placement kernel (the library picks by shape; SB200_TRANSPOSE_PATH forces one)."""
    spec = synth.powerlaw_spec(6000, 3000, 300.0, 91, row_levels=8)
    i, p, x = synth.generate_host(spec)
    monkeypatch.setenv("SB200_TRANSPOSE_BANDS", str(bands))
    monkeypatch.setenv("SB200_TRANSPOSE_PATH", path)
    T = Matrix(x, i, p, np.array([spec.nrow, spec.ncol], np.int32)).transpose()
    ti, tp, tx = checker.transpose(i, p, x, spec.nrow, spec.ncol)
    assert np.array_equal(T.p, tp) and np.array_equal(T.i, ti) and np.array_equal(bits(T.x), bits(tx))


# ---------------------------------------------------------------------------------------------------
# properties that hold at any size (used again at BASELINE sizes in test_fullsize_gpu.py)
# ---------------------------------------------------------------------------------------------------
def test_transpose_round_trip_and_cross_identities():
    spec = synth.config("C3", 0.01)
    with DeviceMatrix.synth(spec) as D:
        i, p, x = D.download_columns()
        with D.transpose_dev() as T, T.transpose_dev() as TT:
            i2, p2, x2 = TT.download_columns()
            assert np.array_equal(p2, p) and np.array_equal(i2, i) and np.array_equal(bits(x2), bits(x))
            # rowSums(A) == colSums(A^T) and A v == (A^T)^T v, within tolerance
            feed_r = np.bincount(i, weights=np.abs(x), minlength=spec.nrow)
            assert np.all(np.abs(D.row_sums() - T.col_sums()) <= 2 * TOL * feed_r)
            v = synth.dense_vector(5, spec.ncol)
            col_of = np.repeat(np.arange(spec.ncol), np.diff(p))
            feed_v = np.bincount(i, weights=np.abs(x * v[col_of]), minlength=spec.nrow)
            assert np.all(np.abs(D.spmv(v) - T.spmv_t(v)) <= 2 * TOL * feed_v)


def test_colsums_bit_stable_run_to_run():
    """The column sweep uses no atomics: identical bits on every run (also a cheap race detector)."""
    spec = synth.config("C4", 0.002)
    with DeviceMatrix.synth(spec) as D:
        first = D.col_sums()
        v = synth.dense_vector(3, spec.nrow)
        first_t = D.spmv_t(v)
        for _ in range(5):
            assert np.array_equal(bits(D.col_sums()), bits(first))
            assert np.array_equal(bits(D.spmv_t(v)), bits(first_t))


def test_spmv_linearity():
    spec = synth.config("C2", 0.02)
    with DeviceMatrix.synth(spec) as D:
        i, p, x = D.download_columns()
        a, b = synth.dense_vector(11, spec.ncol), synth.dense_vector(12, spec.ncol)
        col_of = np.repeat(np.arange(spec.ncol), np.diff(p))
        feed = np.bincount(i, weights=np.abs(x) * (np.abs(2 * a[col_of]) + np.abs(3 * b[col_of])), minlength=spec.nrow)
        lhs = D.spmv(2 * a - 3 * b)
        rhs = 2 * D.spmv(a) - 3 * D.spmv(b)
        assert np.all(np.abs(lhs - rhs) <= 4 * TOL * feed + 1e-300)


# ---------------------------------------------------------------------------------------------------
# reference semantics around the sweeps
# ---------------------------------------------------------------------------------------------------
def test_view_aliases_host_memory_and_refresh():
    """Reference vignettes/Documentation.Rmd:325-347: the Matrix is a view; in-place edits are seen."""
    x = np.array([1.0, 2.0, 3.0])
    A = Matrix(x, np.array([0, 1, 0], np.int32), np.array([0, 2, 3], np.int32), np.array([2, 2], np.int32))
    assert A.x is x
    assert A.colSums().tolist() == [3.0, 3.0]
    x[0] = 999.0
    A.refresh()
    assert A.colSums().tolist() == [1001.0, 3.0]
    B = A.clone()
    B.x[0] = -1.0
    assert A.x[0] == 999.0  # clone() is a deep copy (RcppSparse.h:54-60)


def test_reads_are_live_by_default_and_resident_mirrors_need_refresh():
    """The reference's methods loop over the R vectors on every call (RcppSparse.h:131-156): an in-place edit is seen by the
    next call with no refresh.  resident() keeps the device mirror (and the layouts cached on it): then refresh() is
    what makes an edit visible, and re-pointing a member rebuilds the mirror."""
    x = np.array([1.0, 2.0, 3.0])
    i, p, dim = np.array([0, 1, 0], np.int32), np.array([0, 2, 3], np.int32), np.array([2, 2], np.int32)
    A = Matrix(x, i, p, dim)
    assert A.colSums().tolist() == [3.0, 3.0]
    x[0] = 11.0
    assert A.colSums().tolist() == [13.0, 3.0]       # live read
    assert A._dev is None                            # nothing outlives the call
    A.resident()
    assert A.colSums().tolist() == [13.0, 3.0]
    x[0] = 21.0
    assert A.colSums().tolist() == [13.0, 3.0]       # the mirror still holds the old value
    A.refresh()
    assert A.colSums().tolist() == [23.0, 3.0]
    A.x = np.array([1.0, 1.0, 1.0])                  # re-pointed member: new upload
    assert A.colSums().tolist() == [2.0, 1.0]
    for _ in range(10):                              # resident: the row sums move to the row-ordered copy after 8 calls
        assert A.rowSums().tolist() == [2.0, 1.0]
    assert A._mirror().row_path() == "row-companion"
    A.release()


def test_from_s4_and_exported_function_accept_scipy_csc():
    import scipy.sparse as sp

    a = sp.random(300, 200, density=0.05, format="csc", random_state=3, dtype=np.float64)
    a.sort_indices()
    got = columnSums(a)
    want = np.asarray(a.sum(axis=0)).ravel()
    assert np.allclose(got, want, rtol=0, atol=1e-12 * np.abs(a).sum(axis=0).max())

    class NotS4:
        x = 1

    with pytest.raises(ValueError, match="Cannot construct RcppSparse::Matrix"):
        Matrix.from_S4(NotS4())


@pytest.mark.parametrize("what", ["row_out_of_range", "negative_row", "p0", "p_last", "p_decreasing", "unsorted_rows",
                                  "duplicate_rows"])
def test_corrupt_structure_is_an_error_not_ub(what):
    """Reference: Rcpp::index_out_of_bounds from the checked sums(i[j]) (RcppSparse.h:142).  Here: SB200_E_STRUCTURE."""
    i = np.array([0, 2, 1, 3], np.int32)
    p = np.array([0, 2, 4], np.int32)
    x = np.ones(4)
    if what == "row_out_of_range":
        i[1] = 4
    elif what == "negative_row":
        i[0] = -1
    elif what == "p0":
        p[0] = 1
    elif what == "p_last":
        p[2] = 3
    elif what == "p_decreasing":
        p[1] = 5
    elif what == "unsorted_rows":
        i[:2] = [2, 0]
    elif what == "duplicate_rows":
        i[:2] = [2, 2]
    with pytest.raises(SparseB200Error) as ei:
        Matrix(x, i, p, np.array([4, 2], np.int32)).rowSums()
    assert ei.value.code == _lib.E_STRUCTURE


def test_pinned_upload_path_and_row_path_report():
    """SB200_PIN_HOST (cudaHostRegister on caller-owned pages, what the C++ header uses for R memory)
    gives the same results; the library reports which row-indexed kernel it picked."""
    spec = synth.config("C2", 0.01)
    i, p, x = synth.generate_host(spec)
    args = (i, p, x, spec.nrow, spec.ncol)
    chk = oracle.best()
    with DeviceMatrix.from_host(i, p, x, spec.nrow, spec.ncol, pin=True) as D:
        oracle.assert_within("colSums", D.col_sums(), chk.colSums(*args), *args, tol=TOL)
        oracle.assert_within("rowSums", D.row_sums(), chk.rowSums(*args), *args, tol=TOL)
        assert D.row_path() in ("banded", "l2-atomics")
    small = synth.powerlaw_spec(3000, 500, 50.0, 5)
    si, sp_, sx = synth.generate_host(small)
    with DeviceMatrix.from_host(si, sp_, sx, small.nrow, small.ncol) as D:
        assert D.row_path() == "banded"  # few rows: popular rows would serialise the L2 atomics


@pytest.mark.parametrize("name", ["C1", "pl_rows5", "C2s"])
def test_row_companion_parity_and_lifecycle(name):
    """rowSums / rowMeans from the row-ordered copy of a resident mirror (sparse_b200.h,
    sb200_matrix_row_companion) against the reference, and the copy's lifecycle: built on request or after
    SB200_ROW_COMPANION_AFTER (default 8) row-sum calls, dropped by refresh_values, never built on its own
    for adopted device arrays."""
    spec = {"C1": synth.config("C1"), "pl_rows5": synth.powerlaw_spec(7000, 2000, 80.0, 9, row_levels=5),
            "C2s": synth.config("C2", 0.02)}[name]
    i, p, x = synth.generate_host(spec)
    args = (i, p, x, spec.nrow, spec.ncol)
    chk = oracle.best()
    with DeviceMatrix.from_host(i, p, x, spec.nrow, spec.ncol) as D:
        before = D.row_path()
        assert before in ("banded", "l2-atomics")
        D.row_companion(1)
        assert D.row_path() == "row-companion"
        oracle.assert_within("rowSums", D.row_sums(), chk.rowSums(*args), *args, tol=TOL)
        oracle.assert_within("rowMeans", D.row_means(), chk.rowMeans(*args), *args, tol=TOL)
        v = synth.dense_vector(3, spec.ncol)
        oracle.assert_within("spmv", D.spmv(v), chk.spmv(*args, v), *args, v=v, tol=TOL)  # A v = the gather sweep of the copy
        x2 = x * -0.5 + 1.0
        D.refresh_values(x2)
        assert D.row_path() == before
        args2 = (i, p, x2, spec.nrow, spec.ncol)
        for _ in range(8):
            oracle.assert_within("rowSums", D.row_sums(), chk.rowSums(*args2), *args2, tol=TOL)
        assert D.row_path() == before
        oracle.assert_within("rowMeans", D.row_means(), chk.rowMeans(*args2), *args2, tol=TOL)  # ninth call builds
        assert D.row_path() == "row-companion"
        oracle.assert_within("rowSums", D.row_sums(), chk.rowSums(*args2), *args2, tol=TOL)
        D.row_companion(-1)
        assert D.row_path() == before
        for _ in range(10):
            D.row_sums()
        assert D.row_path() == before
        oracle.assert_within("rowSums", D.row_sums(), chk.rowSums(*args2), *args2, tol=TOL)
    import torch

    di, dp, dx = (torch.from_numpy(a).cuda() for a in (i, p, x))
    with DeviceMatrix.adopt(di, dp, dx, spec.nrow, spec.ncol) as A:
        out = torch.empty(spec.nrow, dtype=torch.float64, device="cuda")
        for _ in range(12):
            A.row_sums_dev(out)
        assert A.row_path() != "row-companion"  # the caller may rewrite dx behind the mirror
        dx.mul_(2.0)
        A.row_sums_dev(out)
        torch.cuda.synchronize()
        oracle.assert_within("rowSums", out.cpu().numpy(), 2.0 * chk.rowSums(*args), i, p, 2.0 * x, spec.nrow, spec.ncol, tol=TOL)


def test_row_companion_golden_edges(golden):
    """The row-ordered copy on the golden fixtures (empty rows/columns, NaN/Inf, 0-dimension shapes)."""
    g = golden
    args = (g["i"], g["p"], g["x"], g["nrow"], g["ncol"])
    with DeviceMatrix.from_host(*args) as D:
        D.row_companion(1)  # a no-op for shapes without entries or rows
        if len(g["x"]) and g["nrow"]:
            assert D.row_path() == "row-companion"
        for _ in range(2):
            oracle.assert_within("rowSums", D.row_sums(), g["rowSums"], *args, tol=TOL)
            oracle.assert_within("rowMeans", D.row_means(), g["rowMeans"], *args, tol=TOL)


# ---------------------------------------------------------------------------------------------------
# band-major companion: A^T v / A v with the operand's band slice in shared memory (bmc.cu)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("band_rows", ["default", "4096", "256", "16"])
@pytest.mark.parametrize("case", sorted(SYNTH_CASES))
def test_band_companion_products_on_synthetic_shapes(case, band_rows, monkeypatch, checker):
    """Both products from the band-major layouts against the reference's iterator sweeps, for the default band height
    (12288 rows) and for small ones (many bands per matrix: band switches inside a CTA, runs cut by tile
    boundaries, empty runs, runs longer than a lane group's reach; where the band-pointer pass takes fewer bands than
    a height gives, the lowest height it allows)."""
    spec = SYNTH_CASES[case]()
    if band_rows != "default":
        rows = int(band_rows)
        while spec.nrow // rows > 20000:  # at most 20000 bands; heights are multiples of 16
            rows += 16
        monkeypatch.setenv("SB200_BMC_ROWS", str(rows))
    i, p, x = synth.generate_host(spec)
    args = (i, p, x, spec.nrow, spec.ncol)
    v_row = synth.dense_vector(spec.seed + 7, spec.nrow)
    v_col = synth.dense_vector(spec.seed + 3, spec.ncol)
    want_t, want = checker.spmv_t(*args, v_row), checker.spmv(*args, v_col)
    with DeviceMatrix.from_host(*args) as D:
        D.band_companion(0, 1)
        assert D.layouts() & 2
        for _ in range(2):
            oracle.assert_within("spmv_t", D.spmv_t(v_row), want_t, *args, v=v_row, tol=TOL)
        D.band_companion(1, 1)
        assert D.layouts() & 5 == 5 and D.row_path() == "row-companion"
        for _ in range(2):
            oracle.assert_within("spmv", D.spmv(v_col), want, *args, v=v_col, tol=TOL)
        oracle.assert_within("rowSums", D.row_sums(), checker.rowSums(*args), *args, tol=TOL)


@pytest.mark.parametrize("block", ["4", "8"])
@pytest.mark.parametrize("regime", ["const_0_1_2", "const_3", "const_10", "const_100", "const_938_939_940", "long_then_dust", "sawtooth"])
def test_band_companion_block_sizes_and_run_lengths(regime, block, monkeypatch, checker):
    """Both block sizes of the band-major layout (entries a thread sums per block; runs are padded to whole blocks with
    entries that point at a dummy 0.0 slot) on every run-length regime, with 1 band and with 24 bands of 256 rows; an
    operand full of NaN / Inf outside the touched rows must not leak through the padding."""
    lengths = LENGTH_REGIMES[regime]
    nrow = 6000
    i, p, x = _columns_of_lengths(lengths, nrow, zlib_seed(regime) + 5)
    args = (i, p, x, nrow, len(lengths))
    v_row = synth.dense_vector(11, nrow)
    want = checker.spmv_t(*args, v_row)
    monkeypatch.setenv("SB200_BS_BLOCK", block)
    for rows in (None, "256"):
        if rows:
            monkeypatch.setenv("SB200_BMC_ROWS", rows)
        with DeviceMatrix.from_host(*args) as D:
            D.band_companion(0, 1)
            oracle.assert_within("spmv_t", D.spmv_t(v_row), want, *args, v=v_row, tol=TOL)
            # rows no entry touches may hold anything: padding entries never read them (they read the dummy slot)
            v_bad = v_row.copy()
            untouched = np.setdiff1d(np.arange(nrow), i)
            v_bad[untouched[::2]] = np.nan
            v_bad[untouched[1::2]] = np.inf
            v_bad[0] = v_row[0] if 0 in i else np.nan
            oracle.assert_within("spmv_t", D.spmv_t(v_bad), checker.spmv_t(*args, v_bad), *args, v=np.where(np.isfinite(v_bad), v_bad, 0.0), tol=TOL)


def test_band_companion_golden_edges(golden, checker):
    """Empty rows / columns, NaN and Inf values, zero-dimension shapes: the companion is a no-op or exact."""
    g = golden
    args = (g["i"], g["p"], g["x"], g["nrow"], g["ncol"])
    with DeviceMatrix.from_host(*args) as D:
        D.band_companion(0, 1)
        D.band_companion(1, 1)
        for _ in range(2):
            oracle.assert_within("spmv", D.spmv(g["v_col"]), g["spmv"], *args, v=g["v_col"], tol=TOL)
            oracle.assert_within("spmv_t", D.spmv_t(g["v_row"]), g["spmv_t"], *args, v=g["v_row"], tol=TOL)


def test_band_companion_lifecycle(checker):
    """Built on its own after SB200_ROW_COMPANION_AFTER (8) A^T v calls on a mirror that owns its arrays, dropped
    by refresh_values (the values it holds are stale), never built on its own for adopted arrays."""
    spec = synth.config("C2", 0.02)
    i, p, x = synth.generate_host(spec)
    args = (i, p, x, spec.nrow, spec.ncol)
    v = synth.dense_vector(4, spec.nrow)
    with DeviceMatrix.from_host(*args) as D:
        for k in range(8):
            oracle.assert_within("spmv_t", D.spmv_t(v), checker.spmv_t(*args, v), *args, v=v, tol=TOL)
            assert not D.layouts() & 2, k
        oracle.assert_within("spmv_t", D.spmv_t(v), checker.spmv_t(*args, v), *args, v=v, tol=TOL)  # ninth call builds
        assert D.layouts() & 2
        x2 = x * 3.0 - 0.25
        D.refresh_values(x2)
        assert not D.layouts() & 2
        args2 = (i, p, x2, spec.nrow, spec.ncol)
        oracle.assert_within("spmv_t", D.spmv_t(v), checker.spmv_t(*args2, v), *args2, v=v, tol=TOL)
        D.band_companion(0, 1)
        oracle.assert_within("spmv_t", D.spmv_t(v), checker.spmv_t(*args2, v), *args2, v=v, tol=TOL)
        D.band_companion(0, -1)
        for _ in range(10):
            D.spmv_t(v)
        assert not D.layouts() & 2
    import torch

    di, dp, dx = (torch.from_numpy(a).cuda() for a in (i, p, x))
    dv = torch.from_numpy(v).cuda()
    with DeviceMatrix.adopt(di, dp, dx, spec.nrow, spec.ncol) as A:
        out = torch.empty(spec.ncol, dtype=torch.float64, device="cuda")
        for _ in range(12):
            A.spmv_t_dev(dv, out)
        assert not A.layouts() & 2  # the caller may rewrite dx behind the mirror


CROSSPROD_CASES = {
    "C1_cols600": lambda: synth.config("C1", 0.06),                 # 10k rows x 600 columns, 100 per column
    "powerlaw_rows": lambda: synth.powerlaw_spec(3000, 900, 40.0, 21, row_levels=5),  # popular rows: long row lists
    "wide_rows": lambda: synth.uniform_spec(40, 1500, 0.5, 22),     # rows of ~750 entries: longer than one staged piece
    "one_column": lambda: synth.uniform_spec(500, 1, 0.3, 23),
}


@pytest.mark.parametrize("case", sorted(CROSSPROD_CASES))
def test_crossprod_against_the_reference(case, checker):
    """Dense A^T A (reference Matrix::crossprod(), RcppSparse.h:158-194) from the row-ordered copy of the mirror:
    within 1e-12 * sum|a_ri a_rj| of the reference's own merges, and exactly symmetric like its result."""
    spec = CROSSPROD_CASES[case]()
    i, p, x = synth.generate_host(spec)
    args = (i, p, x, spec.nrow, spec.ncol)
    want = checker.crossprod(*args)
    with DeviceMatrix.from_host(*args) as D:
        got = D.crossprod()
        oracle.assert_within("crossprod", got, want, *args, tol=TOL)
        assert np.array_equal(bits(got), bits(got.T))
        assert D.row_path() == "row-companion"  # the copy it was computed from stays with the mirror
    import torch

    di, dp, dx = (torch.from_numpy(a).cuda() for a in (i, p, x))
    with DeviceMatrix.adopt(di, dp, dx, spec.nrow, spec.ncol) as A:  # adopted arrays: a temporary copy per call
        out = torch.empty(spec.ncol * spec.ncol, dtype=torch.float64, device="cuda")
        A.crossprod_dev(out)
        A.sync()
        oracle.assert_within("crossprod", out.cpu().numpy().reshape(spec.ncol, spec.ncol), want, *args, tol=TOL)
        assert A.row_path() != "row-companion"


def test_crossprod_golden_edges(golden, checker):
    g = golden
    args = (g["i"], g["p"], g["x"], g["nrow"], g["ncol"])
    A = as_matrix(g)
    got = A.crossprod()
    assert got.shape == (g["ncol"], g["ncol"])
    if g["ncol"]:
        oracle.assert_within("crossprod", got, checker.crossprod(*args), *args, tol=TOL)
    A.release()


@pytest.mark.parametrize("threads", ["1", "default"])
def test_pageable_arrays_travel_through_the_pinned_chunk_workers(threads, checker):
    """Arrays of 32 MB and more in ordinary (pageable) host memory — what R owns — are staged through pinned chunks by
    worker threads in both directions (hostcopy.cu): upload at create and refresh, download of a transposed result.
    Bitwise round trips; chunk boundaries (8 MB) fall inside the arrays many times."""
    import subprocess
    import sys

    code = (
        "import numpy as np\n"
        "from oracle import oracle\n"
        "from rcppsparse_b200 import DeviceMatrix, synth\n"
        "spec = synth.config('C2', 0.09)\n"  # 9e6 entries: i 36 MB, x 72 MB
        "i, p, x = synth.generate_host(spec)\n"
        "assert i.nbytes >= 32 << 20 and x.nbytes >= 32 << 20\n"
        "chk = oracle.best()\n"
        "args = (i, p, x, spec.nrow, spec.ncol)\n"
        "with DeviceMatrix.from_host(*args) as D:\n"
        "    di, dp, dx = D.download_columns()\n"
        "    assert np.array_equal(di, i) and np.array_equal(dp, p) and np.array_equal(dx.view(np.uint64), x.view(np.uint64))\n"
        "    oracle.assert_within('colSums', D.col_sums(), chk.colSums(*args), *args)\n"
        "    ti, tp, tx = D.transpose_host()\n"
        "    ri, rp, rx = chk.transpose(*args)\n"
        "    assert np.array_equal(tp, rp) and np.array_equal(ti, ri) and np.array_equal(tx.view(np.uint64), rx.view(np.uint64))\n"
        "    x2 = x[::-1].copy()\n"
        "    D.refresh_values(x2)\n"
        "    assert np.array_equal(D.download_columns()[2].view(np.uint64), x2.view(np.uint64))\n"
        "print('ok')\n")
    env = dict(os.environ)
    if threads != "default":
        env["SB200_COPY_THREADS"] = threads  # read once per process: hence the subprocess
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600, env=env,
                       cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout[-1500:] + r.stderr[-3000:]


def test_host_ops_write_into_caller_buffers():
    """The C ABI writes results through the caller's pointer; the Python mirror exposes that as out=."""
    import torch

    spec = synth.config("C1")
    i, p, x = synth.generate_host(spec)
    args = (i, p, x, spec.nrow, spec.ncol)
    chk = oracle.best()
    with DeviceMatrix.from_host(*args) as D:
        buf = np.full(spec.nrow, -1.0)
        assert D.row_sums(out=buf) is buf
        oracle.assert_within("rowSums", buf, chk.rowSums(*args), *args, tol=TOL)
        pinned = torch.empty(spec.ncol, dtype=torch.float64).pin_memory()
        D.col_means(out=pinned)
        oracle.assert_within("colMeans", pinned.numpy(), chk.colMeans(*args), *args, tol=TOL)
        with pytest.raises(ValueError):
            D.col_sums(out=np.empty(spec.ncol + 1))
        with pytest.raises(ValueError):
            D.col_sums(out=np.empty(spec.ncol, np.float32))


def test_two_mirrors_and_interleaved_ops_do_not_interfere():
    a, b = synth.config("C1"), synth.powerlaw_spec(7000, 2000, 80.0, 9, row_levels=5)
    ia, pa, xa = synth.generate_host(a)
    ib, pb, xb = synth.generate_host(b)
    chk = oracle.best()
    A = Matrix(xa, ia, pa, np.array([a.nrow, a.ncol], np.int32))
    B = Matrix(xb, ib, pb, np.array([b.nrow, b.ncol], np.int32))
    for _ in range(3):
        ra, rb = A.rowSums(), B.rowSums()
        ca, cb = A.colSums(), B.colSums()
    oracle.assert_within("rowSums", ra, chk.rowSums(ia, pa, xa, a.nrow, a.ncol), ia, pa, xa, a.nrow, a.ncol, tol=TOL)
    oracle.assert_within("rowSums", rb, chk.rowSums(ib, pb, xb, b.nrow, b.ncol), ib, pb, xb, b.nrow, b.ncol, tol=TOL)
    oracle.assert_within("colSums", ca, chk.colSums(ia, pa, xa, a.nrow, a.ncol), ia, pa, xa, a.nrow, a.ncol, tol=TOL)
    oracle.assert_within("colSums", cb, chk.colSums(ib, pb, xb, b.nrow, b.ncol), ib, pb, xb, b.nrow, b.ncol, tol=TOL)
    A.release(), B.release()


def test_launch_counter_counts_kernels():
    before = _lib.lib().sb200_launch_count()
    A = Matrix(np.array([1.0]), np.array([0], np.int32), np.array([0, 1], np.int32), np.array([1, 1], np.int32))
    A.colSums()
    assert _lib.lib().sb200_launch_count() > before
