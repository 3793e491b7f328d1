"""Every reduction and product path, bit for bit against an exact reference, at the CTA geometries it really runs.

The parity tests hold results to |delta| <= 1e-12 * sum|terms| because the paths sum in different orders.  That bar
cannot see a term of magnitude 1 dropped from (or counted twice in) an output whose terms add up to 2^41 or more, and
their shapes mostly leave one sweep tile per CTA.  Here every value is an integer: x = +-{1..7}, about one entry in 64
scaled by 2^E, and operands +-{1..7} with an occasional +-2^F.  E and F are chosen per matrix and per op so that
sum|terms| <= 2^52 for every output; then every partial sum is an integer below 2^53, FP64 addition is exact in any
order, and every path (tile sweep at any geometry, banded kernels, L2 atomics, row-ordered copy, band-major
companions, the block products, the sharded handle) must equal the exact reference, and so each other, bit for bit.
Means are one correctly rounded division of an exact sum, so they must match bit for bit too.

Each op's data plants a "blind" output: the output with the most terms gets a term of 2^E and a term of magnitude 1,
so its sum|terms| >= 2^41 while it holds a term the tolerance bar cannot see.  The CPU-side tests check these
invariants on every shape, hold the C port of the reference (oracle.Port) to the exact reference, and show, per op,
that oracle.assert_within accepts a result missing that term while the exact comparison refuses it.

Knobs that a mirror reads once (row path, gather path, band plans) are set before a fresh mirror is made; the
layouts the library builds on its own after repeated calls are pinned off (row_companion(-1), band_companion(w, -1))
or built on request, and row_path() / layouts() confirm which path served the call.  SB200_SWEEP_CFG is read on
every call.
"""
from __future__ import annotations

import dataclasses
import functools
import os
import zlib

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import oracle
from rcppsparse_b200 import DeviceMatrix, Matrix, ShardedHostMatrix, _lib, columnSums, synth
from test_parity_gpu import LENGTH_REGIMES, _columns_of_lengths

EXACT_MAX = 2.0**52   # every output's sum|terms| stays at or below this: partial sums are exact integers
BLIND_MIN = 2.0**41   # 1e-12 * 2^41 > 2: the tolerance bar cannot see a missing term of magnitude 1 here
MIN_ITEMS = 2_500_000  # merge items (ncol + nnz) of a repeated length regime: 148 CTAs walk ~6 sweep / ~9 gather tiles each
K_MAX = 65             # right-hand sides of the block products' operand; smaller k use its leading columns
F_OPERAND = 10         # operand entries scaled by 2^F (about one in 64)
SPMM_KS = [2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 64, 65]  # every slab width (2, 4, 8, 16, 32) and both sides of each boundary
SWEEP_CFGS = ["256,2,1", "256,3,1", "256,4,1", "256,2,3", "256,4,8"]  # threads, stages, CTAs per SM; 256,2,3 is the default
CP_CAP = 480           # crossprod.cu: entries of a row staged per warp; longer rows are walked in pieces
GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


# ---------------------------------------------------------------------------------------------------------------------
# structures (i, p, nrow, ncol): the values are replaced below
# ---------------------------------------------------------------------------------------------------------------------
def _golden_names():
    return sorted(f[:-4] for f in os.listdir(GOLDEN_DIR) if f.endswith(".npz"))


def _repeat_columns(i, p, reps):
    """The column list repeated `reps` times side by side."""
    nnz = len(i)
    p2 = np.concatenate([p[:-1].astype(np.int64) + r * nnz for r in range(reps)] + [np.array([reps * nnz])])
    return np.tile(i, reps), p2.astype(np.int32)


def _hot_rows_structure():
    """Power-law column lengths plus 12 popular rows, each in ~70 % of the 1500 columns: rows of ~1050 entries, more
    than two CP_CAP pieces, and a row range small enough that rowSums / A v default to the banded scatter."""
    rng = np.random.default_rng(2101)
    nrow, ncol = 20_000, 1500
    lens = np.minimum((rng.pareto(1.5, ncol) + 1.0) * 20.0, nrow // 2).astype(np.int64)
    hot = rng.choice(nrow, 12, replace=False)
    cols = [np.unique(np.concatenate([rng.choice(nrow, n, replace=False), hot[rng.random(12) < 0.7]])) for n in lens]
    p = np.zeros(ncol + 1, np.int64)
    p[1:] = np.cumsum([len(c) for c in cols])
    return np.concatenate(cols).astype(np.int32), p.astype(np.int32), nrow, ncol


def _synth_structure(spec):
    i, p, _ = synth.generate_host(spec)
    return i, p, spec.nrow, spec.ncol


SYNTH_SHAPES = {
    "few_huge_columns": lambda: _synth_structure(synth.uniform_spec(400_000, 7, 0.9, 78)),  # each column spans ~25 CTAs
    "tiny_columns": lambda: _synth_structure(synth.powerlaw_spec(5000, 300_000, 2.0, 77, empty_permille=400)),
    "powerlaw_hot_rows": _hot_rows_structure,
    "tall_short_columns": lambda: _synth_structure(synth.powerlaw_spec(200_000, 60_000, 20.0, 79)),  # row path: L2
}


@functools.lru_cache(maxsize=None)
def structure(shape: str):
    kind, _, name = shape.partition("/")
    if kind == "golden":
        g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        return g["i"].astype(np.int32), g["p"].astype(np.int32), int(g["dim"][0]), int(g["dim"][1])
    if kind == "regime":
        lengths = LENGTH_REGIMES[name]
        i, p, _ = _columns_of_lengths(lengths, 6000, zlib.crc32(name.encode()))
        reps = -(-MIN_ITEMS // (len(lengths) + len(i)))
        i, p = _repeat_columns(i, p, reps)
        return i, p, 6000, len(p) - 1
    return SYNTH_SHAPES[shape]()


def _golden_specials(shape):
    """Positions and values of the NaN / Inf entries of a golden fixture (kept where they are)."""
    if not shape.startswith("golden/"):
        return None
    x = np.load(os.path.join(GOLDEN_DIR, shape[7:] + ".npz"))["x"]
    pos = np.flatnonzero(~np.isfinite(x))
    return (pos, x[pos]) if len(pos) else None


# ---------------------------------------------------------------------------------------------------------------------
# exact data and the exact reference
# ---------------------------------------------------------------------------------------------------------------------
# one data set per key, each with its own E: "col" serves colSums / colMeans / columnSums and the masked column sums,
# "row" rowSums / rowMeans, the others the op of that name
KEYS = ("col", "row", "spmv_t", "spmv", "spmm_t", "spmm", "crossprod")
VECTOR_OP = {"spmm_t": "spmv_t", "spmm": "spmv"}  # the single-vector op of each column of a block product


@dataclasses.dataclass
class Exact:
    shape: str
    key: str
    specials: bool
    i: np.ndarray
    p: np.ndarray
    nrow: int
    ncol: int
    x: np.ndarray
    v: np.ndarray | None      # operand: (n,) for A v / A^T v, Fortran (n, K_MAX) for the block products
    E: int
    feed: np.ndarray          # sum |terms| of every output (finite terms), computed from the integer magnitudes
    want: dict                # op -> exact result
    blind: tuple | None       # (output index, value of its magnitude-1 term), or None where no output has two terms
    max_terms: int = 0        # terms of the output that has the most
    rows_in: np.ndarray | None = None   # "col": index sets of the masked column sums (negate = 0 / 1)
    rows_out: np.ndarray | None = None

    @property
    def args(self):
        return self.i, self.p, self.x, self.nrow, self.ncol


def _pick_E(small, bigw, scale):
    """Largest E with small + bigw * 2^(scale*E) <= 2^52 for every output (small, bigw: integer-valued float64)."""
    if small.size == 0:
        return 30 // scale
    for E in range(60 // scale, -1, -1):
        if (small + bigw * 2.0 ** (scale * E)).max() <= EXACT_MAX:
            return E
    raise AssertionError("the small terms alone exceed 2^52")


def _sum_by(index, weights, n):
    return np.bincount(index, weights=weights, minlength=n).astype(np.float64)


@functools.lru_cache(maxsize=None)
def exact(shape: str, key: str, specials: bool = False) -> Exact:
    i, p, nrow, ncol = structure(shape)
    nnz = len(i)
    rng = np.random.default_rng(zlib.crc32(f"{shape}|{key}|{specials}".encode()))
    col_of = np.repeat(np.arange(ncol), np.diff(p))
    mag = rng.integers(1, 8, nnz).astype(np.float64)
    sgn = np.where(rng.random(nnz) < 0.5, -1.0, 1.0)
    big = rng.random(nnz) < 1.0 / 64
    if key in ("col", "spmv_t", "spmm_t", "crossprod"):
        out, n_out, opi, n_op = col_of, ncol, i, nrow
    else:
        out, n_out, opi, n_op = i, nrow, col_of, ncol
    K = {"spmv_t": 1, "spmv": 1, "spmm_t": K_MAX, "spmm": K_MAX}.get(key, 0)
    if K:
        vmag = rng.integers(1, 8, (n_op, K)).astype(np.float64)
        vsgn = np.where(rng.random((n_op, K)) < 0.5, -1.0, 1.0)
        vbig = rng.random((n_op, K)) < 1.0 / 64

    # the blind output: the one with the most terms gets a 2^E term and a term of magnitude 1 (operand column 0)
    blind_e = None
    counts = np.bincount(out, minlength=n_out) if nnz else np.zeros(n_out, np.int64)
    if counts.size and counts.max() >= 2:
        o = int(np.argmax(counts))
        idx = np.flatnonzero(out == o)
        e_big, e_one = int(idx[0]), int(idx[-1])
        big[e_big], big[e_one], mag[e_one] = True, False, 1.0
        if K:  # the big term is big in both factors: within a few bits of the largest output wherever E lands
            vbig[opi[e_one], 0], vmag[opi[e_one], 0], vbig[opi[e_big], 0] = False, 1.0, True
        blind_e = (o, e_one)

    F = F_OPERAND if K else 0
    w = vmag * 2.0 ** (F * vbig) if K else None  # |operand|
    if key == "crossprod":  # terms x_ra x_rb; sum_r |x_ra x_rb| <= max(diag) (Cauchy-Schwarz): E from the diagonal
        E = _pick_E(_sum_by(col_of, mag**2 * ~big, ncol), _sum_by(col_of, mag**2 * big, ncol), 2)
    elif K == 0:
        E = _pick_E(_sum_by(out, mag * ~big, n_out), _sum_by(out, mag * big, n_out), 1)
    else:
        S = [sp.csr_matrix((mag * sel, (out, opi)), shape=(n_out, n_op)) for sel in (~big, big)]
        E = _pick_E(np.asarray(S[0] @ w), np.asarray(S[1] @ w), 1)
    x = sgn * mag * 2.0 ** (E * big)
    v = None
    if K:
        v = vsgn * w
        v = v[:, 0].copy() if K == 1 else np.asfortranarray(v)
    ax = np.abs(x)
    if key == "crossprod":
        Aa = sp.csc_matrix((ax, i, p), shape=(nrow, ncol))
        feed = (Aa.T @ Aa).toarray()
    elif K == 0:
        feed = _sum_by(out, ax, n_out)
    elif K == 1:
        feed = _sum_by(out, ax * np.abs(v)[opi], n_out)
    else:  # |A| |V| as a sparse product: integers below 2^53, exact in any order
        feed = np.asarray(sp.csr_matrix((ax, (out, opi)), shape=(n_out, n_op)) @ np.abs(v))
    blind = None
    if blind_e is not None:
        o, e = blind_e
        if key == "crossprod":
            blind = ((o, o), x[e] * x[e])
        elif K == 1:
            blind = (o, x[e] * v[opi[e]])
        elif K:
            blind = ((o, 0), x[e] * v[opi[e], 0])
        else:
            blind = (o, x[e])

    # NaN / Inf at fixed positions: the golden fixtures' own, or a fixed stride through x and the operand
    fixed = {blind_e[1], int(np.flatnonzero(out == blind_e[0])[0])} if blind_e else set()
    gs = _golden_specials(shape)
    if gs is not None:
        x[gs[0]] = gs[1]
    if specials and nnz:
        pos = [k for k in range(7, nnz, max(1, nnz // 24)) if k not in fixed]
        x[pos] = np.resize([np.nan, np.inf, -np.inf], len(pos))
        if K:
            keep = {int(opi[e]) for e in fixed}
            vpos = [r for r in range(3, n_op, max(1, n_op // 6)) if r not in keep]
            vals = np.resize([np.inf, -np.inf, np.nan], len(vpos))
            if K == 1:
                v[vpos] = vals
            else:
                v[vpos, 0], v[vpos, K - 1] = vals, vals[::-1]

    d = Exact(shape, key, specials, i, p, nrow, ncol, x, v, E, feed, {}, blind, int(counts.max(initial=0)))
    with np.errstate(invalid="ignore", divide="ignore"):
        if key == "col":
            s = _sum_by(col_of, x, ncol)
            d.want.update(colSums=s, columnSums=s, colMeans=s / np.float64(nrow))
            rows = np.flatnonzero(rng.random(nrow) < 0.5).astype(np.int32)
            must = {int(i[e]) for e in fixed}
            d.rows_in = np.union1d(rows, np.array(sorted(must), np.int32)).astype(np.int32)
            d.rows_out = np.setdiff1d(rows, np.array(sorted(must), np.int32)).astype(np.int32)
            for name, rows_, neg in (("masked_in", d.rows_in, False), ("masked_out", d.rows_out, True)):
                keep = np.isin(i, rows_) != neg
                d.want[name] = _sum_by(col_of[keep], x[keep], ncol)
        elif key == "row":
            s = _sum_by(i, x, nrow)
            d.want.update(rowSums=s, rowMeans=s / np.float64(ncol))
        elif key == "spmv_t":
            d.want["spmv_t"] = _sum_by(col_of, x * v[i], ncol)
        elif key == "spmv":
            d.want["spmv"] = _sum_by(i, x * v[col_of], nrow)
        elif key in ("spmm_t", "spmm"):
            d.want[key] = np.stack([_sum_by(out, x * v[:, j][opi], n_out) for j in range(K)], axis=1) if n_out else \
                np.zeros((0, K))
        else:  # crossprod: the sparse product, exact in any order under the 2^52 invariant
            A = sp.csc_matrix((x, i, p), shape=(nrow, ncol))
            d.want["crossprod"] = (A.T @ A).toarray() if ncol else np.zeros((0, 0))
    return d


def assert_exact(got, want, what):
    """got == want bit for bit, except that +0 and -0 are equal and NaN equals NaN."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape}, exact reference {want.shape}"
    gn, wn = np.isnan(got), np.isnan(want)
    with np.errstate(invalid="ignore"):
        bad = (gn != wn) | (~gn & ~wn & (got != want))
    if bad.any():
        first = "; ".join(f"[{', '.join(map(str, t))}] {got[tuple(t)]!r} instead of {want[tuple(t)]!r}"
                          for t in np.argwhere(bad)[:4])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} outputs differ from the exact reference, hence from "
                             f"every other path of this op; first: {first}")


# ---------------------------------------------------------------------------------------------------------------------
# shapes under test
# ---------------------------------------------------------------------------------------------------------------------
GOLDEN = ["golden/" + n for n in _golden_names()]
REGIMES = ["regime/" + r for r in sorted(LENGTH_REGIMES)]
SHAPES = GOLDEN + REGIMES + sorted(SYNTH_SHAPES)
SPECIALS = ["tiny_columns", "regime/sawtooth"]  # NaN / +-Inf at fixed positions of x and of the operand
CASES = [(s, False) for s in SHAPES] + [(s, True) for s in SPECIALS]
CASE_IDS = [s + ("+specials" if f else "") for s, f in CASES]
SPMM_SHAPES = GOLDEN + ["regime/" + r for r in ("const_0_1_2", "const_3", "const_938_939_940", "long_then_dust", "sawtooth")] + \
    sorted(SYNTH_SHAPES)
CROSSPROD_SHAPES = GOLDEN + ["few_huge_columns", "powerlaw_hot_rows"]
SHARDED_SHAPES = ["golden/max_column_between_empties_300x11", "golden/specials_12x9", "regime/sawtooth", "powerlaw_hot_rows",
                  "tall_short_columns"]


def _keys_of(shape):
    return [k for k in KEYS if (k not in ("spmm_t", "spmm") or shape in SPMM_SHAPES) and (k != "crossprod" or shape in CROSSPROD_SHAPES)]


# ---------------------------------------------------------------------------------------------------------------------
# CPU side: invariants, the C port against the exact reference, why the tolerance bar is not enough
# ---------------------------------------------------------------------------------------------------------------------
def test_shapes_reach_the_geometry_they_are_meant_for():
    for r in REGIMES:
        i, p, nrow, ncol = structure(r)
        assert ncol + len(i) >= MIN_ITEMS and (len(i) + ncol) // 2816 >= 4 * 148, r  # several sweep tiles per CTA at 148 CTAs
    i, p, nrow, ncol = structure("powerlaw_hot_rows")
    assert np.bincount(i, minlength=nrow).max() > 2 * CP_CAP  # rows of three crossprod pieces
    i, p, nrow, ncol = structure("tall_short_columns")
    lens = np.diff(p)
    assert nrow > 65536 and 4 * int(((lens > 0) & (lens < 3 * 148)).sum()) > int((lens > 0).sum())  # decide_row_path: L2
    i, p, nrow, ncol = structure("tiny_columns")
    assert ncol >= 300_000 and (np.diff(p) == 0).sum() > ncol // 4
    i, p, nrow, ncol = structure("few_huge_columns")
    assert np.diff(p).min() > 20 * 2816


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_generator_invariants(case):
    """Integer values, every output's sum|terms| <= 2^52 (so any summation order is exact), and a planted blind output:
    sum|terms| >= 2^41 with a term of magnitude 1 in it, wherever some output has two terms."""
    shape, specials = case
    for key in _keys_of(shape):
        d = exact(shape, key, specials)
        fin = np.isfinite(d.x)
        assert np.array_equal(d.x[fin], np.round(d.x[fin])) and np.abs(d.x[fin]).min(initial=1) >= 1, (shape, key)
        assert d.feed.max(initial=0) <= EXACT_MAX, (shape, key, d.E)
        if d.v is not None:
            vf = d.v[np.isfinite(d.v)]
            assert np.array_equal(vf, np.round(vf)) and np.abs(vf).min(initial=1) >= 1, (shape, key)
        if d.max_terms >= 2:
            o, term = d.blind
            assert abs(term) == 1.0 and d.feed[o] >= BLIND_MIN, (shape, key, d.E, d.feed[o])
        else:
            assert d.blind is None
        if key == "crossprod" and d.ncol:
            assert d.feed.max() == np.diag(d.feed).max()  # so choosing E on the diagonal bounds every output


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_oracle_port_is_exact(case):
    """The C port of the reference (oracle.Port), independent of the golden vectors: bit for bit on every exact case."""
    shape, specials = case
    port = oracle.Port()
    for key in _keys_of(shape):
        d = exact(shape, key, specials)
        a = d.args
        if key == "col":
            for op in ("colSums", "columnSums", "colMeans"):
                assert_exact(getattr(port, op)(*a), d.want[op], f"Port.{op} on {shape}")
        elif key == "row":
            for op in ("rowSums", "rowMeans"):
                assert_exact(getattr(port, op)(*a), d.want[op], f"Port.{op} on {shape}")
        elif key in ("spmv_t", "spmv"):
            assert_exact(getattr(port, key)(*a, d.v), d.want[key], f"Port.{key} on {shape}")
        elif key in ("spmm_t", "spmm"):
            for j in (0, K_MAX - 1):
                assert_exact(getattr(port, VECTOR_OP[key])(*a, d.v[:, j].copy()), d.want[key][:, j],
                             f"Port.{VECTOR_OP[key]} on column {j} of the block operand, {shape}")
        elif d.ncol:
            assert_exact(port.crossprod(*a), d.want["crossprod"], f"Port.crossprod on {shape}")


BLIND_CASES = [(op, shape) for op in ("colSums", "colMeans", "columnSums", "masked_in", "masked_out", "rowSums", "rowMeans",
                                       "spmv_t", "spmv", "spmm_t", "spmm") for shape in ("powerlaw_hot_rows", "regime/const_938_939_940")]
BLIND_CASES += [("crossprod", "few_huge_columns")]  # the tolerance's crossprod denominator is a dense |A|^T |A|: few columns


@pytest.mark.parametrize("op,shape", BLIND_CASES)
def test_tolerance_bar_is_blind_to_a_dropped_term(op, shape):
    """Remove the magnitude-1 term from the blind output: oracle.assert_within still passes, the exact comparison fails.
    That is the class of bug (a dropped or doubled entry, an off-by-one tile edge) these tests exist to catch."""
    key = {"colSums": "col", "colMeans": "col", "columnSums": "col", "masked_in": "col", "masked_out": "col",
           "rowSums": "row", "rowMeans": "row"}.get(op, op)
    d = exact(shape, key)
    want = d.want[op]
    o, term = d.blind
    got = want.copy()
    if op in ("colMeans", "rowMeans"):
        got[o] = (d.want[op[:3] + "Sums"][o] - term) / (d.nrow if op == "colMeans" else d.ncol)
    else:
        got[o] = want[o] - term
    a = d.args
    if op in VECTOR_OP:
        oracle.assert_within(VECTOR_OP[op], got[:, 0], want[:, 0], *a, v=d.v[:, 0])
    elif op.startswith("masked"):
        kept = np.isin(np.arange(d.nrow), d.rows_in if op == "masked_in" else d.rows_out) != (op == "masked_out")
        oracle.assert_within("spmv_t", got, want, *a, v=kept.astype(np.float64))
    elif op in ("spmv_t", "spmv"):
        oracle.assert_within(op, got, want, *a, v=d.v)
    else:
        oracle.assert_within(op, got, want, *a)
    with pytest.raises(AssertionError, match="differ from the exact reference"):
        assert_exact(got, want, f"{op} with the magnitude-1 term of output {o} dropped")


# ---------------------------------------------------------------------------------------------------------------------
# GPU: every path of every op, each against the exact reference
# ---------------------------------------------------------------------------------------------------------------------
def _mirror(d: Exact) -> DeviceMatrix:
    return DeviceMatrix.from_host(d.i, d.p, d.x, d.nrow, d.ncol)


def _has_rows(d: Exact) -> bool:
    return len(d.x) > 0 and d.nrow > 0 and d.ncol > 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_column_sums_every_sweep_geometry(case, monkeypatch):
    """colSums, colMeans, columnSums and the masked column sums (both negate) on the tile sweep at 2, 3 and 4 stages
    and 1, 3 and 8 CTAs per SM (the ring wraps, mbarrier parities flip, carries pass between walk and segment tiles
    and between CTAs)."""
    shape, specials = case
    d = exact(shape, "col", specials)
    for cfg in SWEEP_CFGS:
        monkeypatch.setenv("SB200_SWEEP_CFG", cfg)
        where = f"[tile sweep {cfg}] on {CASE_IDS[CASES.index(case)]}"
        with _mirror(d) as D:
            assert_exact(D.col_sums(), d.want["colSums"], "colSums " + where)
            assert_exact(D.col_means(), d.want["colMeans"], "colMeans " + where)
            assert_exact(D.col_sums_in_rows(d.rows_in), d.want["masked_in"], "col_sums_in_rows(negate=False) " + where)
            assert_exact(D.col_sums_in_rows(d.rows_out, negate=True), d.want["masked_out"], "col_sums_in_rows(negate=True) " + where)
            assert D.layouts() == 0
        A = Matrix(d.x, d.i, d.p, np.array([d.nrow, d.ncol], np.int32), gpus=1)
        assert_exact(columnSums(A), d.want["columnSums"], "columnSums " + where)


def _smallest_bmc_rows(nrow):
    rows = 16  # the band-major companion takes heights of 16 rows and up, and at most 20000 bands
    while nrow // rows > 20000:
        rows += 16
    return str(rows)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_spmv_t_every_path(case, monkeypatch):
    """A^T v on the tile sweep (every geometry), the banded gather, and the band-major companion at the default band
    height, 256 rows and the lowest height allowed, with both block sizes."""
    shape, specials = case
    d = exact(shape, "spmv_t", specials)
    want, cid = d.want["spmv_t"], CASE_IDS[CASES.index(case)]
    monkeypatch.setenv("SB200_GATHER_PLAN", "0")
    for cfg in SWEEP_CFGS:
        monkeypatch.setenv("SB200_SWEEP_CFG", cfg)
        with _mirror(d) as D:
            D.band_companion(0, -1)
            assert_exact(D.spmv_t(d.v), want, f"A^T v [tile sweep {cfg}] on {cid}")
            assert not D.layouts() & 2
    monkeypatch.delenv("SB200_SWEEP_CFG")
    monkeypatch.setenv("SB200_GATHER_PLAN", "1")
    with _mirror(d) as D:
        D.band_companion(0, -1)
        assert_exact(D.spmv_t(d.v), want, f"A^T v [banded gather] on {cid}")
    monkeypatch.delenv("SB200_GATHER_PLAN")
    for rows in (None, "256", _smallest_bmc_rows(d.nrow)):
        for block in ("4", "8"):
            if rows is None:
                monkeypatch.delenv("SB200_BMC_ROWS", raising=False)
            else:
                monkeypatch.setenv("SB200_BMC_ROWS", rows)
            monkeypatch.setenv("SB200_BS_BLOCK", block)
            with _mirror(d) as D:
                D.band_companion(0, 1)
                assert bool(D.layouts() & 2) == _has_rows(d)
                assert_exact(D.spmv_t(d.v), want, f"A^T v [band-major companion, {rows or 'default'} rows, block {block}] on {cid}")


def _scatter_knobs(monkeypatch, d, splits, cluster):
    """Banded scatter with `splits` column splits and clusters of `cluster` bands.  A cluster size that does not divide
    both the band count and the grid is halved by the library, so shapes of 4736 rows and more are given 148 bands (one
    per SM of a B200, 32 rows or more each): 148 and the grid (148 or 296 CTAs, or 148 * splits) are multiples of 4, and
    the size asked for is the size that runs.  Smaller shapes keep the library's band count, and may run a halved size."""
    monkeypatch.setenv("SB200_ROW_PLAN", "1")
    monkeypatch.setenv("SB200_SCATTER_SPLITS", str(splits))
    monkeypatch.setenv("SB200_SCATTER_CLUSTER", str(cluster))
    if d.nrow >= 148 * 32:
        monkeypatch.setenv("SB200_BANDS", "148")
    else:
        monkeypatch.delenv("SB200_BANDS", raising=False)


def _row_paths(d, monkeypatch, run, label):
    """Runs `run(D, where)` on every row-indexed path: the plan-free kernel, the banded scatter at every split and
    cluster size, and the row-ordered copy (two sweep geometries); checks that the intended path served the calls."""
    cid = d.shape + ("+specials" if d.specials else "")
    monkeypatch.setenv("SB200_ROW_PLAN", "0")
    with _mirror(d) as D:
        D.row_companion(-1)
        run(D, f"[{label}] on {cid}")
        assert D.row_path() == "l2-atomics"
    for splits in (1, 4, 64):
        for cluster in (1, 2, 4):
            _scatter_knobs(monkeypatch, d, splits, cluster)
            with _mirror(d) as D:
                D.row_companion(-1)
                run(D, f"[banded scatter, {splits} splits, cluster {cluster}] on {cid}")
                assert D.row_path() == ("banded" if _has_rows(d) else "l2-atomics")
    for v in ("SB200_ROW_PLAN", "SB200_SCATTER_SPLITS", "SB200_SCATTER_CLUSTER", "SB200_BANDS"):
        monkeypatch.delenv(v, raising=False)
    for cfg in ("256,2,3", "256,4,1"):
        monkeypatch.setenv("SB200_SWEEP_CFG", cfg)
        with _mirror(d) as D:
            D.row_companion(1)
            D.band_companion(1, -1)
            run(D, f"[row-ordered copy, sweep {cfg}] on {cid}")
            assert (D.row_path() == "row-companion") == (len(d.x) > 0 and d.nrow > 0) and not D.layouts() & 4
    monkeypatch.delenv("SB200_SWEEP_CFG")


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_row_sums_every_path(case, monkeypatch):
    """rowSums and rowMeans: L2 stream, banded scatter (1 / 4 / 64 splits, clusters of 1 / 2 / 4), row-ordered copy."""
    d = exact(case[0], "row", case[1])

    def run(D, where):
        assert_exact(D.row_sums(), d.want["rowSums"], "rowSums " + where)
        assert_exact(D.row_means(), d.want["rowMeans"], "rowMeans " + where)

    _row_paths(d, monkeypatch, run, "L2 stream")


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_spmv_every_path(case, monkeypatch):
    """A v: the sweep's scatter mode, the banded scatter (every split and cluster size), the gather sweep of the
    row-ordered copy, and that copy's band-major companion."""
    d = exact(case[0], "spmv", case[1])
    _row_paths(d, monkeypatch, lambda D, where: assert_exact(D.spmv(d.v), d.want["spmv"], "A v " + where), "sweep scatter")
    with _mirror(d) as D:
        D.band_companion(1, 1)
        assert (D.layouts() & 5 == 5) == _has_rows(d)
        assert_exact(D.spmv(d.v), d.want["spmv"], f"A v [band-major companion of the row-ordered copy] on {CASE_IDS[CASES.index(case)]}")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SPMM_SHAPES)
def test_block_products_every_path_and_width(shape):
    """A^T B (gather and fold), A B (scatter on the CSC arrays, and gather on the row-ordered copy), k = 2 .. 65: every
    slab width and both sides of each of its boundaries."""
    dt, d = exact(shape, "spmm_t"), exact(shape, "spmm")
    with _mirror(dt) as T, _mirror(d) as S, _mirror(d) as R:
        S.row_companion(-1)
        R.row_companion(1)
        for k in SPMM_KS:
            assert_exact(T.spmm_t(dt.v[:, :k]), dt.want["spmm_t"][:, :k], f"A^T B [gather and fold, k = {k}] on {shape}")
            assert_exact(S.spmm(d.v[:, :k]), d.want["spmm"][:, :k], f"A B [scatter, k = {k}] on {shape}")
            assert_exact(R.spmm(d.v[:, :k]), d.want["spmm"][:, :k], f"A B [gather on the row-ordered copy, k = {k}] on {shape}")
        assert not S.layouts() & 1
        assert bool(R.layouts() & 1) == (len(d.x) > 0 and d.nrow > 0)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", CROSSPROD_SHAPES)
def test_crossprod_exact(shape):
    """Dense A^T A from the row-ordered copy of a resident mirror and from a temporary copy of adopted arrays (rows
    longer than CP_CAP are walked in pieces)."""
    import torch

    d = exact(shape, "crossprod")
    want = d.want["crossprod"]
    with _mirror(d) as D:
        assert_exact(D.crossprod(), want, f"crossprod [row-ordered copy of a resident mirror] on {shape}")
        assert (D.row_path() == "row-companion") == (len(d.x) > 0 and d.nrow > 0)
    if len(d.x) == 0 or d.ncol == 0:
        return
    di, dp, dx = (torch.from_numpy(a).cuda() for a in (d.i, d.p, d.x))
    with DeviceMatrix.adopt(di, dp, dx, d.nrow, d.ncol) as A:
        out = torch.empty(d.ncol * d.ncol, dtype=torch.float64, device="cuda")
        A.crossprod_dev(out)
        A.sync()
        assert_exact(out.cpu().numpy().reshape(d.ncol, d.ncol), want, f"crossprod [temporary copy of adopted arrays] on {shape}")
        assert A.row_path() != "row-companion"


@pytest.mark.gpu
@pytest.mark.parametrize("n_gpus", [1, 2])
@pytest.mark.parametrize("shape", SHARDED_SHAPES)
def test_sharded_handle_exact(shape, n_gpus):
    """The single-process sharded handle (sb200_sharded_*): every sum and product it offers, ten calls each (the ninth
    moves every block to its cached layouts), against the exact reference."""
    if n_gpus > _lib.device_count():
        pytest.skip(f"needs {n_gpus} GPUs")
    for key, calls in (("col", (("colSums", lambda S, d: S.col_sums()), ("colMeans", lambda S, d: S.col_means()))),
                       ("row", (("rowSums", lambda S, d: S.row_sums()), ("rowMeans", lambda S, d: S.row_means()))),
                       ("spmv", (("spmv", lambda S, d: S.spmv(d.v)),)), ("spmv_t", (("spmv_t", lambda S, d: S.spmv_t(d.v)),))):
        d = exact(shape, key)
        with ShardedHostMatrix(d.i, d.p, d.x, d.nrow, d.ncol, n_gpus) as S:
            for rep in range(10):
                for op, call in calls:
                    assert_exact(call(S, d), d.want[op], f"{op} [sharded handle, {n_gpus} GPUs, call {rep + 1}] on {shape}")
