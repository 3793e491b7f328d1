"""Host copies large enough to go through the pinned-chunk workers (hostcopy.cu, host_copies).

Copies of 32 MB and more from or to pageable host memory, which is what R owns, are staged through pinned chunks by
worker threads. Smaller or pinned ones are left to the driver on the stream. These cases put a pageable buffer above
that threshold on the paths no other test takes there:
- the owners' ranges of a sharded transpose, with W >= 2 blocks sharing one GPU;
- the operand and result of a one-GPU block product;
- the row indices a lazily created mirror fetches on its first row-indexed call.
Every result is checked bit for bit: the transposes against scipy's CSR form, the products on integer data whose every
sum is exact, the lazy mirror's row sums on integer data against scipy's."""
import numpy as np
import pytest
import scipy.sparse as sp

from rcppsparse_b200 import DeviceMatrix, ShardedHostMatrix, synth

pytestmark = pytest.mark.gpu

STAGED = 32 << 20  # hostcopy.cu: pageable copies from this size on go through the workers


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


@pytest.fixture(scope="module")
def big():
    """1e6 x 30 000 with ~3e7 entries: i is ~120 MB, x ~240 MB, and every owner's range at W = 3 is above 32 MB."""
    spec = synth.uniform_spec(1_000_000, 30_000, 1e-3, 91)
    i, p, x = synth.generate_host(spec)
    assert i.nbytes // 3 >= 1.1 * STAGED
    return i, p, x, spec.nrow, spec.ncol


@pytest.fixture(scope="module")
def big_csr(big):
    i, p, x, nrow, ncol = big
    return sp.csc_matrix((x, i, p), shape=(nrow, ncol)).tocsr()


@pytest.mark.parametrize("W", [1, 2, 3])
def test_sharded_transpose_stages_every_owners_range(big, big_csr, W):
    i, p, x, nrow, ncol = big
    with ShardedHostMatrix(i, p, x, nrow, ncol, W, devices=[0] * W) as S:
        b = S.bounds()
        assert len(b) == W + 1 and b[-1] == ncol
        ti, tp, tx = S.transpose_host()
    assert np.array_equal(tp, big_csr.indptr)
    assert np.array_equal(ti, big_csr.indices)
    assert np.array_equal(bits(tx), bits(big_csr.data))


def test_lazy_rows_fetch_a_large_pageable_index_array(big):
    """Small integer values: every row sum is exact in any order, so the lazy mirror's row path must give scipy's sums."""
    i, p, _, nrow, ncol = big
    x = np.random.default_rng(93).integers(-4, 5, i.shape[0]).astype(np.float64)
    want = np.asarray(sp.csc_matrix((x, i, p), shape=(nrow, ncol)).sum(axis=1)).ravel()
    with DeviceMatrix.from_host(i, p, x, nrow, ncol, lazy_rows=True) as L:
        got = L.row_sums()  # the first reader of `i`
    assert np.array_equal(got, want)


@pytest.mark.parametrize("op", ["A B", "A^T B"])
def test_block_product_stages_a_large_pageable_operand_and_result(op):
    """400 000 x 400 000 with small integer entries, k = 12: B and Y are 38 MB each. Every sum is an integer far below
    2^53, so any order of the additions gives the exact result."""
    n, k = 400_000, 12
    spec = synth.uniform_spec(n, n, 1e-5, 92)
    i, p, _ = synth.generate_host(spec)
    rng = np.random.default_rng(92)
    x = rng.integers(-4, 5, i.shape[0]).astype(np.float64)
    B = np.asfortranarray(rng.integers(-8, 9, (n, k)).astype(np.float64))
    assert B.nbytes >= STAGED
    A = sp.csc_matrix((x, i, p), shape=(n, n))
    with DeviceMatrix.from_host(i, p, x, n, n) as D:
        Y = D.spmm(B) if op == "A B" else D.spmm_t(B)
    want = A @ B if op == "A B" else A.T @ B
    assert Y.nbytes >= STAGED
    assert np.array_equal(Y, want)
