"""The numpy restatement of SparseArrays' spmatmul (tests/spgemm_ref.py) against a literal pure-Python transcription
of spcolmul!, on small random inputs with signed zeros, NaN and infinities.  CPU only."""

import numpy as np
import pytest

from tests import spgemm_ref as ref

SPECIAL = np.array([0.0, -0.0, np.nan, -np.nan, np.inf, -np.inf, 1.0, -1.0, 1e308, 1e-308])


def random_csc(rng, m, n, density, special=0.2):
    mask = rng.random((n, m)) < density
    cols, rows = np.nonzero(mask)
    nz = rng.standard_normal(len(rows))
    sp = rng.random(len(rows)) < special
    nz[sp] = rng.choice(SPECIAL, int(sp.sum()))
    cp = np.concatenate([[0], np.cumsum(np.bincount(cols, minlength=n))]) + 1
    return cp.astype(np.int64), (rows + 1).astype(np.int64), nz


def spcolmul_literal(m, n, A, B):
    """spcolmul! column by column: the first product of a row is assigned, later ones added; rows then sorted."""
    cpa, rva, nza = A
    cpb, rvb, nzb = B
    cp, rv, nz = [1], [], []
    for j in range(n):
        acc = {}
        for p in range(cpb[j] - 1, cpb[j + 1] - 1):
            k = int(rvb[p]) - 1
            b = float(nzb[p])
            for q in range(cpa[k] - 1, cpa[k + 1] - 1):
                i = int(rva[q])
                prod = float(nza[q]) * b
                acc[i] = prod if i not in acc else acc[i] + prod
        for i in sorted(acc):
            rv.append(i)
            nz.append(acc[i])
        cp.append(len(rv) + 1)
    return np.array(cp, np.int64), np.array(rv, np.int64), np.array(nz, np.float64)


def assert_matches(got, want):
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), "pattern differs"
    a, b = np.asarray(got[2]), np.asarray(want[2])
    assert np.array_equal(np.isnan(a), np.isnan(b)), "NaN positions differ"
    ok = ~np.isnan(a)
    assert np.array_equal(a[ok].view(np.uint64), b[ok].view(np.uint64)), "values differ"


@pytest.mark.parametrize("seed", range(12))
@pytest.mark.parametrize("shape", [(9, 7, 11), (1, 5, 6), (6, 1, 5), (20, 3, 20), (3, 20, 3)])
def test_matches_literal_spcolmul(seed, shape):
    m, k, n = shape
    rng = np.random.default_rng([seed, *shape])
    A = random_csc(rng, m, k, rng.choice([0.1, 0.4, 0.9]))
    B = random_csc(rng, k, n, rng.choice([0.1, 0.4, 0.9]))
    assert_matches(ref.spmatmul(m, n, A, B), spcolmul_literal(m, n, A, B))


def test_left_fold_order_and_signed_zero():
    # column 1 of B = [1e16, 1, -1e16] on rows 1..3; A = [1 1 1] (one row): products in k order 1e16, 1, -1e16
    A = (np.array([1, 2, 3, 4]), np.array([1, 1, 1]), np.array([1.0, 1.0, 1.0]))
    B = (np.array([1, 4, 5]), np.array([1, 2, 3, 1]), np.array([1e16, 1.0, -1e16, -0.0]))
    cp, rv, nz = ref.spmatmul(1, 2, A, B)
    assert cp.tolist() == [1, 2, 3] and rv.tolist() == [1, 1]
    assert nz[0] == 0.0  # (1e16 + 1) - 1e16 rounds to 0; any other order gives 1
    assert nz[1] == 0.0 and np.signbit(nz[1])  # one product 1 * -0.0 is assigned, not added to +0.0


def test_explicit_zeros_create_entries_and_base_zero():
    A = (np.array([1, 3, 4]), np.array([1, 2, 2]), np.array([0.0, 2.0, 3.0]))
    B = (np.array([1, 2, 2]), np.array([1]), np.array([0.0]))
    cp, rv, nz = ref.spmatmul(2, 2, A, B)
    assert cp.tolist() == [1, 3, 3] and rv.tolist() == [1, 2] and nz.tolist() == [0.0, 0.0]
    z = ref.spmatmul(2, 2, tuple(np.asarray(x) - 1 for x in A[:2]) + (A[2],),
                     tuple(np.asarray(x) - 1 for x in B[:2]) + (B[2],), base=0)
    assert z[0].tolist() == [0, 2, 2] and z[1].tolist() == [0, 1]


def test_invalid_products_give_the_negative_default_nan():
    A = (np.array([1, 2]), np.array([1]), np.array([0.0]))
    B = (np.array([1, 2]), np.array([1]), np.array([np.inf]))
    nz = ref.spmatmul(1, 1, A, B)[2]
    assert nz.view(np.uint64)[0] == 0xFFF8000000000000
