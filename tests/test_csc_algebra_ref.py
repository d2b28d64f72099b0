"""The restatement of SparseArrays' map(+/-, A, B) (_map_zeropres!) and dropzeros! (fkeep!), pinned against
answers derived by hand.  CPU only."""

import numpy as np

from tests import csc_algebra_ref as alg


def csc(dense):
    """1-based CSC of a dense array, every position whose entry is not None stored (explicit zeros included)."""
    m, n = len(dense), len(dense[0])
    cp, rv, nz = [1], [], []
    for j in range(n):
        for i in range(m):
            if dense[i][j] is not None:
                rv.append(i + 1)
                nz.append(dense[i][j])
        cp.append(len(rv) + 1)
    return np.array(cp, np.int64), np.array(rv, np.int64), np.array(nz, np.float64)


def bits(x):
    return np.asarray(x, np.float64).view(np.uint64)


def test_difference_keeps_one_entry():
    A = csc([[1.0, None], [None, 2.0]])
    B = csc([[1.0, None], [None, None]])
    cp, rv, nz = alg.map_zeropres("-", 2, 2, A, B)
    assert cp.tolist() == [1, 1, 2] and rv.tolist() == [2] and nz.tolist() == [2.0]


def test_sum_interleaves_rows_and_columns():
    A = csc([[1.0, None, None], [None, None, 3.0], [2.0, None, None]])
    B = csc([[None, 5.0, None], [4.0, None, -3.0], [1.0, None, 7.0]])
    cp, rv, nz = alg.map_zeropres("+", 3, 3, A, B)
    # column 1: rows 1, 2, 3 -> 1, 4, 3; column 2: row 1 -> 5; column 3: row 2 cancels, row 3 -> 7
    assert cp.tolist() == [1, 4, 5, 6]
    assert rv.tolist() == [1, 2, 3, 1, 3]
    assert nz.tolist() == [1.0, 4.0, 3.0, 5.0, 7.0]


def test_explicit_zero_plus_absent_is_not_stored():
    A = csc([[0.0, None], [None, None]])
    B = csc([[None, None], [None, None]])
    for op in "+-":
        cp, rv, nz = alg.map_zeropres(op, 2, 2, A, B)
        assert cp.tolist() == [1, 1, 1] and len(rv) == 0 and len(nz) == 0
        cp, rv, nz = alg.map_zeropres(op, 2, 2, B, A)
        assert cp.tolist() == [1, 1, 1] and len(rv) == 0


def test_signed_zero_dropped_nan_and_inf_minus_inf_kept():
    A = csc([[-0.0, np.nan, np.inf], [1.0, None, 2.0]])
    B = csc([[None, 1.0, np.inf], [-1.0, None, None]])
    cp, rv, nz = alg.map_zeropres("-", 2, 3, A, B)
    # (1,1): -0.0 - 0.0 = -0.0 dropped; (2,1): 1 - (-1) = 2; (1,2): NaN; (1,3): Inf - Inf = NaN; (2,3): 2
    assert cp.tolist() == [1, 2, 3, 5] and rv.tolist() == [2, 1, 1, 2]
    assert nz[0] == 2.0 and np.isnan(nz[1]) and np.isnan(nz[2]) and nz[3] == 2.0
    cp, rv, nz = alg.map_zeropres("+", 2, 3, A, B)
    # (1,1): -0.0 + 0.0 = +0.0 dropped; (2,1): 1 + (-1) = 0 dropped; NaN + 1; Inf + Inf = Inf
    assert cp.tolist() == [1, 1, 2, 4] and rv.tolist() == [1, 1, 2]
    assert np.isnan(nz[0]) and nz[1] == np.inf and nz[2] == 2.0


def test_a_minus_a_is_empty():
    A = csc([[1.5, None], [-2.0, 3.0]])
    cp, rv, nz = alg.map_zeropres("-", 2, 2, A, A)
    assert cp.tolist() == [1, 1, 1] and len(nz) == 0


def test_base_zero_matches_base_one():
    A = csc([[1.0, None, 4.0], [None, 2.0, None]])
    B = csc([[None, 3.0, -4.0], [5.0, None, 6.0]])
    one = alg.map_zeropres("+", 2, 3, A, B)
    A0 = (A[0] - 1, A[1] - 1, A[2])
    B0 = (B[0] - 1, B[1] - 1, B[2])
    zero = alg.map_zeropres("+", 2, 3, A0, B0, base=0)
    assert np.array_equal(one[0] - 1, zero[0]) and np.array_equal(one[1] - 1, zero[1])
    assert np.array_equal(bits(one[2]), bits(zero[2]))


def test_fkeep_drops_signed_zeros_only():
    A = csc([[0.0, np.nan, None], [-0.0, 1.0, -2.0], [3.0, None, 0.0]])
    cp, rv, nz = alg.fkeep_nonzero(3, A)
    assert cp.tolist() == [1, 2, 4, 5] and rv.tolist() == [3, 1, 2, 2]
    assert nz[0] == 3.0 and np.isnan(nz[1]) and nz[2] == 1.0 and nz[3] == -2.0


def test_dropzeros_equals_sum_with_empty_matrix():
    rng = np.random.default_rng(5)
    dense = [[(float(rng.choice([0.0, -0.0, 1.5, -2.25])) if rng.random() < 0.6 else None) for _ in range(7)]
             for _ in range(6)]
    A = csc(dense)
    E = csc([[None] * 7 for _ in range(6)])
    d = alg.fkeep_nonzero(7, A)
    s = alg.map_zeropres("+", 6, 7, A, E)
    assert np.array_equal(d[0], s[0]) and np.array_equal(d[1], s[1]) and np.array_equal(bits(d[2]), bits(s[2]))
