"""The exact reference of the order-free (XSB_FAST) value paths, pinned against answers derived by hand: the
per-entry error bound accepts every summation order and rejects a lost or doubled term, fixed-point sums do not
depend on the order, the colliding keys share one slot of the window table, and the creation rules agree with the
CPU oracle.  CPU only."""
import itertools

import numpy as np
import pytest

from tests import fast_sum_ref as fsr


def bits(x):
    return np.ascontiguousarray(x, np.float64).view(np.uint64)


def one_entry(terms, copies=1):
    """Groups of `copies` entries that all have the same terms (one per column of a 1 x copies matrix)."""
    n = copies
    J = np.repeat(np.arange(1, n + 1), len(terms))
    return fsr.group_contributions(1, n, np.ones(len(J), np.int64), J, np.tile(terms, n), fsr.RAW)


def left_fold(terms):
    acc = 0.0
    for x in terms:
        acc = acc + float(x)
    return acc


def test_gamma_and_exact_sum_by_hand():
    u = 2.0 ** -53
    assert fsr.gamma(0) == 5e-324  # rounded up from 0: never understates
    assert fsr.gamma(1) >= u / (1 - u) and fsr.gamma(1) <= u * (1 + 8 * u)
    assert fsr.gamma(3) >= 3 * u / (1 - 3 * u)
    assert fsr.exact_sum([1e16, 1.0, -1e16]) == 1.0
    assert fsr.exact_sum([0.1] * 10) == 1.0  # correctly rounded, while the left fold gives 0.9999999999999999
    assert left_fold([0.1] * 10) != 1.0
    assert fsr.abs_sum([1e16, 1.0, -1e16]) == 2e16  # 2e16 + 1 rounded to nearest (the ulp there is 4)


def test_cancelling_sum_in_every_order_is_within_the_bound():
    terms = [1e16, 1.0, -1e16]
    orders = list(itertools.permutations(terms))
    got = [left_fold(p) for p in orders]
    # the orders that do not add the pair (1e16, -1e16) first lose the 1 (1e16 + 1 rounds to 1e16): still within
    # the bound
    assert got == [0.0, 1.0, 0.0, 0.0, 1.0, 0.0]
    fsr.assert_within_order_free_bound(np.array(got), one_entry(terms, len(orders)))
    # pairwise trees too: (a + b) + c for every pairing
    trees = [(a + b) + c for a, b, c in orders] + [a + (b + c) for a, b, c in orders]
    fsr.assert_within_order_free_bound(np.array(trees), one_entry(terms, len(trees)))


def test_a_dropped_or_doubled_term_is_outside_the_bound():
    terms = [1e16, 1.0, -1e16]
    g = one_entry(terms)
    dropped = [1.0 - 1e16, 1e16 + 1.0]  # 1e16 dropped, -1e16 dropped
    doubled = [(2e16 + 1.0) - 1e16, (1e16 + 1.0) - 2e16]  # 1e16 doubled, -1e16 doubled
    for wrong in dropped + doubled:
        with pytest.raises(AssertionError, match="outside the order-free bound"):
            fsr.assert_within_order_free_bound(np.array([wrong]), g)
    # the bound is gamma(2) * (2e16 + 1) ~ 4.4: dropping or doubling the 1 beside two terms of 1e16 cannot be seen,
    # which is why the GPU tests also use fixed-point streams and small partners
    fsr.assert_within_order_free_bound(np.array([0.0]), g)
    fsr.assert_within_order_free_bound(np.array([2.0]), g)
    # beside small partners the same lost 1 is far outside
    small = one_entry([3.0, 1.0, -3.0])
    fsr.assert_within_order_free_bound(np.array([1.0]), small)
    for wrong in (0.0, 2.0, -2.0, 4.0):
        with pytest.raises(AssertionError, match="outside the order-free bound"):
            fsr.assert_within_order_free_bound(np.array([wrong]), small)


def test_failure_names_the_worst_entry():
    I = np.array([1, 2, 2, 3])
    J = np.array([1, 1, 1, 2])
    V = np.array([5.0, 1.0, 2.0, 7.0])
    g = fsr.group_contributions(3, 2, I, J, V, fsr.RAW)
    assert g.colptr.tolist() == [1, 3, 4] and g.rowval.tolist() == [1, 2, 3]
    with pytest.raises(AssertionError) as e:
        fsr.assert_within_order_free_bound(np.array([5.0, 2.0, 7.5]), g, "case")
    msg = str(e.value)
    assert "2 entries" in msg and "slot 1 = (2, 1)" in msg and "N = 2" in msg and "exact 3.0" in msg


def test_random_permutations_of_a_cancelling_list():
    rng = np.random.default_rng(1)
    base = rng.standard_normal(40)
    big = np.array([1e8, -1e8, 3e-8, -1e8 + 0.5, 1e8 - 0.25])
    pairs = rng.standard_normal(8)
    terms = np.concatenate([base, big, pairs, -pairs])
    nperm = 10 ** 4
    got = np.empty(nperm)
    for p in range(nperm):
        got[p] = left_fold(terms[rng.permutation(len(terms))])
    assert len(np.unique(got)) > 1  # the order does change the bits
    fsr.assert_within_order_free_bound(got, one_entry(terms, nperm))


@pytest.mark.parametrize("e", [0, 960, -1074])
def test_fixed_point_sums_do_not_depend_on_the_order(e):
    rng = np.random.default_rng(e + 2000)
    terms = fsr.fixed_point_values(rng, 3000, e)
    assert np.all(np.abs(terms) <= np.ldexp(2.0 ** 20, e))
    assert np.any(bits(terms) == bits(-0.0)) and np.any(bits(terms) == bits(0.0))
    k = np.ldexp(terms, -e)
    assert np.all(k == np.round(k)) and np.array_equal(np.ldexp(k, e), terms)
    if e == -1074:
        assert np.all(np.abs(terms) < 2.0 ** -1022)  # every term subnormal
    want = fsr.exact_sum(terms)
    for _ in range(200):
        p = terms[rng.permutation(len(terms))]
        assert bits(left_fold(p)) == bits(want)
        # a pairwise tree as well
        while len(p) > 1:
            p = np.concatenate([p[0:len(p) - 1:2] + p[1::2], p[len(p) - 1:] if len(p) % 2 else []])
        assert bits(p[0] + 0.0) == bits(want)
    # the sign of zero: a sum is -0.0 only if every term is, and a fold that starts from +0.0 never gives it
    assert bits(-0.0 + -0.0) == bits(-0.0) and bits(left_fold([-0.0, -0.0])) == bits(0.0)


def test_colliding_keys_share_one_slot():
    for m, n in ((4096, 4096), (1000, 3000)):
        keys = fsr.colliding_keys(m, n, 512)
        rb = fsr.ceil_log2(m)
        assert keys.shape == (512, 2)
        assert len({(int(i), int(j)) for i, j in keys}) == 512
        assert np.all((keys[:, 0] >= 0) & (keys[:, 0] < m) & (keys[:, 1] >= 0) & (keys[:, 1] < n))
        slots = {fsr.pa_hash((int(j) << rb) | int(i)) for i, j in keys}
        assert slots == {fsr.pa_hash(0)}
    # the hash restated from the kernel: two words mixed, top 9 bits of a multiplicative hash
    assert fsr.pa_hash(1) == (0x9E3779B1 >> 23)
    assert fsr.pa_hash(1 << 32) == ((0x85EBCA6B * 0x9E3779B1) & 0xFFFFFFFF) >> 23
    assert all(0 <= fsr.pa_hash(x) < 512 for x in range(0, 1 << 20, 997))


def assert_same_as_oracle(oracle, m, n, calls, resident=None):
    """calls = [(I, J, V, flavour), ...] applied in order; the reference's pattern and left fold equal the oracle's."""
    A = oracle.OracleExt(m, n)
    if resident is not None:
        A.set_csc(*resident)
    for I, J, V, fl in calls:
        A.insert_batch(np.asarray(I), np.asarray(J), np.asarray(V, np.float64), fl)
    ocp, orv, onz = A.csc()
    I = np.concatenate([np.asarray(c[0]) for c in calls])
    J = np.concatenate([np.asarray(c[1]) for c in calls])
    V = np.concatenate([np.asarray(c[2], np.float64) for c in calls])
    F = np.concatenate([np.full(len(c[0]), c[3]) for c in calls])
    g = fsr.group_contributions(m, n, I, J, V, F, resident)
    assert np.array_equal(g.colptr, ocp) and np.array_equal(g.rowval, orv)
    assert np.array_equal(bits(g.left_fold()), bits(onz))
    fsr.assert_within_order_free_bound(onz, g)
    return g


def test_creation_rules_agree_with_the_oracle(oracle):
    U, R = fsr.UPDATE, fsr.RAW
    # updates that only ever see zeros create nothing (+0.0 and -0.0 alike); a raw zero creates
    g = assert_same_as_oracle(oracle, 3, 3, [([1, 1, 2], [1, 1, 1], [0.0, -0.0, 0.0], U), ([3], [3], [0.0], R)])
    assert g.rowval.tolist() == [3] and g.colptr.tolist() == [1, 1, 1, 2]
    # a zero update before the creating call and after it: the entry holds the sum of all of them
    g = assert_same_as_oracle(oracle, 2, 2, [([1], [2], [0.0], U), ([1], [2], [0.0], R), ([1], [2], [-0.0], U)])
    assert g.counts.tolist() == [3]
    g = assert_same_as_oracle(oracle, 2, 2, [([2, 2, 2], [1, 1, 1], [0.0, 5.0, 0.0], U)])
    assert g.rowval.tolist() == [2]
    # contributions that cancel keep the entry, with +0.0
    g = assert_same_as_oracle(oracle, 2, 2, [([1, 1], [1, 1], [1.5, -1.5], U)])
    assert bits(g.left_fold()).tolist() == [bits(0.0)]
    # on top of a resident CSC: its entries stay whatever arrives, zero updates on a resident entry add to it
    res = (np.array([1, 2, 3]), np.array([2, 1]), np.array([4.0, -0.0]))
    g = assert_same_as_oracle(oracle, 2, 2, [([2, 1, 2], [1, 2, 2], [0.0, -0.0, 0.0], U)], res)
    assert g.rowval.tolist() == [2, 1] and g.has_resident.tolist() == [True, True]
    g = assert_same_as_oracle(oracle, 2, 2, [([1, 2], [1, 2], [0.0, 3.0], U)], res)
    assert g.colptr.tolist() == [1, 2, 4] and g.rowval.tolist() == [2, 1, 2]
    assert g.has_resident.tolist() == [True, True, False]


@pytest.mark.parametrize("seed", [0, 1])
def test_random_streams_agree_with_the_oracle(oracle, seed):
    rng = np.random.default_rng(seed)
    m, n, cnt = 37, 23, 4000
    calls = []
    for b in range(4):
        I = rng.integers(1, m + 1, cnt)
        J = rng.integers(1, n + 1, cnt)
        V = rng.standard_normal(cnt)
        V[rng.random(cnt) < 0.3] = 0.0
        V[rng.random(cnt) < 0.1] = -0.0
        calls.append((I, J, V, b % 2))
    assert_same_as_oracle(oracle, m, n, calls)
    A = oracle.OracleExt(m, n)
    A.insert_batch(rng.integers(1, m + 1, 300), rng.integers(1, n + 1, 300), rng.standard_normal(300), fsr.RAW)
    assert_same_as_oracle(oracle, m, n, calls, A.csc())
