"""Exact reference for the order-free (XSB_FAST) value paths: per-entry contributions, their correctly rounded sum
and the error bound that holds for every summation order.

XSB_FAST may add the contributions of an entry in any order: window partial sums (xsb_preagg.cu) folded per column,
or one atomic add per position of a frozen stream (xsb_values.cu).  No order can promise a relative error once terms
cancel, but every order -- every binary summation tree -- meets the recursive-summation bound (Higham, Accuracy and
Stability of Numerical Algorithms, 2nd ed., eq. 4.4 / 4.6): for N terms x_1..x_N with exact sum s, the computed sum
s^ satisfies  |s^ - s| <= gamma(N-1) * sum|x_i|,  gamma(k) = k u / (1 - k u),  u = 2^-53.  Additions that underflow are
exact, so subnormals need no extra term.  Against the correctly rounded fsum(x) the bound gains half an ulp of fsum.

When every term is k * 2^e with one common e and N * max|k| < 2^53, every partial sum in any order is exact, so an
order-free path must reproduce the deterministic left fold bit for bit (fixed_point_values).

Indices here are 1-based, as in the oracle and the handles' default base."""
import math
from fractions import Fraction

import numpy as np

U = 2.0 ** -53
UPDATE, RAW, ASSIGN = 0, 1, 2  # flavours of include/xsparse_b200.h (and oracle/oracle.py)


def gamma(k):
    """gamma(k) = k u / (1 - k u) as a float (rounded up by one ulp, so it never understates the exact value)."""
    k = np.asarray(k, np.float64)
    return np.nextafter(k * U / (1.0 - k * U), np.inf)


def exact_sum(terms):
    """Correctly rounded sum of the terms (math.fsum)."""
    return math.fsum(terms)


def abs_sum(terms):
    return math.fsum(abs(float(t)) for t in terms)


class Groups:
    """The reference result of one assembly step: the pattern (1-based colptr / rowval) and, per entry in CSC order,
    its contributions in stream order with the resident value first (has_resident[z])."""

    def __init__(self, colptr, rowval, terms, has_resident):
        self.colptr, self.rowval, self.terms, self.has_resident = colptr, rowval, terms, has_resident

    @property
    def counts(self):
        return np.array([len(t) for t in self.terms], np.int64)

    def exact(self):
        return np.array([exact_sum(t) for t in self.terms], np.float64)

    def left_fold(self):
        """The deterministic result: ((x_1 + x_2) + x_3) + ... from +0.0 (a resident value is x_1)."""
        out = np.empty(len(self.terms), np.float64)
        for z, t in enumerate(self.terms):
            r = bool(self.has_resident[z])
            acc = float(t[0]) if r else 0.0
            for x in t[1:] if r else t:
                acc = acc + float(x)
            out[z] = acc
        return out


def group_contributions(m, n, I, J, V, flavours, resident=None):
    """Groups of the stream (I, J, V) (1-based positions; `flavours` one value or one per call) applied to an m x n
    matrix that holds `resident` = (colptr, rowval, nzval) (1-based CSC) or nothing.

    Creation rules of the reference (sparsematrixlnk.jl:210-253): rawupdateindex! always creates, updateindex!
    creates only with v != 0 (so -0.0 creates nothing either), an entry whose contributions cancel stays.  Every
    contribution of an entry that exists in the end is one of its terms, zeros included: a zero update that came
    before the entry existed adds +0.0 to a sum that starts from +0.0, which changes nothing."""
    I = np.asarray(I, np.int64).ravel()
    J = np.asarray(J, np.int64).ravel()
    V = np.asarray(V, np.float64).ravel()
    F = np.broadcast_to(np.asarray(flavours, np.int64), V.shape)
    assert len(I) == len(J) == len(V)
    if np.any(F == ASSIGN):
        raise ValueError("A[i,j] = v does not commute: not an order-free stream")
    assert np.all((I >= 1) & (I <= m) & (J >= 1) & (J <= n)), "positions out of bounds"
    if resident is not None:
        cp, rv, nz = (np.asarray(a) for a in resident)
        rcol = np.repeat(np.arange(1, n + 1, dtype=np.int64), np.diff(cp).astype(np.int64))
        rrow = np.asarray(rv, np.int64)
        rval = np.asarray(nz, np.float64)
    else:
        rcol = rrow = np.empty(0, np.int64)
        rval = np.empty(0, np.float64)
    nres = len(rval)
    cols = np.concatenate([rcol, J])
    rows = np.concatenate([rrow, I])
    vals = np.concatenate([rval, V])
    creates = np.concatenate([np.ones(nres, bool), (F != UPDATE) | (V != 0.0)])
    # lexsort is stable: resident value first, then the calls in stream order
    order = np.lexsort((rows, cols))
    cs, rs = cols[order], rows[order]
    first = np.ones(len(order), bool)
    first[1:] = (cs[1:] != cs[:-1]) | (rs[1:] != rs[:-1])
    starts = np.flatnonzero(first)
    gid = np.cumsum(first) - 1
    made = np.zeros(len(starts), bool)
    np.logical_or.at(made, gid, creates[order])
    keep = np.flatnonzero(made)
    bounds = np.append(starts, len(order))
    terms = [vals[order[bounds[g]:bounds[g + 1]]] for g in keep]
    kcol, krow = cs[starts[keep]], rs[starts[keep]]
    colptr = np.ones(n + 1, np.int64)
    colptr[1:] += np.cumsum(np.bincount(kcol - 1, minlength=n))
    return Groups(colptr, krow.copy(), terms, order[starts[keep]] < nres)


def _exact_check(got, terms):
    """The bound of one entry in rational arithmetic: (holds, fsum, bound as a float)."""
    fs = exact_sum(terms)
    a = sum((Fraction(abs(float(t))) for t in terms), Fraction(0))
    k = max(len(terms) - 1, 0)
    bound = Fraction(k, 2 ** 53 - k) * a + Fraction(math.ulp(fs)) / 2  # gamma(k) = k u / (1 - k u)
    if math.isnan(got) or math.isinf(got):
        return False, fs, float(bound)
    return abs(Fraction(float(got)) - Fraction(fs)) <= bound, fs, float(bound)


def assert_within_order_free_bound(got, groups, what=""):
    """Every entry z with N terms: |got[z] - fsum| <= gamma(N-1) * sum|x| + ulp(fsum)/2.  A float pre-check finds the
    candidates, an exact rational check decides; the worst offender is reported."""
    got = np.asarray(got, np.float64)
    assert len(got) == len(groups.terms), f"{what}: {len(got)} values for {len(groups.terms)} entries"
    if len(got) == 0:
        return
    ex = groups.exact()
    S = np.array([abs_sum(t) for t in groups.terms], np.float64)
    N = groups.counts
    bound = gamma(np.maximum(N - 1, 0)) * S + 0.5 * np.array([math.ulp(x) for x in ex])
    err = np.abs(got - ex)
    cand = np.flatnonzero(~(err <= bound))  # NaN counts as a failure
    bad = []
    for z in cand:
        ok, fs, b = _exact_check(float(got[z]), groups.terms[z])
        if not ok:
            bad.append((abs(float(got[z]) - fs) / max(b, 5e-324), int(z), fs, b))
    if bad:
        ratio, z, fs, b = max(bad)
        cp = groups.colptr
        col = int(np.searchsorted(cp, z + 1, side="right"))  # 1-based column of CSC slot z
        raise AssertionError(
            f"{what}: {len(bad)} entries outside the order-free bound; worst at slot {z} = "
            f"({int(groups.rowval[z])}, {col}): N = {len(groups.terms[z])}, got {float(got[z])!r}, "
            f"exact {fs!r}, bound {b!r} ({ratio:.3g} x the bound)")


def fixed_point_values(rng, cnt, e, kmax=2 ** 20):
    """cnt values k * 2^e, integer |k| <= kmax, about one in eight an exact +0.0 or -0.0.  While N * kmax < 2^53 every
    partial sum of N such values is exact in any order.  e = 0: integers; e = 960: close to overflow (sums stay
    below 2^1024 while N < 2^43); e = -1074: all subnormal (the partial sums stay below 2^-1021, where every
    multiple of 2^-1074 is a double)."""
    k = rng.integers(-kmax, kmax + 1, cnt).astype(np.float64)
    z = rng.random(cnt) < 0.125
    k[z] = 0.0
    neg = z & (rng.random(cnt) < 0.5)
    k[neg] = -0.0
    return np.ldexp(k, e)


# ---------------------------------------------------------------- the pre-aggregation table (xsb_preagg.cu)
PA_HBITS = 9
PA_H = 1 << PA_HBITS
PA_W = 512


def pa_hash(cr):
    """xsb_preagg.cu pa_hash: slot of the (column, row) key cr = key >> low in the 512-slot window table."""
    cr = int(cr)
    x = ((cr & 0xFFFFFFFF) ^ (((cr >> 32) & 0xFFFFFFFF) * 0x85EBCA6B)) & 0xFFFFFFFF
    return ((x * 0x9E3779B1) & 0xFFFFFFFF) >> (32 - PA_HBITS)


def ceil_log2(x):
    """xsb_api.cu ceil_log2: bits of a row or column field (at least 1)."""
    b = 0
    while (1 << b) < x:
        b += 1
    return max(b, 1)


def colliding_keys(m, n, count, slot=None):
    """`count` distinct 0-based (row, col) pairs of an m x n plain single-partition handle whose window keys
    cr = col << ceil_log2(m) | row all hash to one slot (the slot of (0, 0) unless given).  Inserted into one window
    they fill the table along one probe chain that wraps around it.  Written from the kernel's hash: if that hash
    changes, a test using these keys stays correct but stops being adversarial."""
    rb = ceil_log2(m)
    want = pa_hash(0) if slot is None else slot
    out = []
    for j in range(n):
        for i in range(m):
            if pa_hash((j << rb) | i) == want:
                out.append((i, j))
                if len(out) == count:
                    return np.array(out, np.int64)
    raise ValueError(f"only {len(out)} keys of an {m} x {n} matrix share slot {want}")
