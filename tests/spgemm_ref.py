"""Restatement of SparseArrays' spmatmul (C = A * B) from its published semantics, in numpy: the reference the tests
compare xsb_matmul with.

spcolmul! walks, for every column j of B, B[:, j]'s entries (k, b) in stored order and, for each, A[:, k]'s entries
(i, a); the first product a * b of row i is assigned and every later one added, acc = acc + p.  So C stores the
structural pattern and each value is the left fold in ascending k of separately rounded products.  Here the products
are expanded in (j, B position, A position) order as array-by-array a * b, stably sorted by (j, i), and every segment
is folded with a depth loop: acc = first product, then acc = acc + next, one depth at a time.

NaN results carry the bits a scalar x86-64 multiply or add gives them (as Julia's do): the first NaN operand,
quieted; an invalid operation on non-NaN operands (0 * Inf, Inf - Inf) gives the negative default NaN.  numpy's own
vector loops do not keep that operand order for two NaN operands, so every result is passed through x86_nan.

CSCs are (colptr, rowval, nzval) with index base `base` (1 as in Julia), rows sorted within each column.
"""
import numpy as np

QUIET = np.uint64(0x0008000000000000)
DEFAULT_NAN = np.uint64(0xFFF8000000000000)


def x86_nan(r, a, b):
    """r = a op b elementwise, its NaN results replaced by x86-64's: quiet(a) if a is NaN, else quiet(b) if b is
    NaN, else the negative default NaN."""
    bad = np.isnan(r)
    if not bad.any():
        return r
    out = r.view(np.uint64).copy()
    a, b = np.broadcast_to(a, r.shape), np.broadcast_to(b, r.shape)
    na, nb = np.isnan(a) & bad, np.isnan(b) & bad & ~np.isnan(a)
    out[bad] = DEFAULT_NAN
    out[nb] = b[nb].view(np.uint64) | QUIET
    out[na] = a[na].view(np.uint64) | QUIET
    return out.view(np.float64)


def expand(m, n, A, B, base=1):
    """(rows, cols, products) of every product in (j, B position, A position) order, 0-based."""
    cpa, rva, nza = (np.asarray(A[0], np.int64) - base, np.asarray(A[1], np.int64) - base, np.asarray(A[2], np.float64))
    cpb, rvb, nzb = (np.asarray(B[0], np.int64) - base, np.asarray(B[1], np.int64) - base, np.asarray(B[2], np.float64))
    lens = cpa[rvb + 1] - cpa[rvb]  # products of every B position
    pidx = np.repeat(np.arange(len(rvb), dtype=np.int64), lens)
    first = np.cumsum(lens) - lens
    q = cpa[rvb][pidx] + (np.arange(len(pidx), dtype=np.int64) - first[pidx])
    cols = np.repeat(np.arange(n, dtype=np.int64), np.diff(cpb))[pidx]
    a = nza[q]
    b = nzb[pidx]
    with np.errstate(invalid="ignore", over="ignore", under="ignore"):
        p = x86_nan(a * b, a, b)
    return rva[q], cols, p


def spmatmul(m, n, A, B, base=1):
    """C = A * B for A m x k and B k x n: (colptr, rowval, nzval) in the same base."""
    rows, cols, p = expand(m, n, A, B, base)
    order = np.lexsort((rows, cols))  # stable: equal (j, i) keep (B position, A position) order
    rows, cols, p = rows[order], cols[order], p[order]
    key = cols * m + rows
    start = np.flatnonzero(np.r_[True, key[1:] != key[:-1]]) if len(key) else np.zeros(0, np.int64)
    seglen = np.diff(np.r_[start, len(key)])
    acc = p[start].copy()
    # longest segments first, so that the segments still open at depth d are a prefix
    byl = np.argsort(-seglen, kind="stable")
    sl, st = seglen[byl], start[byl]
    fold = acc[byl]
    with np.errstate(invalid="ignore", over="ignore"):
        for d in range(1, int(sl[0]) if len(sl) else 0):
            live = int(np.searchsorted(-sl, -d, side="left"))  # segments longer than d
            acc_d, p_d = fold[:live], p[st[:live] + d]
            fold[:live] = x86_nan(acc_d + p_d, acc_d, p_d)
    acc[byl] = fold
    cp = np.concatenate([[0], np.cumsum(np.bincount(cols[start], minlength=n))]) + base
    return cp.astype(np.int64), (rows[start] + base).astype(np.int64), acc
