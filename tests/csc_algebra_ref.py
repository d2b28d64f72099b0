"""Restatement of SparseArrays' map(+/-, A, B) (_map_zeropres!) and dropzeros! (fkeep!) from their published
semantics, in numpy: the reference the tests compare xsb_add and xsb_dropzeros with.

CSCs are (colptr, rowval, nzval) with index base `base` (1 as in Julia), rows sorted within each column.
"""
import numpy as np


def map_zeropres(op, m, n, A, B, base=1):
    """C = map(op, A, B) for op in {"+", "-"}: column by column over the sorted rows of both, a row in both gives
    op(a, b), a row in A only op(a, 0.0), a row in B only op(0.0, b); the result is stored only if !(x == 0)."""
    def keys(M):
        cp, rv, _ = M
        cols = np.repeat(np.arange(n, dtype=np.int64), np.diff(np.asarray(cp, np.int64)))
        return cols * m + (np.asarray(rv, np.int64) - base)

    ka, kb = keys(A), keys(B)
    k = np.union1d(ka, kb)
    a = np.zeros(len(k))
    b = np.zeros(len(k))
    a[np.searchsorted(k, ka)] = A[2]
    b[np.searchsorted(k, kb)] = B[2]
    with np.errstate(invalid="ignore", over="ignore"):
        x = a + b if op == "+" else a - b
    keep = ~(x == 0)
    k, x = k[keep], x[keep]
    cp = np.concatenate([[0], np.cumsum(np.bincount(k // m, minlength=n))]) + base
    return cp.astype(np.int64), (k % m + base).astype(np.int64), x


def fkeep_nonzero(n, A, base=1):
    """dropzeros!(A) = fkeep!(A, (i, j, x) -> !iszero(x)): drops +-0.0, keeps the order and the other bits."""
    cp, rv, nz = (np.asarray(A[0], np.int64), np.asarray(A[1], np.int64), np.asarray(A[2], np.float64))
    keep = ~(nz == 0)
    cols = np.repeat(np.arange(n, dtype=np.int64), np.diff(cp))
    cp2 = np.concatenate([[0], np.cumsum(np.bincount(cols[keep], minlength=n))]) + base
    return cp2.astype(np.int64), rv[keep], nz[keep]
