"""Host-side mirror of the reference's matrix interface for the assembly path.

Same names, argument order and error behaviour as ExtendableSparse.jl (the `!` of Julia
mutators is dropped):

    ExtendableSparseMatrix(m, n)                      src/matrix/extendable.jl:10-41
    updateindex(A, op, v, i, j)                       extendable.jl:159-174
    rawupdateindex(A, op, v, i, j[, tid])             extendable.jl:181-197, genericmt...:87-99
    A[i, j] = v ; A[i, j]                             extendable.jl:205-238
    pointblock(A, blocksize)                          extendable.jl:292-318
    A + B ; A - B ; dropzeros(A)                      abstractextendablesparsematrixcsc.jl
    flush(A) ; sparse(A) ; nnz(A) ; reset(A)          extendable.jl:248-272
    MTExtendableSparseMatrix(m, n, nparts)            src/ExtendableSparse.jl:35-39, genericmt...:1-114

Indices are 1-based like the reference's.  Per-entry calls are appended to a host buffer of
16-byte triplets {u32 row, u32 col, f64 val} and shipped to the device in batches through the
C ABI (xsb_insert_triplets; xsb_insert_batch for the bulk (I, J, V) variants); everything else
happens on the GPU.  There is no CPU fallback.
"""
from __future__ import annotations

import operator

import numpy as np

from . import capi

_CHUNK = 1 << 16


class _HostBuffer:
    """Insert calls of one partition, in call order, waiting to be shipped."""

    def __init__(self):
        self.T = np.empty(_CHUNK, capi.TRIPLET_DTYPE)
        self.n = 0
        self.flavour = capi.UPDATE


class ExtendableSparseMatrix:
    """ExtendableSparseMatrixCSC{Float64,Int64} backed by libxsparse_b200 (one partition)."""

    _n_tid = 1

    def __init__(self, m, n=None, *, mode=capi.DETERMINISTIC, device=0):
        if n is None:
            n = m
        self._h = capi.Handle(int(m), int(n), capi.I64, 1, self._n_tid, device)
        self.m, self.n = int(m), int(n)
        self.mode = mode
        self._buf = [_HostBuffer() for _ in range(self._n_tid)]
        self.pattern_changes = 0  # stands in for "phash changed" (extendable.jl:252)

    # -- construction from CSC: extendable.jl:61-67
    @classmethod
    def from_csc(cls, m, n, colptr, rowval, nzval, **kw):
        A = cls(m, n, **kw)
        A._h.set_csc(np.ascontiguousarray(colptr, np.int64), np.ascontiguousarray(rowval, np.int64),
                     np.ascontiguousarray(nzval, np.float64))
        return A

    @property
    def handle(self) -> capi.Handle:
        return self._h

    @property
    def shape(self):
        return (self.m, self.n)

    # -- staging
    def _ship(self, t):
        b = self._buf[t]
        if b.n:
            n = b.n
            b.n = 0  # a rejected batch is dropped, like the failing call in the reference
            self._h.insert_triplets(b.T, b.flavour, t, n)

    def _push(self, flavour, v, i, j, t=0):
        if not (1 <= i <= self.m and 1 <= j <= self.n):
            raise capi.XsbBoundsError(capi.EBOUNDS, f"BoundsError: attempt to access {self.m}x{self.n} matrix at [{i}, {j}]")
        b = self._buf[t]
        if b.n and (b.flavour != flavour or b.n == _CHUNK):
            self._ship(t)
        b.flavour = flavour
        b.T[b.n] = (i, j, v)
        b.n += 1

    @staticmethod
    def _signed(op, v):
        if op is operator.add or op == "+":
            return v
        if op is operator.sub or op == "-":
            return -v
        raise NotImplementedError("the device path implements op in {+,-}; other ops stay on the CPU path")

    def updateindex(self, op, v, i, j):
        self._push(capi.UPDATE, self._signed(op, v), i, j)
        return self

    def rawupdateindex(self, op, v, i, j, part=1):
        self._push(capi.RAW, self._signed(op, v), i, j)
        return self

    def __setitem__(self, ij, v):
        self._push(capi.ASSIGN, v, ij[0], ij[1])

    def __getitem__(self, ij):
        i, j = ij
        if not (1 <= i <= self.m and 1 <= j <= self.n):
            raise capi.XsbBoundsError(capi.EBOUNDS, f"BoundsError at [{i}, {j}]")
        self.flush()
        return float(self._h.get_values(np.array([i], np.int64), np.array([j], np.int64))[0])

    # -- bulk variants of the same calls (k-th element == k-th call)
    def insert_batch(self, I, J, V, flavour=capi.UPDATE, tid=0):
        self._ship(tid)
        self._h.insert_batch(I, J, V, flavour, tid)

    def insert_elements(self, dofs, Aloc, flavour=capi.RAW, tid=0, col_dofs=None):
        """Element loop (test/femtools.jl:45-72): for every element c, for jl, for il,
        rawupdateindex!(A, +, Aloc[c, jl, il], dofs[c, il], dofs[c, jl]) (or the `flavour`'s call).
        dofs (ncells, k), 1-based; Aloc (ncells, k, k).  With col_dofs (ncells, kc) the columns come from col_dofs:
        rawupdateindex!(A, +, Aloc[c, jl, il], dofs[c, il], col_dofs[c, jl]), dofs (ncells, kr), Aloc (ncells, kc, kr)."""
        self._ship(tid)
        self._h.insert_elements(dofs, Aloc, flavour, tid, col_dofs=col_dofs)

    # -- flush!/sparse/nnz/reset!
    def flush(self):
        for t in range(self._n_tid):
            self._ship(t)
        if self._h.pending:
            _, changed = self._h.flush(self.mode)
            self.pattern_changes += int(changed)
        return self

    def csc(self):
        """sparse(A) as Julia-style (colptr, rowval, nzval), 1-based."""
        self.flush()
        return self._h.fetch_csc_numpy()

    def sparse(self):
        import scipy.sparse as sp

        cp, rv, nz = self.csc()
        return sp.csc_matrix((nz, rv - 1, cp - 1), shape=(self.m, self.n))

    def mul(self, x):
        """A*x: flush, then the column-order kernel (abstractextendablesparsematrixcsc.jl:170-181)."""
        self.flush()
        return self._h.mul(np.ascontiguousarray(x, np.float64))

    def __matmul__(self, x):
        return self.mul(x)

    @property
    def nnz(self):
        self.flush()  # abstractextendablesparsematrixcsc.jl:24
        return self._h.nnz

    def reset(self):
        for b in self._buf:
            b.n = 0
        self._h.reset()

    def zero_values(self):
        """nonzeros(A) .= 0 (sprand.jl:80-85)."""
        self.flush()
        self._h.zero_values()

    def dropzeros(self):
        """dropzeros!(A) (abstractextendablesparsematrixcsc.jl:110): the stored +-0.0 removed on the device, in place."""
        self.flush()
        _, changed = self._h.dropzeros()
        self.pattern_changes += int(changed)
        return self

    def _combine(self, other, op):
        if not isinstance(other, ExtendableSparseMatrix):
            return NotImplemented
        self.flush()
        other.flush()
        hc = self._h.add(other._h, op)
        C = ExtendableSparseMatrix.__new__(ExtendableSparseMatrix)
        C._h, C.m, C.n, C.mode = hc, self.m, self.n, self.mode
        C._buf = [_HostBuffer()]
        C.pattern_changes = 0
        return C

    def __add__(self, other):
        """A + B (abstractextendablesparsematrixcsc.jl: flush both, then SparseArrays' +): a new matrix."""
        return self._combine(other, capi.OP_ADD)

    def __sub__(self, other):
        """A - B: a new matrix."""
        return self._combine(other, capi.OP_SUB)

    def mark_dirichlet(self, penalty=1.0e20):
        self.flush()
        return self._h.mark_dirichlet(penalty)

    def eliminate_dirichlet(self, marker):
        self.flush()
        self._h.eliminate_dirichlet(marker)
        return self

    def pointblock(self, blocksize):
        """pointblock(A, blocksize) (extendable.jl:292-318): (colptr, rowval, blocks) of the block matrix,
        1-based, blocks[k] the k-th stored blocksize x blocksize block (blocks[k][ii-1, jj-1] = block[ii, jj])."""
        self.flush()
        hb = self._h.pointblock(blocksize)
        try:
            cp, rv, _ = hb.fetch_csc_numpy()
            blocks = hb.fetch_blocks_numpy().transpose(0, 2, 1).copy()
        finally:
            hb.close()
        return cp, rv, blocks


class MTExtendableSparseMatrix(ExtendableSparseMatrix):
    """MTExtendableSparseMatrixCSC: one insert buffer per partition (genericmt...:1-114)."""

    def __init__(self, m, n=None, nparts=1, **kw):
        self._n_tid = int(nparts)
        super().__init__(m, n, **kw)

    def rawupdateindex(self, op, v, i, j, tid=1):
        self._push(capi.RAW, self._signed(op, v), i, j, tid - 1)
        return self

    def updateindex(self, op, v, i, j, tid=1):
        self._push(capi.UPDATE, self._signed(op, v), i, j, tid - 1)
        return self

    @property
    def nnznew(self):
        """Upper bound of nnznew(A) (genericmt...:84): the staged insertions."""
        return self._h.pending + sum(b.n for b in self._buf)


# function-style spellings, as in the reference's exports (src/ExtendableSparse.jl:42-58)
def updateindex(A, op, v, i, j, *tid):
    return A.updateindex(op, v, i, j, *tid)


def rawupdateindex(A, op, v, i, j, *tid):
    return A.rawupdateindex(op, v, i, j, *tid)


def pointblock(A, blocksize):
    return A.pointblock(blocksize)


def dropzeros(A):
    return A.dropzeros()


def flush(A):
    return A.flush()


def sparse(A):
    return A.sparse()


def nnz(A):
    return A.nnz


def reset(A):
    return A.reset()


def fdrand(A, nx, ny=1, nz=1, *, update=None, rand=None):
    """fdrand!(A,nx,ny,nz;update,rand): src/matrix/sprand.jl:58-126, driving A through `update`."""
    if update is None:
        update = lambda A, v, i, j: A.updateindex(operator.add, v, i, j)  # noqa: E731
    if rand is None:
        rng = np.random.default_rng(0)
        rand = rng.random
    N = nx * ny * nz
    if A.shape != (N, N):
        raise ValueError("Matrix size mismatch")
    A.zero_values()

    def update_pair(v, i, j):
        update(A, -v, i, j)
        update(A, -v, j, i)
        update(A, v, i, i)
        update(A, v, j, j)

    hx, hy, hz = 1.0 / nx, 1.0 / ny, 1.0 / nz
    nxy = nx * ny
    l = 1
    for k in range(1, nz + 1):
        for j in range(1, ny + 1):
            for i in range(1, nx + 1):
                if i < nx:
                    update_pair(rand() * hy * hz / hx, l, l + 1)
                if i == 1 or i == nx:
                    update(A, rand() * hy * hz, l, l)
                if j < ny:
                    update_pair(rand() * hx * hz / hy, l, l + nx)
                if ny > 2 and (j == 1 or j == ny):
                    update(A, rand() * hx * hz, l, l)
                if k < nz:
                    update_pair(rand() * hx * hy / hz, l, l + nxy)
                if nz > 2 and (k == 1 or k == nz):
                    update(A, rand() * hx * hy, l, l)
                l += 1
    return A.flush()
