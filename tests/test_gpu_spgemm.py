"""GPU tests of A * B (xsb_matmul): colptr / rowval exact and nzval bit for bit against the numpy restatement of
SparseArrays' spmatmul (tests/spgemm_ref.py)."""

import operator
import threading

import numpy as np
import pytest

from tests import spgemm_ref as ref

pytestmark = pytest.mark.gpu

SPECIAL = np.array([0.0, -0.0, np.nan, -np.nan, np.inf, -np.inf, 1.0, -1.0])
# f(j), the products of a column, decides its path: warp tables up to 256, 1024 and 4096 products, row tiles above
BIN_EDGES = (256, 1024, 4096)


@pytest.fixture(scope="module")
def xsb():
    import __graft_entry__ as ge

    ge.build()
    import xsparse_b200

    assert xsparse_b200.capi.device_count() > 0
    return xsparse_b200


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def assert_same(got, want):
    cp, rv, nz = got
    assert np.array_equal(np.asarray(cp, np.int64), np.asarray(want[0], np.int64)), "colptr differs"
    assert np.array_equal(np.asarray(rv, np.int64), np.asarray(want[1], np.int64)), "rowval differs"
    bad = np.nonzero(bits(nz) != bits(want[2]))[0]
    assert bad.size == 0, f"{bad.size} nzval entries differ, first at {bad[:5]}"


def random_csc(rng, m, n, density, base=1, special=0.1):
    mask = rng.random((n, m)) < density
    cols, rows = np.nonzero(mask)
    nz = rng.standard_normal(len(rows))
    sp = rng.random(len(rows)) < special
    nz[sp] = rng.choice(SPECIAL, int(sp.sum()))
    cp = np.concatenate([[0], np.cumsum(np.bincount(cols, minlength=n))]) + base
    return cp.astype(np.int64), (rows + base).astype(np.int64), nz


def columns_csc(m, cols, base=1):
    """CSC from a list of (rows, values) per column, rows 0-based and sorted."""
    cp = np.concatenate([[0], np.cumsum([len(r) for r, _ in cols])]) + base
    rv = np.concatenate([np.asarray(r, np.int64) for r, _ in cols] + [np.zeros(0, np.int64)]) + base
    nz = np.concatenate([np.asarray(v, np.float64) for _, v in cols] + [np.zeros(0)])
    return cp.astype(np.int64), rv.astype(np.int64), nz


def handle(xsb, m, n, A, idx=None, base=1):
    idx = xsb.I64 if idx is None else idx
    h = xsb.Handle(m, n, idx, base)
    dt = np.int64 if idx == xsb.I64 else np.int32
    h.set_csc(np.ascontiguousarray(A[0], dt), np.ascontiguousarray(A[1], dt), np.ascontiguousarray(A[2], np.float64))
    return h


def products_per_column(A, B, base=1):
    la = np.diff(np.asarray(A[0], np.int64))
    k = np.asarray(B[1], np.int64) - base
    cols = np.repeat(np.arange(len(B[0]) - 1), np.diff(np.asarray(B[0], np.int64)))
    return np.bincount(cols, weights=la[k], minlength=len(B[0]) - 1).astype(np.int64)


def check_product(xsb, m, k, n, A, B, idx=None, base=1):
    ha, hb = handle(xsb, m, k, A, idx, base), handle(xsb, k, n, B, idx, base)
    hc = ha.matmul(hb)
    assert (hc.m, hc.n) == (m, n)
    assert_same(hc.fetch_csc_numpy(), ref.spmatmul(m, n, A, B, base))
    assert_same(ha.fetch_csc_numpy(), A)
    assert_same(hb.fetch_csc_numpy(), B)
    for h in (ha, hb, hc):
        h.close()


@pytest.mark.parametrize("density", [0.02, 0.2, 0.7, 1.0])
@pytest.mark.parametrize("idx,base", [(1, 1), (1, 0), (0, 1), (0, 0)])
@pytest.mark.parametrize("shape", [(60, 45, 50), (1, 40, 7), (40, 1, 40), (500, 7, 500), (7, 500, 7)])
def test_random_pairs(xsb, density, idx, base, shape):
    m, k, n = shape
    rng = np.random.default_rng([int(density * 100), idx, base, *shape])
    A = random_csc(rng, m, k, density, base)
    B = random_csc(rng, k, n, density, base)
    check_product(xsb, m, k, n, A, B, idx, base)


def test_empty_operands_and_columns(xsb):
    rng = np.random.default_rng(1)
    m, k, n = 30, 20, 25
    E = lambda r, c: (np.ones(c + 1, np.int64), np.zeros(0, np.int64), np.zeros(0))  # noqa: E731
    A = random_csc(rng, m, k, 0.3)
    B = random_csc(rng, k, n, 0.3)
    check_product(xsb, m, k, n, E(m, k), B)
    check_product(xsb, m, k, n, A, E(k, n))
    check_product(xsb, m, k, n, E(m, k), E(k, n))
    # empty columns of A hit by B, and empty columns of B
    A2 = columns_csc(m, [([], []) if c % 3 == 0 else (np.sort(rng.choice(m, 5, replace=False)), rng.standard_normal(5))
                         for c in range(k)])
    B2 = columns_csc(k, [([], []) if c % 4 == 0 else (np.sort(rng.choice(k, 6, replace=False)), rng.standard_normal(6))
                         for c in range(n)])
    check_product(xsb, m, k, n, A2, B2)


def test_square_of_itself(xsb):
    rng = np.random.default_rng(2)
    n = 300
    A = random_csc(rng, n, n, 0.05)
    ha = handle(xsb, n, n, A)
    hc = ha.matmul(ha)  # a is b
    assert_same(hc.fetch_csc_numpy(), ref.spmatmul(n, n, A, A))
    assert_same(ha.fetch_csc_numpy(), A)
    ha.close()
    hc.close()


def test_explicit_zeros_signed_zero_and_nan(xsb):
    snan = np.array([0x7FF0000000000001], np.uint64).view(np.float64)[0]
    # A: column 1 rows {1, 2} = (-1.0, 0.0); column 2 row 1 = +inf; column 3 row 1 = -inf; column 4 row 2 = sNaN
    A = columns_csc(3, [([0, 1], [-1.0, 0.0]), ([0], [np.inf]), ([0], [-np.inf]), ([1], [snan])])
    # B: column 1 = explicit zero at k=1 -> (-1 * 0, 0 * 0) both stored; column 2: k=1 x 0.0 and k=2 x 0.0 (0 * Inf);
    # column 3: k=2, k=3 with 1.0 (Inf + -Inf); column 4: k=4 x 2.0 (quieted payload)
    B = columns_csc(4, [([0], [0.0]), ([0, 1], [0.0, 0.0]), ([1, 2], [1.0, 1.0]), ([3], [2.0])])
    want = ref.spmatmul(3, 4, A, B)
    check_product(xsb, 3, 4, 4, A, B)
    ha, hb = handle(xsb, 3, 4, A), handle(xsb, 4, 4, B)
    cp, rv, nz = ha.matmul(hb).fetch_csc_numpy()
    assert cp.tolist() == want[0].tolist() == [1, 3, 5, 6, 7]
    u = bits(nz)
    assert u[0] == 0x8000000000000000  # -1.0 * 0.0 assigned: -0.0 with the sign bit set
    assert u[1] == 0  # +0.0 * 0.0
    assert u[2] == 0xFFF8000000000000  # 0 * Inf in row 1 of column 2 (then + 0 * -0: NaN stays)
    assert u[4] == 0xFFF8000000000000  # Inf + -Inf
    assert u[5] == 0x7FF8000000000001  # the payload of A's NaN, quieted


def test_bin_thresholds(xsb):
    """Columns whose product counts sit on both sides of every bin edge, in one product."""
    rng = np.random.default_rng(3)
    m = 9000
    lens = [1, 2, 255, 256, 257, 1023, 1024, 1025, 4095, 4096, 4097, 8192, 9000]
    A = columns_csc(m, [(np.sort(rng.choice(m, L, replace=False)), rng.standard_normal(L)) for L in lens])
    k = len(lens)
    cols = [([c], [rng.standard_normal()]) for c in range(k)]
    cols += [([0, 2, 3], rng.standard_normal(3)), ([3, 4], rng.standard_normal(2)), ([5, 6, 9], [1.0, -1.0, 0.5])]
    cols += [([], [])] * 3 + [(list(range(k)), rng.standard_normal(k))]
    B = columns_csc(k, cols)
    f = products_per_column(A, B)
    for e in BIN_EDGES:
        assert (f == e).any() and (f == e + 1).any()
    check_product(xsb, m, k, len(cols), A, B)
    zero = lambda M: (M[0] - 1, M[1] - 1, M[2])  # noqa: E731
    check_product(xsb, m, k, len(cols), zero(A), zero(B), xsb.I32, 0)


# f(j) = 100 per_col: counted in a warp table, then in row tiles; u(j) > 4096 at m = 9000: written by the row tiles
@pytest.mark.parametrize("per_col,m", [(20, 200), (60, 200), (5000, 9000)])
def test_left_fold_order_across_batches(xsb, per_col, m):
    """Products in k order like [1e16, 1, -1e16, ...]: the left fold gives 0, any other order does not."""
    rng = np.random.default_rng(4)
    k, n = 100, 6
    vals = np.array([1e16, 1.0, -1e16])
    A = columns_csc(m, [(np.sort(rng.choice(m, per_col, replace=False)), rng.choice(vals, per_col)) for _ in range(k)])
    B = columns_csc(k, [(np.arange(k), np.ones(k)) for _ in range(n - 1)] + [(np.arange(0, k, 3), np.ones(34))])
    # row m is met at k = 5, 37, 70 only, with 1e16, 1, -1e16: its products straddle 32-product batches
    cols = []
    cp, rv, nz = A
    for c in range(k):
        r, v = rv[cp[c] - 1:cp[c + 1] - 1] - 1, nz[cp[c] - 1:cp[c + 1] - 1]
        keep = r != m - 1
        r, v = list(r[keep]), list(v[keep])
        if c in (5, 37, 70):
            r.append(m - 1)
            v.append({5: 1e16, 37: 1.0, 70: -1e16}[c])
        cols.append((r, v))
    A = columns_csc(m, cols)
    want = ref.spmatmul(m, n, A, B)
    assert want[1][want[0][1] - 2] == m and want[2][want[0][1] - 2] == 0.0  # row m of column 1 folds to 0
    check_product(xsb, m, k, n, A, B)


def test_long_column_beside_empty_columns(xsb):
    rng = np.random.default_rng(5)
    m, k, n, L = 1 << 22, 3, 4096, 1 << 20
    A = columns_csc(m, [(np.sort(rng.choice(m, L, replace=False)), rng.standard_normal(L)) for _ in range(2)] +
                    [([0, m - 1], [1.0, 2.0])])
    cols = [([], [])] * n
    cols[1000] = ([0], [1.5])
    cols[3000] = ([0, 1, 2], [-0.5, 2.0, 3.0])
    B = columns_csc(k, cols)
    check_product(xsb, m, k, n, A, B)
    check_product(xsb, m, k, n, A, B, xsb.I32, 1)


def test_long_b_column_on_short_a_columns(xsb):
    """A B column with 2^14 entries on A columns of 1-4 rows: f(j) large, each row met many times."""
    rng = np.random.default_rng(6)
    m, k, n = 5000, 1 << 14, 3
    lens = rng.integers(1, 5, k)
    A = columns_csc(m, [(np.sort(rng.choice(m, L, replace=False)), rng.choice([1e16, 1.0, -1e16, 0.5], L))
                        for L in lens])
    B = columns_csc(k, [(np.arange(k), np.ones(k)), ([], []), (np.arange(0, k, 7), rng.standard_normal(len(range(0, k, 7))))])
    assert products_per_column(A, B)[0] > BIN_EDGES[-1]
    check_product(xsb, m, k, n, A, B)


def test_emitted_fem_squared(xsb):
    nxn = 33  # FEM 32^3 cells
    n = nxn ** 3
    h = xsb.Handle(n, n)
    h.emit_p1fem(nxn, nxn, nxn, flavour=xsb.RAW)
    h.flush()
    F = h.fetch_csc_numpy()
    hc = h.matmul(h)
    assert_same(hc.fetch_csc_numpy(), ref.spmatmul(n, n, F, F))
    h.close()
    hc.close()


def kuhn_cells(xsb, mesh):
    """(ncells, 4) 1-based node numbers of the FEM emitter's Kuhn mesh: node jl of cell t is the column of its
    stream's call 20 t + 1 + jl."""
    nn = (mesh + 1) ** 3
    g = xsb.Handle(nn, nn)
    g.set_precount(False)
    g.emit_p1fem(mesh + 1, mesh + 1, mesh + 1, flavour=xsb.RAW)
    J = g.debug_fetch_staged()[1]
    g.close()
    return np.ascontiguousarray(J.reshape(-1, 4, 5)[:, 0, 1:5].astype(np.int64)), nn


def test_rectangular_element_operators(xsb):
    cells, nn = kuhn_cells(xsb, 6)
    nc = len(cells)
    rng = np.random.default_rng(7)
    own = np.arange(1, nc + 1, dtype=np.int64)[:, None]
    d1 = xsb.Handle(nc, nn)  # p0xp1: row the cell, columns its nodes
    d1.insert_elements(own, rng.standard_normal((nc, 4, 1)), xsb.RAW, col_dofs=cells)
    d1.flush()
    d2 = xsb.Handle(nn, nc)  # p1xp0
    d2.insert_elements(cells, rng.standard_normal((nc, 1, 4)), xsb.RAW, col_dofs=own)
    d2.flush()
    D1, D2 = d1.fetch_csc_numpy(), d2.fetch_csc_numpy()
    for a, b, A, B, m, n in ((d1, d2, D1, D2, nc, nc), (d2, d1, D2, D1, nn, nn)):
        hc = a.matmul(b)
        assert (hc.m, hc.n) == (m, n)
        assert_same(hc.fetch_csc_numpy(), ref.spmatmul(m, n, A, B))
        hc.close()
    d1.close()
    d2.close()


def test_result_is_an_assembly_target(xsb, oracle):
    rng = np.random.default_rng(8)
    m, k, n = 200, 150, 180
    A = random_csc(rng, m, k, 0.03, special=0.0)
    B = random_csc(rng, k, n, 0.03, special=0.0)
    ha, hb = handle(xsb, m, k, A), handle(xsb, k, n, B)
    hc = ha.matmul(hb)
    C0 = ref.spmatmul(m, n, A, B)
    ha.close()
    hb.close()  # C owns its arrays
    x = rng.standard_normal(n)
    y = hc.mul(x)
    want = np.zeros(m)
    cols = np.repeat(np.arange(n), np.diff(C0[0]))
    for q in range(len(C0[2])):  # the column-order left fold of mul!
        want[C0[1][q] - 1] += C0[2][q] * x[cols[q]]
    assert np.array_equal(bits(y), bits(want))
    I = rng.integers(1, m + 1, 3000)
    J = rng.integers(1, n + 1, 3000)
    V = rng.standard_normal(3000)
    hc.insert_batch(I, J, V, xsb.UPDATE)
    hc.flush()
    o = oracle.OracleExt(m, n)
    o.set_csc(*C0)
    o.insert_batch(I, J, V, oracle.UPDATE)
    assert_same(hc.fetch_csc_numpy(), o.csc())
    hc.freeze_pattern(I, J)
    V2 = rng.standard_normal(3000)
    hc.reassemble_values(V2, zero_first=True)
    o.zero_values()
    o.insert_batch(I, J, V2, oracle.UPDATE)
    assert_same(hc.fetch_csc_numpy(), o.csc())
    hd = hc.add(hc)  # and an operand of +
    assert hd.nnz > 0
    hd.close()
    hc.close()


def test_errors_leave_inputs_unchanged(xsb):
    rng = np.random.default_rng(9)
    m, k = 40, 30
    A = random_csc(rng, m, k, 0.2, special=0.0)
    ha = handle(xsb, m, k, A)

    def refused(code, other, left=None):
        with pytest.raises(xsb.XsbError) as e:
            (left or ha).matmul(other)
        assert e.value.code == code
        assert_same(ha.fetch_csc_numpy(), A)

    def empty(r, c, idx=None, base=1):
        return handle(xsb, r, c, (np.full(c + 1, base, np.int64), np.zeros(0, np.int64), np.zeros(0)), idx, base)

    refused(xsb.capi.ESIZE, empty(k + 1, 5))
    refused(xsb.capi.ESIZE, empty(m, k), empty(m, k))  # A.n != B.m
    with pytest.raises(xsb.XsbError, match="DimensionMismatch"):
        ha.matmul(empty(k - 1, 5))
    refused(xsb.capi.EINVAL, empty(k, 5, xsb.I32))
    refused(xsb.capi.EINVAL, empty(k, 5, xsb.I64, 0))
    hp = empty(k, 5)
    hp.insert_batch(np.array([1]), np.array([1]), np.array([1.0]))
    refused(xsb.capi.ESTATE, hp)
    with pytest.raises(xsb.XsbError) as e:
        empty(5, m).matmul(hp)
    assert e.value.code == xsb.capi.ESTATE
    hp.flush()
    assert ha.matmul(hp).nnz >= 1
    refused(xsb.capi.ESTATE, xsb.Handle(k, 20, slab=(2, 0, [0, 10, 20])))
    hb = empty(2 * k, 2 * k).pointblock(2)  # k x k
    refused(xsb.capi.ESTATE, hb)
    hs = xsb.Handle(m, k, slab=(2, 1, [0, 10, k]))
    with pytest.raises(xsb.XsbError) as e:
        hs.matmul(empty(k, 5))
    assert e.value.code == xsb.capi.ESTATE


def test_result_too_large_for_int32(xsb):
    """A dense 65536 x 1 column times a dense 1 x 32768 row: C would hold 2^31 entries."""
    a_rows, b_cols = 1 << 16, 1 << 15
    A = (np.array([1, a_rows + 1], np.int32), np.arange(1, a_rows + 1, dtype=np.int32), np.ones(a_rows))
    B = (np.arange(1, b_cols + 2, dtype=np.int32), np.ones(b_cols, np.int32), np.ones(b_cols))
    ha, hb = handle(xsb, a_rows, 1, A, xsb.I32), handle(xsb, 1, b_cols, B, xsb.I32)
    with pytest.raises(xsb.XsbError) as e:
        ha.matmul(hb)
    assert e.value.code == xsb.capi.EINVAL and "Int32" in str(e.value)
    assert ha.nnz == a_rows and hb.nnz == b_cols
    ha.close()
    hb.close()


def test_two_threads_opposite_order(xsb):
    rng = np.random.default_rng(10)
    n = 150
    A = random_csc(rng, n, n, 0.05, special=0.0)
    B = random_csc(rng, n, n, 0.05, special=0.0)
    ha, hb = handle(xsb, n, n, A), handle(xsb, n, n, B)
    errors = []

    def run(x, y):
        try:
            for _ in range(20):
                x.matmul(y).close()
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    ts = [threading.Thread(target=run, args=(ha, hb)), threading.Thread(target=run, args=(hb, ha))]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=120)
    assert not any(t.is_alive() for t in ts), "deadlock"
    assert not errors
    ha.close()
    hb.close()


def test_matrix_wrapper(xsb):
    m, k, n = 50, 40, 30
    A = xsb.ExtendableSparseMatrix(m, k)
    B = xsb.ExtendableSparseMatrix(k, n)
    rng = np.random.default_rng(11)
    for M, (r, c) in ((A, (m, k)), (B, (k, n))):
        for _ in range(300):
            M.rawupdateindex(operator.add, float(rng.choice([0.0, 1.0, -2.5])), int(rng.integers(1, r + 1)),
                             int(rng.integers(1, c + 1)))
    A.rawupdateindex(operator.add, 3.0, m, k)  # pending: @ flushes first
    B.rawupdateindex(operator.add, -1.0, k, n)
    C = A @ B
    assert isinstance(C, xsb.ExtendableSparseMatrix) and C.shape == (m, n)
    Ac, Bc = A.csc(), B.csc()
    assert_same(C.csc(), ref.spmatmul(m, n, Ac, Bc))
    x = rng.standard_normal(k)
    y = A @ x
    assert isinstance(y, np.ndarray) and np.array_equal(bits(y), bits(A.mul(x)))
    C.rawupdateindex(operator.add, 1.0, 1, 1)  # C is an assembly target
    assert C.nnz >= 1
