"""GPU tests of A + B, A - B (xsb_add) and dropzeros! (xsb_dropzeros): colptr / rowval exact and nzval bit for bit
against the numpy restatement of SparseArrays' map(+/-, A, B) and fkeep! (tests/csc_algebra_ref.py)."""

import socket

import numpy as np
import pytest

from tests import csc_algebra_ref as alg

pytestmark = pytest.mark.gpu

SPECIAL = np.array([0.0, -0.0, np.nan, -np.nan, np.inf, -np.inf, 1.0, -1.0])


@pytest.fixture(scope="module")
def xsb():
    import __graft_entry__ as ge

    ge.build()
    import xsparse_b200

    assert xsparse_b200.capi.device_count() > 0
    return xsparse_b200


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def assert_same(got, ref):
    cp, rv, nz = got
    ocp, orv, onz = ref
    assert np.array_equal(np.asarray(cp, np.int64), ocp), "colptr differs"
    assert np.array_equal(np.asarray(rv, np.int64), orv), "rowval differs"
    bad = np.nonzero(bits(nz) != bits(onz))[0]
    assert bad.size == 0, f"{bad.size} nzval entries differ, first at {bad[:5]}"


def random_csc(rng, m, n, density, base=1, special=0.1, values=None):
    """Sorted CSC with `density` of the positions stored; a fraction `special` of the values from SPECIAL."""
    mask = rng.random((n, m)) < density
    cols, rows = np.nonzero(mask)
    nz = rng.standard_normal(len(rows)) if values is None else values(len(rows))
    sp = rng.random(len(rows)) < special
    nz[sp] = rng.choice(SPECIAL, int(sp.sum()))
    cp = np.concatenate([[0], np.cumsum(np.bincount(cols, minlength=n))]) + base
    return cp.astype(np.int64), (rows + base).astype(np.int64), nz


def handle(xsb, m, n, A, idx=None, base=1):
    idx = xsb.I64 if idx is None else idx
    h = xsb.Handle(m, n, idx, base)
    dt = np.int64 if idx == xsb.I64 else np.int32
    h.set_csc(np.ascontiguousarray(A[0], dt), np.ascontiguousarray(A[1], dt), np.ascontiguousarray(A[2], np.float64))
    return h


def shift(A, d):
    return (np.asarray(A[0]) + d, np.asarray(A[1]) + d, A[2])


def check_pair(xsb, oracle, m, n, A, B, op, idx, base):
    ha, hb = handle(xsb, m, n, A, idx, base), handle(xsb, m, n, B, idx, base)
    hc = ha.add(hb, op)
    got = hc.fetch_csc_numpy()
    ref = alg.map_zeropres("+" if op == xsb.OP_ADD else "-", m, n, A, B, base=base)
    assert_same(got, ref)
    # A and B untouched
    assert_same(ha.fetch_csc_numpy(), A)
    assert_same(hb.fetch_csc_numpy(), B)
    for h in (ha, hb, hc):
        h.close()


@pytest.mark.parametrize("kind", ["overlap", "disjoint", "identical"])
@pytest.mark.parametrize("op", [0, 1])
@pytest.mark.parametrize("idx,base", [(1, 1), (1, 0), (0, 1), (0, 0)])
@pytest.mark.parametrize("shape", [(60, 50), (1, 40), (40, 1), (500, 7), (7, 500)])
def test_random_pairs(xsb, oracle, kind, op, idx, base, shape):
    m, n = shape
    rng = np.random.default_rng([["overlap", "disjoint", "identical"].index(kind), op, idx, base, *shape])
    A = random_csc(rng, m, n, 0.3, base)
    if kind == "overlap":
        B = random_csc(rng, m, n, 0.3, base)
    elif kind == "identical":
        B = (A[0], A[1], rng.standard_normal(len(A[2])))
        same = rng.random(len(B[2])) < 0.3
        B[2][same] = A[2][same]  # cancellations
    else:  # B stores exactly the positions A does not
        full = random_csc(rng, m, n, 1.1, base)
        ka = set(zip(np.repeat(np.arange(n), np.diff(A[0])), A[1]))
        cols = np.repeat(np.arange(n), np.diff(full[0]))
        keep = np.array([(c, r) not in ka for c, r in zip(cols, full[1])], bool)
        B = (np.concatenate([[0], np.cumsum(np.bincount(cols[keep], minlength=n))]) + base, full[1][keep], full[2][keep])
    check_pair(xsb, oracle, m, n, A, B, op, idx, base)


def test_empty_and_full_cancellation(xsb, oracle):
    rng = np.random.default_rng(1)
    m, n = 30, 20
    E = (np.ones(n + 1, np.int64), np.zeros(0, np.int64), np.zeros(0))
    A = random_csc(rng, m, n, 0.4, special=0.0)
    for op in (xsb.OP_ADD, xsb.OP_SUB):
        check_pair(xsb, oracle, m, n, E, E, op, xsb.I64, 1)
        check_pair(xsb, oracle, m, n, A, E, op, xsb.I64, 1)
        check_pair(xsb, oracle, m, n, E, A, op, xsb.I64, 1)
    check_pair(xsb, oracle, m, n, A, A, xsb.OP_SUB, xsb.I64, 1)
    ha = handle(xsb, m, n, A)
    hc = ha.add(ha, xsb.OP_SUB)  # a is b
    assert hc.nnz == 0 and np.all(hc.fetch_csc_numpy()[0] == 1)
    hd = ha.add(ha, xsb.OP_ADD)
    assert_same(hd.fetch_csc_numpy(), alg.map_zeropres("+", m, n, A, A))
    for h in (ha, hc, hd):
        h.close()


def test_long_column_beside_empty_columns(xsb, oracle):
    rng = np.random.default_rng(2)
    m, n, L = 1 << 22, 4096, 1 << 20

    def one_column(col, rows, vals):
        cp = np.zeros(n + 1, np.int64)
        cp[col + 1:] = len(rows)
        return cp + 1, np.sort(rows).astype(np.int64) + 1, vals
    A = one_column(1000, rng.choice(m, L, replace=False), rng.standard_normal(L))
    B = one_column(1000, rng.choice(m, L, replace=False), rng.standard_normal(L))
    B2 = one_column(3000, rng.choice(m, L, replace=False), rng.standard_normal(L))
    for op in (xsb.OP_ADD, xsb.OP_SUB):
        check_pair(xsb, oracle, m, n, A, B, op, xsb.I64, 1)
        check_pair(xsb, oracle, m, n, A, B2, op, xsb.I32, 1)


def test_full_size_emitted_pair(xsb, oracle):
    nxn = 65  # FEM 64^3 cells
    n = nxn ** 3
    hf = xsb.Handle(n, n)
    hf.emit_p1fem(nxn, nxn, nxn, flavour=xsb.RAW)
    hf.flush()
    hd = xsb.Handle(n, n)
    hd.emit_fdrand(nxn, nxn, nxn, seed=11)
    hd.flush()
    F, D = hf.fetch_csc_numpy(), hd.fetch_csc_numpy()
    for op, sym in ((xsb.OP_ADD, "+"), (xsb.OP_SUB, "-")):
        hc = hf.add(hd, op)
        assert_same(hc.fetch_csc_numpy(), alg.map_zeropres(sym, n, n, F, D))
        hc.close()
    hc = hf.add(hf, xsb.OP_SUB)
    assert hc.nnz == 0
    for h in (hf, hd, hc):
        h.close()


def test_result_is_an_assembly_target(xsb, oracle):
    rng = np.random.default_rng(3)
    m = n = 200
    A = random_csc(rng, m, n, 0.05, special=0.0)
    B = random_csc(rng, m, n, 0.05, special=0.0)
    ha, hb = handle(xsb, m, n, A), handle(xsb, m, n, B)
    hc = ha.add(hb, xsb.OP_SUB)
    C0 = alg.map_zeropres("-", m, n, A, B)
    ha.close()
    hb.close()  # C owns its arrays
    x = rng.standard_normal(n)
    y = hc.mul(x)
    ref = np.zeros(m)
    cols = np.repeat(np.arange(n), np.diff(C0[0]))
    for k in range(len(C0[2])):  # the column-order left fold of mul!
        ref[C0[1][k] - 1] += C0[2][k] * x[cols[k]]
    assert np.array_equal(bits(y), bits(ref))
    # insert + flush into C
    I = rng.integers(1, m + 1, 3000)
    J = rng.integers(1, n + 1, 3000)
    V = rng.standard_normal(3000)
    hc.insert_batch(I, J, V, xsb.UPDATE)
    hc.flush()
    o = oracle.OracleExt(m, n)
    o.set_csc(*C0)
    o.insert_batch(I, J, V, oracle.UPDATE)
    C1 = o.csc()
    assert_same(hc.fetch_csc_numpy(), C1)
    # freeze and re-assemble on C
    hc.freeze_pattern(I, J)
    V2 = rng.standard_normal(3000)
    hc.reassemble_values(V2, zero_first=True)
    o.zero_values()
    o.insert_batch(I, J, V2, oracle.UPDATE)
    assert_same(hc.fetch_csc_numpy(), o.csc())
    hc.close()


def test_errors_leave_inputs_unchanged(xsb):
    rng = np.random.default_rng(4)
    m, n = 40, 30
    A = random_csc(rng, m, n, 0.2, special=0.0)
    ha = handle(xsb, m, n, A)

    def refused(code, other, op=0):
        with pytest.raises(xsb.XsbError) as e:
            ha.add(other, op)
        assert e.value.code == code
        assert_same(ha.fetch_csc_numpy(), A)

    def empty(m, n):
        return handle(xsb, m, n, (np.ones(n + 1, np.int64), np.zeros(0, np.int64), np.zeros(0)))

    refused(xsb.capi.ESIZE, empty(m, n + 1))
    refused(xsb.capi.ESIZE, empty(m + 1, n))
    with pytest.raises(xsb.XsbError, match="DimensionMismatch"):
        ha.add(empty(m + 1, n))
    refused(xsb.capi.EINVAL, handle(xsb, m, n, A, xsb.I32))
    refused(xsb.capi.EINVAL, handle(xsb, m, n, shift(A, -1), xsb.I64, 0))
    refused(xsb.capi.EINVAL, ha, 2)
    hp = handle(xsb, m, n, A)
    hp.insert_batch(np.array([1]), np.array([1]), np.array([1.0]))
    refused(xsb.capi.ESTATE, hp)
    with pytest.raises(xsb.XsbError) as e:
        hp.add(ha)
    assert e.value.code == xsb.capi.ESTATE
    hp.flush()
    assert hp.add(ha).nnz >= 1
    hs = xsb.Handle(m, n, slab=(2, 0, [0, 10, n]))
    refused(xsb.capi.ESTATE, hs)
    hb = empty(n, n).pointblock(2)
    hq = empty(n // 2, n // 2)
    with pytest.raises(xsb.XsbError) as e:
        hq.add(hb)
    assert e.value.code == xsb.capi.ESTATE
    with pytest.raises(xsb.XsbError) as e:
        hb.dropzeros()
    assert e.value.code == xsb.capi.ESTATE
    with pytest.raises(xsb.XsbError) as e:
        hs2 = xsb.Handle(m, n)
        hs2.insert_batch(np.array([1]), np.array([1]), np.array([0.0]), xsb.RAW)
        hs2.dropzeros()
    assert e.value.code == xsb.capi.ESTATE


def test_result_too_large_for_int32(xsb):
    """Two disjoint columns of 1.1e9 entries each: C would need 2.2e9 Int32 positions."""
    torch = pytest.importorskip("torch")
    L = 1_100_000_000
    m, n = L + 1, 2

    def big(col):
        cp = torch.tensor([1, 1 + (L if col == 0 else 0), 1 + L], dtype=torch.int32, device="cuda")
        rv = torch.arange(1, L + 1, dtype=torch.int32, device="cuda")
        nz = torch.ones(L, dtype=torch.float64, device="cuda")
        h = xsb.Handle(m, n, xsb.I32, 1)
        h.set_csc(cp, rv, nz)
        del rv, nz
        return h

    ha = big(0)
    hb = big(1)
    with pytest.raises(xsb.XsbError) as e:
        ha.add(hb)
    assert e.value.code == xsb.capi.EINVAL and "Int32" in str(e.value)
    assert ha.nnz == L and hb.nnz == L
    ha.close()
    hb.close()
    torch.cuda.empty_cache()


# ---- dropzeros! ----
@pytest.mark.parametrize("idx,base", [(1, 1), (0, 0)])
def test_dropzeros_plain(xsb, oracle, idx, base):
    rng = np.random.default_rng(6)
    m, n = 300, 250
    A = random_csc(rng, m, n, 0.1, base, special=0.3)
    h = handle(xsb, m, n, A, idx, base)
    nnz, changed = h.dropzeros()
    ref = alg.fkeep_nonzero(n, A, base)
    assert changed and nnz == len(ref[2])
    assert_same(h.fetch_csc_numpy(), ref)
    assert h.dropzeros() == (nnz, False)
    assert_same(h.fetch_csc_numpy(), ref)
    h.close()


def test_dropzeros_frozen_and_mul(xsb, oracle):
    rng = np.random.default_rng(7)
    m = n = 120
    A = random_csc(rng, m, n, 0.1, special=0.0)
    h = handle(xsb, m, n, A)
    cols = np.repeat(np.arange(n), np.diff(A[0])) + 1
    I, J = A[1], cols
    h.freeze_pattern(I, J)
    x = rng.standard_normal(n)
    y0 = h.mul(x)  # builds the row-major view
    assert h.dropzeros() == (len(A[2]), False)
    V = rng.standard_normal(len(I))
    V[::5] = 0.0
    h.reassemble_values(V, zero_first=True)  # still frozen
    vals = h.fetch_csc_numpy()[2]
    assert np.array_equal(bits(vals), bits(V + 0.0))
    nnz, changed = h.dropzeros()
    ref = alg.fkeep_nonzero(n, (A[0], A[1], V + 0.0))
    assert changed and nnz == len(ref[2])
    assert_same(h.fetch_csc_numpy(), ref)
    with pytest.raises(xsb.XsbError):  # the frozen map is gone
        h.reassemble_values(V)
    y = h.mul(x)
    refy = np.zeros(m)
    rc = np.repeat(np.arange(n), np.diff(ref[0]))
    for k in range(len(ref[2])):
        refy[ref[1][k] - 1] += ref[2][k] * x[rc[k]]
    assert np.array_equal(bits(y), bits(refy))
    assert y0.shape == y.shape
    h.close()


@pytest.mark.parametrize("splits", [[0, 40, 90], [0, 1, 60, 90]])
def test_dropzeros_slabs(xsb, oracle, splits):
    rng = np.random.default_rng(8)
    m, n = 70, 90
    A = random_csc(rng, m, n, 0.2, special=0.4)
    ref = alg.fkeep_nonzero(n, A)
    world = len(splits) - 1
    for r in range(world):
        lo, hi = splits[r], splits[r + 1]
        a0, a1 = A[0][lo] - 1, A[0][hi] - 1
        hs = xsb.Handle(m, n, slab=(world, r, splits))
        hs.set_csc(A[0][lo:hi + 1] - a0, np.ascontiguousarray(A[1][a0:a1]), np.ascontiguousarray(A[2][a0:a1]))
        nnz, changed = hs.dropzeros()
        r0, r1 = ref[0][lo] - 1, ref[0][hi] - 1
        assert nnz == r1 - r0 and changed == (r1 - r0 != a1 - a0)
        assert_same(hs.fetch_csc_numpy(), (ref[0][lo:hi + 1] - r0, ref[1][r0:r1], ref[2][r0:r1]))
        hs.close()


def test_matrix_wrapper(xsb, oracle):
    import operator

    m, n = 50, 40
    A = xsb.ExtendableSparseMatrix(m, n)
    B = xsb.ExtendableSparseMatrix(m, n)
    rng = np.random.default_rng(9)
    for M in (A, B):
        for _ in range(300):
            M.rawupdateindex(operator.add, float(rng.choice([0.0, 1.0, -2.5])), int(rng.integers(1, m + 1)),
                             int(rng.integers(1, n + 1)))
    Ac, Bc = A.csc(), B.csc()  # flushes
    A.rawupdateindex(operator.add, 0.0, 1, 1)  # pending: + flushes first
    Ac2 = oracle.OracleExt(m, n)
    Ac2.set_csc(*Ac)
    Ac2.rawupdateindex(0.0, 1, 1)
    Ac = Ac2.csc()
    S, D = A + B, A - B
    assert_same(S.csc(), alg.map_zeropres("+", m, n, Ac, Bc))
    assert_same(D.csc(), alg.map_zeropres("-", m, n, Ac, Bc))
    S.rawupdateindex(operator.add, 1.0, m, n)  # C is an assembly target
    o = oracle.OracleExt(m, n)
    o.set_csc(*alg.map_zeropres("+", m, n, Ac, Bc))
    o.rawupdateindex(1.0, m, n)
    assert_same(S.csc(), o.csc())
    before = A.pattern_changes
    A.dropzeros()
    ref = alg.fkeep_nonzero(n, Ac)
    assert_same(A.csc(), ref)
    assert len(ref[2]) < len(Ac[2]) and A.pattern_changes == before + 1
    A.dropzeros()
    assert A.pattern_changes == before + 1


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def test_dist_dropzeros_world_one(xsb, oracle):
    torch = pytest.importorskip("torch")
    import torch.distributed as dist

    from xsparse_b200.dist import DistExtendableSparseMatrix

    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{_free_port()}", rank=0, world_size=1,
                            device_id=torch.device("cuda", 0))
    try:
        m = n = 60
        D = DistExtendableSparseMatrix(m, n)
        rng = np.random.default_rng(10)
        I = np.concatenate([np.arange(1, n + 1), rng.integers(1, m + 1, 400)])
        J = np.concatenate([np.arange(1, n + 1), rng.integers(1, n + 1, 400)])
        V = rng.choice([0.0, 1.0, 2.0], len(I))
        D.insert_batch(I, J, V, xsb.RAW)
        D.flush()
        A = D.h.fetch_csc_numpy()
        D.freeze_pattern(I, J)
        nnz, changed = D.dropzeros()
        ref = alg.fkeep_nonzero(n, A)
        assert changed and nnz == len(ref[2]) == D.nnz_global and D.nnz_offset == 0
        assert not D._frozen
        assert_same(D.h.fetch_csc_numpy(), ref)
        assert D.dropzeros() == (nnz, False)
        D.close()
    finally:
        dist.destroy_process_group()
