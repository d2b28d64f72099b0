"""GPU tests of rectangular element matrices (xsb_insert_elements_rect / xsb_freeze_elements_rect /
xsb_freeze_slab_elements_rect): an element loop whose rows come from one connectivity (kr dofs per element) and whose
columns come from another (kc dofs) stages exactly the loop's call stream, and gives the CSC that xsb_insert_batch of
the expanded stream and the CPU oracle give, bit for bit."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHAPES = [(1, 1), (1, 64), (64, 1), (3, 7), (7, 3), (4, 12), (12, 4), (64, 64)]


@pytest.fixture(scope="module")
def xsb():
    import __graft_entry__ as ge

    ge.build()
    import xsparse_b200

    assert xsparse_b200.capi.device_count() > 0
    return xsparse_b200


@pytest.fixture(scope="module")
def torch():
    import torch

    assert torch.cuda.is_available()
    return torch


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def expand(rdofs, cdofs, Aloc):
    """The call stream: call kr kc c + kr jl + il = (rdofs[c, il], cdofs[c, jl], Aloc[c, jl, il])."""
    rdofs, cdofs = np.asarray(rdofs), np.asarray(cdofs)
    nc, kr = rdofs.shape
    kc = cdofs.shape[1]
    I = np.broadcast_to(rdofs[:, None, :], (nc, kc, kr)).reshape(-1).copy()
    J = np.broadcast_to(cdofs[:, :, None], (nc, kc, kr)).reshape(-1).copy()
    return I, J, np.ascontiguousarray(Aloc, np.float64).reshape(-1).copy()


def assert_same(got, ref):
    cp, rv, nz = got
    ocp, orv, onz = ref
    assert np.array_equal(cp, ocp), "colptr differs"
    assert np.array_equal(rv, orv), "rowval differs"
    bad = np.nonzero(bits(nz) != bits(onz))[0]
    assert bad.size == 0, f"{bad.size} nzval entries differ, first at {bad[:5]}"


def window_dofs(rng, size, ncells, k, repeat=False):
    """k dofs per element near a window that moves over [0, size): neighbouring elements share dofs; distinct inside
    an element unless `repeat`."""
    lo = (np.arange(ncells) * max(1, size // max(ncells, 1)))[:, None]
    span = 3 * k + 2
    dofs = (lo + rng.integers(0, span, (ncells, k))) % size
    if not repeat:
        for c in range(ncells):
            if len(set(dofs[c].tolist())) < k:
                dofs[c] = (lo[c, 0] + rng.permutation(span)[:k]) % size
    return dofs


def element_values(rng, ncells, kr, kc):
    """(ncells, kc, kr) values with exact zeros and entries that cancel next to Gaussian noise, so that RAW, UPDATE
    and ASSIGN give different matrices."""
    A = rng.choice(np.array([-1.5, -1.0, -0.5, 0.0, 0.5, 1.0, 1.5]), (ncells, kc, kr))
    noisy = rng.random(ncells) < 0.5
    A[noisy] = rng.standard_normal((int(noisy.sum()), kc, kr))
    A[rng.random((ncells, kc, kr)) < 0.1] = 0.0
    return A


def random_rect(rng, m, n, ncells, kr, kc, base=1, repeat=False):
    rdofs = window_dofs(rng, m, ncells, kr, repeat) + base
    cdofs = window_dofs(rng, n, ncells, kc, repeat) + base
    return rdofs.astype(np.int64), cdofs.astype(np.int64), element_values(rng, ncells, kr, kc)


def to_dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("kr,kc", SHAPES)
def test_random_connectivity_matches_batch_and_oracle(xsb, oracle, torch, kr, kc):
    rng = np.random.default_rng(100 * kr + kc)
    ncells = max(3, 1500 // (kr * kc))
    cases = [(xsb.I64, 1, False), (xsb.I32, 0, True), (xsb.I32, 1, False), (xsb.I64, 0, True)]
    for (idx, base, device), (m, n) in zip(cases, [(530, 230), (230, 530), (530, 230), (230, 530)]):
        # tall (rows beyond n) and wide (columns beyond m)
        dt = np.int64 if idx == xsb.I64 else np.int32
        h = xsb.Handle(m, n, idx_type=idx, index_base=base)
        ref = xsb.Handle(m, n, idx_type=idx, index_base=base)
        ora = oracle.OracleExt(m, n)
        for step in range(2):  # element batches with plain batches between them, then spliced onto the resident CSC
            for fl in (xsb.RAW, xsb.UPDATE, xsb.ASSIGN):
                rd, cd, A = random_rect(rng, m, n, ncells, kr, kc, base)
                rd, cd = rd.astype(dt), cd.astype(dt)
                I, J, V = expand(rd, cd, A)
                if device:
                    h.insert_elements(to_dev(torch, rd), to_dev(torch, A), fl, col_dofs=to_dev(torch, cd))
                else:
                    h.insert_elements(rd, A, fl, col_dofs=cd)
                ref.insert_batch(I, J, V, fl)
                ora.insert_batch(I.astype(np.int64) + (1 - base), J.astype(np.int64) + (1 - base), V, fl)
                Ib = rng.integers(base, m + base, 50).astype(dt)
                Jb = rng.integers(base, n + base, 50).astype(dt)
                Vb = rng.standard_normal(50)
                h.insert_batch(Ib, Jb, Vb, xsb.UPDATE)
                ref.insert_batch(Ib, Jb, Vb, xsb.UPDATE)
                ora.insert_batch(Ib.astype(np.int64) + (1 - base), Jb.astype(np.int64) + (1 - base), Vb, xsb.UPDATE)
            assert h.pending == ref.pending
            h.flush()
            ref.flush()
            got = h.fetch_csc_numpy()
            assert_same(got, ref.fetch_csc_numpy())
            ocp, orv, onz = ora.csc()
            assert_same(got, (ocp - 1 + base, orv - 1 + base, onz))


@pytest.mark.parametrize("precount", [True, False])
@pytest.mark.parametrize("k", [1, 4, 9, 64])
def test_square_call_is_the_same_loop(xsb, precount, k):
    """kr == kc with one connectivity for rows and columns stages what xsb_insert_elements stages -- through the same
    array and through an equal copy -- and flushes to the same CSC."""
    rng = np.random.default_rng(k)
    n = 300
    dofs = window_dofs(rng, n, max(4, 3000 // (k * k)), k) + 1
    A = element_values(rng, len(dofs), k, k)
    handles = [xsb.Handle(n, n) for _ in range(3)]
    for h in handles:
        h.set_precount(precount)
    handles[0].insert_elements(dofs, A, xsb.UPDATE)
    handles[1].insert_elements(dofs, A, xsb.UPDATE, col_dofs=dofs)
    handles[2].insert_elements(dofs, A, xsb.UPDATE, col_dofs=dofs.copy())
    staged = [h.debug_fetch_staged() for h in handles]
    for s in staged[1:]:
        for x, y in zip(staged[0], s):
            assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8))
    for h in handles:
        h.flush()
    for h in handles[1:]:
        assert_same(h.fetch_csc_numpy(), handles[0].fetch_csc_numpy())


@pytest.mark.parametrize("precount", [True, False])
@pytest.mark.parametrize("kr,kc", [(16, 16), (64, 32), (5, 9)])
def test_repeated_dofs(xsb, oracle, precount, kr, kc):
    """Repeats inside an element's row list and inside its column list.  Elements 16 .. 23 name one column dof kc
    times: (16, 16) gives a full chunk of eight such elements, 2048 records of one column; (64, 32) two elements per
    chunk, 2048 records of one column from one element -- more than one run of the grouped flush holds (2047).  The
    matrix stays small and poor enough for the grouped flush, so that it reads what the producer published."""
    m, n, ncells = 48, 40, 64
    rng = np.random.default_rng(kr * kc)
    rdofs = (np.arange(ncells)[:, None] + np.arange(kr)[None, :] % 3) % m + 1
    cdofs = (np.arange(ncells)[:, None] + np.arange(kc)[None, :] % 2) % n + 1
    cdofs[16:24] = 23
    rdofs[30, :] = 7
    A = rng.standard_normal((ncells, kc, kr))
    A[rng.random(A.shape) < 0.1] = 0.0
    h = xsb.Handle(m, n)
    h.set_precount(precount)
    h.insert_elements(rdofs, A, xsb.RAW, col_dofs=cdofs)
    h.flush()
    ora = oracle.OracleExt(m, n)
    ora.insert_batch(*expand(rdofs, cdofs, A), oracle.RAW)
    assert_same(h.fetch_csc_numpy(), ora.csc())
    st = h.flush_stats()
    assert st["column_path"] == 4
    if precount:
        assert st["precounted"] > 0.99
    h.insert_elements(rdofs[::-1].copy(), -A, xsb.UPDATE, col_dofs=cdofs[::-1].copy())  # onto the resident matrix
    h.flush()
    ora.insert_batch(*expand(rdofs[::-1].copy(), cdofs[::-1].copy(), -A), oracle.UPDATE)
    assert_same(h.fetch_csc_numpy(), ora.csc())


def test_staged_order_is_the_call_order(xsb):
    rng = np.random.default_rng(3)
    m, n, kr, kc = 70, 110, 5, 3
    rd, cd, A = random_rect(rng, m, n, 77, kr, kc)
    h = xsb.Handle(m, n)
    h.set_precount(False)
    h.insert_elements(rd, A, xsb.UPDATE, col_dofs=cd)
    I, J, V, F = h.debug_fetch_staged()
    I0, J0, V0 = expand(rd, cd, A)
    assert np.array_equal(I, I0) and np.array_equal(J, J0)
    assert np.array_equal(bits(V), bits(V0))


def test_bounds(xsb, oracle):
    rng = np.random.default_rng(11)
    m, n, kr, kc = 120, 200, 3, 5  # a row dof in [m, n) would be a good column dof, and the other way round
    rd, cd, A = random_rect(rng, m, n, 500, kr, kc)
    h = xsb.Handle(m, n)
    h.insert_elements(rd[:250], A[:250], xsb.RAW, col_dofs=cd[:250])  # a grouped batch ahead of the rejected ones
    before = h.pending
    for c, what, bad in [(37, "row", m + 1), (301, "column", n + 1), (88, "row", 0), (499, "column", -4)]:
        r2, c2 = rd.copy(), cd.copy()
        (r2 if what == "row" else c2)[c, 1] = bad
        if c + 1 < len(rd):  # a later offending element does not hide the first
            r2[c + 1, 0] = m + 7
            c2[c + 1, 0] = n + 7
        with pytest.raises(IndexError, match=f"element {c} of the batch has a {what} dof"):
            h.insert_elements(r2, A, xsb.RAW, col_dofs=c2)
        assert h.pending == before
    h.insert_elements(rd[250:], A[250:], xsb.RAW, col_dofs=cd[250:])
    h.flush()
    ora = oracle.OracleExt(m, n)
    ora.insert_batch(*expand(rd, cd, A), oracle.RAW)
    assert_same(h.fetch_csc_numpy(), ora.csc())
    for kr2, kc2 in [(0, 4), (4, 0), (65, 4), (4, 65)]:
        with pytest.raises(xsb.XsbError) as e:
            h.insert_elements(np.ones((3, kr2), np.int64), np.zeros((3, kc2, kr2)), xsb.RAW,
                              col_dofs=np.ones((3, kc2), np.int64))
        assert e.value.code == xsb.capi.EINVAL
        with pytest.raises(xsb.XsbError) as e:
            h.freeze_elements(np.ones((3, kr2), np.int64), col_dofs=np.ones((3, kc2), np.int64))
        assert e.value.code == xsb.capi.EINVAL


def test_multi_partition_handle(xsb, oracle):
    rng = np.random.default_rng(5)
    m, n, kr, kc, parts = 90, 150, 4, 6, 3
    h = xsb.Handle(m, n, n_tid=parts)
    ref = xsb.Handle(m, n, n_tid=parts)
    ora = oracle.OracleMT(m, n, parts)
    batches = []
    for t in range(parts):
        rd, cd, A = random_rect(rng, m, n, 120, kr, kc)
        fl = (xsb.RAW, xsb.UPDATE)[t % 2]
        h.insert_elements(rd, A, fl, tid=t, col_dofs=cd)
        ref.insert_batch(*expand(rd, cd, A), fl, tid=t)
        ora.insert_batch(*expand(rd, cd, A), tid=t + 1, flavour=fl)
        batches.append((rd, cd))
    h.flush()
    ref.flush()
    ora.flush()
    assert_same(h.fetch_csc_numpy(), ora.csc())
    assert_same(h.fetch_csc_numpy(), ref.fetch_csc_numpy())
    # setindex! of positions already in the CSC is accepted, like xsb_insert_batch of the same calls ...
    A2 = rng.standard_normal((40, kc, kr))
    rd, cd = batches[0][0][:40], batches[0][1][:40]
    h.insert_elements(rd, A2, xsb.ASSIGN, tid=2, col_dofs=cd)
    ref.insert_batch(*expand(rd, cd, A2), xsb.ASSIGN, tid=2)
    h.flush()
    ref.flush()
    assert_same(h.fetch_csc_numpy(), ref.fetch_csc_numpy())
    # ... a new position is an error (genericmt...:63-68)
    with pytest.raises(xsb.capi.XsbIllegalError):
        h.insert_elements(np.array([[1, m, 2, m - 1]], np.int64), np.ones((1, 2, 4)), xsb.ASSIGN, tid=1,
                          col_dofs=np.array([[n, 1]], np.int64))
    assert h.pending == 0


@pytest.mark.parametrize("world", [2, 3])
def test_slab_handles(xsb, torch, world):
    from tests.test_gpu_dist import route_and_flush

    rng = np.random.default_rng(world)
    m, n, kr, kc = 180, 240, 4, 12
    splits = [0, 100, 240] if world == 2 else [0, 70, 71, 240]
    handles = [xsb.Handle(m, n, slab=(world, r, splits)) for r in range(world)]
    single = xsb.Handle(m, n)
    for splice in range(2):
        for r in range(world):  # rank r assembles elements of every slab; the single handle sees the ranks in order
            rd, cd, A = random_rect(rng, m, n, 150 + 30 * r, kr, kc)
            fl = (xsb.RAW, xsb.UPDATE)[(splice + r) % 2]
            if r % 2:
                handles[r].insert_elements(to_dev(torch, rd), to_dev(torch, A), fl, col_dofs=to_dev(torch, cd))
            else:
                handles[r].insert_elements(rd, A, fl, col_dofs=cd)
            single.insert_elements(rd, A, fl, col_dofs=cd)
        route_and_flush(xsb, torch, handles)
        single.flush()
        cp, rv, nz = single.fetch_csc_numpy()
        for r in range(world):
            lcp, lrv, lnz = handles[r].fetch_csc_numpy()
            lo, hi = splits[r], splits[r + 1]
            assert np.array_equal(lcp - 1, cp[lo:hi + 1] - cp[lo])
            assert np.array_equal(lrv, rv[cp[lo] - 1:cp[hi] - 1])
            assert np.array_equal(bits(lnz), bits(nz[cp[lo] - 1:cp[hi] - 1]))


@pytest.mark.parametrize("kr,kc", [(1, 4), (4, 1), (12, 4)])
def test_freeze_from_rect_elements(xsb, torch, kr, kc):
    rng = np.random.default_rng(9 + kr)
    m, n = (300, 200) if kr > kc else (200, 300)
    rd, cd, A1 = random_rect(rng, m, n, 700, kr, kc)
    A2 = rng.standard_normal(A1.shape)
    A2[:, 0, 0] = 0.0

    def assembled(*steps):
        g = xsb.Handle(m, n)
        for s in steps:
            if s is None:
                g.zero_values()
            else:
                g.insert_elements(rd, s, xsb.RAW, col_dofs=cd)
                g.flush()
        return g.fetch_csc_numpy()

    onto = assembled(A1, A2)
    zeroed = assembled(A1, None, A2)
    h = xsb.Handle(m, n)
    h.insert_elements(rd, A1, xsb.RAW, col_dofs=cd)
    h.flush()
    h.freeze_elements(to_dev(torch, rd), col_dofs=to_dev(torch, cd))
    h.reassemble_values(A2.reshape(-1))  # the element matrices as they are: V = vec(Aloc)
    assert_same(h.fetch_csc_numpy(), onto)
    h.unfreeze()
    h.freeze_elements(rd, col_dofs=cd)
    for _ in range(2):  # deterministic: the same bits every time
        h.reassemble_values(A2.reshape(-1), zero_first=True)
        assert_same(h.fetch_csc_numpy(), zeroed)
    h.reassemble_values(A2.reshape(-1), mode=xsb.FAST, zero_first=True)
    cp, rv, nz = h.fetch_csc_numpy()
    assert np.array_equal(cp, zeroed[0]) and np.array_equal(rv, zeroed[1])
    assert np.allclose(nz, zeroed[2], rtol=1e-14, atol=1e-14 * np.abs(zeroed[2]).max())
    # a position the pattern does not hold: a row that column 1 lacks; a dof outside the matrix
    absent = min(set(range(1, m + 1)) - set(rv[cp[0] - 1:cp[1] - 1].tolist()))
    with pytest.raises(xsb.capi.XsbIllegalError):
        h.freeze_elements(np.concatenate([rd, np.full((1, kr), absent)]),
                          col_dofs=np.concatenate([cd, np.ones((1, kc), np.int64)]))
    bad = cd.copy()
    bad[3, 0] = n + 1
    with pytest.raises(IndexError):
        h.freeze_elements(rd, col_dofs=bad)


@pytest.mark.parametrize("world,splits", [(2, [0, 50, 110]), (3, [0, 30, 31, 110])])
def test_slab_freeze_of_rect_elements(xsb, torch, world, splits):
    """The slab freeze of every rank's rectangular element loop equals one plain handle that froze the concatenated
    streams, bit for bit, step after step."""
    from tests.test_gpu_dist_values import check_slabs, freeze_all, route_and_flush, signed_values, step_all

    m, n, kr, kc = 80, 110, 3, 5
    rng = np.random.default_rng(world)
    conn = [random_rect(rng, m, n, 40 + 9 * r, kr, kc)[:2] for r in range(world)]
    handles = [xsb.Handle(m, n, slab=(world, r, splits)) for r in range(world)]
    P = xsb.Handle(m, n)
    for h, (rd, cd) in zip(handles, conn):
        ones = np.ones((len(rd), kc, kr))
        h.insert_elements(rd, ones, col_dofs=cd)
        P.insert_elements(rd, ones, col_dofs=cd)
    route_and_flush(torch, handles)
    P.flush()
    freeze_all(torch, handles, [(lambda h=h, c=c: h.freeze_slab_elements(c[0], col_dofs=c[1]))
                                for h, c in zip(handles, conn)])
    P.freeze_elements(np.concatenate([c[0] for c in conn]), col_dofs=np.concatenate([c[1] for c in conn]))
    for zero_first in (True, False):
        Vs = [signed_values(rng, len(c[0]) * kr * kc) for c in conn]
        step_all(torch, handles, Vs, 0, zero_first)
        P.reassemble_values(np.concatenate(Vs), zero_first=zero_first)
        pcp, _, pnz = P.fetch_csc_numpy()
        check_slabs(handles, splits, pcp, pnz)


def test_matrix_wrapper(xsb, oracle):
    """ExtendableSparseMatrix.insert_elements takes col_dofs."""
    from xsparse_b200.matrix import ExtendableSparseMatrix

    rng = np.random.default_rng(21)
    m, n, kr, kc = 60, 45, 4, 2
    rd, cd, A = random_rect(rng, m, n, 80, kr, kc)
    M = ExtendableSparseMatrix(m, n)
    M.insert_elements(rd, A, col_dofs=cd)
    ora = oracle.OracleExt(m, n)
    ora.insert_batch(*expand(rd, cd, A), oracle.RAW)
    assert_same(M.csc(), ora.csc())
    with pytest.raises(ValueError):
        M.insert_elements(rd, A.transpose(0, 2, 1).copy(), col_dofs=cd)  # (ncells, kr, kc): the wrong order


def test_fem_p0_p1_device(xsb, oracle, torch):
    """A P0 x P1 operator (kr = 1, kc = 4) on the Kuhn mesh of the oracle, device connectivity, against device
    triplets of the expanded stream."""
    nx = 24
    _, J, _ = oracle.fem_stream(nx, nx, nx)
    cd = np.ascontiguousarray(J.reshape(-1, 4, 5)[:, 0, 1:5]).astype(np.int64)
    ncells = len(cd)
    rd = np.arange(1, ncells + 1, dtype=np.int64)[:, None]
    A = np.random.default_rng(1).standard_normal((ncells, 4, 1))
    h = xsb.Handle(ncells, nx ** 3)
    h.insert_elements(to_dev(torch, rd), to_dev(torch, A), xsb.RAW, col_dofs=to_dev(torch, cd))
    h.flush()
    I, Jx, V = expand(rd, cd, A)
    T = np.zeros(len(V), dtype=[("r", np.uint32), ("c", np.uint32), ("v", np.float64)])
    T["r"], T["c"], T["v"] = I, Jx, V
    g = xsb.Handle(ncells, nx ** 3)
    g.insert_triplets(to_dev(torch, T.view(np.int64)), xsb.RAW, 0, len(V))
    g.flush()
    assert_same(h.fetch_csc_numpy(), g.fetch_csc_numpy())
