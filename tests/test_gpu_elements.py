"""GPU tests of element-by-element insertion (xsb_insert_elements / xsb_freeze_elements): connectivity plus dense
element matrices stage exactly the call stream of the element loop (test/femtools.jl:45-72), and give the CSC that
xsb_insert_batch of the expanded stream and the CPU oracle give, bit for bit."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


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


def expand(dofs, Aloc):
    """The call stream of the element loop: call k^2 c + k jl + il = (dofs[c, il], dofs[c, jl], Aloc[c, jl, il])."""
    dofs = np.asarray(dofs)
    nc, k = dofs.shape
    I = np.broadcast_to(dofs[:, None, :], (nc, k, k)).reshape(-1).copy()
    J = np.broadcast_to(dofs[:, :, None], (nc, k, k)).reshape(-1).copy()
    return I, J, np.ascontiguousarray(Aloc, np.float64).reshape(-1).copy()


def assert_same(got, ref):
    cp, rv, nz = got
    ocp, orv, onz = ref
    assert np.array_equal(cp, ocp), "colptr differs"
    assert np.array_equal(rv, orv), "rowval differs"
    bad = np.nonzero(bits(nz) != bits(onz))[0]
    assert bad.size == 0, f"{bad.size} nzval entries differ, first at {bad[:5]}"


def random_elements(rng, n, ncells, k, base=1, repeat=False):
    """Elements of k dofs near a moving window (neighbours share columns); values with exact zeros and entries that
    cancel: small halves and their negatives next to Gaussian noise."""
    lo = (np.arange(ncells) * max(1, n // max(ncells, 1)))[:, None]
    dofs = (lo + rng.integers(0, 3 * k + 2, (ncells, k))) % n
    if not repeat:  # distinct dofs inside an element (the common mesh case); repeats get their own test
        for c in range(ncells):
            if len(set(dofs[c].tolist())) < k:
                dofs[c] = (lo[c, 0] + rng.permutation(max(3 * k + 2, k))[:k]) % n
    A = rng.choice(np.array([-1.5, -1.0, -0.5, 0.0, 0.5, 1.0, 1.5]), (ncells, k, k))
    noisy = rng.random(ncells) < 0.5
    A[noisy] = rng.standard_normal((int(noisy.sum()), k, k))
    A[rng.random((ncells, k, k)) < 0.1] = 0.0
    return (dofs + base).astype(np.int64), A


def to_dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("k", [1, 2, 3, 4, 8, 10, 16, 27, 64])
def test_random_connectivity_matches_batch_and_oracle(xsb, oracle, torch, k):
    rng = np.random.default_rng(k)
    for idx, base, device in [(xsb.I64, 1, False), (xsb.I32, 0, True), (xsb.I32, 1, False), (xsb.I64, 0, True)]:
        n = 400 + 13 * k
        dt = np.int64 if idx == xsb.I64 else np.int32
        h = xsb.Handle(n, n, idx_type=idx, index_base=base)
        ref = xsb.Handle(n, n, idx_type=idx, index_base=base)
        ora = oracle.OracleExt(n, n)
        for step in range(3):  # element batches with plain batches between them, then splices onto the resident CSC
            for fl in (xsb.RAW, xsb.UPDATE, xsb.ASSIGN):
                dofs, A = random_elements(rng, n, max(1, 600 // k), k, base)
                dofs = dofs.astype(dt)
                I, J, V = expand(dofs, A)
                if device:
                    h.insert_elements(to_dev(torch, dofs), to_dev(torch, A), fl)
                else:
                    h.insert_elements(dofs, A, fl)
                ref.insert_batch(I, J, V, fl)
                ora.insert_batch(I.astype(np.int64) + (1 - base), J.astype(np.int64) + (1 - base), V, fl)
                Ib = rng.integers(base, n + base, 50).astype(dt)
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
@pytest.mark.parametrize("k", [2, 5, 16, 32, 46, 64])
def test_repeated_dofs_inside_an_element(xsb, oracle, precount, k):
    """Periodic identification / collapsed nodes: an element may name a dof several times.  Elements 16 .. 23 name
    one dof k times each: a column then holds up to (elements of the chunk) x k^2 records of a chunk -- k = 16: a
    full chunk of eight such elements, 2048 records; k = 32: two of them; k = 46, 64: one element is already more than
    2047 records -- which is more than one run of the grouped flush holds."""
    rng = np.random.default_rng(7 + k)
    n = 60 + 3 * k
    dofs, A = random_elements(rng, n, 300 if k < 32 else 60, k, repeat=True)
    dofs[16:24] = 23
    dofs[40, 1:3] = dofs[40, 0]
    h = xsb.Handle(n, n)
    h.set_precount(precount)
    h.insert_elements(dofs, A, xsb.RAW)
    h.insert_elements(dofs[::-1].copy(), -A, xsb.UPDATE)  # and a second batch on top, staged behind the first
    h.flush()
    ora = oracle.OracleExt(n, n)
    ora.insert_batch(*expand(dofs, A), oracle.RAW)
    ora.insert_batch(*expand(dofs[::-1].copy(), -A), oracle.UPDATE)
    assert_same(h.fetch_csc_numpy(), ora.csc())


@pytest.mark.parametrize("precount", [True, False])
@pytest.mark.parametrize("k", [16, 32, 46, 64])
def test_long_runs_take_the_grouped_flush(xsb, oracle, precount, k):
    """Columns with more than 2047 records in one chunk (one run of the grouped flush holds at most 2047) on a matrix
    whose columns stay short and poor enough for the grouped flush, so that it reads what the producer published.
    Element c names the dofs c and c + 1, k / 2 times each: k = 46, 64 give a column k^2 records in a chunk; elements
    16 .. 23 name one dof k times: k = 16 (a full chunk of them) 2048 records, k = 32 4096."""
    n, ncells = 40, 64
    rng = np.random.default_rng(k)
    dofs = (np.arange(ncells)[:, None] + np.arange(k)[None, :] % 2) % n + 1
    dofs[16:24] = 23
    A = rng.standard_normal((ncells, k, k))
    A[rng.random(A.shape) < 0.1] = 0.0
    h = xsb.Handle(n, n)
    h.set_precount(precount)
    h.insert_elements(dofs, A, xsb.RAW)
    h.flush()
    ora = oracle.OracleExt(n, n)
    ora.insert_batch(*expand(dofs, A), oracle.RAW)
    assert_same(h.fetch_csc_numpy(), ora.csc())
    st = h.flush_stats()
    assert st["column_path"] == 4
    if precount:
        assert st["precounted"] > 0.99
    h.insert_elements(dofs, -A, xsb.UPDATE)  # the same onto the resident matrix
    h.flush()
    ora.insert_batch(*expand(dofs, -A), oracle.UPDATE)
    assert_same(h.fetch_csc_numpy(), ora.csc())


def test_staged_order_is_the_call_order(xsb):
    rng = np.random.default_rng(3)
    n, k = 90, 6
    dofs, A = random_elements(rng, n, 77, k)
    h = xsb.Handle(n, n)
    h.set_precount(False)
    h.insert_elements(dofs, A, xsb.UPDATE)
    h.insert_elements(dofs[:5], -A[:5], xsb.ASSIGN)
    I, J, V, F = h.debug_fetch_staged()
    I0, J0, V0 = expand(dofs, A)
    I1, J1, V1 = expand(dofs[:5], -A[:5])
    assert np.array_equal(I, np.concatenate([I0, I1])) and np.array_equal(J, np.concatenate([J0, J1]))
    assert np.array_equal(bits(V), bits(np.concatenate([V0, V1])))
    assert np.array_equal(F, np.array([xsb.UPDATE] * len(V0) + [xsb.ASSIGN] * len(V1), np.int32))


def fem_elements(oracle, nx):
    """The Kuhn mesh stream of the oracle in element form: node jl of tetrahedron t is the column of its calls
    20 t + 1 + jl, its element matrix the stiffness calls (the mass terms are dropped)."""
    I, J, V = oracle.fem_stream(nx, nx, nx)
    J4 = J.reshape(-1, 4, 5)
    V4 = V.reshape(-1, 4, 5)  # call 20 t + 5 il + w
    dofs = np.ascontiguousarray(J4[:, 0, 1:5])
    A = np.ascontiguousarray(V4[:, :, 1:5].transpose(0, 2, 1))  # [t, jl, il] = V[20 t + 5 il + 1 + jl]
    return dofs, A


def test_kuhn_mesh_takes_the_grouped_path(xsb, oracle):
    nx = 30
    dofs, A = fem_elements(oracle, nx)
    n = nx ** 3
    h = xsb.Handle(n, n)
    h.insert_elements(dofs, A, xsb.RAW)
    h.flush()
    st = h.flush_stats()
    assert st["column_path"] == 4 and st["precounted"] > 0.99
    ora = oracle.OracleExt(n, n)
    ora.insert_batch(*expand(dofs, A), oracle.RAW)
    assert_same(h.fetch_csc_numpy(), ora.csc())


def test_bounds(xsb, oracle):
    rng = np.random.default_rng(11)
    n, k = 200, 4
    dofs, A = random_elements(rng, n, 500, k)
    h = xsb.Handle(n, n)
    h.insert_elements(dofs[:250], A[:250], xsb.RAW)  # a grouped batch ahead of the rejected one
    before = h.pending
    for c, bad in [(37, n + 1), (301, 0), (499, -4)]:
        d = dofs.copy()
        d[c, 2] = bad
        d[c + 1 if c + 1 < len(d) else c, 0] = n + 7  # a later offending element does not hide the first
        with pytest.raises(IndexError, match=f"element {c} "):
            h.insert_elements(d, A, xsb.RAW)
        assert h.pending == before
    h.insert_elements(dofs[250:], A[250:], xsb.RAW)
    h.flush()
    ora = oracle.OracleExt(n, n)
    ora.insert_batch(*expand(dofs, A), oracle.RAW)
    assert_same(h.fetch_csc_numpy(), ora.csc())
    for kk in (0, 65):
        with pytest.raises(xsb.XsbError) as e:
            h.insert_elements(np.ones((3, kk), np.int64), np.zeros((3, kk, kk)), xsb.RAW)
        assert e.value.code == xsb.capi.EINVAL
        with pytest.raises(xsb.XsbError) as e:
            h.freeze_elements(np.ones((3, kk), np.int64))
        assert e.value.code == xsb.capi.EINVAL


def test_multi_partition_handle(xsb, oracle):
    rng = np.random.default_rng(5)
    n, k, parts = 150, 4, 3
    h = xsb.Handle(n, n, n_tid=parts)
    ref = xsb.Handle(n, n, n_tid=parts)
    ora = oracle.OracleMT(n, n, parts)
    batches = []
    for t in range(parts):
        dofs, A = random_elements(rng, n, 120, k)
        fl = (xsb.RAW, xsb.UPDATE)[t % 2]
        h.insert_elements(dofs, A, fl, tid=t)
        ref.insert_batch(*expand(dofs, A), fl, tid=t)
        ora.insert_batch(*expand(dofs, A), tid=t + 1, flavour=fl)
        batches.append(dofs)
    h.flush()
    ref.flush()
    ora.flush()
    assert_same(h.fetch_csc_numpy(), ora.csc())
    # setindex! of positions already in the CSC (the rawupdateindex! batch of tid 0 stored all of its positions) is
    # accepted, like xsb_insert_batch of the same calls ...
    A2 = rng.standard_normal((40, k, k))
    h.insert_elements(batches[0][:40], A2, xsb.ASSIGN, tid=2)
    ref.insert_batch(*expand(batches[0][:40], A2), xsb.ASSIGN, tid=2)
    h.flush()
    ref.flush()
    assert_same(h.fetch_csc_numpy(), ref.fetch_csc_numpy())
    # ... a new position is an error (genericmt...:63-68)
    fresh = np.array([[1, n, 2, n - 1]], np.int64)
    with pytest.raises(xsb.capi.XsbIllegalError):
        h.insert_elements(fresh, np.ones((1, k, k)), xsb.ASSIGN, tid=1)
    assert h.pending == 0


@pytest.mark.parametrize("world", [2, 3])
def test_slab_handles(xsb, oracle, torch, world):
    from tests.test_gpu_dist import route_and_flush

    rng = np.random.default_rng(world)
    n, k = 240, 4
    splits = [0, 100, 240] if world == 2 else [0, 70, 71, 240]
    handles = [xsb.Handle(n, n, slab=(world, r, splits)) for r in range(world)]
    single = xsb.Handle(n, n)
    for splice in range(2):
        for r in range(world):  # rank r assembles elements of every slab; the single handle sees the ranks in order
            dofs, A = random_elements(rng, n, 200 + 30 * r, k)
            fl = (xsb.RAW, xsb.UPDATE)[(splice + r) % 2]
            handles[r].insert_elements(to_dev(torch, dofs) if r % 2 else dofs, A, fl)
            single.insert_elements(dofs, A, fl)
        route_and_flush(xsb, torch, handles)
        single.flush()
        cp, rv, nz = single.fetch_csc_numpy()
        for r in range(world):
            lcp, lrv, lnz = handles[r].fetch_csc_numpy()
            lo, hi = splits[r], splits[r + 1]
            assert np.array_equal(lcp - 1, cp[lo:hi + 1] - cp[lo])
            assert np.array_equal(lrv, rv[cp[lo] - 1:cp[hi] - 1])
            assert np.array_equal(bits(lnz), bits(nz[cp[lo] - 1:cp[hi] - 1]))


def test_freeze_from_elements(xsb, oracle):
    rng = np.random.default_rng(9)
    n, k = 300, 4
    dofs, A1 = random_elements(rng, n, 700, k)
    A2 = rng.standard_normal(A1.shape)
    A2[:, 0, 0] = 0.0

    def assembled(*steps):
        g = xsb.Handle(n, n)
        for s in steps:
            if s is None:
                g.zero_values()
            else:
                g.insert_elements(dofs, s, xsb.RAW)
                g.flush()
        return g.fetch_csc_numpy()

    onto = assembled(A1, A2)
    zeroed = assembled(A1, None, A2)
    h = xsb.Handle(n, n)
    h.insert_elements(dofs, A1, xsb.RAW)
    h.flush()
    first = h.fetch_csc_numpy()
    h.freeze_elements(dofs)
    h.reassemble_values(A2.reshape(-1))  # the element matrices as they are: V = vec(Aloc)
    assert_same(h.fetch_csc_numpy(), onto)
    for _ in range(2):  # deterministic: the same bits every time
        h.reassemble_values(A2.reshape(-1), zero_first=True)
        assert_same(h.fetch_csc_numpy(), zeroed)
    h.reassemble_values(A2.reshape(-1), mode=xsb.FAST, zero_first=True)
    cp, rv, nz = h.fetch_csc_numpy()
    assert np.array_equal(cp, zeroed[0]) and np.array_equal(rv, zeroed[1])
    assert np.allclose(nz, zeroed[2], rtol=1e-14, atol=1e-14 * np.abs(zeroed[2]).max())
    assert np.array_equal(first[0], cp)
    # a position the pattern does not hold
    far = np.array([[1, n, 2, 3]], np.int64)
    with pytest.raises(xsb.capi.XsbIllegalError):
        h.freeze_elements(np.concatenate([dofs, far]))
    bad = dofs.copy()
    bad[3, 1] = n + 1
    with pytest.raises(IndexError):
        h.freeze_elements(bad)


def fem128_on_device(xsb, torch, nx):
    """FEM nx^3 in element form, resident in HBM: generated by the emitter, staged in call order, converted."""
    n = nx ** 3
    g = xsb.Handle(n, n)
    g.set_precount(False)
    g.emit_p1fem(nx, nx, nx, flavour=xsb.RAW)
    cnt = g.pending
    dJ = torch.empty(cnt, dtype=torch.int64, device="cuda")
    dI = torch.empty_like(dJ)
    dV = torch.empty(cnt, dtype=torch.float64, device="cuda")
    got = C.c_int64(0)
    c = xsb.capi
    c.check(c.lib().xsb_debug_fetch_staged(g._h, 0, dI.data_ptr(), dJ.data_ptr(), dV.data_ptr(), None, cnt,
                                           C.byref(got)), g._h)
    g.close()
    del dI
    dofs = dJ.view(-1, 4, 5)[:, 0, 1:5].contiguous()
    del dJ
    A = dV.view(-1, 4, 5)[:, :, 1:5].transpose(1, 2).contiguous()
    del dV
    return dofs, A


def test_full_size_fem128(xsb, torch):
    nx = 128
    n = nx ** 3
    dofs, A = fem128_on_device(xsb, torch, nx)
    ncells, k = dofs.shape
    assert (ncells, k) == (12290298, 4)
    h = xsb.Handle(n, n)
    h.insert_elements(dofs, A, xsb.RAW)
    h.flush()
    assert h.flush_stats()["column_path"] == 4
    # the expanded 196.6 M-call stream as 16-byte device triplets {u32 row, u32 col, f64 val}
    T = torch.empty((ncells, k, k, 2), dtype=torch.int64, device="cuda")
    T[..., 0] = dofs[:, None, :] | (dofs[:, :, None] << 32)
    T[..., 1] = A.view(torch.int64)
    del A
    g = xsb.Handle(n, n)
    g.insert_triplets(T, xsb.RAW, 0, ncells * k * k)
    del T
    g.flush()
    assert g.nnz == h.nnz
    for x, y in zip(device_csc(torch, h), device_csc(torch, g)):
        assert torch.equal(x.view(torch.int64), y.view(torch.int64))


def device_csc(torch, h):
    nnz = h.nnz
    cp = torch.empty(h.n + 1, dtype=torch.int64, device="cuda")
    rv = torch.empty(nnz, dtype=torch.int64, device="cuda")
    nz = torch.empty(nnz, dtype=torch.float64, device="cuda")
    h.fetch_csc(cp, rv, nz)
    h.synchronize()
    return cp, rv, nz
