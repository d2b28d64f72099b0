"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same
seeded inputs.  Bar: colptr/rowval bit-exact; nzval bit-exact in deterministic mode and
within 1e-14 relative in fast mode.  Cases follow the reference's own tests (SURVEY.md 4)."""
import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def xsb():
    import __graft_entry__ as ge

    ge.build()
    import xsparse_b200

    assert xsparse_b200.capi.device_count() > 0, "no CUDA device: GPU tests need the real extension on a GPU"
    return xsparse_b200


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def assert_csc_equal(got, ref, exact=True, rtol=1e-14):
    cp, rv, nz = got
    ocp, orv, onz = ref
    assert np.array_equal(cp, ocp), "colptr differs"
    assert np.array_equal(rv, orv), "rowval differs"
    if exact:
        bad = np.nonzero(bits(nz) != bits(onz))[0]
        assert bad.size == 0, f"{bad.size} nzval entries not bit-exact, first at {bad[:5]}: {nz[bad[:5]]} vs {onz[bad[:5]]}"
    else:
        assert np.allclose(nz, onz, rtol=rtol, atol=0.0)


# ---------------------------------------------------------------- known-answer tests
def test_micro_vector(xsb):
    """SURVEY.md 8(c')."""
    h = xsb.Handle(3, 3)
    I = np.array([2, 3, 2, 1], np.int64)
    J = np.array([1, 1, 1, 2], np.int64)
    V = np.array([1.0, 2.0, 0.5, 0.0])
    h.insert_batch(I, J, V, xsb.UPDATE)
    h.insert_batch(np.array([1], np.int64), np.array([3], np.int64), np.array([0.0]), xsb.RAW)
    nnz, changed = h.flush()
    assert (nnz, changed) == (3, True)
    cp, rv, nz = h.fetch_csc_numpy()
    assert cp.tolist() == [1, 3, 3, 4] and rv.tolist() == [2, 3, 1] and nz.tolist() == [1.5, 2.0, 0.0]
    h.insert_batch(np.array([2, 1], np.int64), np.array([1, 1], np.int64), np.array([-1.5, 4.0]), xsb.UPDATE)
    nnz, changed = h.flush()
    assert (nnz, changed) == (4, True)
    cp, rv, nz = h.fetch_csc_numpy()
    assert cp.tolist() == [1, 4, 4, 5] and rv.tolist() == [1, 2, 3, 1] and nz.tolist() == [4.0, 0.0, 2.0, 0.0]
    # values-only update: pattern (phash) unchanged
    h.insert_batch(np.array([1], np.int64), np.array([1], np.int64), np.array([1.0]), xsb.UPDATE)
    assert h.flush() == (4, False)
    assert h.flush() == (4, False)  # nothing pending: no-op


def test_updates_zero_semantics(xsb):
    """test/test_updates.jl:10-25 through the host mirror."""
    import operator

    A = xsb.ExtendableSparseMatrix(10, 10)
    assert A.nnz == 0
    A[1, 3] = 5
    A.updateindex(operator.add, 6.0, 4, 5)
    A.updateindex(operator.add, 0.0, 2, 3)
    assert A.nnz == 2
    A.rawupdateindex(operator.add, 0.0, 2, 3)
    assert A.nnz == 3
    A.dropzeros()
    assert A.nnz == 2
    A.rawupdateindex(operator.add, 0.1, 2, 3)
    assert A.nnz == 3
    A.dropzeros()
    assert A.nnz == 3
    assert A[1, 3] == 5.0 and A[4, 5] == 6.0 and A[2, 3] == 0.1 and A[7, 7] == 0.0


def test_readme_example(xsb):
    """README.md:15-27 with A[i,j] += v spelled through getindex/setindex!."""
    A = xsb.ExtendableSparseMatrix(10, 10)
    A[1, 1] = 1
    for i in range(1, 10):
        A[i + 1, i] = A[i + 1, i] - 1
        A[i, i + 1] = A[i, i + 1] - 1
        A[i + 1, i + 1] = A[i + 1, i + 1] + 1
        A[i, i] = A[i, i] + 1
    S = A.sparse().toarray()
    T = 2 * np.eye(10) - np.eye(10, k=1) - np.eye(10, k=-1)
    T[9, 9] = 1
    assert A.nnz == 28 and np.array_equal(S, T)


def triplets(xsb, I, J, V):
    T = np.empty(len(V), xsb.capi.TRIPLET_DTYPE)
    T["row"], T["col"], T["val"] = I, J, V
    return T


@pytest.mark.parametrize("where", ["host", "device"])
def test_insert_triplets_equals_insert_batch(xsb, oracle, where):
    """xsb_insert_triplets: the k-th 16-byte triplet is the k-th updateindex!/rawupdateindex!/setindex!
    call (extendable.jl:159-218); host arrays land in the staging buffer and are rewritten in place."""
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(77)
    m, n, cnt = 57, 43, 20000
    I = rng.integers(1, m + 1, cnt)
    J = rng.integers(1, n + 1, cnt)
    V = rng.standard_normal(cnt)
    V[rng.random(cnt) < 0.1] = 0.0
    h = xsb.Handle(m, n)
    A = oracle.OracleExt(m, n)
    for k, fl in enumerate((xsb.UPDATE, xsb.RAW, xsb.ASSIGN, xsb.UPDATE)):
        sl = slice(k * cnt // 4, (k + 1) * cnt // 4)
        T = triplets(xsb, I[sl], J[sl], V[sl])
        if where == "device":
            dT = torch.from_numpy(T.view(np.uint8)).cuda()
            h.insert_triplets(dT, fl, 0, len(T))
        else:
            h.insert_triplets(T, fl)
        if k == 1:  # a (I, J, V) batch between two triplet batches keeps the call order
            h.insert_batch(I[:50], J[:50], V[:50], xsb.UPDATE)
            A.insert_batch(I[sl], J[sl], V[sl], fl)
            A.insert_batch(I[:50], J[:50], V[:50], oracle.UPDATE)
        else:
            A.insert_batch(I[sl], J[sl], V[sl], fl)
        if k == 2:
            h.flush()
            A.flush()
    h.flush()
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())


def test_insert_triplets_fem_stream_and_bounds(xsb, oracle):
    I, J, V = oracle.fem_stream(9, 8, 7)
    n = 9 * 8 * 7
    h = xsb.Handle(n, n)
    h.insert_triplets(triplets(xsb, I, J, V), xsb.RAW)
    assert h.pending == len(V)
    h.flush()
    A = oracle.OracleExt(n, n)
    A.insert_batch(I, J, V, oracle.RAW)
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())
    bad = triplets(xsb, [1, n + 1, 1], [1, 1, 1], [1.0, 1.0, 1.0])
    with pytest.raises(IndexError) as e:
        h.insert_triplets(bad, xsb.UPDATE)
    assert "entry 1" in str(e.value) and h.pending == 0
    for i, j in [(0, 1), (1, 0), (1, n + 1), (2 ** 32 - 1, 1)]:
        with pytest.raises(IndexError):
            h.insert_triplets(triplets(xsb, [i], [j], [1.0]), xsb.RAW)
    assert h.flush()[1] is False
    # 0-based handles: index 0 is valid, n is not
    h0 = xsb.Handle(4, 4, index_base=0)
    h0.insert_triplets(triplets(xsb, [0, 3], [0, 3], [1.0, 2.0]), xsb.UPDATE)
    with pytest.raises(IndexError):
        h0.insert_triplets(triplets(xsb, [4], [0], [1.0]), xsb.UPDATE)
    assert h0.flush() == (2, True)
    cp, rv, nz = h0.fetch_csc_numpy()
    assert cp.tolist() == [0, 1, 1, 1, 2] and rv.tolist() == [0, 3] and nz.tolist() == [1.0, 2.0]


def test_bounds_error_rejects_batch(xsb):
    h = xsb.Handle(4, 5)
    I = np.array([1, 2, 5, 1], np.int64)
    J = np.array([1, 1, 1, 1], np.int64)
    with pytest.raises(IndexError) as e:
        h.insert_batch(I, J, np.ones(4), xsb.UPDATE)
    assert "entry 2" in str(e.value) and h.pending == 0
    for i, j in [(0, 1), (1, 0), (1, 6)]:
        with pytest.raises(IndexError):
            h.insert_batch(np.array([i], np.int64), np.array([j], np.int64), np.ones(1), xsb.RAW)
    h.insert_batch(np.array([4], np.int64), np.array([5], np.int64), np.ones(1), xsb.RAW)
    assert h.flush() == (1, True)


# ---------------------------------------------------------------- random streams
@pytest.mark.parametrize(
    "m,n,xnnz,nsplice",
    [(10, 10, 5, 1), (100, 100, 500, 2), (1000, 1000, 5000, 3), (20, 10, 5, 1), (200, 100, 500, 2),
     (2000, 1000, 5000, 3), (10, 20, 5, 1), (100, 200, 500, 2), (1000, 2000, 5000, 3), (37, 9001, 7000, 5),
     (1, 1, 10, 2), (1, 50, 200, 2), (50, 1, 200, 2), (5000, 7000, 200000, 3)],
)
def test_assembly_random_splices(xsb, oracle, m, n, xnnz, nsplice):
    """test/test_assembly.jl:6-35: sorted columns, equal nnz, exactly equal values, after every splice."""
    rng = np.random.default_rng(1000 * m + n)
    h = xsb.Handle(m, n)
    A = oracle.OracleExt(m, n)
    for _ in range(nsplice):
        I = rng.integers(1, m + 1, xnnz)
        J = rng.integers(1, n + 1, xnnz)
        V = 1.0 + rng.random(xnnz)
        h.insert_batch(I, J, V, xsb.UPDATE)
        A.insert_batch(I, J, V, oracle.UPDATE)
        nnz_before = h.nnz
        nnz, changed = h.flush()
        got = h.fetch_csc_numpy()
        ref = A.csc()
        assert nnz == len(ref[2]) and changed == (nnz != nnz_before)
        assert_csc_equal(got, ref)
        cols = np.repeat(np.arange(n), np.diff(got[0]))
        order = np.lexsort((got[1], cols))
        assert np.array_equal(order, np.arange(len(order)))  # rows strictly sorted per column


@pytest.mark.parametrize("seed", range(6))
def test_mixed_flavours_and_zeros(xsb, oracle, seed):
    """All three insert flavours interleaved, with +0.0/-0.0 values, cancellations and splices."""
    rng = np.random.default_rng(seed)
    m, n = int(rng.integers(5, 60)), int(rng.integers(5, 60))
    h = xsb.Handle(m, n)
    A = oracle.OracleExt(m, n)
    for _ in range(4):
        for _ in range(int(rng.integers(1, 12))):
            cnt = int(rng.integers(1, 400))
            I = rng.integers(1, m + 1, cnt)
            J = rng.integers(1, n + 1, cnt)
            V = rng.choice([0.0, -0.0, 1.0, -1.0, 0.5, 1e-3, 1e30, -1e30], cnt) * rng.choice([1.0, rng.random()], cnt)
            fl = int(rng.integers(0, 3))
            h.insert_batch(I, J, V, fl)
            A.insert_batch(I, J, V, fl)
        h.flush()
        assert_csc_equal(h.fetch_csc_numpy(), A.csc())


def test_cancellation_keeps_entry(xsb, oracle):
    h = xsb.Handle(3, 3)
    A = oracle.OracleExt(3, 3)
    I, J, V = np.array([2, 2], np.int64), np.array([2, 2], np.int64), np.array([1.5, -1.5])
    h.insert_batch(I, J, V, xsb.UPDATE)
    A.insert_batch(I, J, V, oracle.UPDATE)
    assert h.flush() == (1, True)
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())


@pytest.mark.parametrize("idx,base", [(0, 0), (0, 1), (1, 0)])
def test_index_types_and_bases(xsb, oracle, idx, base):
    rng = np.random.default_rng(5)
    m, n, cnt = 300, 200, 5000
    dt = np.int64 if idx == 1 else np.int32
    h = xsb.Handle(m, n, idx_type=idx, index_base=base)
    A = oracle.OracleExt(m, n)
    for _ in range(2):
        I = rng.integers(1, m + 1, cnt)
        J = rng.integers(1, n + 1, cnt)
        V = rng.standard_normal(cnt)
        h.insert_batch((I - 1 + base).astype(dt), (J - 1 + base).astype(dt), V, xsb.RAW)
        A.insert_batch(I, J, V, oracle.RAW)
        h.flush()
        cp, rv, nz = h.fetch_csc_numpy()
        assert cp.dtype == dt and rv.dtype == dt
        assert_csc_equal((cp.astype(np.int64) + 1 - base, rv.astype(np.int64) + 1 - base, nz), A.csc())


def test_device_pointers(xsb, oracle):
    torch = pytest.importorskip("torch")
    rng = np.random.default_rng(9)
    m = n = 4000
    cnt = 300000
    I = rng.integers(1, m + 1, cnt)
    J = rng.integers(1, n + 1, cnt)
    V = rng.standard_normal(cnt)
    h = xsb.Handle(m, n)
    dI, dJ, dV = (torch.from_numpy(x).cuda() for x in (I, J, V))
    torch.cuda.synchronize()
    h.insert_batch(dI, dJ, dV, xsb.UPDATE, count=cnt)
    nnz, _ = h.flush()
    cp = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    rv = torch.empty(nnz, dtype=torch.int64, device="cuda")
    nz = torch.empty(nnz, dtype=torch.float64, device="cuda")
    h.fetch_csc(cp, rv, nz)
    A = oracle.OracleExt(m, n)
    A.insert_batch(I, J, V, oracle.UPDATE)
    assert_csc_equal((cp.cpu().numpy(), rv.cpu().numpy(), nz.cpu().numpy()), A.csc())


# ---------------------------------------------------------------- reference constructors / operations
@pytest.mark.parametrize("seed", range(4))
def test_csc_plus_lnk_is_twice(xsb, seed):
    """test/test_operations.jl:8-13: csc + SparseMatrixLNK(csc) == 2*csc (COMBINE_ADD)."""
    rng = np.random.default_rng(seed)
    m, n = int(rng.integers(1, 400)), int(rng.integers(1, 400))
    S = sp.random(m, n, density=0.3 * rng.random(), format="csc", random_state=seed)
    S.sort_indices()
    cp, rv, nz = S.indptr.astype(np.int64) + 1, S.indices.astype(np.int64) + 1, S.data.copy()
    h = xsb.Handle(m, n)
    h.set_csc(cp, rv, nz)
    cols = np.repeat(np.arange(1, n + 1), np.diff(cp)).astype(np.int64)
    h.insert_batch(rv, cols, nz, xsb.ASSIGN)  # SparseMatrixLNK(csc): setindex! per entry, sparsematrixlnk.jl:109-118
    h.flush(xsb.DETERMINISTIC, xsb.COMBINE_ADD)
    cp2, rv2, nz2 = h.fetch_csc_numpy()
    assert np.array_equal(cp2, cp) and np.array_equal(rv2, rv) and np.array_equal(nz2, 2 * nz)


@pytest.mark.parametrize("seed", range(4))
def test_csc_roundtrip(xsb, seed):
    """test/test_constructors.jl:26-31, :44: CSC -> extension -> CSC is exact."""
    rng = np.random.default_rng(50 + seed)
    m, n = int(rng.integers(1, 400)), int(rng.integers(1, 400))
    S = sp.random(m, n, density=0.3 * rng.random(), format="csc", random_state=seed)
    S.sort_indices()
    cp, rv, nz = S.indptr.astype(np.int64) + 1, S.indices.astype(np.int64) + 1, S.data.copy()
    cols = np.repeat(np.arange(1, n + 1), np.diff(cp)).astype(np.int64)
    h = xsb.Handle(m, n)
    perm = rng.permutation(len(nz))
    h.insert_batch(rv[perm], cols[perm], nz[perm], xsb.ASSIGN)
    h.flush()
    cp2, rv2, nz2 = h.fetch_csc_numpy()
    assert np.array_equal(cp2, cp) and np.array_equal(rv2, rv) and np.array_equal(nz2, nz)
    h2 = xsb.Handle(m, n)
    h2.set_csc(cp, rv, nz)
    cp3, rv3, nz3 = h2.fetch_csc_numpy()
    assert np.array_equal(cp3, cp) and np.array_equal(rv3, rv) and np.array_equal(nz3, nz)


def assert_same_entry_streams(got, ref):
    """Grouping at insertion reorders a chunk by column but must keep, for every (i, j), its insertions in
    stream order: stable-sort both streams by (j, i) and compare."""
    gI, gJ, gV = got
    I, J, V = ref
    assert len(gV) == len(V)
    kg = np.lexsort((gI, gJ))  # stable
    kr = np.lexsort((I, J))
    assert np.array_equal(gI[kg], I[kr]) and np.array_equal(gJ[kg], J[kr])
    assert np.array_equal(bits(gV[kg]), bits(V[kr]))


# ---------------------------------------------------------------- generated streams
@pytest.mark.parametrize("dims", [(100, 100, 1), (100, 1, 1), (10, 10, 1), (5, 5, 5), (2, 2, 2), (3, 1, 1), (1, 1, 1),
                                  (2, 1, 1), (1, 4, 1), (1, 1, 3), (17, 33, 9), (40, 40, 40)])
@pytest.mark.parametrize("ones", [False, True])
def test_emit_fdrand_stream_and_matrix(xsb, oracle, dims, ones):
    """cfg 1 (fdrand 2D 100x100 via updateindex! + flush!, test_fdrand.jl) and friends."""
    nx, ny, nz_ = dims
    N = nx * ny * nz_
    I, J, V = oracle.fdrand_stream(nx, ny, nz_, seed=20240717, ones=ones)
    A = oracle.OracleExt(N, N)
    A.insert_batch(I, J, V, oracle.UPDATE)
    for grouped in (False, True):  # stream order as staged / chunks grouped by column while they are staged
        h = xsb.Handle(N, N)
        h.set_precount(grouped)
        h.emit_fdrand(nx, ny, nz_, seed=20240717, ones=ones, flavour=xsb.UPDATE)
        gI, gJ, gV, gF = h.debug_fetch_staged()
        if not grouped:
            assert np.array_equal(gI, I) and np.array_equal(gJ, J) and np.array_equal(bits(gV), bits(V))
        assert_same_entry_streams((gI, gJ, gV), (I, J, V))
        assert np.all(gF == xsb.UPDATE)
        h.flush()
        assert_csc_equal(h.fetch_csc_numpy(), A.csc())
        h.close()


def test_fdrand_ones_analytic(xsb):
    """SURVEY 8c(v): fdrand(100,100; rand=()->1) is analytic."""
    nx = ny = 100
    h = xsb.Handle(nx * ny, nx * ny)
    h.emit_fdrand(nx, ny, 1, ones=True)
    assert h.pending == 79600
    assert h.flush() == (49600, True)
    cp, rv, nz = h.fetch_csc_numpy()
    cols = np.repeat(np.arange(1, nx * ny + 1), np.diff(cp))
    off = rv != cols
    assert np.all(nz[off] == -1.0)
    ix, iy = (cols[~off] - 1) % nx + 1, (cols[~off] - 1) // nx + 1
    interior = (ix > 1) & (ix < nx) & (iy > 1) & (iy < ny)
    assert np.all(nz[~off][interior] == 4.0)
    assert np.array_equal(np.diff(cp), 1 + (ix > 1) + (ix < nx) + (iy > 1) + (iy < ny))


@pytest.mark.parametrize("dims", [(2, 2, 2), (3, 4, 5), (9, 9, 9), (17, 5, 3)])
def test_emit_p1fem(xsb, oracle, dims):
    """cfg 2 at oracle-sized meshes: testassemble! stream (femtools.jl:45-72), rawupdateindex!."""
    N = dims[0] * dims[1] * dims[2]
    I, J, V = oracle.fem_stream(*dims)
    A = oracle.OracleExt(N, N)
    A.insert_batch(I, J, V, oracle.RAW)
    for grouped in (False, True):
        h = xsb.Handle(N, N)
        h.set_precount(grouped)
        h.emit_p1fem(*dims, flavour=xsb.RAW)
        gI, gJ, gV, gF = h.debug_fetch_staged()
        if not grouped:
            assert np.array_equal(gI, I) and np.array_equal(gJ, J) and np.array_equal(bits(gV), bits(V))
        assert_same_entry_streams((gI, gJ, gV), (I, J, V))
        h.flush()
        assert_csc_equal(h.fetch_csc_numpy(), A.csc())
        h.close()


@pytest.mark.parametrize("dims", [(2, 2, 2, 4), (5, 4, 3, 4), (6, 6, 6, 2), (3, 1, 1, 3), (4, 3, 2, 1), (3, 3, 2, 6), (2, 2, 2, 7)])
def test_emit_blockrd_with_dirichlet(xsb, oracle, dims):
    """cfg 4 at oracle size: block system, then Dirichlet penalty rows (A[d,d]=1e30) and elimination."""
    nx, ny, nz_, ns = dims
    N = nx * ny * nz_ * ns
    I, J, V = oracle.blockrd_stream(nx, ny, nz_, ns, seed=7)
    # Dirichlet on the two x-faces: test/test_dirichlet.jl:9-11
    node = np.arange(nx * ny * nz_)
    face = (node % nx == 0) | (node % nx == nx - 1)
    d = (ns * node[face][:, None] + np.arange(1, ns + 1)[None, :]).ravel().astype(np.int64)
    pen = np.full(len(d), 1.0e30)
    for grouped in (False, True):  # stream order as staged / chunks grouped by column while they are staged
        h = xsb.Handle(N, N)
        h.set_precount(grouped)
        h.emit_blockrd(nx, ny, nz_, ns, seed=7, flavour=xsb.UPDATE)
        gI, gJ, gV, _ = h.debug_fetch_staged()
        if not grouped:
            assert np.array_equal(gI, I) and np.array_equal(gJ, J) and np.array_equal(bits(gV), bits(V))
        assert_same_entry_streams((gI, gJ, gV), (I, J, V))
        A = oracle.OracleExt(N, N)
        A.insert_batch(I, J, V, oracle.UPDATE)
        h.insert_batch(d, d, pen, xsb.ASSIGN)
        A.insert_batch(d, d, pen, oracle.ASSIGN)
        h.flush()
        assert_csc_equal(h.fetch_csc_numpy(), A.csc())
        mk = h.mark_dirichlet()
        omk = A.mark_dirichlet()
        assert np.array_equal(mk, omk) and mk.sum() == len(d)
        h.eliminate_dirichlet(mk)
        A.eliminate_dirichlet(omk)
        assert_csc_equal(h.fetch_csc_numpy(), A.csc())
        h.close()


# ---------------------------------------------------------------- multi-partition
@pytest.mark.parametrize("nparts", [1, 3, 8])
def test_mt_partitions(xsb, oracle, nparts):
    """MTExtendableSparseMatrixCSC: per-partition buffers summed in partition order
    (sparsematrixdilnkc.jl:397-435), then a second assembly that only hits the CSC."""
    I, J, V = oracle.fem_stream(5, 5, 5)
    N = 125
    h = xsb.Handle(N, N, n_tid=nparts)
    A = oracle.OracleMT(N, N, nparts)
    rng = np.random.default_rng(nparts)
    chunks = np.array_split(np.arange(len(V)), nparts)
    order = rng.permutation(nparts)  # partitions deliver their batches in arbitrary order
    for t in order:
        c = chunks[t]
        for part in np.array_split(c, 3):
            h.insert_batch(I[part], J[part], V[part], xsb.RAW, tid=int(t))
    for t in range(nparts):
        A.insert_batch(I[chunks[t]], J[chunks[t]], V[chunks[t]], t + 1, oracle.RAW)
    h.flush()
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())
    h.zero_values()
    A.zero_values()
    for t in range(nparts):
        c = chunks[t]
        h.insert_batch(I[c], J[c], V[c], xsb.RAW, tid=t)
        A.insert_batch(I[c], J[c], V[c], t + 1, oracle.RAW)
    assert h.flush()[1] is False
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())


# ---------------------------------------------------------------- values-only path
@pytest.mark.parametrize("dims", [(20, 20, 1), (12, 11, 10)])
def test_frozen_reassembly(xsb, oracle, dims):
    """cfg 3 at oracle size: build, then re-assemblies into the frozen pattern (Newton loop)."""
    nx, ny, nz_ = dims
    N = nx * ny * nz_
    h = xsb.Handle(N, N)
    h.emit_fdrand(nx, ny, nz_, seed=1)
    h.flush()
    A = oracle.OracleExt(N, N)
    I, J, V = oracle.fdrand_stream(nx, ny, nz_, seed=1)
    A.insert_batch(I, J, V, oracle.UPDATE)
    A.flush()
    hash0 = h.pattern_hash()
    h.freeze_pattern(I, J)
    for it in range(3):
        _, _, Vn = oracle.fdrand_stream(nx, ny, nz_, seed=2 + it)
        h.zero_values()
        h.reassemble_values(Vn, xsb.DETERMINISTIC)
        A.zero_values()
        A.insert_batch(I, J, Vn, oracle.UPDATE)
        assert A.nflush == 1
        assert_csc_equal(h.fetch_csc_numpy(), A.csc())
        # accumulate on top without zeroing: ((old + v1) + v2) order
        h.reassemble_values(Vn, xsb.DETERMINISTIC)
        A.insert_batch(I, J, Vn, oracle.UPDATE)
        assert_csc_equal(h.fetch_csc_numpy(), A.csc())
        h.zero_values()
        h.reassemble_values(Vn, xsb.FAST)
        A.zero_values()
        A.insert_batch(I, J, Vn, oracle.UPDATE)
        assert_csc_equal(h.fetch_csc_numpy(), A.csc(), exact=False, rtol=1e-14)
        # nonzeros(A) .= 0 fused into the re-assembly (xsb_reassemble_values_zeroed): same bits as the two calls
        h.reassemble_values(Vn, xsb.DETERMINISTIC, zero_first=True)
        assert_csc_equal(h.fetch_csc_numpy(), A.csc())
        h.reassemble_values(Vn, xsb.FAST, zero_first=True)
        assert_csc_equal(h.fetch_csc_numpy(), A.csc(), exact=False, rtol=1e-14)
    assert h.pattern_hash() == hash0
    # the same re-assembly through the general path (keys re-searched) gives the same bits
    h.zero_values()
    h.insert_batch(I, J, Vn, xsb.UPDATE)
    assert h.flush()[1] is False
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())
    # a position outside the pattern is refused
    with pytest.raises(xsb.XsbIllegalError):
        h.freeze_pattern(np.array([1], np.int64), np.array([N], np.int64))
    with pytest.raises(xsb.XsbSizeError):
        h.freeze_pattern(I, J)
        h.reassemble_values(Vn[:-1])


def test_fast_mode_flush(xsb, oracle):
    I, J, V = oracle.fem_stream(7, 7, 7)
    N = 343
    h = xsb.Handle(N, N)
    h.insert_batch(I, J, V, xsb.RAW)
    h.flush(xsb.FAST)
    A = oracle.OracleExt(N, N)
    A.insert_batch(I, J, V, oracle.RAW)
    cp, rv, nz = h.fetch_csc_numpy()
    ocp, orv, onz = A.csc()
    assert np.array_equal(cp, ocp) and np.array_equal(rv, orv)
    scale = np.abs(onz).max()
    assert np.max(np.abs(nz - onz)) <= 1e-14 * scale


@pytest.mark.parametrize("flavour", ["raw", "update"])
def test_fast_mode_preaggregation(xsb, oracle, flavour):
    """XSB_FAST with accumulate-on-insert inside windows of the stream: same pattern as the reference
    (zeros of updateindex! create nothing, cancelled entries stay), values within 1e-14, also on top
    of a resident CSC."""
    I, J, V = oracle.fem_stream(9, 9, 9)
    N = 729
    V = V.copy()
    fl, ofl = (xsb.RAW, oracle.RAW) if flavour == "raw" else (xsb.UPDATE, oracle.UPDATE)
    if flavour == "update":  # rows of node 5 only ever receive zeros: updateindex! must not create them
        V[I == 5] = 0.0
    h = xsb.Handle(N, N)
    h.set_preaggregation(True)
    A = oracle.OracleExt(N, N)
    for rnd in range(2):
        h.insert_batch(I, J, V * (rnd + 1), fl)
        h.flush(xsb.FAST)
        st = h.flush_stats()
        assert 0 < st["preagg_records"] < len(V) // 2
        A.insert_batch(I, J, V * (rnd + 1), ofl)
        A.flush()
        cp, rv, nz = h.fetch_csc_numpy()
        ocp, orv, onz = A.csc()
        assert np.array_equal(cp, ocp) and np.array_equal(rv, orv)
        assert np.max(np.abs(nz - onz)) <= 1e-14 * np.abs(onz).max()
    # a stream that does not repeat itself inside a window: tried twice, then left alone
    rng = np.random.default_rng(9)
    Ir = rng.integers(1, N + 1, 20000)
    Jr = rng.integers(1, N + 1, 20000)
    Vr = rng.standard_normal(20000)
    B = oracle.OracleExt(N, N)
    g = xsb.Handle(N, N)
    g.set_preaggregation(True)
    for rnd in range(3):
        g.insert_batch(Ir, Jr, Vr, xsb.UPDATE)
        g.flush(xsb.FAST)
        assert (g.flush_stats()["preagg_records"] > 0) == (rnd < 2)
        B.insert_batch(Ir, Jr, Vr, oracle.UPDATE)
        B.flush()
    cp, rv, nz = g.fetch_csc_numpy()
    ocp, orv, onz = B.csc()
    assert np.array_equal(cp, ocp) and np.array_equal(rv, orv)
    assert np.max(np.abs(nz - onz)) <= 1e-14 * np.abs(onz).max()


def test_get_values_and_pattern_hash(xsb, oracle):
    rng = np.random.default_rng(3)
    m, n, cnt = 500, 400, 20000
    I = rng.integers(1, m + 1, cnt)
    J = rng.integers(1, n + 1, cnt)
    V = rng.standard_normal(cnt)
    h = xsb.Handle(m, n)
    h.insert_batch(I, J, V, xsb.UPDATE)
    with pytest.raises(xsb.XsbError):
        h.get_values(I[:3], J[:3])  # pending inserts: flush first
    h.flush()
    A = oracle.OracleExt(m, n)
    A.insert_batch(I, J, V, oracle.UPDATE)
    qI = rng.integers(1, m + 1, 1000)
    qJ = rng.integers(1, n + 1, 1000)
    got = h.get_values(qI, qJ)
    ref = np.array([A[int(i), int(j)] for i, j in zip(qI, qJ)])
    assert np.array_equal(bits(got), bits(ref))
    h0 = h.pattern_hash()
    h.insert_batch(I[:100], J[:100], V[:100], xsb.UPDATE)
    h.flush()
    assert h.pattern_hash() == h0  # values-only update keeps the fingerprint (test_lu.jl:7-31)
    free = np.setdiff1d(np.arange(1, m + 1), I[J == 1])[:1]
    h.insert_batch(free, np.array([1], np.int64), np.array([1.0]), xsb.UPDATE)
    assert h.flush()[1] is True and h.pattern_hash() != h0  # new entry changes it (test_lu.jl:33-45)


def reference_mul(cp, rv, nz, x, m):
    """The stdlib kernel behind mul!(y, A, x): columns ascending, y[rowval[k]] += nzval[k] * x[j]."""
    y = np.zeros(m)
    for j in range(len(cp) - 1):
        xj = x[j]
        for k in range(cp[j] - 1, cp[j + 1] - 1):
            y[rv[k] - 1] += nz[k] * xj
    return y


def test_mul_bit_exact_and_tracks_the_matrix(xsb, oracle):
    """y = A*x (SURVEY 8f rank 3): bit-identical to the reference's column-order kernel, follows
    values-only updates without rebuilding its row-major view, rebuilds it when the pattern grows,
    handles empty rows/columns and a rectangular matrix."""
    rng = np.random.default_rng(12)
    m, n, cnt = 700, 500, 30000
    I = rng.integers(1, m + 1, cnt)
    J = rng.integers(1, n + 1, cnt)
    I[I % 50 == 0] = 1  # rows 50, 100, ... stay empty
    J[J % 40 == 0] = 2  # columns 40, 80, ... stay empty
    V = rng.standard_normal(cnt)
    h = xsb.Handle(m, n)
    x = rng.standard_normal(n)
    assert np.array_equal(h.mul(x), np.zeros(m))  # empty matrix
    h.insert_batch(I, J, V, xsb.UPDATE)
    with pytest.raises(xsb.XsbError):
        h.mul(x)  # pending inserts: flush first
    h.flush()
    cp, rv, nz = h.fetch_csc_numpy()
    y = h.mul(x)
    assert np.array_equal(bits(y), bits(reference_mul(cp, rv, nz, x, m)))
    S = sp.csc_matrix((nz, rv - 1, cp - 1), shape=(m, n))
    assert np.allclose(y, S @ x, rtol=1e-12, atol=1e-12)
    # same pattern, new values
    h.insert_batch(I[:5000], J[:5000], V[:5000], xsb.UPDATE)
    assert h.flush()[1] is False
    cp2, rv2, nz2 = h.fetch_csc_numpy()
    assert np.array_equal(bits(h.mul(x)), bits(reference_mul(cp2, rv2, nz2, x, m)))
    # pattern grows: the view is rebuilt
    h.insert_batch(np.array([50, 100]), np.array([40, 80]), np.array([2.5, -1.0]), xsb.UPDATE)
    assert h.flush()[1] is True
    cp3, rv3, nz3 = h.fetch_csc_numpy()
    y3 = h.mul(x)
    assert np.array_equal(bits(y3), bits(reference_mul(cp3, rv3, nz3, x, m)))
    assert y3[49] == 2.5 * x[39]
    # Int32 / 0-based handle and the host mirror
    g = xsb.Handle(m, n, idx_type=xsb.capi.I32, index_base=0)
    g.insert_batch((I - 1).astype(np.int32), (J - 1).astype(np.int32), V, xsb.UPDATE)
    g.flush()
    assert np.array_equal(bits(g.mul(x)), bits(y))
    A = xsb.ExtendableSparseMatrix(30, 30)
    xsb.fdrand(A, 30, 1, 1, rand=lambda: 1.0)
    assert np.allclose(A @ np.ones(30), A.sparse() @ np.ones(30))


def test_mul_slab_contributions_add_up(xsb):
    torch = pytest.importorskip("torch")
    nx = 20
    N = nx ** 3
    world = 3
    splits = [0, 3000, 5500, N]
    full = xsb.Handle(N, N)
    full.emit_fdrand(nx, nx, nx, seed=9)
    full.flush()
    x = np.random.default_rng(3).standard_normal(N)
    y = full.mul(x)
    from tests.test_gpu_dist import route_and_flush

    handles = [xsb.Handle(N, N, slab=(world, r, splits)) for r in range(world)]
    for r, h in enumerate(handles):
        h.emit_fdrand(nx, nx, nx, seed=9, l_range=(splits[r], splits[r + 1]))
    route_and_flush(xsb, torch, handles)
    parts = [h.mul(x[splits[r]:splits[r + 1]]) for r, h in enumerate(handles)]
    assert np.allclose(sum(parts), y, rtol=1e-13, atol=1e-13)


def test_reset_and_reuse(xsb, oracle):
    h = xsb.Handle(50, 50)
    I, J, V = oracle.fdrand_stream(50, 1, 1, seed=4)
    h.insert_batch(I, J, V, xsb.UPDATE)
    h.flush()
    h.reset()
    assert h.nnz == 0 and h.pending == 0
    cp, rv, nz = h.fetch_csc_numpy()
    assert np.all(cp == 1) and len(rv) == 0
    h.insert_batch(I, J, V, xsb.UPDATE)
    h.flush()
    A = oracle.OracleExt(50, 50)
    A.insert_batch(I, J, V, oracle.UPDATE)
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())


def test_host_mirror_fdrand(xsb, oracle):
    """test/test_fdrand.jl:29-53: A[i,j]+=v vs rawupdateindex! vs updateindex! with rand=()->1."""
    import operator

    def run(update):
        A = xsb.ExtendableSparseMatrix(25, 25)
        xsb.fdrand(A, 5, 5, 1, update=update, rand=lambda: 1.0)
        return A.csc()

    a2 = run(lambda A, v, i, j: A.rawupdateindex(operator.add, v, i, j))
    a3 = run(lambda A, v, i, j: A.updateindex(operator.add, v, i, j))
    I, J, V = oracle.fdrand_stream(5, 5, 1, ones=True)
    O = oracle.OracleExt(25, 25)
    O.insert_batch(I, J, V, oracle.UPDATE)
    assert_csc_equal(a2, O.csc())
    assert_csc_equal(a3, O.csc())


# ---------------------------------------------------------------- full-size properties (no oracle)
def test_full_size_fd_properties(xsb):
    """fdrand 3D 128^3 (25 M insertions): size-independent properties of the result."""
    nx = 128
    N = nx ** 3
    h = xsb.Handle(N, N)
    h.emit_fdrand(nx, nx, nx, seed=11)
    n_ins = h.pending
    nnz, changed = h.flush()
    assert changed and nnz == 7 * N - 6 * nx * nx
    cp, rv, nz = h.fetch_csc_numpy()
    assert cp[0] == 1 and cp[-1] == nnz + 1 and np.all(np.diff(cp) >= 4) and np.all(np.diff(cp) <= 7)
    cols = np.repeat(np.arange(1, N + 1), np.diff(cp))
    assert np.all((np.diff(rv) > 0) | (np.diff(cols) > 0))  # strictly sorted rows inside each column
    S = sp.csc_matrix((nz, rv - 1, cp - 1), shape=(N, N))
    assert abs(S - S.T).max() == 0.0  # update_pair inserts -v at (i,j) and (j,i)
    rs = np.asarray(S.sum(axis=0)).ravel()
    assert rs.min() > -1e-12  # weakly diagonally dominant M-matrix
    # idempotence: flushing the same stream on top doubles every value, pattern unchanged
    h.emit_fdrand(nx, nx, nx, seed=11)
    assert h.pending == n_ins
    assert h.flush() == (nnz, False)
    _, _, nz2 = h.fetch_csc_numpy()
    assert np.array_equal(nz2[rv != cols], 2 * nz[rv != cols])  # one contribution each: exact
    assert np.allclose(nz2, 2 * nz, rtol=1e-14, atol=0.0)


# ---------------------------------------------------------------- flush strategies
def test_strategies_agree_and_long_columns_fall_back(xsb, oracle):
    """Column sort + hash fold (AUTO) and the (col,row) sort (FULLSORT) give the same bits; a column too
    rich for the in-warp path makes AUTO finish with the general path.  No other strategy is accepted."""
    rng = np.random.default_rng(77)
    m, n, cnt = 3000, 500, 60000
    I = rng.integers(1, m + 1, cnt)
    J = rng.integers(1, n + 1, cnt)
    V = rng.standard_normal(cnt)
    A = oracle.OracleExt(m, n)
    A.insert_batch(I, J, V, oracle.UPDATE)
    ref = A.csc()
    for strat, expect_col in ((xsb.capi.STRATEGY_AUTO, 2), (xsb.capi.STRATEGY_FULLSORT, 0)):
        h = xsb.Handle(m, n)
        h.set_strategy(strat)
        h.insert_batch(I, J, V, xsb.UPDATE)
        h.flush()
        assert h.flush_stats()["column_path"] == expect_col
        assert_csc_equal(h.fetch_csc_numpy(), ref)
    # one dense column (3000 records in column 7) -> overflow -> fallback, same result
    J2 = J.copy()
    J2[:3000] = 7
    A = oracle.OracleExt(m, n)
    A.insert_batch(I, J2, V, oracle.UPDATE)
    h = xsb.Handle(m, n)
    h.set_strategy(xsb.capi.STRATEGY_AUTO)
    h.insert_batch(I, J2, V, xsb.UPDATE)
    h.flush()
    st = h.flush_stats()
    assert st["column_path"] == 0 and st["sort_passes"] > 3
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())
    # columns of every length around the warp-sort sizes (31..257 records), duplicates included
    lens = [1, 2, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256]
    Jl = np.concatenate([np.full(L, k + 1) for k, L in enumerate(lens)])
    Il = rng.integers(1, 40, len(Jl))
    Vl = rng.standard_normal(len(Jl))
    perm = rng.permutation(len(Jl))
    A = oracle.OracleExt(50, len(lens))
    A.insert_batch(Il[perm], Jl[perm], Vl[perm], oracle.RAW)
    h = xsb.Handle(50, len(lens))
    h.set_strategy(xsb.capi.STRATEGY_AUTO)
    h.insert_batch(Il[perm], Jl[perm], Vl[perm], xsb.RAW)
    h.flush()
    assert h.flush_stats()["column_path"] == 2
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())
    # any value but AUTO (0) and FULLSORT (1) is rejected
    h = xsb.Handle(m, n)
    with pytest.raises(xsb.capi.XsbError) as e:
        h.set_strategy(2)
    assert e.value.code == xsb.capi.EINVAL


def test_hash_fold_groups_of_columns(xsb, oracle):
    """The hash-fold kernel on shapes that stress its grouping: many short columns per group, columns
    around the group size, a long column with few distinct rows, empty columns in between, all three
    flavours, several partitions and a second flush on top of the first (old entries seed the fold)."""
    rng = np.random.default_rng(4242)
    m, n = 5000, 4000
    lens = np.concatenate([rng.integers(0, 6, 1500), rng.integers(100, 140, 40), [2000, 1, 0, 0, 700],
                           rng.integers(20, 70, 300)])
    cols = rng.permutation(n)[: len(lens)] + 1
    J = np.repeat(cols, lens)
    I = np.empty(len(J), dtype=np.int64)
    pos = 0
    for L in lens:
        I[pos:pos + L] = rng.integers(1, min(150, max(3, int(L) // 3) + 8), L)  # plenty of duplicates
        pos += L
    V = rng.standard_normal(len(J))
    V[rng.random(len(J)) < 0.05] = 0.0
    perm = rng.permutation(len(J))
    I, J, V = I[perm], J[perm], V[perm]
    for n_tid, grouping in ((1, xsb.capi.GROUPING_OFF), (3, xsb.capi.GROUPING_OFF), (1, xsb.capi.GROUPING_ON)):
        A = oracle.OracleMT(m, n, n_tid) if n_tid > 1 else oracle.OracleExt(m, n)
        h = xsb.Handle(m, n, n_tid=n_tid)
        h.set_grouping(grouping)
        for rnd in range(2):
            parts = np.array_split(np.arange(len(J)), 3 * n_tid)
            for q, idx in enumerate(parts):
                fl = (xsb.UPDATE, xsb.RAW, xsb.ASSIGN)[q % 3] if n_tid == 1 else (xsb.UPDATE, xsb.RAW)[q % 2]
                ofl = {xsb.UPDATE: oracle.UPDATE, xsb.RAW: oracle.RAW, xsb.ASSIGN: oracle.ASSIGN}[fl]
                if n_tid > 1:  # partitions deliver in tid order: CSC hits are applied in call order
                    A.insert_batch(I[idx], J[idx], V[idx] * (rnd + 1), q // 3 + 1, ofl)
                    h.insert_batch(I[idx], J[idx], V[idx] * (rnd + 1), fl, tid=q // 3)
                else:
                    A.insert_batch(I[idx], J[idx], V[idx] * (rnd + 1), ofl)
                    h.insert_batch(I[idx], J[idx], V[idx] * (rnd + 1), fl)
            A.flush()
            h.flush()
            assert h.flush_stats()["column_path"] in ((2,) if grouping == xsb.capi.GROUPING_OFF else (2, 3, 4))
            assert_csc_equal(h.fetch_csc_numpy(), A.csc())


# ---------------------------------------------------------------- two-pass grouping by column
def test_grouping_by_column_fem_and_fallback(xsb, oracle):
    """Streams with column locality take the two-pass grouping (sparse per-chunk column histograms);
    a stream without locality is detected after the counting pass and takes the radix sort.  Same bits
    either way, also on top of a resident CSC and with several partitions."""
    I, J, V = oracle.fem_stream(12, 12, 12)
    N = 12 ** 3
    assert len(V) >= 32768
    A = oracle.OracleExt(N, N)
    A.insert_batch(I, J, V, oracle.RAW)
    ref = A.csc()
    got = {}
    for grouping in (xsb.capi.GROUPING_AUTO, xsb.capi.GROUPING_OFF):
        h = xsb.Handle(N, N)
        h.set_grouping(grouping)
        h.insert_batch(I, J, V, xsb.RAW)
        h.flush()
        st = h.flush_stats()
        assert st["column_path"] == (4 if grouping == xsb.capi.GROUPING_AUTO else 2)
        if grouping == xsb.capi.GROUPING_AUTO:
            assert 0 < st["group_pairs"] < len(V) // 4
        got[grouping] = h.fetch_csc_numpy()
        assert_csc_equal(got[grouping], ref)
        # second assembly on top of the resident CSC, scaled values, update flavour with some zeros
        V2 = V * 0.5
        V2[::7] = 0.0
        h.insert_batch(I, J, V2, xsb.UPDATE)
        h.flush()
        A2 = oracle.OracleExt(N, N)
        A2.insert_batch(I, J, V, oracle.RAW)
        A2.flush()
        A2.insert_batch(I, J, V2, oracle.UPDATE)
        assert_csc_equal(h.fetch_csc_numpy(), A2.csc())
    # no locality: random columns -> about one pair per record -> radix sort
    rng = np.random.default_rng(5)
    m, n, cnt = 30000, 30000, 80000
    Ir = rng.integers(1, m + 1, cnt)
    Jr = rng.integers(1, n + 1, cnt)
    Vr = rng.standard_normal(cnt)
    B = oracle.OracleExt(m, n)
    B.insert_batch(Ir, Jr, Vr, oracle.UPDATE)
    h = xsb.Handle(m, n)
    h.set_grouping(xsb.capi.GROUPING_ON)
    h.insert_batch(Ir, Jr, Vr, xsb.UPDATE)
    h.flush()
    st = h.flush_stats()
    assert st["column_path"] == 2 and st["group_pairs"] > cnt // 4
    assert_csc_equal(h.fetch_csc_numpy(), B.csc())
    # several partitions (general fold) through the grouping
    nparts = 3
    hm = xsb.Handle(N, N, n_tid=nparts)
    M = oracle.OracleMT(N, N, nparts)
    for t, c in enumerate(np.array_split(np.arange(len(V)), nparts)):
        hm.insert_batch(I[c], J[c], V[c], xsb.RAW, tid=t)
        M.insert_batch(I[c], J[c], V[c], t + 1, oracle.RAW)
    hm.flush()
    assert hm.flush_stats()["column_path"] == 3
    assert_csc_equal(hm.fetch_csc_numpy(), M.csc())


def test_grouping_fdrand_large(xsb, oracle):
    """fdrand 3-D 40^3 through the generator kernel: short columns, little duplication."""
    nx = 40
    N = nx ** 3
    h = xsb.Handle(N, N)
    h.emit_fdrand(nx, nx, nx, seed=3)
    h.flush()
    assert h.flush_stats()["column_path"] == 4
    I, J, V = oracle.fdrand_stream(nx, nx, nx, seed=3)
    A = oracle.OracleExt(N, N)
    A.insert_batch(I, J, V, oracle.UPDATE)
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())


# ---------------------------------------------------------------- pointblock (SURVEY.md 8f rank 4)
@pytest.mark.parametrize("case", ["fd_bs4_i64", "fem_bs3_i32", "rd_bs4_big"])
def test_pointblock_matches_oracle(xsb, oracle, case):
    """pointblock(A, blocksize), src/matrix/extendable.jl:292-318: pattern and blocks bit for bit."""
    if case == "fd_bs4_i64":
        I, J, V = oracle.fdrand_stream(6, 4, 2, seed=5)
        n, bs, idx = 48, 4, xsb.I64
    elif case == "fem_bs3_i32":
        I, J, V = oracle.fem_stream(6, 5, 4)
        n, bs, idx = 120, 3, xsb.I32
    else:  # enough entries for the grouping path of the block-pattern flush
        I, J, V = oracle.blockrd_stream(12, 10, 8, 4, seed=3)
        n, bs, idx = 4 * 960, 4, xsb.I64
    V = V.copy()
    V[::97] = -0.0
    h = xsb.Handle(n, n, idx_type=idx)
    dt = np.int64 if idx == xsb.I64 else np.int32
    h.insert_batch(I.astype(dt), J.astype(dt), V, xsb.RAW)
    h.flush()
    A = oracle.OracleExt(n, n)
    A.insert_batch(I, J, V, oracle.RAW)
    ocp, orv, obl = A.pointblock(bs)
    hb = h.pointblock(bs)
    cp, rv, _ = hb.fetch_csc_numpy()
    bl = hb.fetch_blocks_numpy().reshape(hb.nnz, bs * bs)
    assert hb.nnz == len(orv)
    assert np.array_equal(cp, ocp) and np.array_equal(rv, orv)
    assert np.array_equal(bits(bl), bits(obl)), "blocks not bit-exact"
    hb.close()
    # the source matrix is untouched and can be converted again
    hb2 = h.pointblock(1)
    assert hb2.nnz == h.nnz
    hb2.close()


def test_pointblock_errors_and_mirror(xsb, oracle):
    h = xsb.Handle(5, 5)
    h.insert_batch(np.array([1, 2], np.int64), np.array([1, 5], np.int64), np.ones(2), xsb.RAW)
    with pytest.raises(xsb.XsbError):  # pending inserts
        h.pointblock(2)
    h.flush()
    with pytest.raises(IndexError) as e:  # column 5 -> block row 3 of a 2x2 block matrix
        h.pointblock(2)
    assert "entry 1" in str(e.value)
    with pytest.raises(xsb.XsbError):
        h.pointblock(6)
    # host mirror on the hand vector of tests/test_oracle_kat.py::test_pointblock_hand_vector
    import operator

    A = xsb.ExtendableSparseMatrix(4, 4)
    for v, i, j in [(1.0, 1, 1), (2.0, 2, 1), (3.0, 3, 2), (4.0, 1, 4), (-0.0, 4, 4)]:
        A.rawupdateindex(operator.add, v, i, j)
    cp, rv, blocks = xsb.pointblock(A, 2)
    assert cp.tolist() == [1, 3, 5] and rv.tolist() == [1, 2, 1, 2]
    assert blocks[0].tolist() == [[1.0, 2.0], [0.0, 0.0]] and blocks[1].tolist() == [[0.0, 0.0], [4.0, 0.0]]
    assert blocks[2].tolist() == [[0.0, 0.0], [3.0, 0.0]] and not np.signbit(blocks).any()
    # an empty matrix gives an empty block matrix
    E = xsb.Handle(6, 6)
    hb = E.pointblock(3)
    assert hb.nnz == 0 and hb.fetch_csc_numpy()[0].tolist() == [1, 1, 1]
    hb.close()


# ---------------------------------------------------------------- counting at insertion (pre-count)
def _fem_case(oracle, n1=30):
    I, J, V = oracle.fem_stream(n1, n1, n1)
    n = n1 ** 3
    A = oracle.OracleExt(n, n)
    A.insert_batch(I, J, V, oracle.RAW)
    return I, J, V, n, A.csc()


@pytest.mark.parametrize("producer", ["emit", "batch", "triplets"])
def test_precount_equals_flush_time_count(xsb, oracle, producer):
    """The column histograms taken by the staging kernels (xsb_set_precount, default on) give the bits
    of the flush-time counting pass and of the oracle; the flush then counts (almost) nothing."""
    n1 = 30
    I, J, V, n, ref = _fem_case(oracle, n1)
    out = {}
    for on in (True, False):
        h = xsb.Handle(n, n)
        h.set_precount(on)
        if producer == "emit":
            h.emit_p1fem(n1, n1, n1, flavour=xsb.RAW)
        elif producer == "batch":
            h.insert_batch(I, J, V, xsb.RAW)
        else:
            h.insert_triplets(triplets(xsb, I, J, V), xsb.RAW)
        h.flush()
        st = h.flush_stats()
        assert st["column_path"] == 4
        if on:
            assert st["precounted"] > 0.99
        else:
            assert st["precounted"] == 0.0
        out[on] = h.fetch_csc_numpy()
        assert_csc_equal(out[on], ref)
        h.close()


def test_precount_ragged_batches_and_rejections(xsb, oracle):
    """Batches that end off a chunk boundary stop the counting at insertion (the flush counts the rest);
    a rejected batch or a stage that grows under counted chunks makes the flush count everything."""
    n1 = 30
    I, J, V, n, ref = _fem_case(oracle, n1)
    cnt = len(V)
    W = 512
    cuts = {
        "aligned_then_ragged": [0, 200 * W, 200 * W + 777, 300 * W + 777, cnt],
        "all_aligned": [0, 64 * W, 640 * W, cnt],
        "ragged_first": [0, 100, 100 + 300 * W, cnt],
    }
    for name, cut in cuts.items():
        h = xsb.Handle(n, n)
        h.reserve(0, cnt)
        for a, b in zip(cut[:-1], cut[1:]):
            h.insert_batch(I[a:b], J[a:b], V[a:b], xsb.RAW)
        h.flush()
        st = h.flush_stats()
        assert st["column_path"] == 4, name
        assert st["precounted"] > 0.99, name  # a batch of any length is grouped while it is packed
        assert_csc_equal(h.fetch_csc_numpy(), ref)
        h.close()
    # rejected batch after counted chunks
    h = xsb.Handle(n, n)
    h.reserve(0, cnt)
    h.insert_batch(I[:400 * W], J[:400 * W], V[:400 * W], xsb.RAW)
    badI = I[400 * W:500 * W].copy()
    badI[12345] = n + 7
    with pytest.raises(IndexError) as e:
        h.insert_batch(badI, J[400 * W:500 * W], V[400 * W:500 * W], xsb.RAW)
    assert "entry 12345" in str(e.value)
    badI[12345] = I[400 * W + 12345]
    badI[-3] = 0  # in the tail handled by the plain kernel? no: whole chunks -> fused kernel reports it too
    with pytest.raises(IndexError) as e:
        h.insert_batch(badI, J[400 * W:500 * W], V[400 * W:500 * W], xsb.RAW)
    assert f"entry {100 * W - 3}" in str(e.value)
    h.insert_batch(I[400 * W:], J[400 * W:], V[400 * W:], xsb.RAW)
    h.flush()
    assert h.flush_stats()["precounted"] == 0.0
    assert_csc_equal(h.fetch_csc_numpy(), ref)
    h.close()
    # the stage grows under counted chunks (no reserve)
    h = xsb.Handle(n, n)
    for a, b in [(0, 128 * W), (128 * W, 1024 * W), (1024 * W, cnt)]:
        h.insert_batch(I[a:b], J[a:b], V[a:b], xsb.RAW)
    h.flush()
    assert_csc_equal(h.fetch_csc_numpy(), ref)
    # second assembly into the now non-empty matrix: grouped at insertion as well, merged with the resident columns
    h.insert_batch(I, J, V, xsb.RAW)
    h.flush()
    assert h.flush_stats()["precounted"] > 0.99 and h.flush_stats()["column_path"] == 4
    A = oracle.OracleExt(n, n)
    A.insert_batch(I, J, V, oracle.RAW)
    A.flush()
    A.insert_batch(I, J, V, oracle.RAW)
    assert_csc_equal(h.fetch_csc_numpy(), A.csc())
    # reset! starts over: counting at insertion again
    h.reset()
    h.insert_batch(I, J, V, xsb.RAW)
    h.flush()
    assert h.flush_stats()["precounted"] > 0.99
    assert_csc_equal(h.fetch_csc_numpy(), ref)
    h.close()


def test_precount_tail_bounds_error(xsb):
    """An out-of-range entry in the ragged tail of a batch (plain kernel) is reported at its batch position."""
    h = xsb.Handle(1000, 1000)
    cnt = 3 * 512 + 100
    I = np.ones(cnt, np.int64)
    J = np.ones(cnt, np.int64)
    I[3 * 512 + 40] = 1001
    with pytest.raises(IndexError) as e:
        h.insert_batch(I, J, np.ones(cnt), xsb.UPDATE)
    assert f"entry {3 * 512 + 40}" in str(e.value) and h.pending == 0
    T = triplets(xsb, I, J, np.ones(cnt))
    with pytest.raises(IndexError) as e:
        h.insert_triplets(T, xsb.UPDATE)
    assert f"entry {3 * 512 + 40}" in str(e.value) and h.pending == 0
    I[3 * 512 + 40] = 1
    h.insert_batch(I, J, np.ones(cnt), xsb.UPDATE)
    assert h.flush() == (1, True)
    assert h.fetch_csc_numpy()[2].tolist() == [float(cnt)]


def test_column_met_by_many_chunks_uses_pair_sort(xsb, oracle):
    """The bucketed pair path orders a column's (chunk, column) pairs inside one thread; a column that more
    than 128 chunks write to sends the flush to the radix sort of the pairs instead.  Same bits either way."""
    n1 = 30
    I, J, V, n, _ = _fem_case(oracle, n1)
    I, J = I.copy(), J.copy()
    hot = np.arange(0, len(V), 300)
    I[hot] = (hot % n) + 1
    J[hot] = 7
    A = oracle.OracleExt(n, n)
    A.insert_batch(I, J, V, oracle.RAW)
    ref = A.csc()
    for pre in (True, False):
        h = xsb.Handle(n, n)
        h.set_precount(pre)
        h.insert_batch(I, J, V, xsb.RAW)
        h.flush()
        st = h.flush_stats()
        assert st["column_path"] == 3 and st["sort_passes"] > 0  # pairs went through the sort
        assert_csc_equal(h.fetch_csc_numpy(), ref)
        h.close()
    # the plain FEM stream takes the bucketed path: no sort passes at all
    h = xsb.Handle(n, n)
    h.emit_p1fem(n1, n1, n1, flavour=xsb.RAW)
    h.flush()
    st = h.flush_stats()
    assert st["column_path"] == 4 and st["sort_passes"] == 0
    h.close()


@pytest.mark.parametrize("stream,batch", [("fd", 700), ("fd", 96), ("fem", 300), ("fem", 64)])
def test_columns_met_by_many_small_chunks(xsb, oracle, stream, batch):
    """Small insertion batches make small chunks: a column then collects more run descriptors than the merge kernel
    keeps in registers (4 with the small table shape, 8 otherwise) and orders its bucket in place instead."""
    if stream == "fd":
        nx = 24
        n = nx ** 3
        I, J, V = oracle.fdrand_stream(nx, nx, nx, seed=11)
        fl, ofl = xsb.UPDATE, oracle.UPDATE
    else:
        n1 = 16
        n = n1 ** 3
        I, J, V = oracle.fem_stream(n1, n1, n1)
        fl, ofl = xsb.RAW, oracle.RAW
    A = oracle.OracleExt(n, n)
    A.insert_batch(I, J, V, ofl)
    ref = A.csc()
    h = xsb.Handle(n, n)
    for rnd in range(2):  # second round: the table shape follows the first flush's hint
        h.reset()
        h.reserve(0, len(V))
        for a in range(0, len(V), batch * 37):
            b = min(a + batch * 37, len(V))
            for c in range(a, b, batch):
                h.insert_batch(I[c:min(c + batch, b)], J[c:min(c + batch, b)], V[c:min(c + batch, b)], fl)
        h.flush()
        assert h.flush_stats()["column_path"] == 4
        assert_csc_equal(h.fetch_csc_numpy(), ref)
    h.close()


def test_fold_table_shape_follows_previous_flush(xsb, oracle):
    """The thread fold picks its table from the distinct rows per column the previous flush saw (15 for a P1
    mesh: the 32-slot / 16-accumulator shape).  A following assembly with richer columns overflows that table once,
    is folded by the fallback path, and the result is the oracle's both times."""
    n1 = 30
    I, J, V, n, ref = _fem_case(oracle, n1)
    h = xsb.Handle(n, n)
    for _ in range(3):  # first flush: no hint; later ones: the slim table
        h.reset()
        h.insert_batch(I, J, V, xsb.RAW)
        h.flush()
        assert h.flush_stats()["column_path"] == 4
        assert_csc_equal(h.fetch_csc_numpy(), ref)
    # 22 distinct rows in every column
    rng = np.random.default_rng(5)
    cols = np.repeat(np.arange(1, n + 1), 44)
    rows = ((cols[:, None].reshape(-1, 44) * 7 + np.arange(44)[None, :] % 22 * 131) % n + 1).reshape(-1)
    vals = rng.standard_normal(len(cols))
    perm = np.argsort(rng.integers(0, 64, len(cols)) + (cols // 40) * 64, kind="stable")  # keep column locality
    I2, J2, V2 = rows[perm], cols[perm], vals[perm]
    A = oracle.OracleExt(n, n)
    A.insert_batch(I2, J2, V2, oracle.RAW)
    for _ in range(2):
        h.reset()
        h.insert_batch(I2, J2, V2, xsb.RAW)
        h.flush()
        assert_csc_equal(h.fetch_csc_numpy(), A.csc())
    h.close()
