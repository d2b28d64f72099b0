"""Pins the CPU oracle against the reference's own known-answer tests.

The reference (pure Julia) holds no stored golden vectors; these are the
known-answer and property tests of its test-suite restated (SURVEY.md 8c).
"""
import numpy as np
import pytest
import scipy.sparse as sp


def dense_accumulate(stream):
    """Sequential S[i,j] += a on a dict: the test_assembly.jl:16 oracle."""
    acc = {}
    for (i, j, a) in stream:
        acc[(i, j)] = acc.get((i, j), 0.0) + a
    return acc


def csc_to_dict(cp, rv, nz):
    out = {}
    for j in range(len(cp) - 1):
        for k in range(cp[j] - 1, cp[j + 1] - 1):
            out[(int(rv[k]), j + 1)] = float(nz[k])
    return out


def test_philox_known_answer(oracle):
    # Random123 kat_vectors: philox4x32 10 rounds, counter 0, key 0
    assert [hex(x) for x in oracle.philox(0, 0)] == ["0x6627e8d5", "0xe169c58d", "0xbc57ac4c", "0x9b00dbd8"]
    u = oracle.uniform(0, 0)
    bits = (0xE169C58D << 32) | 0x6627E8D5
    assert u == (bits >> 11) * 2.0 ** -53


def test_micro_vector(oracle):
    """SURVEY.md 8(c'): hand-stepped through sparsematrixlnk.jl."""
    A = oracle.OracleExt(3, 3)
    A.updateindex(1.0, 2, 1)
    A.updateindex(2.0, 3, 1)
    A.updateindex(0.5, 2, 1)
    A.updateindex(0.0, 1, 2)
    A.rawupdateindex(0.0, 1, 3)
    assert A.nnz_lnk == 3
    cp, rv, nz = A.csc()
    assert cp.tolist() == [1, 3, 3, 4]
    assert rv.tolist() == [2, 3, 1]
    assert nz.tolist() == [1.5, 2.0, 0.0]
    A.updateindex(-1.5, 2, 1)
    A.updateindex(4.0, 1, 1)
    cp, rv, nz = A.csc()
    assert cp.tolist() == [1, 4, 4, 5]
    assert rv.tolist() == [1, 2, 3, 1]
    assert nz.tolist() == [4.0, 0.0, 2.0, 0.0]
    assert A.nflush == 2


def test_updates_zero_semantics(oracle):
    """test/test_updates.jl:10-25."""
    A = oracle.OracleExt(10, 10)
    assert A.nnz == 0
    A[1, 3] = 5
    A.updateindex(6.0, 4, 5)
    A.updateindex(0.0, 2, 3)
    assert A.nnz == 2
    A.rawupdateindex(0.0, 2, 3)
    assert A.nnz == 3
    # dropzeros!(A) acts on the flushed CSC (stdlib); restated with numpy
    cp, rv, nz = A.csc()
    keep = nz != 0
    cols = np.repeat(np.arange(10), np.diff(cp))
    cp2 = np.concatenate([[1], 1 + np.cumsum(np.bincount(cols[keep], minlength=10))])
    A.set_csc(cp2, rv[keep], nz[keep])
    assert A.nnz == 2
    A.rawupdateindex(0.1, 2, 3)
    assert A.nnz == 3


@pytest.mark.parametrize(
    "m,n,xnnz,nsplice",
    [(10, 10, 5, 1), (100, 100, 500, 2), (1000, 1000, 5000, 3), (20, 10, 5, 1), (200, 100, 500, 2),
     (2000, 1000, 5000, 3), (10, 20, 5, 1), (100, 200, 500, 2), (1000, 2000, 5000, 3), (37, 9001, 7000, 5)],
)
def test_assembly_exact(oracle, m, n, xnnz, nsplice):
    """test/test_assembly.jl:6-35: A[i,j] += a  ==  sequential accumulation, exactly."""
    rng = np.random.default_rng(1000 * m + n)
    A = oracle.OracleExt(m, n)
    stream = []
    for _ in range(nsplice):
        I = rng.integers(1, m + 1, xnnz)
        J = rng.integers(1, n + 1, xnnz)
        V = 1.0 + rng.random(xnnz)
        for i, j, a in zip(I, J, V):
            # A[i,j] += a  ->  setindex!(A, A[i,j]+a, i, j)   (README.md:82-94)
            A[i, j] = A[i, j] + a
            stream.append((int(i), int(j), float(a)))
        cp, rv, nz = A.csc()
        for j in range(n):
            col = rv[cp[j] - 1:cp[j + 1] - 1]
            assert np.all(np.diff(col) > 0)
        ref = dense_accumulate(stream)
        got = csc_to_dict(cp, rv, nz)
        assert got == ref  # exact ==, both directions


def test_update_equals_plus_equals(oracle):
    rng = np.random.default_rng(7)
    m = n = 50
    A, B = oracle.OracleExt(m, n), oracle.OracleExt(m, n)
    I = rng.integers(1, m + 1, 2000)
    J = rng.integers(1, n + 1, 2000)
    V = rng.standard_normal(2000)
    V[::7] = 0.0
    for i, j, a in zip(I, J, V):
        A[i, j] = A[i, j] + a
    B.insert_batch(I, J, V, oracle.UPDATE)
    for x, y in zip(A.csc(), B.csc()):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("seed", range(5))
def test_csc_plus_lnk_is_twice(oracle, seed):
    """test/test_operations.jl:8-13."""
    rng = np.random.default_rng(seed)
    m, n = int(rng.integers(1, 300)), int(rng.integers(1, 300))
    S = sp.random(m, n, density=0.3 * rng.random(), format="csc", random_state=seed)
    S.sort_indices()
    cp, rv, nz = S.indptr.astype(np.int64) + 1, S.indices.astype(np.int64) + 1, S.data
    L = oracle.OracleLNK.from_csc(m, n, cp, rv, nz)
    cp2, rv2, nz2 = L.plus_csc(m, n, cp, rv, nz)
    assert np.array_equal(cp2, cp) and np.array_equal(rv2, rv) and np.array_equal(nz2, 2 * nz)


@pytest.mark.parametrize("seed", range(5))
def test_lnk_roundtrip(oracle, seed):
    """test/test_constructors.jl:26-31."""
    rng = np.random.default_rng(100 + seed)
    m, n = int(rng.integers(1, 300)), int(rng.integers(1, 300))
    S = sp.random(m, n, density=0.3 * rng.random(), format="csc", random_state=seed)
    S.sort_indices()
    cp, rv, nz = S.indptr.astype(np.int64) + 1, S.indices.astype(np.int64) + 1, S.data
    L = oracle.OracleLNK.from_csc(m, n, cp, rv, nz)
    empty = np.ones(n + 1, np.int64)
    cp2, rv2, nz2 = L.plus_csc(m, n, empty, np.zeros(0, np.int64), np.zeros(0))
    assert np.array_equal(cp2, cp) and np.array_equal(rv2, rv) and np.array_equal(nz2, nz)


def test_readme_example(oracle):
    """README.md:15-27: 10x10 tridiagonal."""
    A = oracle.OracleExt(10, 10)
    A[1, 1] = 1
    for i in range(1, 10):
        A[i + 1, i] = A[i + 1, i] + (-1)
        A[i, i + 1] = A[i, i + 1] + (-1)
        A[i + 1, i + 1] = A[i + 1, i + 1] + 1
        A[i, i] = A[i, i] + 1
    cp, rv, nz = A.csc()
    assert len(nz) == 28
    d = csc_to_dict(cp, rv, nz)
    for i in range(1, 11):
        assert d[(i, i)] == (1.0 if i == 10 else 2.0)
    for i in range(1, 10):
        assert d[(i, i + 1)] == -1.0 and d[(i + 1, i)] == -1.0


@pytest.mark.parametrize("flavour", [0, 1, 2])
def test_fdrand_ones_analytic(oracle, flavour):
    """fdrand(100,100; rand=()->1): test/test_fdrand.jl:22-53, SURVEY 8c(v)."""
    nx = ny = 100
    assert oracle.fdrand_count(nx, ny, 1) == 79600
    I, J, V = oracle.fdrand_stream(nx, ny, 1, ones=True)
    A = oracle.OracleExt(nx * ny, nx * ny)
    if flavour == 2:  # A[i,j] += v
        for i, j, v in zip(I, J, V):
            A[i, j] = A[i, j] + v
    else:
        A.insert_batch(I, J, V, flavour)
    cp, rv, nz = A.csc()
    assert len(nz) == 49600
    cols = np.repeat(np.arange(1, nx * ny + 1), np.diff(cp))
    off = rv != cols
    assert np.all(nz[off] == -1.0)
    ix = (cols[~off] - 1) % nx + 1
    iy = (cols[~off] - 1) // nx + 1
    interior = (ix > 1) & (ix < nx) & (iy > 1) & (iy < ny)
    assert np.all(nz[~off][interior] == 4.0)
    corner = ((ix == 1) | (ix == nx)) & ((iy == 1) | (iy == ny))
    assert np.allclose(nz[~off][corner], 2.02, rtol=1e-14)
    edge = ~interior & ~corner
    assert np.allclose(nz[~off][edge], 3.01, rtol=1e-14)
    # closed-form colptr: 3/4/5 entries per column
    per_col = 1 + (ix > 1) + (ix < nx) + (iy > 1) + (iy < ny)
    assert np.array_equal(np.diff(cp), per_col)


def test_fdrand_sizes(oracle):
    assert oracle.fdrand_count(200, 200, 200) == 95_760_000
    assert oracle.fdrand_count(400, 400, 400) == 767_040_000
    assert oracle.fem_count(128, 128, 128) == 245_805_960
    assert oracle.blockrd_count(96, 96, 96, 4) == 182_255_616


def test_fdrand_3d_vs_scipy(oracle):
    I, J, V = oracle.fdrand_stream(7, 6, 5, seed=3)
    A = oracle.OracleExt(210, 210)
    A.insert_batch(I, J, V, oracle.UPDATE)
    cp, rv, nz = A.csc()
    S = sp.coo_matrix((V, (I - 1, J - 1)), shape=(210, 210)).tocsc()
    S.sort_indices()
    assert np.array_equal(S.indptr + 1, cp) and np.array_equal(S.indices + 1, rv)
    assert np.allclose(S.data, nz, rtol=1e-13)
    # M-matrix: positive diagonal, non-positive off-diagonal, weakly diagonally dominant
    D = S.toarray()
    assert np.all(np.diag(D) > 0) and np.all(D - np.diag(np.diag(D)) <= 0)
    assert np.all(D.sum(axis=1) >= -1e-12)


def test_fem_stream_properties(oracle):
    n = 5
    I, J, V = oracle.fem_stream(n, n, n)
    assert len(V) == 20 * 6 * (n - 1) ** 3
    A = oracle.OracleExt(n ** 3, n ** 3)
    A.insert_batch(I, J, V, oracle.RAW)
    cp, rv, nz = A.csc()
    S = sp.csc_matrix((nz, rv - 1, cp - 1), shape=(n ** 3, n ** 3))
    assert abs(S - S.T).max() < 1e-13
    # stiffness rows sum to zero; what remains is the lumped mass 0.1*vol/4 per tet-vertex: total 0.1*|Omega|
    assert abs(S.sum() - 0.1) < 1e-12
    # interior node of a Kuhn mesh has 14 neighbours
    mid = (n // 2) * (1 + n + n * n)
    assert cp[mid + 1] - cp[mid] == 15


def test_lu_pattern_contract(oracle):
    """test/test_lu.jl:7-45: diagonal update keeps the pattern, (i,i+-3) changes it."""
    I, J, V = oracle.fdrand_stream(20, 1, 1, ones=True)
    A = oracle.OracleExt(20, 20)
    A.insert_batch(I, J, V, oracle.UPDATE)
    cp0, rv0, _ = A.csc()
    nf = A.nflush
    for i in range(1, 21):
        A[i, i] = A[i, i] + 1.0
    cp1, rv1, _ = A.csc()
    assert A.nflush == nf and np.array_equal(cp0, cp1) and np.array_equal(rv0, rv1)
    for i in range(4, 18):
        A[i, i + 3] = A[i, i + 3] - 1.0e-4
        A[i - 3, i] = A[i - 3, i] - 1.0e-4
    cp2, rv2, _ = A.csc()
    assert A.nflush == nf + 1 and len(rv2) > len(rv1)


def test_bounds_error(oracle):
    A = oracle.OracleExt(4, 5)
    for ij in [(0, 1), (5, 1), (1, 0), (1, 6)]:
        with pytest.raises(IndexError):
            A.updateindex(1.0, *ij)


def test_mt_matches_ext(oracle):
    """test/test_parallel.jl:18-26: sparse(A0) ~ sparse(A); exact for one partition."""
    I, J, V = oracle.fem_stream(4, 4, 4)
    n = 64
    A0 = oracle.OracleExt(n, n)
    A0.insert_batch(I, J, V, oracle.RAW)
    A1 = oracle.OracleMT(n, n, 1)
    A1.insert_batch(I, J, V, 1, oracle.RAW)
    for x, y in zip(A0.csc(), A1.csc()):
        assert np.array_equal(x, y)
    # 3 partitions: contiguous chunks of the stream; values agree to rounding, pattern exactly
    A3 = oracle.OracleMT(n, n, 3)
    chunks = np.array_split(np.arange(len(V)), 3)
    for t, c in enumerate(chunks):
        A3.insert_batch(I[c], J[c], V[c], t + 1, oracle.RAW)
    assert A3.nnznew > 0
    cp, rv, nz = A3.csc()
    cp0, rv0, nz0 = A0.csc()
    assert np.array_equal(cp, cp0) and np.array_equal(rv, rv0)
    assert np.allclose(nz, nz0, rtol=1e-12, atol=1e-15)
    # second assembly into the now-frozen pattern: every insert is a CSC hit
    A3.zero_values()
    for t, c in enumerate(chunks):
        A3.insert_batch(I[c], J[c], V[c], t + 1, oracle.RAW)
    assert A3.nnznew == 0
    A0.zero_values()
    A0.insert_batch(I, J, V, oracle.RAW)
    assert np.array_equal(A3.csc()[2], A0.csc()[2])


def test_mt_setindex_of_stored_entry_overwrites(oracle):
    """setindex! of an entry the CSC already holds overwrites it (genericmt...:63-68); a new one is an error.
    The oracle used to add the value, which the GPU key-layout tests caught."""
    A = oracle.OracleMT(3, 3, 2)
    A.update(1.5, 2, 2, 1, oracle.RAW)
    A.flush()
    A.update(4.0, 2, 2, 2, oracle.ASSIGN)
    A.update(0.5, 2, 2, 1, oracle.UPDATE)
    assert A.csc()[2].tolist() == [4.5]
    with pytest.raises(RuntimeError):
        A.update(1.0, 1, 1, 1, oracle.ASSIGN)


def test_mt_threaded_matches_serial(oracle):
    """testassemble_parallel! (test/femtools.jl:75-110): partitions of a colour inserted by concurrent
    threads give the bits of the serial tid-wise insertion; second assembly = CSC hits only."""
    nn = 12
    I, J, V = oracle.fem_stream(nn, nn, nn)
    n = nn ** 3
    nparts = 6
    ncells = len(V) // 20
    pb = 20 * (np.arange(nparts + 1) * ncells // nparts)
    A = oracle.OracleMT(n, n, nparts)
    for t in range(nparts):
        sl = slice(pb[t], pb[t + 1])
        A.insert_batch(I[sl], J[sl], V[sl], t + 1, oracle.RAW)
    ref = A.csc()
    for nthreads in (1, 3, 8):
        B = oracle.OracleMT(n, n, nparts)
        B.insert_partitioned(I, J, V, pb, nthreads, oracle.RAW)
        got = B.csc()
        for x, y in zip(ref, got):
            assert np.array_equal(x.view(np.int64), y.view(np.int64))
        B.zero_values()
        B.insert_partitioned(I, J, V, pb, nthreads, oracle.RAW)
        assert B.nnznew == 0
    A0 = oracle.OracleExt(n, n)
    A0.insert_batch(I, J, V, oracle.RAW)
    cp0, rv0, nz0 = A0.csc()
    assert np.array_equal(ref[0], cp0) and np.array_equal(ref[1], rv0)
    assert np.allclose(ref[2], nz0, rtol=1e-12, atol=1e-15)


def test_dirichlet(oracle):
    """test/test_dirichlet.jl:7-28 (values-only passes, sparsematrixcsc.jl:97-148)."""
    I, J, V = oracle.fdrand_stream(6, 5, 1, seed=11)
    n = 30
    A = oracle.OracleExt(n, n)
    A.insert_batch(I, J, V, oracle.UPDATE)
    A.flush()
    for i in range(1, n + 1, 10):
        A[i, i] = 1.0e30
    mk = A.mark_dirichlet()
    assert mk.nonzero()[0].tolist() == [0, 10, 20]
    A.eliminate_dirichlet(mk)
    cp, rv, nz = A.csc()
    D = sp.csc_matrix((nz, rv - 1, cp - 1), shape=(n, n)).toarray()
    for d in (0, 10, 20):
        assert D[d, d] == 1.0 and np.count_nonzero(D[d, :]) == 1 and np.count_nonzero(D[:, d]) == 1


def test_pointblock_hand_vector(oracle):
    """pointblock (src/matrix/extendable.jl:292-318), stepped through by hand on a 4x4 matrix with
    blocksize 2: the block index of A's COLUMN becomes the block row, single-entry blocks are summed."""
    A = oracle.OracleExt(4, 4)
    for v, i, j in [(1.0, 1, 1), (2.0, 2, 1), (3.0, 3, 2), (4.0, 1, 4), (-0.0, 4, 4)]:
        A.rawupdateindex(v, i, j)
    cp, rv, bl = A.pointblock(2)
    assert cp.tolist() == [1, 3, 5] and rv.tolist() == [1, 2, 1, 2]
    # column-major blocks: [b11, b21, b12, b22]
    assert bl.tolist() == [[1.0, 0.0, 2.0, 0.0], [0.0, 4.0, 0.0, 0.0], [0.0, 3.0, 0.0, 0.0], [0.0, 0.0, 0.0, 0.0]]
    assert not np.signbit(bl).any()  # zero(Tb) + block: -0.0 becomes +0.0
    # blocksize 1: Ab[i,j] = A[j,i]
    cp1, rv1, bl1 = A.pointblock(1)
    S = sp.csc_matrix((A.csc()[2], A.csc()[1] - 1, A.csc()[0] - 1), shape=(4, 4))
    T = sp.csc_matrix((bl1[:, 0], rv1 - 1, cp1 - 1), shape=(4, 4))
    assert np.array_equal(T.toarray(), S.toarray().T)
    # an entry beyond nblock*blocksize is the reference's BoundsError
    B = oracle.OracleExt(5, 5)
    B.rawupdateindex(1.0, 1, 1)
    B.rawupdateindex(1.0, 2, 5)
    with pytest.raises(IndexError):
        B.pointblock(2)
    B2 = oracle.OracleExt(5, 5)
    B2.rawupdateindex(1.0, 4, 3)
    assert B2.pointblock(2)[1].tolist() == [2]


def test_pointblock_dense_property(oracle):
    """Every stored A[j,i] lands at Ab[(i-1)/bs+1, (j-1)/bs+1][(i-1)%bs+1, (j-1)%bs+1]; nothing else is set."""
    I, J, V = oracle.fdrand_stream(6, 4, 2, seed=5)
    n, bs = 48, 4
    A = oracle.OracleExt(n, n)
    A.insert_batch(I, J, V, oracle.UPDATE)
    cp, rv, nz = A.csc()
    D = sp.csc_matrix((nz, rv - 1, cp - 1), shape=(n, n)).toarray()
    bcp, brv, bl = A.pointblock(bs)
    nb = n // bs
    R = np.zeros((n, n))
    for jb in range(nb):
        for k in range(bcp[jb] - 1, bcp[jb + 1] - 1):
            ib = brv[k] - 1
            R[ib * bs:(ib + 1) * bs, jb * bs:(jb + 1) * bs] = bl[k].reshape(bs, bs).T  # column-major block
    assert np.array_equal(R, D.T)


def _esmp_case(seed, n=60, nt=4, cnt=3000):
    """Random assembly through the ESMP restatement: columns owned by slab threads, separator columns by two."""
    rng = np.random.default_rng(seed)
    owners = []
    for j in range(n):
        t = j * nt // n + 1
        owners.append([t] if j % 7 else sorted({t, t % nt + 1}))
    calls = []
    for _ in range(cnt):
        j = int(rng.integers(1, n + 1))
        tid = int(rng.choice(owners[j - 1]))
        v = float(rng.standard_normal()) if rng.random() > 0.05 else 0.0
        calls.append((int(rng.integers(1, n + 1)), j, tid, v))
    return owners, calls


def test_esmp_restatement_matches_dense_accumulation():
    """oracle/esmp.py (ExtendableSparseMatrixParallel: addtoentry! + sparse flush!, local column remap) against a
    dense accumulator over two splices: test/ExperimentalParallel.jl:273-343 asks for `≈` and the CSC invariants."""
    from oracle.esmp import ESMP

    n, nt = 60, 4
    owners, calls = _esmp_case(5, n, nt)
    A = ESMP(n, nt, owners)
    D = np.zeros((n, n))
    touched = np.zeros((n, n), bool)
    for part in (calls[:1500], calls[1500:]):
        for i, j, tid, v in part:
            A.addtoentry(i, j, tid, v)
            D[i - 1, j - 1] += v
            touched[i - 1, j - 1] |= (v != 0.0)
        A.flush()
        cp, rv, nz = A.csc()
        assert cp[0] == 1 and cp[-1] == len(rv) + 1
        got = np.zeros((n, n))
        for j in range(n):
            rows = rv[cp[j] - 1:cp[j + 1] - 1]
            assert np.all(np.diff(rows) > 0)
            got[rows - 1, j] = nz[cp[j] - 1:cp[j + 1] - 1]
        assert np.allclose(got, D, rtol=1e-13, atol=1e-13)
        # the pattern holds every entry that received a non-zero value (zero-sum entries stay: keep_zeros)
        pat = np.zeros((n, n), bool)
        for j in range(n):
            pat[rv[cp[j] - 1:cp[j + 1] - 1] - 1, j] = True
        assert np.all(pat[touched])
