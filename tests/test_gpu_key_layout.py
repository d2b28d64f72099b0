"""GPU tests of assembly at the limits of the packed record key.

A staged record's 64-bit key packs, from the bottom up, [flavour:2][tid:tidbits][row:rowbits][col:colbits]
[owner:ownerbits] (xsb_common.cuh); xsb_create sizes every field with ceil_log2 and accepts any layout up to 64 bits.
Which flush runs depends on that layout:
  - column_path 4 (grouped chunks, and grouping at insertion): rowbits <= 26, no tid bits, colbits + ownerbits <= 31;
  - column_path 2 / 3 (column sort or grouping, then a hash fold per column): rowbits <= 26;
  - column_path 0 ((col,row) radix sort of up to 62 bits, flat reduction): everything else.
Every case here sits on one side of one of these gates: matrices of 2^26 .. 2^32 rows, a full 64-bit key through
65536 partitions, the owner bit of a slab handle as key bit 63.  Device memory and the CPU oracle are O(n + records),
never O(m), so a matrix with 2^32 rows and a few hundred columns costs a few MB.

Bar (as in test_gpu_parity.py): colptr / rowval exact, nzval bit-exact in XSB_DETERMINISTIC, within 1e-14 relative
in XSB_FAST with the pattern exact."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def xsb():
    import __graft_entry__ as ge

    ge.build()
    import xsparse_b200

    assert xsparse_b200.capi.device_count() > 0, "no CUDA device: GPU tests need the real extension on a GPU"
    return xsparse_b200


@pytest.fixture(scope="module")
def torch():
    import torch

    assert torch.cuda.is_available()
    return torch


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


VALUES = np.array([0.0, -0.0, 1.0, -1.0, 0.5, 1e-3, 1e30, -1e30])


def special_rows(m):
    """0-based rows at the field boundaries that exist in an m-row matrix."""
    cand = [0, 1, 2 ** 26 - 1, 2 ** 26, 2 ** 26 + 1, 2 ** 31 - 1, 2 ** 31, 2 ** 31 + 1, 2 ** 32 - 1, m - 2, m - 1]
    return np.array(sorted({r for r in cand if 0 <= r < m}), np.int64)


def make_batch(rng, m, n, cnt, wrap=True):
    """0-based (rows, cols, values).  A quarter of the rows come from special_rows, so each of them repeats; the
    columns of every 512 consecutive calls lie in a window of 128 (the column locality grouped flushes need); values
    are signed zeros, small numbers and +-1e30 that cancel."""
    rows = rng.integers(0, m, cnt, dtype=np.int64)
    pick = rng.random(cnt) < 0.25
    rows[pick] = rng.choice(special_rows(m), int(pick.sum()))
    start = rng.integers(0, n, (cnt + 511) // 512)
    if wrap:  # the first window holds the last and the first columns
        start[0] = n - 64
    cols = (np.repeat(start, 512)[:cnt] + rng.integers(0, 128, cnt)) % n
    vals = rng.choice(VALUES, cnt) * rng.choice([1.0, rng.random()], cnt)
    return rows, cols.astype(np.int64), vals


class Layout:
    """One matrix shape: m rows, n (owned) columns, index type and base, the partitions it uses (tids) or the slab
    splits of which it is rank 1 of 2."""

    def __init__(self, m, n, idx, base, tids=None, splits=None):
        self.m, self.idx, self.base, self.tids, self.splits = m, idx, base, tids, splits
        self.n = n if splits is None else splits[2] - splits[1]
        self.col_begin = 0 if splits is None else splits[1]
        self.dt = np.int64 if idx == 1 else np.int32

    def handle(self, xsb):
        if self.splits is not None:
            return xsb.Handle(self.m, self.splits[2], self.idx, self.base, slab=(2, 1, self.splits))
        return xsb.Handle(self.m, self.n, self.idx, self.base, n_tid=65536 if self.tids else 1)

    def index(self, rows, cols):
        """Handle indices of 0-based rows and owned columns (slab handles insert global columns)."""
        return (rows + self.base).astype(self.dt), (cols + self.col_begin + self.base).astype(self.dt)

    def one_based(self, csc):
        cp, rv, nz = csc
        return cp.astype(np.int64) + 1 - self.base, rv.astype(np.int64) + 1 - self.base, nz


class Reference:
    """The oracle of one layout (0-based indices in, 1-based CSC out).  A multi-partition handle is checked against
    OracleMT over the partitions it uses, numbered in order (empty partitions add nothing); a slab handle against
    OracleExt over its own columns (a slab's columns do not depend on the others)."""

    def __init__(self, oracle, lay):
        self.oracle, self.m, self.n = oracle, lay.m, lay.n
        self.parts = sorted(lay.tids) if lay.tids else None
        self.A = oracle.OracleMT(lay.m, lay.n, len(self.parts)) if self.parts else oracle.OracleExt(lay.m, lay.n)

    def insert(self, calls):
        """calls: [(tid, rows, cols, vals, flavour)] in call order; the partitions are summed in partition order."""
        if self.parts is None:
            for _, r, c, v, fl in calls:
                self.A.insert_batch(r + 1, c + 1, v, fl)
            return
        for p, t in enumerate(self.parts):
            for tt, r, c, v, fl in calls:
                if tt == t:
                    self.A.insert_batch(r + 1, c + 1, v, tid=p + 1, flavour=fl)

    def csc(self):
        return self.A.flush().csc() if self.parts else self.A.csc()

    def plus(self, calls):
        """The CSC after a COMBINE_ADD flush of `calls`: SparseMatrixLNK of the calls + the resident CSC."""
        L = self.oracle.OracleLNK(self.m, self.n)
        op = {0: L.updateindex, 1: L.rawupdateindex}
        for _, rows, cols, vals, fl in calls:
            for i, j, v in zip(rows.tolist(), cols.tolist(), vals.tolist()):
                if fl == 2:
                    L[i + 1, j + 1] = v
                else:
                    op[fl](v, i + 1, j + 1)
        return L.plus_csc(self.m, self.n, *self.csc())


def route_and_flush(h, torch, mode=0, combine=0):
    """A slab handle staged only its own columns: route nothing out, receive nothing from rank 0, flush."""
    if getattr(h, "n_ranks", 0):
        cnt = h.pending
        assert h.route_count() == [0, cnt]
        buf = torch.empty(2, dtype=torch.int64, device="cuda")
        assert h.route_prepare(buf, 0) == [0, cnt]
        h.route_finish(0, buf, 0)
    return h.flush(mode, combine)


def device_csc(torch, h):
    dt = torch.int64 if h.idx_dtype == np.int64 else torch.int32
    cp = torch.empty(h.n + 1, dtype=dt, device="cuda")
    rv = torch.empty(max(h.nnz, 1), dtype=dt, device="cuda")
    nz = torch.empty(max(h.nnz, 1), dtype=torch.float64, device="cuda")
    h.fetch_csc(cp, rv, nz)
    return cp.cpu().numpy(), rv[: h.nnz].cpu().numpy(), nz[: h.nnz].cpu().numpy()


def assemble_and_check(xsb, oracle, torch, lay, paths, seed):
    """Three splicing flushes of interleaved flavours, host and device arrays and outputs, get_values in the highest
    rows, the pattern of a STRATEGY_FULLSORT twin, XSB_FAST with and without pre-aggregation, a frozen pattern's
    re-assembly, a COMBINE_ADD flush and y = A*x -- each against the oracle."""
    rng = np.random.default_rng(seed)
    m, n = lay.m, lay.n
    h = lay.handle(xsb)
    g = lay.handle(xsb)
    g.set_strategy(xsb.capi.STRATEGY_FULLSORT)
    ref = Reference(oracle, lay)
    tids = lay.tids or [0]
    cnt = min(256, 3 * n // 2)  # calls per batch: columns stay short enough for the grouped flush's per-thread tables

    def insert(handles, calls, device=False):
        for t, r, c, v, fl in calls:
            I, J = lay.index(r, c)
            if device:
                I, J, v = (torch.from_numpy(a).cuda() for a in (I, J, v))
            for x in handles:
                x.insert_batch(I, J, v, fl, tid=t)
        ref.insert(calls)

    resident = None
    for step in range(3):
        calls = []
        for b in range(4):
            fl = (xsb.UPDATE, xsb.RAW, xsb.ASSIGN, xsb.UPDATE)[(b + step) % 4]
            t = tids[(b + step) % len(tids)]  # partitions deliver out of order: 65535 first
            rows, cols, vals = make_batch(rng, m, n, cnt, wrap=b == 0)
            if fl == xsb.ASSIGN and lay.tids:  # A[i,j] = v of a multi-partition matrix: only positions already stored
                if resident is None:
                    fl = xsb.RAW
                else:
                    k = rng.integers(0, len(resident[1]), len(vals))
                    rows = resident[1][k] - 1
                    cols = np.repeat(np.arange(n), np.diff(resident[0]))[k]
            calls.append((t, rows, cols, vals, fl))
        insert((h, g), calls, device=step == 1)
        route_and_flush(h, torch)
        assert h.flush_stats()["column_path"] in paths
        route_and_flush(g, torch)
        assert g.flush_stats()["column_path"] == 0
        resident = ref.csc()
        got = h.fetch_csc_numpy()
        assert_csc_equal(lay.one_based(got), resident)
    dev = device_csc(torch, h)
    for a, b in zip(dev, got):
        assert np.array_equal(a, b) and a.dtype == b.dtype
    assert h.pattern_hash() == g.pattern_hash() and h.pattern_equal(g)
    g.close()

    # get_values at present and absent positions of the highest rows (absent reads 0.0)
    ocp, orv, onz = resident
    ocol = np.repeat(np.arange(n), np.diff(ocp))
    stored = dict(zip(zip((orv - 1).tolist(), ocol.tolist()), onz))
    top = np.argsort(orv, kind="stable")[-200:]  # entries of the highest rows
    qr = np.concatenate([orv[top] - 1] + [np.full(n, m - d) for d in (1, 2, 3)])
    qc = np.concatenate([ocol[top]] + [np.arange(n)] * 3)
    want = np.array([stored.get((i, j), 0.0) for i, j in zip(qr.tolist(), qc.tolist())])
    assert sum((i, j) not in stored for i, j in zip(qr.tolist(), qc.tolist())) >= n // 2  # absent positions too
    I, J = lay.index(qr, qc)
    J = J - lay.col_begin  # lookups take the owned (local) columns of a slab handle, like fetch_csc
    out = torch.empty(len(qr), dtype=torch.float64, device="cuda")
    h.get_values(torch.from_numpy(I).cuda(), torch.from_numpy(J).cuda(), out)
    assert np.array_equal(bits(h.get_values(I, J)), bits(want))
    assert np.array_equal(bits(out.cpu().numpy()), bits(want))

    # XSB_FAST, then XSB_FAST with pre-aggregation on a stream of at least 4096 calls.  The values are positive: a
    # reordered sum stays within 1e-14 of the serial one only without cancellation.
    for preagg in (False, True):
        h.zero_values()
        ref.A.zero_values()
        h.set_preaggregation(preagg)
        calls = []
        for b, fl in enumerate((xsb.UPDATE, xsb.RAW, xsb.UPDATE)):
            rows, cols, _ = make_batch(rng, m, n, 1400)
            calls.append((tids[b % len(tids)], rows, cols, 1.0 + rng.random(len(rows)), fl))
        insert((h,), calls)
        route_and_flush(h, torch, xsb.FAST)
        if preagg:
            assert h.flush_stats()["preagg_records"] > 0
        assert_csc_equal(lay.one_based(h.fetch_csc_numpy()), ref.csc(), exact=False)
    h.set_preaggregation(False)
    h.zero_values()  # back to bit-exact values on both sides
    ref.A.zero_values()

    # freeze the pattern, re-assemble values into it
    ocp, orv, _ = ref.csc()
    ocol = np.repeat(np.arange(n), np.diff(ocp))
    perm = rng.permutation(len(orv))
    top = np.argsort(orv, kind="stable")[-100:]
    fr = np.concatenate([orv[perm], orv[top]]) - 1
    fc = np.concatenate([ocol[perm], ocol[top]])
    FV = rng.choice(VALUES, len(fr)) * rng.random(len(fr))
    I, J = lay.index(fr, fc)
    h.freeze_pattern(I, J - lay.col_begin)
    upd = [(lay.tids[0] if lay.tids else 0, fr, fc, FV, xsb.UPDATE)]
    h.zero_values()
    h.reassemble_values(FV, xsb.DETERMINISTIC)
    ref.A.zero_values()
    ref.insert(upd)
    assert_csc_equal(lay.one_based(h.fetch_csc_numpy()), ref.csc())
    h.reassemble_values(FV, xsb.DETERMINISTIC)  # on top, without zeroing
    ref.insert(upd)
    assert_csc_equal(lay.one_based(h.fetch_csc_numpy()), ref.csc())
    h.reassemble_values(FV, xsb.FAST, zero_first=True)
    ref.A.zero_values()
    ref.insert(upd)
    assert_csc_equal(lay.one_based(h.fetch_csc_numpy()), ref.csc(), exact=False)
    h.reassemble_values(FV, xsb.DETERMINISTIC, zero_first=True)
    assert_csc_equal(lay.one_based(h.fetch_csc_numpy()), ref.csc())
    h.unfreeze()

    # COMBINE_ADD: the staged calls as a SparseMatrixLNK, added to the resident CSC
    calls = []
    for b, fl in enumerate((xsb.UPDATE, xsb.RAW, xsb.UPDATE) if lay.tids else (xsb.UPDATE, xsb.ASSIGN, xsb.RAW)):
        rows, cols, vals = make_batch(rng, m, n, cnt)
        calls.append((tids[-1], rows, cols, vals, fl))
    for t, r, c, v, fl in calls:
        h.insert_batch(*lay.index(r, c), v, fl, tid=t)
    want = ref.plus(calls)
    route_and_flush(h, torch, xsb.DETERMINISTIC, xsb.COMBINE_ADD)
    got = h.fetch_csc_numpy()
    assert_csc_equal(lay.one_based(got), want)

    # y = A*x where the 32-bit row-major map is allowed and its O(m) arrays are affordable
    if m <= 2 ** 27 + 1:
        x = rng.standard_normal(n)
        cp, rv, nz = lay.one_based(got)
        y_ref = np.zeros(m)
        np.add.at(y_ref, rv - 1, nz * x[np.repeat(np.arange(n), np.diff(cp))])  # columns ascending, unbuffered
        assert np.array_equal(bits(h.mul(x)), bits(y_ref))
    h.close()


I32, I64 = 0, 1
W = 40  # columns of the narrow slab
S31 = [0, 2 ** 30, 2 ** 30 + W]  # widest slab 2^30 columns: colbits + ownerbits = 31
S32 = [0, 2 ** 30 + 1, 2 ** 30 + 1 + W]  # widest slab 2^30 + 1 columns: colbits + ownerbits = 32
TIDS = [65535, 0, 1]

LAYOUTS = {
    # row gate: rowbits 26 | 27 .. 32
    "rows26-i64-b1": (Layout(2 ** 26, 1000, I64, 1), (4,)),
    "rows26-i32-b0": (Layout(2 ** 26, 1000, I32, 0), (4,)),
    "rows27-i64-b0": (Layout(2 ** 26 + 1, 1000, I64, 0), (0,)),
    "rows27-i32-b1": (Layout(2 ** 26 + 1, 1000, I32, 1), (0,)),
    "rows31-i32-limit-b1": (Layout(2 ** 31 - 2, 1000, I32, 1), (0,)),
    "rows31-i32-limit-b0": (Layout(2 ** 31 - 2, 1000, I32, 0), (0,)),
    "rows31-i64-b0": (Layout(2 ** 31 - 1, 1000, I64, 0), (0,)),
    "rows31-i64-b1": (Layout(2 ** 31, 1000, I64, 1), (0,)),
    "rows32-i64-b0": (Layout(2 ** 32 - 1, 1000, I64, 0), (0,)),
    "rows32-i64-b1": (Layout(2 ** 32 - 1, 1000, I64, 1), (0,)),
    "rows32-full-i64-b0": (Layout(2 ** 32, 1000, I64, 0), (0,)),
    "rows32-full-i64-b1": (Layout(2 ** 32, 1000, I64, 1), (0,)),
    # 65536 partitions: 2 + 16 + 26 + 20 = 64 key bits on the hash-fold path, 2 + 16 + 27 + 19 = 64 on the sort
    "tid16-colfold-i32-b1": (Layout(2 ** 26, 2 ** 20, I32, 1, tids=TIDS), (2, 3)),
    "tid16-sort-i64-b0": (Layout(2 ** 26 + 1, 2 ** 19, I64, 0, tids=TIDS), (0,)),
    # owner bit on top of a slab handle's key
    "owner31-i32-b0": (Layout(2 ** 26, None, I32, 0, splits=S31), (4,)),
    "owner32-i64-b1": (Layout(2 ** 26, None, I64, 1, splits=S32), (2, 3)),
    "owner-bit63-i32-b1": (Layout(2 ** 30, None, I32, 1, splits=S32), (0,)),  # 2 + 30 + 31 + 1 = 64
}


@pytest.mark.parametrize("name", list(LAYOUTS))
def test_layout_matches_oracle(xsb, oracle, torch, name):
    lay, paths = LAYOUTS[name]
    assemble_and_check(xsb, oracle, torch, lay, paths, seed=sum(map(ord, name)))


def test_key_wider_than_64_bits_is_refused(xsb):
    """The 64-bit layouts of the partition cases with one more column bit."""
    for m, n in [(2 ** 26, 2 ** 21), (2 ** 26 + 1, 2 ** 20)]:
        with pytest.raises(xsb.XsbError) as e:
            xsb.Handle(m, n, n_tid=65536)
        assert e.value.code == xsb.capi.EINVAL
    with pytest.raises(xsb.XsbError) as e:
        xsb.Handle(2 ** 30 + 1, S32[2], slab=(2, 1, S32))  # 2 + 31 + 31 + 1 = 65
    assert e.value.code == xsb.capi.EINVAL


# ---------------------------------------------------------------- rejections at the bit boundaries
def bad_indices(m, idx, base):
    """Indices outside the matrix: the first one past the end, negatives, and (64-bit) values whose low 32 bits
    are an index in range."""
    r = base + 3
    bad = [m + base, -1]
    if idx == I64:
        bad += [2 ** 32 + r, 2 ** 31 + r, -(2 ** 63)]
    else:
        bad += [-(2 ** 31)]
    return [b for b in bad if idx == I64 or -(2 ** 31) <= b < 2 ** 31]


@pytest.mark.parametrize("idx,base,m", [(I64, 0, 1000), (I64, 1, 1000), (I64, 1, 2 ** 31 - 2), (I32, 0, 2 ** 31 - 2),
                                        (I32, 1, 2 ** 31 - 2), (I32, 1, 1000)])
def test_rejections_leave_the_handle_intact(xsb, oracle, idx, base, m):
    """insert_batch, insert_elements, get_values and freeze_pattern refuse every bad index with IndexError
    (XSB_EBOUNDS), leave the pending calls as they were, and the next flush is right."""
    rng = np.random.default_rng(m + 10 * idx + base)
    n = 600
    lay = Layout(m, n, idx, base)
    dt = lay.dt
    h = lay.handle(xsb)
    ref = oracle.OracleExt(m, n)
    rows, cols, vals = make_batch(rng, m, n, 3000)
    h.insert_batch(*lay.index(rows, cols), vals, xsb.UPDATE)
    ref.insert_batch(rows + 1, cols + 1, vals, oracle.UPDATE)
    h.flush()
    rows, cols, vals = make_batch(rng, m, n, 2000)
    I, J = lay.index(rows, cols)
    h.insert_batch(I, J, vals, xsb.RAW)
    ref.insert_batch(rows + 1, cols + 1, vals, oracle.RAW)
    pending = h.pending
    dofs = (rng.integers(0, min(m, n), (50, 4)) + base).astype(dt)
    A = rng.standard_normal((50, 4, 4))
    for bad in bad_indices(m, idx, base):
        for which in (0, 1):
            Ib, Jb = I.copy(), J.copy()
            (Ib, Jb)[which][17] = bad
            with pytest.raises(IndexError, match="entry 17"):
                h.insert_batch(Ib, Jb, vals, xsb.UPDATE)
            assert h.pending == pending
        d = dofs.copy()
        d[5, 2] = bad
        with pytest.raises(IndexError, match="element 5 "):
            h.insert_elements(d, A, xsb.RAW)
        assert h.pending == pending
    h.flush()
    assert_csc_equal(lay.one_based(h.fetch_csc_numpy()), ref.csc())
    nnz = h.nnz
    qI, qJ = I[:40].copy(), J[:40].copy()
    for bad in bad_indices(m, idx, base):
        for which in (0, 1):
            Ib, Jb = qI.copy(), qJ.copy()
            (Ib, Jb)[which][3] = bad
            with pytest.raises(IndexError):
                h.get_values(Ib, Jb)
            with pytest.raises(IndexError):
                h.freeze_pattern(Ib, Jb)
            assert h.pending == 0 and h.nnz == nnz
    # the handle still assembles correctly, and a freeze of good positions works
    rows, cols, vals = make_batch(rng, m, n, 2000)
    h.insert_batch(*lay.index(rows, cols), vals, xsb.ASSIGN)
    ref.insert_batch(rows + 1, cols + 1, vals, oracle.ASSIGN)
    h.flush()
    ocp, orv, onz = ref.csc()
    assert_csc_equal(lay.one_based(h.fetch_csc_numpy()), (ocp, orv, onz))
    want = np.array([ref[int(i) + 1 - base, int(j) + 1 - base] for i, j in zip(qI, qJ)])
    assert np.array_equal(bits(h.get_values(qI, qJ)), bits(want))


def triplets(xsb, I, J, V):
    T = np.empty(len(V), xsb.capi.TRIPLET_DTYPE)
    T["row"], T["col"], T["val"] = I, J, V
    return T


def test_triplets_at_32_bit_rows(xsb, oracle):
    """Triplets carry 32-bit indices: m = 2^32 - 1 is accepted, and row 0xFFFFFFFF is valid under base 1;
    m = 2^32 is refused with XSB_EINVAL."""
    rng = np.random.default_rng(32)
    m, n = 2 ** 32 - 1, 300
    h = xsb.Handle(m, n)
    ref = oracle.OracleExt(m, n)
    for fl in (xsb.RAW, xsb.UPDATE, xsb.ASSIGN):
        rows, cols, vals = make_batch(rng, m, n, 3000)
        rows[:5] = m - 1  # index 0xFFFFFFFF
        h.insert_triplets(triplets(xsb, rows + 1, cols + 1, vals), fl)
        ref.insert_batch(rows + 1, cols + 1, vals, fl)
        h.flush()
        assert h.flush_stats()["column_path"] == 0
        assert_csc_equal(h.fetch_csc_numpy(), ref.csc())
    assert h.fetch_csc_numpy()[1].max() == 2 ** 32 - 1
    g = xsb.Handle(2 ** 32, n)
    with pytest.raises(xsb.XsbError) as e:
        g.insert_triplets(triplets(xsb, [1], [1], [1.0]), xsb.RAW)
    assert e.value.code == xsb.capi.EINVAL and g.pending == 0


# ---------------------------------------------------------------- producers that group at insertion
def spread_elements(rng, m, ncells, k, ends):
    """0-based dofs of elements spread over [0, m): each element's dofs lie near its own random point, so that a
    chunk meets few columns; with `ends` the first element holds dof 0, the last dof m - 1."""
    lo = np.sort(rng.integers(0, m - 3 * k - 2, ncells))
    dofs = lo[:, None] + np.stack([rng.permutation(3 * k + 2)[:k] for _ in range(ncells)])
    if ends:
        dofs[0, 0] = 0
        dofs[-1, -1] = m - 1
    A = rng.choice(VALUES, (ncells, k, k)) * rng.choice([1.0, rng.random()], (ncells, k, k))
    return dofs.astype(np.int64), A


def expand(dofs, Aloc):
    """The call stream of the element loop: call k^2 c + k jl + il = (dofs[c, il], dofs[c, jl], Aloc[c, jl, il])."""
    nc, k = dofs.shape
    I = np.broadcast_to(dofs[:, None, :], (nc, k, k)).reshape(-1).copy()
    J = np.broadcast_to(dofs[:, :, None], (nc, k, k)).reshape(-1).copy()
    return I, J, np.ascontiguousarray(Aloc, np.float64).reshape(-1).copy()


@pytest.mark.parametrize("nzn", [2 ** 24, 2 ** 24 + 1])
def test_grouping_producers_above_26_row_bits(xsb, oracle, torch, nzn):
    """insert_elements (k = 4, 27; Int32 and Int64 dofs), insert_triplets and emit_p1fem_range on a square matrix of
    2 x 2 x nzn nodes: 2^26 (grouped at insertion, column_path 4) against 2^26 + 4 (27 row bits: neither producer
    nor flush may group)."""
    m = 4 * nzn
    tall = m > 2 ** 26
    rng = np.random.default_rng(nzn)
    h64 = xsb.Handle(m, m, I64, 1)
    h32 = xsb.Handle(m, m, I32, 0)
    ref = oracle.OracleExt(m, m)

    def check():
        for h, base in ((h64, 1), (h32, 0)):
            h.flush()
            st = h.flush_stats()
            assert st["column_path"] == (0 if tall else 4)
            if not tall:
                assert st["precounted"] > 0.99
        want = ref.csc()
        for h, base in ((h64, 1), (h32, 0)):
            cp, rv, nz = h.fetch_csc_numpy()
            assert_csc_equal((cp.astype(np.int64) + 1 - base, rv.astype(np.int64) + 1 - base, nz), want)
        return want

    frozen = None
    for k, ncells, fl in ((4, 3000, xsb.RAW), (27, 40, xsb.UPDATE)):
        dofs, A = spread_elements(rng, m, ncells, k, ends=k == 4)  # a column of both would be too rich for path 4
        h64.insert_elements(dofs + 1, A, fl)
        h32.insert_elements(torch.from_numpy((dofs).astype(np.int32)).cuda(), torch.from_numpy(A).cuda(), fl)
        I, J, V = expand(dofs + 1, A)
        ref.insert_batch(I, J, V, fl)
        check()
        frozen = frozen or (dofs, A)
    rows, cols, vals = make_batch(rng, m, m, 20000, wrap=False)
    h64.insert_triplets(triplets(xsb, rows + 1, cols + 1, vals), xsb.UPDATE)
    h32.insert_triplets(triplets(xsb, rows, cols, vals), xsb.UPDATE)
    ref.insert_batch(rows + 1, cols + 1, vals, oracle.UPDATE)
    check()
    # the emitter's top cube layers; the oracle has no ranged FEM stream, so a handle that does not group stages it
    cz = (nzn - 301, nzn - 1)
    r = xsb.Handle(m, m)
    r.set_precount(False)
    r.emit_p1fem(2, 2, nzn, flavour=xsb.RAW, cz_range=cz)
    I, J, V, _ = r.debug_fetch_staged()
    r.close()
    assert len(V) == 120 * 300 and I.max() == m
    for h in (h64, h32):
        h.emit_p1fem(2, 2, nzn, flavour=xsb.RAW, cz_range=cz)
    ref.insert_batch(I, J, V, oracle.RAW)
    check()
    # freeze from the connectivity of the first element batch, re-assemble into it
    dofs, A = frozen
    A2 = rng.standard_normal(A.shape)
    I, J, V = expand(dofs + 1, A2)  # V: the element matrices as they are, call after call
    h64.freeze_elements(dofs + 1)
    h32.freeze_elements(dofs.astype(np.int32))
    for mode, exact in ((xsb.DETERMINISTIC, True), (xsb.FAST, False)):
        for h in (h64, h32):
            h.reassemble_values(V, mode, zero_first=True)
        ref.zero_values()
        ref.insert_batch(I, J, V, oracle.UPDATE)
        want = ref.csc()
        for h, base in ((h64, 1), (h32, 0)):
            cp, rv, nz = h.fetch_csc_numpy()
            assert_csc_equal((cp.astype(np.int64) + 1 - base, rv.astype(np.int64) + 1 - base, nz), want, exact=exact)
    h64.zero_values()
    h64.reassemble_values(V, xsb.DETERMINISTIC)
    cp, rv, nz = h64.fetch_csc_numpy()
    assert_csc_equal((cp, rv, nz), want)
    h64.close()
    h32.close()
