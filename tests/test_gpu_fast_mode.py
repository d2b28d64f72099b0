"""GPU tests of the order-free value paths (XSB_FAST) against exact sums, entry by entry.

Two kinds of stream run through every path:
  * fixed-point values k * 2^e (one common e, N * max|k| < 2^53): every partial sum is exact in any order, so FAST
    must equal the deterministic left fold -- the oracle's and the GPU's own DETERMINISTIC result -- bit for bit;
  * cancelling values (N(0,1), terms of 1e+-8, pairs that cancel to zero): the pattern must be exact and every entry
    within gamma(N-1) * sum|terms| of the exact sum of its N contributions (tests/fast_sum_ref.py).
A lost, doubled or misrouted contribution fails both, wherever it sits in the matrix.

Paths: the window pre-aggregation of a FAST flush (xsb_preagg.cu; its windows are 512 consecutive staged records,
its table 512 slots), the exact merge a FAST flush runs without it, and the atomic re-assembly of frozen streams
(plain, element, rectangular element and slab-frozen).  flush_stats()["preagg_records"] shows whether the windows
ran: 0 when they did not."""
import ctypes as C

import numpy as np
import pytest

from tests import fast_sum_ref as fsr

pytestmark = pytest.mark.gpu

WINDOW = fsr.PA_W
MIN_PREAGG = 4096  # a FAST flush pre-aggregates only streams of at least this many staged records


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


def cancelling_values(rng, cnt):
    """N(0,1) with one term in 16 scaled by 1e8 or 1e-8 and one in 16 an exact zero."""
    V = rng.standard_normal(cnt)
    pick = rng.random(cnt)
    V[pick < 1 / 32] *= 1e8
    V[(pick >= 1 / 32) & (pick < 1 / 16)] *= 1e-8
    V[(pick >= 1 / 16) & (pick < 1 / 8)] = 0.0
    return V


def values(rng, cnt, kind):
    """'fixed' (e = 0), 'fixed960', 'fixed-1074' or 'random' (cancelling)."""
    if kind == "random":
        return cancelling_values(rng, cnt)
    e = {"fixed": 0, "fixed960": 960, "fixed-1074": -1074}[kind]
    return fsr.fixed_point_values(rng, cnt, e)


def check(got, groups, exact, what="", base=1):
    """got = (colptr, rowval, nzval) in the handle's base against the reference groups: the pattern exactly; the
    values as the left fold's bits (exact=True, fixed-point streams) or within the order-free bound."""
    cp, rv, nz = got
    assert np.array_equal(np.asarray(cp, np.int64) - base + 1, groups.colptr), f"{what}: colptr differs"
    assert np.array_equal(np.asarray(rv, np.int64) - base + 1, groups.rowval), f"{what}: rowval differs"
    if exact:
        want = groups.left_fold()
        bad = np.flatnonzero(bits(nz) != bits(want))
        assert bad.size == 0, f"{what}: {bad.size} entries differ from the exact sum, first {bad[:4]}: " \
                              f"{nz[bad[:4]]} vs {want[bad[:4]]}"
    else:
        fsr.assert_within_order_free_bound(nz, groups, what)


def same_bits(a, b, what=""):
    for x, y, name in zip(a, b, ("colptr", "rowval", "nzval")):
        x, y = np.asarray(x), np.asarray(y)
        assert x.shape == y.shape and np.array_equal(x.view(np.uint64) if x.dtype == np.float64 else x,
                                                     y.view(np.uint64) if y.dtype == np.float64 else y), \
            f"{what}: {name} differs"


def insert_runs(h, I, J, V, F):
    """The calls in order, one batch per run of equal flavour (a handle or an OracleExt)."""
    F = np.broadcast_to(np.asarray(F), np.shape(V))
    cut = np.flatnonzero(np.diff(F)) + 1
    for a, b in zip(np.r_[0, cut], np.r_[cut, len(V)]):
        h.insert_batch(np.ascontiguousarray(I[a:b]), np.ascontiguousarray(J[a:b]), np.ascontiguousarray(V[a:b]),
                       int(F[a]))


def random_stream(rng, m, n, cnt, kind, keys=None):
    """cnt calls on `keys` distinct positions (default cnt / 16, so that a window of 512 calls meets about 300
    positions), mixed UPDATE / RAW calls with some zeros, and three pairs (v, -v) of consecutive raw calls on the last
    rows and columns."""
    nkeys = keys or max(cnt // 16, 1)
    kI = rng.integers(1, m + 1, nkeys)
    kJ = rng.integers(1, n + 1, nkeys)
    k = rng.integers(0, nkeys, cnt)
    I, J = kI[k].copy(), kJ[k].copy()
    V = values(rng, cnt, kind)
    F = rng.integers(0, 2, cnt)  # UPDATE or RAW
    for t in range(3):
        p = rng.integers(0, cnt - 1)
        I[p] = I[p + 1] = m - t
        J[p] = J[p + 1] = n - t
        V[p + 1] = -V[p]
        F[p] = F[p + 1] = fsr.RAW
    return I, J, V, F


# ================================================================ 1. FAST without pre-aggregation is the exact merge
@pytest.mark.parametrize("variant", ["product", "fullsort", "three_partitions"])
def test_fast_without_preaggregation_is_the_exact_merge(xsb, oracle, variant):
    """DESIGN.md 5: without window pre-aggregation a FAST flush is the exact merge, the same bits as DETERMINISTIC
    and the oracle, even for random values, on the product path (column_path 4) and on the fallbacks."""
    rng = np.random.default_rng(1)
    m, n = 300, 280
    ntid = 3 if variant == "three_partitions" else 1
    h = xsb.Handle(m, n, n_tid=ntid)
    if variant == "fullsort":
        h.set_strategy(xsb.capi.STRATEGY_FULLSORT)
    A = oracle.OracleMT(m, n, ntid) if ntid > 1 else oracle.OracleExt(m, n)
    for step in range(3):  # the second and third land on a resident CSC
        I, J, V, F = random_stream(rng, m, n, 20000, "random")
        if ntid > 1:
            F = np.full(len(V), fsr.RAW)
            parts = np.array_split(np.arange(len(V)), ntid)
            for t in rng.permutation(ntid):
                p = parts[t]
                h.insert_batch(I[p], J[p], V[p], xsb.RAW, tid=int(t))
            for t in range(ntid):
                p = parts[t]
                A.insert_batch(I[p], J[p], V[p], t + 1, oracle.RAW)
        else:
            insert_runs(h, I, J, V, F)
            insert_runs(A, I, J, V, F)
        h.flush(xsb.FAST)
        st = h.flush_stats()
        assert st["preagg_records"] == 0
        if variant == "product":
            assert st["column_path"] == 4
        elif variant == "fullsort":
            assert st["column_path"] == 0
        if ntid > 1:
            A.flush()
        same_bits(h.fetch_csc_numpy(), A.csc(), f"{variant} step {step}")


def test_fast_combine_add_equals_deterministic(xsb):
    """COMBINE_ADD (old + ((0 + v1) + v2)) has no oracle counterpart: FAST equals DETERMINISTIC of the same inputs."""
    rng = np.random.default_rng(2)
    m, n = 200, 220
    hs = [xsb.Handle(m, n) for _ in range(2)]
    for step in range(3):
        I, J, V, F = random_stream(rng, m, n, 12000, "random")
        for h, mode in zip(hs, (xsb.DETERMINISTIC, xsb.FAST)):
            insert_runs(h, I, J, V, F)
            h.flush(mode, xsb.capi.COMBINE_ADD)
            assert h.flush_stats()["preagg_records"] == 0
        same_bits(hs[1].fetch_csc_numpy(), hs[0].fetch_csc_numpy(), f"COMBINE_ADD step {step}")


def test_fast_wrappers_equal_deterministic(xsb, oracle):
    """ExtendableSparseMatrix(mode=FAST) and the drop-in wrapper with mode=FAST: the exact merge, bit for bit."""
    from xsparse_b200 import dropin
    from xsparse_b200.matrix import ExtendableSparseMatrix

    rng = np.random.default_rng(3)
    m, n = 150, 150
    A = ExtendableSparseMatrix(m, n, mode=xsb.FAST)
    O = oracle.OracleExt(m, n)
    D = [dropin.GenericMTExtendableSparseMatrixCSC(m, n, 1, mode=mode) for mode in (xsb.DETERMINISTIC, xsb.FAST)]
    for step in range(3):
        I, J, V, F = random_stream(rng, m, n, 6000, "random")
        F[:] = fsr.RAW
        A.insert_batch(I, J, V, xsb.RAW)
        O.insert_batch(I, J, V, oracle.RAW)
        same_bits(A.csc(), O.csc(), f"ExtendableSparseMatrix step {step}")
        for d in D:
            d.update_batch(xsb.RAW, I, J, V)
            d.flush()
        same_bits(D[1].sparse(), D[0].sparse(), f"drop-in step {step}")
    dropin.release_handles()


# ================================================================ 2. window edges
def edge_stream(rng, m, n, kind):
    """One stream (1-based I, J, V, F) of 9 * 512 + 1 calls that puts the pre-aggregation's edges at known windows
    when staged in call order.  Windows (512 calls each, numbered from 0):
      0        one position repeated 512 times
      1        512 distinct positions of one hash slot (full table, probe chains that wrap around it)
      2.5-3.5  the same 512 positions again, straddling the boundary of windows 2 and 3
      5        position P0 receives only zero updates; window 6 creates it with a raw call
      5-7      position P1 receives only zero updates (+0.0 and -0.0): it must not appear
      7        position P2 receives v and -v, nothing else: it stays, with +0.0
      8        random traffic
      9        a single call (the last, partial window)
    The rest is random traffic on the left half of the matrix.  The calls that end the truncations TRUNCATIONS
    (the last call of each) are raw calls on positions nobody else has, so a stream cut there misses a whole entry if
    its last record is lost."""
    W = WINDOW
    cnt = 9 * W + 1
    I = rng.integers(1, m // 2, cnt)
    J = rng.integers(1, n // 2, cnt)
    F = rng.integers(0, 2, cnt)
    V = values(rng, cnt, kind)
    hot = (m - 1, n - 1)
    I[0:W], J[0:W] = hot
    coll = fsr.colliding_keys(m, n, W) + 1
    coll = coll[rng.permutation(W)]
    I[W:2 * W], J[W:2 * W] = coll[:, 0], coll[:, 1]
    mid = 2 * W + W // 2
    coll2 = coll[rng.permutation(W)]
    I[mid:mid + W], J[mid:mid + W] = coll2[:, 0], coll2[:, 1]
    P0, P1, P2 = (m, n // 2 + 1), (m, n // 2 + 2), (m, n // 2 + 3)
    for p in (5 * W + 3, 5 * W + 100):
        I[p], J[p], V[p], F[p] = P0[0], P0[1], 0.0, fsr.UPDATE
    p = 6 * W + 7
    I[p], J[p], F[p] = P0[0], P0[1], fsr.RAW
    V[p] = V[p] if V[p] != 0 else 3.0
    for k, p in enumerate((5 * W + 1, 6 * W + 1, 7 * W + 2)):
        I[p], J[p], V[p], F[p] = P1[0], P1[1], (0.0, -0.0, 0.0)[k], fsr.UPDATE
    p, q = 7 * W + 10, 7 * W + 400
    v = V[p] if V[p] != 0 else 5.0
    I[p], J[p], V[p], F[p] = P2[0], P2[1], v, fsr.UPDATE
    I[q], J[q], V[q], F[q] = P2[0], P2[1], -v, fsr.UPDATE
    for t, c in enumerate(TRUNCATIONS):
        I[c - 1], J[c - 1], F[c - 1] = m - 3 - t, n - 5, fsr.RAW
    assert TRUNCATIONS[-1] == cnt
    return I, J, V, F, (P0, P1, P2)


# stream lengths around the size limit of the windows: the last window short by one, exactly 8 windows, a last
# window of 1, 511 (one lane of its last batch of 32 idle) and 512 calls, and the whole edge stream
TRUNCATIONS = (4095, 4096, 4097, 4096 + 511, 4096 + 512, 9 * WINDOW + 1)


@pytest.mark.parametrize("precount", [False, True])
@pytest.mark.parametrize("kind", ["fixed", "random"])
def test_window_edges(xsb, oracle, precount, kind):
    rng = np.random.default_rng(10 + int(precount))
    m = n = 4096
    I, J, V, F, (P0, P1, P2) = edge_stream(rng, m, n, kind)
    for cnt in TRUNCATIONS:
        assert cnt <= len(V)  # a truncation is never silently the whole stream
        h = xsb.Handle(m, n)
        h.set_precount(precount)
        h.set_preaggregation(True)
        insert_runs(h, I[:cnt], J[:cnt], V[:cnt], F[:cnt])
        h.flush(xsb.FAST)
        kept = h.flush_stats()["preagg_records"]
        if cnt < MIN_PREAGG:
            assert kept == 0
        else:
            assert 0 < kept < cnt
        got = h.fetch_csc_numpy()
        g = fsr.group_contributions(m, n, I[:cnt], J[:cnt], V[:cnt], F[:cnt])
        check(got, g, kind != "random", f"{cnt} calls, precount {precount}")
        if cnt == len(V):
            A = oracle.OracleExt(m, n)
            insert_runs(A, I, J, V, F)
            ocp, orv, onz = A.csc()
            assert np.array_equal(got[0], ocp) and np.array_equal(got[1], orv)
            if kind != "random":
                assert np.array_equal(bits(got[2]), bits(onz))
            vals = h.get_values(np.array([P0[0], P2[0]]), np.array([P0[1], P2[1]]))
            assert bits(vals[1]) == bits(0.0)  # cancelled: stays, as +0.0
            # the zero-update-only position is absent, the late-created one present
            cp, rv = got[0], got[1]
            col = lambda j: rv[cp[j - 1] - 1: cp[j] - 1]
            assert P1[0] not in col(P1[1]) and P0[0] in col(P0[1]) and P2[0] in col(P2[1])
        h.close()


# ================================================================ 3. state a FAST flush leaves behind
def test_fast_and_deterministic_flushes_alternate_on_one_handle(xsb, oracle):
    """FAST + pre-aggregation flushes onto a resident CSC, alternating with DETERMINISTIC ones on one handle.  After
    each FAST step the oracle is seeded with the GPU's CSC; the next DETERMINISTIC flush must equal it bit for bit --
    a stale staging buffer (the swapped A/B buffers), capacity or fold-table hint left by the FAST flush would show."""
    rng = np.random.default_rng(20)
    m, n = 700, 650
    h = xsb.Handle(m, n)
    h.set_preaggregation(True)
    A = oracle.OracleExt(m, n)
    resident = None
    for step in range(6):
        cnt = 9000 + 1500 * step
        fixed = step < 4  # fixed-point values while the resident values stay on their lattice, then random ones
        I, J, V, F = random_stream(rng, m, n, cnt, "fixed" if fixed else "random")
        if step % 2 == 0:
            insert_runs(h, I, J, V, F)
            h.flush(xsb.FAST)
            assert 0 < h.flush_stats()["preagg_records"] < cnt
            got = h.fetch_csc_numpy()
            check(got, fsr.group_contributions(m, n, I, J, V, F, resident), fixed, f"FAST step {step}")
            A.set_csc(*got)
        else:
            insert_runs(h, I, J, V, F)
            h.flush(xsb.DETERMINISTIC)
            insert_runs(A, I, J, V, F)
            got = h.fetch_csc_numpy()
            same_bits(got, A.csc(), f"DETERMINISTIC step {step}")
        resident = got


def test_preaggregation_misses_turn_it_off(xsb):
    """Current behaviour, pinned: a FAST flush whose windows keep more than 3/4 of the records is a miss; after two
    misses in a row the handle stops pre-aggregating, also for streams that repeat themselves, until
    set_preaggregation is called again.  A hit in between resets the count.  Every result stays within the bound."""
    rng = np.random.default_rng(21)
    m, n = 3000, 3000
    h = xsb.Handle(m, n)
    h.set_preaggregation(True)
    resident = None

    def step(distinct, expect_preagg):
        nonlocal resident
        cnt = 8192
        I, J, V, F = random_stream(rng, m, n, cnt, "random", keys=cnt * 50 if distinct else cnt // 32)
        insert_runs(h, I, J, V, F)
        h.flush(xsb.FAST)
        kept = h.flush_stats()["preagg_records"]
        assert (kept > 0) == expect_preagg, (distinct, kept)
        got = h.fetch_csc_numpy()
        check(got, fsr.group_contributions(m, n, I, J, V, F, resident), False)
        resident = got
        return kept, cnt

    kept, cnt = step(True, True)
    assert kept * 4 > cnt * 3  # a miss
    step(False, True)  # a hit: the count starts again
    step(True, True)
    step(True, True)  # second miss in a row
    step(False, False)  # off for good on this handle
    step(False, False)
    h.set_preaggregation(True)  # switching it on again forgets the misses
    step(False, True)


# ================================================================ 4. multi-partition handles
@pytest.mark.parametrize("ntid", [3, 8])
@pytest.mark.parametrize("kind", ["fixed", "random"])
def test_multi_partition_preaggregation(xsb, oracle, ntid, kind):
    """Partial sums are folded into partition 0 by the windows: the pattern still equals OracleMT's, the values
    its bits (fixed point) or the bound; also on top of the resident CSC."""
    rng = np.random.default_rng(30 + ntid)
    m, n = 500, 480
    h = xsb.Handle(m, n, n_tid=ntid)
    h.set_preaggregation(True)
    A = oracle.OracleMT(m, n, ntid)
    resident = None
    for step in range(2):
        I, J, V, _ = random_stream(rng, m, n, 16000, kind)
        parts = np.array_split(np.arange(len(V)), ntid)
        for t in rng.permutation(ntid):  # partitions deliver in any order, in pieces
            for p in np.array_split(parts[t], 3):
                h.insert_batch(I[p], J[p], V[p], xsb.RAW, tid=int(t))
        for t in range(ntid):
            p = parts[t]
            A.insert_batch(I[p], J[p], V[p], t + 1, oracle.RAW)
        A.flush()
        h.flush(xsb.FAST)
        assert 0 < h.flush_stats()["preagg_records"] < len(V)
        got = h.fetch_csc_numpy()
        ocp, orv, onz = A.csc()
        assert np.array_equal(got[0], ocp) and np.array_equal(got[1], orv)
        if kind != "random":
            assert np.array_equal(bits(got[2]), bits(onz))
        order = np.concatenate(parts)
        g = fsr.group_contributions(m, n, I[order], J[order], V[order], fsr.RAW, resident)
        check(got, g, kind != "random", f"{ntid} partitions step {step}")
        resident = got


# ================================================================ 5. slab handles
SLABS = [(2, [0, 1, 300]), (3, [0, 150, 151, 300]), (4, [0, 75, 76, 200, 300])]


@pytest.mark.parametrize("world,splits", SLABS)
@pytest.mark.parametrize("kind", ["fixed", "random"])
def test_slab_preaggregation(xsb, oracle, torch, world, splits, kind):
    """Pre-aggregation on every rank: the partial sums keep their owner bits, the records received from lower and
    higher ranks are mixed into one stream, drop_foreign runs after the windows.  Every slab equals the same columns
    of the plain handle's pattern, its values the bits (fixed point) or the bound.  The last rank stages nothing."""
    from tests.test_gpu_dist import route_and_flush

    rng = np.random.default_rng(40 + world)
    m, n = 200, 300
    handles = [xsb.Handle(m, n, slab=(world, r, splits)) for r in range(world)]
    for h in handles:
        h.set_preaggregation(True)
    resident = None
    for step in range(2):
        streams = []
        for r in range(world):
            cnt = 0 if r == world - 1 else 7000 + 1000 * r
            I, J, V, F = random_stream(rng, m, n, max(cnt, 64), kind)
            J[:world] = np.asarray(splits[:-1]) + 1  # every slab, the one-column ones included, owns records
            streams.append((I[:cnt], J[:cnt], V[:cnt], F[:cnt]))
            if cnt:
                insert_runs(handles[r], *streams[-1])
        route_and_flush(xsb, torch, handles, xsb.FAST)
        kept = [h.flush_stats()["preagg_records"] for h in handles]
        I, J, V, F = (np.concatenate([s[k] for s in streams]) for k in range(4))
        g = fsr.group_contributions(m, n, I, J, V, F, resident)
        full_nz = np.empty(len(g.terms))
        for r, h in enumerate(handles):
            lcp, lrv, lnz = h.fetch_csc_numpy()
            lo, hi = splits[r], splits[r + 1]
            a, b = g.colptr[lo] - 1, g.colptr[hi] - 1
            assert np.array_equal(lcp - 1, g.colptr[lo:hi + 1] - g.colptr[lo]), f"rank {r} colptr"
            assert np.array_equal(lrv, g.rowval[a:b]), f"rank {r} rowval"
            full_nz[a:b] = lnz
        check((g.colptr, g.rowval, full_nz), g, kind != "random", f"world {world} step {step}")
        assert any(k > 0 for k in kept), kept
        resident = (g.colptr, g.rowval, full_nz)
    for h in handles:
        h.close()


@pytest.mark.parametrize("exchange", ["fixed", "peer"])
def test_fixed_and_peer_exchanges_do_not_preaggregate(xsb, torch, exchange):
    """Both block exchanges set the handle's fixed-exchange state, which turns the windows off: preagg_records is 0
    and a FAST flush equals the DETERMINISTIC one of the same streams bit for bit, random values included."""
    from tests.test_gpu_dist import exchange_fixed_and_flush, peer_step

    world, splits = 3, [0, 7, 8, 300]
    m, n = 200, 300
    rng = np.random.default_rng(50)
    pairs = {mode: [xsb.Handle(m, n, slab=(world, r, splits)) for r in range(world)]
             for mode in (xsb.DETERMINISTIC, xsb.FAST)}
    caps = [[0 if s == d else 8000 for d in range(world)] for s in range(world)]
    for hs in pairs.values():
        for h in hs:
            h.set_preaggregation(True)
        if exchange == "peer":
            capsT = [[caps[s][d] for s in range(world)] for d in range(world)]
            for h in hs:
                h.peer_exchange_create(capsT)
            for h in hs:
                h.peer_exchange_connect_local(hs)
    for step in range(2):
        streams = [random_stream(rng, m, n, 6000 + 500 * r, "random") for r in range(world)]
        for mode, hs in pairs.items():
            for h, s in zip(hs, streams):
                insert_runs(h, *s)
            if exchange == "fixed":
                exchange_fixed_and_flush(xsb, torch, hs, caps, mode)
            else:
                peer_step(hs, mode)
            assert all(h.flush_stats()["preagg_records"] == 0 for h in hs)
        for r in range(world):
            same_bits(pairs[xsb.FAST][r].fetch_csc_numpy(), pairs[xsb.DETERMINISTIC][r].fetch_csc_numpy(),
                      f"{exchange} rank {r} step {step}")
    for hs in pairs.values():
        if exchange == "peer":
            for h in hs:
                h.peer_exchange_disconnect()
            for h in hs:
                h.peer_exchange_destroy()
        for h in hs:
            h.close()


# ================================================================ 6. reassemble_values(FAST)
def element_positions(rd, cd):
    """(I, J) of the element stream: call kr*kc*c + kr*jl + il is (rd[c, il], cd[c, jl])."""
    nc, kr = rd.shape
    kc = cd.shape[1]
    I = np.broadcast_to(rd[:, None, :], (nc, kc, kr)).ravel()
    J = np.broadcast_to(cd[:, :, None], (nc, kc, kr)).ravel()
    return np.ascontiguousarray(I), np.ascontiguousarray(J)


def reassembly_case(xsb, torch, h, I, J, m, n, freeze, rng, base=1, on_device=False):
    """Frozen stream (I, J) (1-based) on handle h: FAST re-assemblies, from zero and on top of resident values,
    with fixed-point values (== DETERMINISTIC bits) and cancelling ones (bound)."""
    freeze()
    cnt = len(I)

    def dev(V):
        return torch.from_numpy(V).cuda() if on_device else V

    for kind in ("fixed", "random"):
        V = values(rng, cnt, kind)
        R = values(rng, cnt, kind)  # resident values: on the lattice of the fixed-point stream
        for zero_first in (True, False):

            def run(mode):
                if not zero_first:
                    h.reassemble_values(dev(R), xsb.DETERMINISTIC, zero_first=True)
                h.synchronize()
                before = h.fetch_csc_numpy()
                h.reassemble_values(dev(V), mode, zero_first=zero_first)
                h.synchronize()
                return before, h.fetch_csc_numpy()

            before, fast = run(xsb.FAST)
            resident = (before[0] - base + 1, before[1] - base + 1, before[2])
            g = fsr.group_contributions(m, n, I, J, V, fsr.UPDATE, resident)
            if zero_first:  # every entry is resident; its value is replaced by +0.0
                g.terms = [t[1:] for t in g.terms]
                g.has_resident = np.zeros(len(g.terms), bool)
            check(fast, g, kind != "random", f"{kind} zero_first={zero_first}", base)
            if kind != "random":
                same_bits(fast, run(xsb.DETERMINISTIC)[1], f"FAST vs DETERMINISTIC zero_first={zero_first}")


@pytest.mark.parametrize("idx,base,on_device", [(1, 1, False), (0, 0, True), (0, 1, False), (1, 0, True)])
def test_reassemble_fast_frozen_pattern(xsb, torch, idx, base, on_device):
    rng = np.random.default_rng(60 + 2 * idx + base)
    m, n = 400, 380
    dt = np.int64 if idx == xsb.I64 else np.int32
    nk = 20000
    kI, kJ = rng.integers(1, m + 1, nk), rng.integers(1, n + 1, nk)
    k = rng.integers(0, nk, 100000)
    I, J = kI[k], kJ[k]
    h = xsb.Handle(m, n, idx, base)
    h.insert_batch((I - 1 + base).astype(dt), (J - 1 + base).astype(dt), np.ones(len(I)), xsb.RAW)
    h.flush()
    Ib, Jb = (I - 1 + base).astype(dt), (J - 1 + base).astype(dt)
    if on_device:
        Ib, Jb = torch.from_numpy(Ib).cuda(), torch.from_numpy(Jb).cuda()
    reassembly_case(xsb, torch, h, I, J, m, n, lambda: h.freeze_pattern(Ib, Jb, count=len(I)), rng, base, on_device)


def test_reassemble_fast_hot_entry(xsb, torch):
    """One entry with 2^20 contributions beside 10^5 cold ones: every atomic on the hot entry collides."""
    rng = np.random.default_rng(61)
    m = n = 1000
    cold = 100000
    I = np.concatenate([rng.integers(1, m + 1, cold), np.full(1 << 20, 17)])
    J = np.concatenate([rng.integers(1, n + 1, cold), np.full(1 << 20, 23)])
    p = rng.permutation(len(I))
    I, J = I[p], J[p]
    h = xsb.Handle(m, n)
    h.insert_batch(I, J, np.ones(len(I)), xsb.RAW)
    h.flush()
    reassembly_case(xsb, torch, h, I, J, m, n, lambda: h.freeze_pattern(I, J), rng, on_device=True)


@pytest.mark.parametrize("kr,kc", [(4, 4), (27, 27), (1, 4), (12, 4)])
def test_reassemble_fast_elements(xsb, torch, kr, kc):
    rng = np.random.default_rng(62 + kr + kc)
    nn, ncells = 300, 700
    rd = np.stack([rng.choice(np.arange(1, nn + 1), kr, replace=False) for _ in range(ncells)])
    cd = rd if kr == kc else np.stack([rng.choice(np.arange(1, nn + 1), kc, replace=False) for _ in range(ncells)])
    I, J = element_positions(rd, cd)
    h = xsb.Handle(nn, nn)
    square = kr == kc
    if square:
        h.insert_elements(rd, np.ones((ncells, kc, kr)))
        freeze = lambda: h.freeze_elements(rd)  # noqa: E731
    else:
        h.insert_elements(rd, np.ones((ncells, kc, kr)), col_dofs=cd)
        freeze = lambda: h.freeze_elements(rd, col_dofs=cd)  # noqa: E731
    h.flush()
    reassembly_case(xsb, torch, h, I, J, nn, nn, freeze, rng)


# ================================================================ 7. slab-frozen streams
@pytest.mark.parametrize("world,splits", [(1, [0, 60]), (2, [0, 31, 60]), (3, [0, 1, 2, 60]), (4, [0, 10, 11, 45, 60])])
def test_slab_frozen_fast(xsb, oracle, torch, world, splits):
    """xsb_reassemble_slab_values(FAST): positions of the own stream in other ranks' columns contribute nothing here,
    every received value exactly once.  Fixed point: the bits of the DETERMINISTIC step; random: the bound against
    the rank-ordered concatenation of the streams."""
    from tests.test_gpu_dist_values import build, entries_of, freeze_all, step_all

    m, n = 50, 60
    rng = np.random.default_rng(70 + world)
    handles, P, A, cp, rv, nz = build(xsb, torch, oracle, rng, m, n, world, splits, xsb.I64, 1)
    streams = []
    for r in range(world):
        cnt = 0 if (world > 2 and r == world - 1) else 2000 + 300 * r
        I1, J1 = entries_of(rng, cp, rv, range(splits[r], splits[r + 1]), cnt // 2)
        I2, J2 = entries_of(rng, cp, rv, range(n), cnt - cnt // 2)
        I, J = np.concatenate([I1, I2]), np.concatenate([J1, J2])
        p = rng.permutation(len(I))
        streams.append((I[p], J[p]))
    freeze_all(torch, handles, [(lambda h=h, s=s: h.freeze_slab(*s)) for h, s in zip(handles, streams)])
    Icat = np.concatenate([s[0] for s in streams])
    Jcat = np.concatenate([s[1] for s in streams])

    def slabs():
        out = [h.fetch_csc_numpy() for h in handles]
        return cp, rv, np.concatenate([o[2] for o in out])

    for kind in ("fixed", "random"):
        Vs = [values(rng, len(s[0]), kind) for s in streams]
        Rs = [values(rng, len(s[0]), kind) for s in streams]  # resident values, on the same lattice
        for zero_first in (True, False):

            def run(mode):
                if not zero_first:
                    step_all(torch, handles, [torch.from_numpy(v).cuda() for v in Rs], 0, True)
                before = slabs()
                step_all(torch, handles, [torch.from_numpy(v).cuda() for v in Vs], mode, zero_first)
                return before, slabs()

            resident, got = run(xsb.capi.FAST)
            g = fsr.group_contributions(m, n, Icat, Jcat, np.concatenate(Vs), fsr.UPDATE, resident)
            if zero_first:
                g.terms = [t[1:] for t in g.terms]
                g.has_resident = np.zeros(len(g.terms), bool)
            check(got, g, kind != "random", f"world {world} {kind} zero_first={zero_first}")
            if kind != "random":  # the DETERMINISTIC step from the same resident values gives the same bits
                same_bits(run(0)[1], got, f"world {world} FAST vs DETERMINISTIC")


def test_dist_matrix_reassemble_fast_world_one(xsb, torch):
    """DistExtendableSparseMatrix.reassemble_values(V, mode=FAST) on a one-rank process group: from zero and on top of
    resident values, fixed point (the bits of the DETERMINISTIC step) and cancelling values (the bound)."""
    import socket

    import torch.distributed as dist
    from xsparse_b200.dist import DistExtendableSparseMatrix

    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1)
    try:
        rng = np.random.default_rng(75)
        m, n = 90, 80
        I = np.concatenate([np.arange(1, n + 1), rng.integers(1, m + 1, 700)])
        J = np.concatenate([np.arange(1, n + 1), rng.integers(1, n + 1, 700)])
        D = DistExtendableSparseMatrix(m, n)
        D.insert_batch(I, J, np.ones(len(I)))
        D.flush()
        pick = rng.integers(0, len(I), 5000)
        Is, Js = I[pick], J[pick]
        D.freeze_pattern(Is, Js)
        for kind in ("fixed", "random"):
            V = values(rng, len(Is), kind)
            R = values(rng, len(Is), kind)
            for zero_first in (True, False):

                def run(mode):
                    if not zero_first:
                        D.reassemble_values(torch.from_numpy(R).cuda(), 0, zero_first=True)
                    D.h.synchronize()
                    before = D.h.fetch_csc_numpy()
                    D.reassemble_values(torch.from_numpy(V).cuda(), mode, zero_first=zero_first)
                    D.h.synchronize()
                    return before, D.h.fetch_csc_numpy()

                before, fast = run(xsb.FAST)
                g = fsr.group_contributions(m, n, Is, Js, V, fsr.UPDATE, before)
                if zero_first:
                    g.terms = [t[1:] for t in g.terms]
                    g.has_resident = np.zeros(len(g.terms), bool)
                check(fast, g, kind != "random", f"world 1 {kind} zero_first={zero_first}")
                if kind != "random":
                    same_bits(fast, run(xsb.DETERMINISTIC)[1], "world 1 FAST vs DETERMINISTIC")
        D.close()
    finally:
        dist.destroy_process_group()


# ================================================================ 8. full size, fixed point
def staged_arrays(xsb, torch, h):
    cnt = h.pending
    dI = torch.empty(cnt, dtype=torch.int64, device="cuda")
    dJ = torch.empty(cnt, dtype=torch.int64, device="cuda")
    dV = torch.empty(cnt, dtype=torch.float64, device="cuda")
    got = C.c_int64(0)
    c = xsb.capi
    c.check(c.lib().xsb_debug_fetch_staged(h._h, 0, dI.data_ptr(), dJ.data_ptr(), dV.data_ptr(), None, cnt,
                                           C.byref(got)), h._h)
    h.synchronize()
    return dI, dJ, dV


def device_csc(torch, h):
    nnz = h.nnz
    cp = torch.empty(h.n + 1, dtype=torch.int64, device="cuda")
    rv = torch.empty(nnz, dtype=torch.int64, device="cuda")
    nz = torch.empty(nnz, dtype=torch.float64, device="cuda")
    h.fetch_csc(cp, rv, nz)
    h.synchronize()
    return cp, rv, nz


def device_fixed_point(torch, cnt, e, seed, kmax=2 ** 20):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    k = torch.randint(-kmax, kmax + 1, (cnt,), generator=g, device="cuda", dtype=torch.int64).to(torch.float64)
    return torch.ldexp(k, torch.tensor(float(e), device="cuda", dtype=torch.float64))


@pytest.mark.parametrize("mesh,e", [(128, 0), (64, -1074)])
def test_full_size_fem_fixed_point_preaggregation(xsb, torch, mesh, e):
    """The FEM stream with fixed-point values: a FAST flush with pre-aggregation equals the DETERMINISTIC flush of
    the same arrays bit for bit (at e = -1074 every value and every sum is subnormal)."""
    n = mesh ** 3
    g = xsb.Handle(n, n)
    g.set_precount(False)
    g.emit_p1fem(mesh, mesh, mesh, flavour=xsb.RAW)
    dI, dJ, _ = staged_arrays(xsb, torch, g)
    g.close()
    dV = device_fixed_point(torch, len(dI), e, seed=mesh)
    out = {}
    for mode in (xsb.DETERMINISTIC, xsb.FAST):
        h = xsb.Handle(n, n)
        h.set_preaggregation(True)
        h.insert_batch(dI, dJ, dV, xsb.RAW, count=len(dV))
        h.flush(mode)
        kept = h.flush_stats()["preagg_records"]
        assert (kept > 0) == (mode == xsb.FAST)
        out[mode] = device_csc(torch, h)
        h.close()
    a, b = out[xsb.DETERMINISTIC], out[xsb.FAST]
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert torch.equal(a[2].view(torch.int64), b[2].view(torch.int64)), "FAST differs from DETERMINISTIC"
    if e < -1000:
        assert float(a[2].abs().max()) < 2.0 ** -1021 and bool((a[2] != 0).any())


@pytest.mark.parametrize("nx,e", [(200, 0), (64, -1074)])
def test_full_size_fdrand_reassembly_fixed_point(xsb, torch, nx, e):
    """fdrand frozen, re-assembled with fixed-point values: FAST equals DETERMINISTIC bit for bit."""
    n = nx ** 3
    g = xsb.Handle(n, n)
    g.set_precount(False)
    g.emit_fdrand(nx, nx, nx, seed=7)
    dI, dJ, dV0 = staged_arrays(xsb, torch, g)
    g.close()
    h = xsb.Handle(n, n)
    h.insert_batch(dI, dJ, dV0, xsb.UPDATE, count=len(dV0))
    h.flush()
    h.freeze_pattern(dI, dJ, count=len(dI))
    V = device_fixed_point(torch, len(dI), e, seed=nx)
    del dI, dJ, dV0
    res = {}
    for mode in (xsb.DETERMINISTIC, xsb.FAST):
        h.reassemble_values(V, mode, count=len(V), zero_first=True)
        res[mode] = device_csc(torch, h)[2]
    assert torch.equal(res[0].view(torch.int64), res[1].view(torch.int64))
    if e < -1000:
        assert float(res[0].abs().max()) < 2.0 ** -1021
    h.close()
