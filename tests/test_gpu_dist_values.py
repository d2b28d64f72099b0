"""GPU tests of values-only re-assembly on column slabs: a stream of GLOBAL positions frozen across the ranks
(xsb_freeze_slab* + xsb_reassemble_slab_*).  The ranks are simulated inside one process on one GPU, the exchanges
are done by hand with device copies in source-rank order (what all_to_all_single produces).  Every result is
compared with one plain handle that froze the rank-ordered concatenation of the streams, bit for bit, and with the
CPU oracle applying the same values in the same order."""
import os
import socket

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


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def route_and_flush(torch, handles):
    world = len(handles)
    sends, counts = [], []
    for r, h in enumerate(handles):
        c = h.route_count()
        leaving = sum(c) - c[r]
        buf = torch.empty(2 * max(leaving, 1), dtype=torch.int64, device="cuda")
        h.route_prepare(buf, leaving)
        sends.append(buf)
        counts.append(c)
    torch.cuda.synchronize()
    for dst in range(world):
        for src in range(world):
            if src != dst:
                off = sum(c for d, c in enumerate(counts[src][:dst]) if d != src)
                handles[dst].route_finish(src, sends[src][2 * off: 2 * (off + counts[src][dst])], counts[src][dst])
        handles[dst].flush()


def _gather(torch, sends, offs, dst, dtype):
    """What rank dst receives: the buckets for it, sources ascending, own rank left out."""
    parts, rc = [], [0] * len(sends)
    for src in range(len(sends)):
        if src == dst:
            continue
        o = sum(offs[src][:dst])
        rc[src] = offs[src][dst]
        parts.append(sends[src][o: o + offs[src][dst]])
    recv = torch.cat(parts) if parts and sum(rc) else torch.empty(1, dtype=dtype, device="cuda")
    return recv, rc


def freeze_all(torch, handles, firsts):
    """firsts[r]() = the first step of rank r's freeze (returns its counts); then prepare, exchange, finish."""
    world = len(handles)
    counts = [f() for f in firsts]
    sends, offs = [], []
    for r, h in enumerate(handles):
        off = [0 if d == r else c for d, c in enumerate(counts[r])]
        buf = torch.empty(max(sum(off), 1), dtype=torch.int64, device="cuda")
        h.freeze_slab_prepare(buf, sum(off))
        sends.append(buf)
        offs.append(off)
    torch.cuda.synchronize()
    for dst in range(world):
        recv, rc = _gather(torch, sends, offs, dst, torch.int64)
        handles[dst].freeze_slab_finish(recv, rc)
        sent, got = handles[dst].frozen_slab_counts()
        assert sent == counts[dst] and got == rc
    return counts


def step_all(torch, handles, Vs, mode=0, zero_first=True):
    world = len(handles)
    sends, offs = [], []
    for r, h in enumerate(handles):
        sc, _ = h.frozen_slab_counts()
        off = [0 if d == r else c for d, c in enumerate(sc)]
        buf = torch.empty(max(sum(off), 1), dtype=torch.float64, device="cuda")
        h.reassemble_slab_pack(Vs[r], buf)
        h.synchronize()
        sends.append(buf)
        offs.append(off)
    for dst in range(world):
        recv, _ = _gather(torch, sends, offs, dst, torch.float64)
        torch.cuda.synchronize()
        handles[dst].reassemble_slab_values(Vs[dst], recv, mode, zero_first)
        handles[dst].synchronize()


def make_pattern(rng, m, n, extra):
    I = np.concatenate([np.arange(1, min(m, n) + 1), rng.integers(1, m + 1, extra)])
    J = np.concatenate([np.arange(1, min(m, n) + 1), rng.integers(1, n + 1, extra)])
    return I, J


def slab_nz(h):
    return h.fetch_csc_numpy()[2]


def check_slabs(handles, splits, cp, nz, exact=True):
    for r, h in enumerate(handles):
        lnz = slab_nz(h)
        want = nz[cp[splits[r]] - 1: cp[splits[r + 1]] - 1]
        if exact:
            assert np.array_equal(bits(lnz), bits(want)), f"rank {r}"
        else:
            # within 1e-14 of the entries' magnitude: cancellations leave sums far below their terms
            np.testing.assert_allclose(lnz, want, rtol=1e-14, atol=1e-14 * max(1.0, float(np.abs(want).max(initial=0.0))))


def build(xsb, torch, oracle, rng, m, n, world, splits, idx, base):
    """Slabs built by a routed flush, a plain handle and the oracle holding the same matrix."""
    I, J = make_pattern(rng, m, n, 6 * n)
    V = rng.standard_normal(len(I))
    handles = [xsb.Handle(m, n, idx, base, slab=(world, r, splits)) for r in range(world)]
    P = xsb.Handle(m, n, idx, base)
    dt = np.int64 if idx == xsb.I64 else np.int32
    parts = np.array_split(np.arange(len(I)), world)
    for r, h in enumerate(handles):
        p = parts[r]
        h.insert_batch((I[p] - 1 + base).astype(dt), (J[p] - 1 + base).astype(dt), V[p])
    route_and_flush(torch, handles)
    P.insert_batch((I - 1 + base).astype(dt), (J - 1 + base).astype(dt), V)
    P.flush()
    A = oracle.OracleExt(m, n)
    A.insert_batch(I, J, V)
    cp, rv, nz = A.csc()
    check_slabs(handles, splits, cp, nz)
    return handles, P, A, cp, rv, nz


def entries_of(rng, cp, rv, cols, cnt):
    """cnt positions (1-based) drawn from the pattern's entries in the given columns (with duplicates)."""
    cols = np.asarray(cols)
    ent = np.concatenate([np.stack([rv[cp[c] - 1: cp[c + 1] - 1], np.full(cp[c + 1] - cp[c], c + 1)], 1) for c in cols])
    pick = ent[rng.integers(0, len(ent), cnt)]
    return pick[:, 0].copy(), pick[:, 1].copy()


def signed_values(rng, cnt):
    V = rng.standard_normal(cnt)
    V[::7] = -0.0
    V[3::11] = 0.0
    return V


CASES = [(1, [0, 60]), (2, [0, 31, 60]), (3, [0, 1, 2, 60]), (4, [0, 10, 11, 45, 60])]


@pytest.mark.parametrize("world,splits", CASES)
@pytest.mark.parametrize("idx,base,on_device", [(1, 1, False), (0, 0, True), (0, 1, False), (1, 0, True)])
def test_slab_frozen_stream_matches_single_handle(xsb, oracle, world, splits, idx, base, on_device):
    torch = pytest.importorskip("torch")
    m, n = 50, 60
    rng = np.random.default_rng(world * 10 + idx * 2 + base)
    handles, P, A, cp, rv, nz = build(xsb, torch, oracle, rng, m, n, world, splits, idx, base)
    dt = np.int64 if idx == xsb.I64 else np.int32
    # rank r's stream mixes its own columns with everybody's (duplicates included); the last rank of a world > 2 has
    # an empty stream
    streams = []
    for r in range(world):
        cnt = 0 if (world > 2 and r == world - 1) else 700 + 90 * r
        I1, J1 = entries_of(rng, cp, rv, range(splits[r], splits[r + 1]), cnt // 2)
        I2, J2 = entries_of(rng, cp, rv, range(n), cnt - cnt // 2)
        I, J = np.concatenate([I1, I2]), np.concatenate([J1, J2])
        perm = rng.permutation(len(I))
        streams.append((I[perm], J[perm]))

    def dev(a, dtype):
        a = np.ascontiguousarray(a, dtype)
        return torch.from_numpy(a).cuda() if on_device else a

    firsts = [(lambda h=h, I=I, J=J: h.freeze_slab(dev(I - 1 + base, dt), dev(J - 1 + base, dt)))
              for h, (I, J) in zip(handles, streams)]
    counts = freeze_all(torch, handles, firsts)
    for r in range(world):
        assert sum(counts[r]) == len(streams[r][0])
    Icat = np.concatenate([s[0] for s in streams])
    Jcat = np.concatenate([s[1] for s in streams])
    P.freeze_pattern((Icat - 1 + base).astype(dt), (Jcat - 1 + base).astype(dt))
    A.set_csc(cp, rv, nz)
    # deterministic: zeroed, on top of the resident values, zeroed again
    for step, zero_first in enumerate((True, False, True)):
        Vs = [signed_values(rng, len(s[0])) for s in streams]
        step_all(torch, handles, [dev(v, np.float64) for v in Vs], 0, zero_first)
        Vcat = np.concatenate(Vs)
        P.reassemble_values(Vcat, zero_first=zero_first)
        pcp, _, pnz = P.fetch_csc_numpy()
        check_slabs(handles, splits, pcp - base + 1, pnz)
        if zero_first:
            A.zero_values()
        A.insert_batch(Icat, Jcat, Vcat, oracle.RAW)
        _, _, onz = A.csc()
        assert np.array_equal(bits(pnz), bits(onz))
    # fast mode: the same sums in any order
    Vs = [rng.standard_normal(len(s[0])) for s in streams]
    step_all(torch, handles, [dev(v, np.float64) for v in Vs], xsb.capi.FAST, True)
    P.reassemble_values(np.concatenate(Vs), xsb.capi.DETERMINISTIC, zero_first=True)
    pcp, _, pnz = P.fetch_csc_numpy()
    check_slabs(handles, splits, pcp - base + 1, pnz, exact=False)


@pytest.mark.parametrize("world,splits", [(2, [0, 30, 60]), (3, [0, 20, 21, 60])])
def test_slab_streams_that_exchange_nothing(xsb, oracle, world, splits):
    torch = pytest.importorskip("torch")
    m, n = 40, 60
    rng = np.random.default_rng(5)
    handles, P, A, cp, rv, nz = build(xsb, torch, oracle, rng, m, n, world, splits, xsb.I64, 1)
    streams = [entries_of(rng, cp, rv, range(splits[r], splits[r + 1]), 300) for r in range(world)]
    counts = freeze_all(torch, handles, [(lambda h=h, s=s: h.freeze_slab(*s)) for h, s in zip(handles, streams)])
    for r in range(world):
        assert counts[r][r] == 300 and sum(counts[r]) == 300
        sent, got = handles[r].frozen_slab_counts()
        assert sum(got) == 0
    Vs = [signed_values(rng, 300) for _ in range(world)]
    step_all(torch, handles, Vs)
    P.freeze_pattern(np.concatenate([s[0] for s in streams]), np.concatenate([s[1] for s in streams]))
    P.reassemble_values(np.concatenate(Vs), zero_first=True)
    pcp, _, pnz = P.fetch_csc_numpy()
    check_slabs(handles, splits, pcp, pnz)


def _elements_case(xsb, torch, oracle, handles, splits, P, dofs_per_rank, rng):
    firsts = [(lambda h=h, d=d: h.freeze_slab_elements(d)) for h, d in zip(handles, dofs_per_rank)]
    freeze_all(torch, handles, firsts)
    P.freeze_elements(np.concatenate(dofs_per_rank))
    for zero_first in (True, False):
        Alocs = [signed_values(rng, d.shape[0] * d.shape[1] ** 2).reshape(d.shape[0], d.shape[1], d.shape[1])
                 for d in dofs_per_rank]
        step_all(torch, handles, [a.reshape(-1) for a in Alocs], 0, zero_first)
        P.reassemble_values(np.concatenate([a.reshape(-1) for a in Alocs]), zero_first=zero_first)
        pcp, _, pnz = P.fetch_csc_numpy()
        check_slabs(handles, splits, pcp, pnz)


@pytest.mark.parametrize("k", [4, 27])
def test_slab_frozen_elements_random(xsb, oracle, k):
    torch = pytest.importorskip("torch")
    world, nn, ncells = 3, 90, 40
    splits = [0, 30, 31, nn]
    rng = np.random.default_rng(k)
    dofs = [np.stack([rng.choice(np.arange(1, nn + 1), k, replace=False) for _ in range(ncells + 7 * r)])
            for r in range(world)]
    handles = [xsb.Handle(nn, nn, slab=(world, r, splits)) for r in range(world)]
    P = xsb.Handle(nn, nn)
    for r, h in enumerate(handles):
        h.insert_elements(dofs[r], np.ones((len(dofs[r]), k, k)))
        P.insert_elements(dofs[r], np.ones((len(dofs[r]), k, k)))
    route_and_flush(torch, handles)
    P.flush()
    _elements_case(xsb, torch, oracle, handles, splits, P, dofs, rng)


def test_slab_frozen_elements_fem_layout(xsb, oracle):
    """The z-slab layout of the FEM weak-scaling bench: rank r holds the cube layers of its slab; only the interface
    plane's entries travel."""
    torch = pytest.importorskip("torch")
    world, nx, ny, layers = 3, 6, 5, 4
    nz_nodes = layers * world + 1
    N = nx * ny * nz_nodes
    plane = nx * ny
    splits = [plane * layers * r for r in range(world)] + [N]
    handles = [xsb.Handle(N, N, slab=(world, r, splits)) for r in range(world)]
    for r, h in enumerate(handles):
        h.emit_p1fem(nx, ny, nz_nodes, flavour=xsb.RAW, cz_range=(layers * r, layers * (r + 1)))
    route_and_flush(torch, handles)
    I, J, V = oracle.fem_stream(nx, ny, nz_nodes)
    P = xsb.Handle(N, N)
    P.insert_batch(I, J, V, xsb.RAW)
    P.flush()
    # the stream of rank r = the calls of its cube layers (6 tetrahedra of 4 nodes per cube)
    per_layer = len(I) // (layers * world)
    streams = [(I[per_layer * layers * r: per_layer * layers * (r + 1)], J[per_layer * layers * r: per_layer * layers * (r + 1)])
               for r in range(world)]
    counts = freeze_all(torch, handles, [(lambda h=h, s=s: h.freeze_slab(*s)) for h, s in zip(handles, streams)])
    for r in range(world):
        for d in range(world):
            if d not in (r, r + 1):
                assert counts[r][d] == 0
    P.freeze_pattern(I, J)
    rng = np.random.default_rng(3)
    for zero_first in (True, True, False):
        Vs = [signed_values(rng, len(s[0])) for s in streams]
        step_all(torch, handles, Vs, 0, zero_first)
        P.reassemble_values(np.concatenate(Vs), zero_first=zero_first)
        pcp, _, pnz = P.fetch_csc_numpy()
        check_slabs(handles, splits, pcp, pnz)
    # the same layout in element form: the connectivity of rank r's tetrahedra (a tetrahedron's 20 calls visit its
    # nodes row by row, 5 calls per node), frozen with xsb_freeze_slab_elements against xsb_freeze_elements
    dofs = [np.ascontiguousarray(s[0].reshape(-1, 20)[:, ::5]) for s in streams]
    for d, s in zip(dofs, streams):  # node il's calls after its mass term go to the columns of the 4 nodes
        assert np.array_equal(s[1].reshape(-1, 4, 5)[:, :, 1:], np.broadcast_to(d[:, None, :], (len(d), 4, 4)))
    counts = freeze_all(torch, handles, [(lambda h=h, d=d: h.freeze_slab_elements(d)) for h, d in zip(handles, dofs)])
    for r in range(world):
        assert counts[r][r] > 0 and all(counts[r][d] == 0 for d in range(world) if d not in (r, r + 1))
        if r + 1 < world:
            assert counts[r][r + 1] > 0
    P.freeze_elements(np.concatenate(dofs))
    for zero_first in (True, False, True):
        Alocs = [signed_values(rng, 16 * len(d)) for d in dofs]
        step_all(torch, handles, Alocs, 0, zero_first)
        P.reassemble_values(np.concatenate(Alocs), zero_first=zero_first)
        pcp, _, pnz = P.fetch_csc_numpy()
        check_slabs(handles, splits, pcp, pnz)


def test_slab_freeze_errors_and_states(xsb, oracle):
    torch = pytest.importorskip("torch")
    world, splits, m, n = 2, [0, 25, 50], 40, 50
    rng = np.random.default_rng(11)
    handles, P, A, cp, rv, nz = build(xsb, torch, oracle, rng, m, n, world, splits, xsb.I64, 1)
    h0, h1 = handles
    I, J = entries_of(rng, cp, rv, range(n), 200)
    # not a slab handle
    with pytest.raises(xsb.XsbError) as e:
        P.freeze_slab(I, J)
    assert e.value.code == xsb.capi.ESTATE
    # out of the matrix: the message names the stream position
    Ib = I.copy()
    Ib[17] = m + 1
    with pytest.raises(IndexError, match="position 17"):
        h0.freeze_slab(Ib, J)
    # own position not in the pattern
    col = 3  # a column of rank 0 with a row that is not an entry
    absent = next(i for i in range(1, m + 1) if i not in set(rv[cp[col - 1] - 1: cp[col] - 1]))
    with pytest.raises(xsb.XsbIllegalError):
        h0.freeze_slab(np.append(I, absent), np.append(J, col))
    # count at or above 2^32
    with pytest.raises(xsb.XsbError) as e:
        h0.freeze_slab(I, J, count=1 << 32)
    assert e.value.code == xsb.capi.EINVAL
    # the half-frozen state: re-assembly refused; every dropping call drops it
    for drop in (lambda h: h.unfreeze(), lambda h: h.flush(), lambda h: h.insert_batch(np.array([1]), np.array([1]), np.array([0.0]))):
        h0.freeze_slab(I, J)
        with pytest.raises(xsb.XsbError) as e:
            h0.reassemble_slab_values(np.zeros(len(I)), None)
        assert e.value.code == xsb.capi.ESTATE
        with pytest.raises(xsb.XsbError) as e:
            h0.reassemble_slab_pack(np.zeros(len(I)), torch.empty(len(I), dtype=torch.float64, device="cuda"))
        assert e.value.code == xsb.capi.ESTATE
        drop(h0)
        with pytest.raises(xsb.XsbError) as e:
            h0.freeze_slab_prepare(torch.empty(len(I), dtype=torch.int64, device="cuda"), len(I))
        assert e.value.code == xsb.capi.ESTATE
    # the insert above is pending: every new call refuses
    with pytest.raises(xsb.XsbError) as e:
        h0.freeze_slab(I, J)
    assert e.value.code == xsb.capi.ESTATE
    route_and_flush(torch, handles)  # (1,1) already exists: the pattern stays
    # a received position that is not in the owner's pattern fails the finish on the owner, which stays unfrozen
    c0 = h0.freeze_slab(I, J)
    h1.freeze_slab(np.array([], np.int64), np.array([], np.int64))
    bad = torch.tensor([(absent - 1) | ((col - 1) << 32)], dtype=torch.int64, device="cuda")
    with pytest.raises(xsb.XsbIllegalError):
        h0.freeze_slab_finish(bad, [0, 1])
    with pytest.raises(xsb.XsbError) as e:
        h0.frozen_slab_counts()
    assert e.value.code == xsb.capi.ESTATE
    outside = torch.tensor([(m + 3) | (0 << 32)], dtype=torch.int64, device="cuda")
    h0.freeze_slab(I, J)
    with pytest.raises(IndexError):
        h0.freeze_slab_finish(outside, [0, 1])
    h0.freeze_slab(I, J)
    with pytest.raises(xsb.XsbError) as e:
        h0.freeze_slab_finish(bad, [0, 1 << 32])
    assert e.value.code == xsb.capi.EINVAL
    # usable afterwards: a correct freeze, then a wrong value count and the plain re-assembly are refused
    h1.unfreeze()
    Is = [I, I[:50]]
    Js = [J, J[:50]]
    freeze_all(torch, handles, [(lambda h=h, a=a, b=b: h.freeze_slab(a, b)) for h, a, b in zip(handles, Is, Js)])
    assert c0 == h0.frozen_slab_counts()[0]
    with pytest.raises(xsb.XsbSizeError):
        h0.reassemble_slab_values(np.zeros(len(I) + 1), None)
    with pytest.raises(xsb.XsbError) as e:
        h0.reassemble_values(np.zeros(len(I)))
    assert e.value.code == xsb.capi.ESTATE
    Vs = [signed_values(rng, len(a)) for a in Is]
    step_all(torch, handles, Vs)
    P.freeze_pattern(np.concatenate(Is), np.concatenate(Js))
    P.reassemble_values(np.concatenate(Vs), zero_first=True)
    pcp, _, pnz = P.fetch_csc_numpy()
    check_slabs(handles, splits, pcp, pnz)
    # a flush that does not change the pattern keeps the map; one that changes it drops it
    h0.insert_batch(np.array([1]), np.array([1]), np.array([1.0]))
    route_and_flush(torch, handles)
    h0.frozen_slab_counts()
    h0.insert_batch(np.array([absent]), np.array([col]), np.array([1.0]))
    route_and_flush(torch, handles)
    with pytest.raises(xsb.XsbError) as e:
        h0.frozen_slab_counts()
    assert e.value.code == xsb.capi.ESTATE
    h1.frozen_slab_counts()  # its own pattern did not change
    # re-freezing after unfreeze
    h1.unfreeze()
    P2 = xsb.Handle(m, n)
    gcp = np.concatenate([handles[0].fetch_csc_numpy()[0][:-1],
                          handles[1].fetch_csc_numpy()[0] + handles[0].nnz])
    P2.set_csc(gcp, np.concatenate([h.fetch_csc_numpy()[1] for h in handles]),
               np.concatenate([h.fetch_csc_numpy()[2] for h in handles]))
    freeze_all(torch, handles, [(lambda h=h, a=a, b=b: h.freeze_slab(a, b)) for h, a, b in zip(handles, Is, Js)])
    P2.freeze_pattern(np.concatenate(Is), np.concatenate(Js))
    Vs = [signed_values(rng, len(a)) for a in Is]
    step_all(torch, handles, Vs, 0, False)
    P2.reassemble_values(np.concatenate(Vs))
    pcp, _, pnz = P2.fetch_csc_numpy()
    check_slabs(handles, splits, pcp, pnz)


# ---- two processes over NCCL: DistExtendableSparseMatrix.freeze_pattern + reassemble_values ----
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, world, port, out_q):
    import sys

    import torch
    import torch.distributed as dist

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from xsparse_b200.dist import DistExtendableSparseMatrix

        m = n = 80
        splits = [0, 37, 80]
        D = DistExtendableSparseMatrix(m, n, splits=splits)
        rng = np.random.default_rng(7)  # the same pattern on both ranks
        I = np.concatenate([np.arange(1, n + 1), rng.integers(1, m + 1, 500)])
        J = np.concatenate([np.arange(1, n + 1), rng.integers(1, n + 1, 500)])
        half = len(I) // 2
        sl = slice(0, half) if rank == 0 else slice(half, len(I))
        D.insert_batch(I[sl], J[sl], np.ones(len(I[sl])))
        D.flush()
        rng = np.random.default_rng(100 + rank)
        pick = rng.integers(0, len(I), 900 + 100 * rank)
        Is, Js = I[pick], J[pick]
        D.freeze_pattern(Is, Js)
        results = []
        for step in range(3):
            V = torch.from_numpy(signed_values(rng, len(Is))).cuda()
            D.reassemble_values(V, zero_first=step != 1)
            results.append((V.cpu().numpy(), D.h.fetch_csc_numpy()[2]))
        out_q.put((rank, I, J, Is, Js, results))
        D.close()
    finally:
        dist.destroy_process_group()


def test_dist_frozen_stream_over_nccl(xsb):
    torch = pytest.importorskip("torch")
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(2):
        r, I, J, Is, Js, res = q.get(timeout=300)
        got[r] = (I, J, Is, Js, res)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    I, J = got[0][0], got[0][1]
    P = xsb.Handle(80, 80)
    P.insert_batch(I, J, np.ones(len(I)))
    P.flush()
    P.freeze_pattern(np.concatenate([got[0][2], got[1][2]]), np.concatenate([got[0][3], got[1][3]]))
    splits = [0, 37, 80]
    for step in range(3):
        P.reassemble_values(np.concatenate([got[0][4][step][0], got[1][4][step][0]]), zero_first=step != 1)
        cp, _, nz = P.fetch_csc_numpy()
        for r in range(2):
            assert np.array_equal(bits(got[r][4][step][1]), bits(nz[cp[splits[r]] - 1: cp[splits[r + 1]] - 1]))
