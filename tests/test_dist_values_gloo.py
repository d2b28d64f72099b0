"""world_size-2/3 gloo tests (CPU) of the choreography of values-only re-assembly in dist.py
(DistExtendableSparseMatrix.freeze_pattern / reassemble_values / unfreeze): the count exchange, the all-to-all-v of
the positions, the per-step point-to-point of the values, the fold order, the freeze that fails on every rank when
one rank fails, and the unfreeze after a pattern-changing flush.  The per-rank slab object is a numpy TEST DOUBLE of
the slab calls of capi.Handle (the product backend is the CUDA library and needs a GPU)."""
import ctypes
import os
import re
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EBOUNDS, EILLEGAL, ESTATE = 1, 3, 7


class DoubleError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(msg)
        self.code = code


class NumpySlabValues:
    """Stands in for capi.Handle(slab=...): a slab of the pattern (1-based global positions) with its values, and the
    slab-freeze calls with the semantics of include/xsparse_b200.h."""

    def __init__(self, m, n, world, rank, splits, entries, values):
        self.m, self.n, self.world, self.rank, self.splits = m, n, world, rank, list(splits)
        lo, hi = splits[rank], splits[rank + 1]
        own = sorted((j, i) for (i, j) in entries if lo < j <= hi)  # CSC order
        self.slot = {(i, j): s for s, (j, i) in enumerate(own)}
        self.nz = np.array([values[(i, j)] for (j, i) in own], np.float64)
        self.staged = []
        self.plain_failure = False
        self.unfreeze()

    # --- the slab freeze
    def unfreeze(self):
        self.state = 0
        self.map = None

    def _owner(self, j):
        return int(np.searchsorted(np.asarray(self.splits[1:]), j - 1, side="right"))

    def freeze_slab(self, I, J):
        assert not self.staged
        self.unfreeze()
        if self.plain_failure:  # a bad argument caught in Python, before the library is called: no status code
            raise ValueError("dofs must have shape (ncells, k)")
        own, send = [], [[] for _ in range(self.world)]
        for k, (i, j) in enumerate(zip(np.asarray(I).tolist(), np.asarray(J).tolist())):
            if not (1 <= i <= self.m and 1 <= j <= self.n):
                raise DoubleError(EBOUNDS, f"position {k} is outside the matrix")
            o = self._owner(j)
            if o == self.rank:
                if (i, j) not in self.slot:
                    raise DoubleError(EILLEGAL, "own position not in the pattern")
                own.append(self.slot[(i, j)])
            else:
                own.append(None)
                send[o].append((k, i - 1, j - 1 - self.splits[o]))
        self.own, self.count = own, len(own)
        self.send = [q for d in range(self.world) for q in send[d]]
        self.send_counts = [len(send[d]) if d != self.rank else sum(x is not None for x in own) for d in range(self.world)]
        self.state = 1
        return list(self.send_counts)

    def freeze_slab_prepare(self, buf, capacity):
        assert self.state == 1 and capacity >= len(self.send)
        b = buf.numpy()
        for q, (_, i, lc) in enumerate(self.send):
            b[q] = i | (lc << 32)

    def freeze_slab_finish(self, recv, rcounts):
        if self.state != 1:
            raise DoubleError(ESTATE, "no slab freeze in progress")
        b = recv.numpy()
        lo = self.splits[self.rank]
        got = []
        for q in range(sum(rcounts)):
            i, lc = int(b[q]) & 0xFFFFFFFF, int(b[q]) >> 32
            if (i + 1, lo + lc + 1) not in self.slot:
                self.unfreeze()
                raise DoubleError(EILLEGAL, "received position not in the pattern")
            got.append(self.slot[(i + 1, lo + lc + 1)])
        low = sum(rcounts[: self.rank])
        self.map = got[:low] + self.own + got[low:]  # [lower ranks | own stream | higher ranks]
        self.low, self.rcounts = low, list(rcounts)
        self.state = 2

    def frozen_slab_counts(self):
        return list(self.send_counts), list(self.rcounts)

    def reassemble_slab_pack(self, V, send):
        assert self.state == 2 and len(V) == self.count
        s = send.numpy()
        for q, (k, _, _) in enumerate(self.send):
            s[q] = np.asarray(V)[k]

    def reassemble_slab_values(self, V, recv, mode=0, zero_first=False):
        if self.state != 2:
            raise DoubleError(ESTATE, "no frozen slab stream")
        r = recv.numpy()
        vals = list(r[: self.low]) + list(np.asarray(V)) + list(r[self.low: len(self.map) - self.count])
        nz = np.zeros_like(self.nz) if zero_first else self.nz
        for s, v in zip(self.map, vals):
            if s is not None:
                nz[s] = nz[s] + v
        self.nz = nz

    # --- just enough of the assembly path for a flush that only this rank's columns see
    def insert_batch(self, I, J, V, flavour=0):
        self.staged += list(zip(I, J, V))

    @property
    def pending(self):
        return len(self.staged)

    def route_count(self):
        return [len(self.staged) if d == self.rank else 0 for d in range(self.world)]

    def route_prepare(self, send, capacity):
        return self.route_count()

    def route_finish(self, src, recv, count):
        assert count == 0

    def flush(self, mode=0):
        changed = False
        for (i, j, v) in self.staged:
            assert self._owner(j) == self.rank
            if (i, j) not in self.slot:
                changed = True
                self.slot[(i, j)] = len(self.nz)
                self.nz = np.append(self.nz, v)
        self.staged = []
        if changed:
            self.unfreeze()  # the library drops the map of a slab whose pattern changed
        return len(self.nz), changed


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _pattern(m, n):
    rng = np.random.default_rng(42)
    ent = {(i, i) for i in range(1, min(m, n) + 1)}
    ent |= set(zip(rng.integers(1, m + 1, 150).tolist(), rng.integers(1, n + 1, 150).tolist()))
    ent = sorted(ent)
    values = {e: float(v) for e, v in zip(ent, rng.standard_normal(len(ent)))}
    return ent, values


def _worker(rank, world, port, m, n, splits, out_q):
    import importlib.util
    import sys

    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        spec = importlib.util.spec_from_file_location("xsb_dist", os.path.join(ROOT, "extendablesparse.jl_b200", "dist.py"))
        xd = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(xd)
        ent, values = _pattern(m, n)
        h = NumpySlabValues(m, n, world, rank, splits, ent, values)
        D = xd.DistExtendableSparseMatrix(m, n, splits=splits, backend=h)
        rng = np.random.default_rng(7 + rank)
        pick = rng.integers(0, len(ent), 200 + 30 * rank)
        I = np.array([ent[p][0] for p in pick])
        J = np.array([ent[p][1] for p in pick])
        res = {"stream": (I, J), "steps": []}
        D.freeze_pattern(I, J)
        for step in range(3):
            V = rng.standard_normal(len(I))
            V[::5] = -0.0
            D.reassemble_values(V if step != 2 else torch.from_numpy(V), zero_first=step != 1)
            res["steps"].append((V, h.nz.copy()))
        # an own position absent from the pattern on rank 1 fails the freeze on every rank
        bad_I, bad_J = I.copy(), J.copy()
        lo, hi = splits[rank], splits[rank + 1]
        missing = next((i, j) for j in range(lo + 1, hi + 1) for i in range(1, m + 1) if (i, j) not in h.slot)
        if rank == 1:
            bad_I[0], bad_J[0] = missing
        res["fail_first"] = _expect_failure(D, h, bad_I, bad_J)
        # a position rank 0 sends to the last rank that the last rank's pattern lacks: fails at finish, everywhere
        last = world - 1
        lmiss = next((i, j) for j in range(splits[last] + 1, splits[last + 1] + 1) for i in range(1, m + 1)
                     if (i, j) not in set(ent))
        bad_I, bad_J = I.copy(), J.copy()
        if rank == 0:
            bad_I, bad_J = np.append(bad_I, lmiss[0]), np.append(bad_J, lmiss[1])
        res["fail_finish"] = _expect_failure(D, h, bad_I, bad_J)
        # an exception without a library status on rank 1 fails the freeze everywhere too
        h.plain_failure = rank == 1
        res["fail_plain"] = _expect_failure(D, h, I, J)
        h.plain_failure = False
        # re-freeze, then a flush that changes the pattern on rank 0 only unfreezes every rank
        D.freeze_pattern(I, J)
        assert h.state == 2 and D._frozen
        if rank == 0:
            D.insert_batch([missing[0]], [missing[1]], [1.0])
        D.flush()
        res["after_change"] = (D.changed_any, h.state, D._frozen)
        try:
            D.reassemble_values(np.zeros(len(I)))
            res["refused"] = False
        except RuntimeError:
            res["refused"] = True
        out_q.put((rank, res))
    finally:
        dist.destroy_process_group()


def _expect_failure(D, h, I, J):
    try:
        D.freeze_pattern(I, J)
    except DoubleError as e:
        return ("own", e.code, h.state, D._frozen)
    except ValueError as e:
        return ("plain", str(e)[:40], h.state, D._frozen)
    except RuntimeError as e:
        return ("other", str(e), h.state, D._frozen)
    return ("none", None, h.state, D._frozen)


@pytest.mark.parametrize("world,splits", [(2, [0, 17, 40]), (3, [0, 1, 22, 40])])
def test_dist_frozen_stream_choreography(world, splits):
    m, n = 30, 40
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, m, n, splits, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(world):
        r, res = q.get(timeout=180)
        got[r] = res
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0

    # serial reference: one matrix folding the rank-ordered concatenation of the streams, step after step
    ent, values = _pattern(m, n)
    glob = dict(values)
    for step in range(3):
        if step != 1:
            glob = {e: 0.0 for e in glob}
        for r in range(world):
            I, J = got[r]["stream"]
            for i, j, v in zip(I.tolist(), J.tolist(), got[r]["steps"][step][0].tolist()):
                glob[(i, j)] = glob[(i, j)] + v
        for r in range(world):
            lo, hi = splits[r], splits[r + 1]
            want = np.array([glob[(i, j)] for (j, i) in sorted((j, i) for (i, j) in ent if lo < j <= hi)])
            assert np.array_equal(got[r]["steps"][step][1].view(np.uint64), want.view(np.uint64)), (step, r)

    for r in range(world):
        kind, code, state, frozen = got[r]["fail_first"]
        assert (kind, code) == (("own", EILLEGAL) if r == 1 else ("other", code)) and state == 0 and not frozen
        kind, code, state, frozen = got[r]["fail_finish"]
        assert kind == ("own" if r == world - 1 else "other") and state == 0 and not frozen
        kind, msg, state, frozen = got[r]["fail_plain"]
        assert state == 0 and not frozen
        if r == 1:
            assert kind == "plain"
        else:
            assert kind == "other" and "rank 1" in msg and "without a library status" in msg, msg
        changed, state, frozen = got[r]["after_change"]
        assert changed and state == 0 and not frozen
        assert got[r]["refused"]


def test_slab_freeze_symbols_are_declared_and_exported():
    import __graft_entry__ as ge

    ge.build()
    import xsparse_b200

    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "xsparse_b200.h")).read(), flags=re.S)
    lib = ctypes.CDLL(xsparse_b200.capi.LIB_PATH)
    for name in ("xsb_freeze_slab", "xsb_freeze_slab_elements", "xsb_freeze_slab_prepare", "xsb_freeze_slab_finish",
                 "xsb_frozen_slab_counts", "xsb_reassemble_slab_pack", "xsb_reassemble_slab_values"):
        assert re.search(r"\b" + name + r"\s*\(", text), name
        assert hasattr(lib, name), name
        assert name in xsparse_b200.capi.SIGNATURES
