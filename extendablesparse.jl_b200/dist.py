"""Column-slab multi-GPU assembly: one process per GPU, torch.distributed for the exchange.

Rank r owns the contiguous column slab [splits[r], splits[r+1]).  Every rank stages the
insertions it generates (any column).  A staged record carries its owner and its column
relative to the owner's slab, so routing only copies OUT what other ranks own
(xsb_route_count + xsb_route_prepare: one read of the keys, the records a rank keeps never
move); those buckets travel with ONE all-to-all-v (NCCL over NVLink), are appended behind the
rank's own records (xsb_route_finish per source, ascending) and xsb_flush merges everything
into the rank's CSC slab.  The fold meets the records of an entry as [resident CSC | lower
ranks | own | higher ranks], each in stream order -- the distributed result equals the serial
reference applied to the rank-ordered concatenation of the ranks' streams.

That is the COUNTED exchange of the first step.  An assembly loop repeats its step: from the second
flush on the blocks have fixed capacities (twice what the counted step moved) and -- on one node --
travel without any collective: the routing kernel stores every block straight into the receiving
rank's mailbox over NVLink peer memory and raises a flag there (xsb_route_pack_peer /
xsb_route_unpack_peer, mailboxes exchanged once through CUDA IPC); NCCL grouped send / receive is
the fallback (XSB_EXCHANGE=nccl, ranks on several nodes, GPUs without peer access).

Reference analogue: the per-partition buffers of GenericMTExtendableSparseMatrixCSC
(genericmtextendablesparsematrixcsc.jl:45-51) summed in partition order
(sparsematrixdilnkc.jl:416-426).  The reference itself is single-process.
"""
from __future__ import annotations

from typing import List, Sequence, Tuple

import torch
import torch.distributed as dist


_ROUTE_MAGIC = 0x5853425F524F5554  # header word of a fixed-capacity block ("XSB_ROUT", xsb_route.cu)
_FAILED_WITHOUT_STATUS = 1000  # a rank's freeze failed with an exception that has no library status code


def uniform_splits(n: int, world: int) -> List[int]:
    """Contiguous column slabs of (almost) equal width."""
    return [(n * r) // world for r in range(world)] + [n]


def exchange_off_rank(send: torch.Tensor, send_counts: Sequence[int], rank: int, group=None
                      ) -> Tuple[torch.Tensor, List[int]]:
    """All-to-all-v of the OFF-RANK buckets of 16-byte records (2 int64 words each).

    `send` holds the buckets for the other ranks, destination after destination (nothing for the
    own rank: those records never left the staging buffer).  Returns the received records, source
    rank after source rank, and the per-source record counts (own rank: 0)."""
    world = dist.get_world_size(group)
    assert len(send_counts) == world
    off = [int(c) if r != rank else 0 for r, c in enumerate(send_counts)]
    sc = torch.tensor(off, dtype=torch.int64, device=send.device)
    rc = torch.empty(world, dtype=torch.int64, device=send.device)
    dist.all_to_all_single(rc, sc, group=group)
    recv_counts = [int(x) for x in rc.cpu().tolist()]
    recv = torch.empty(2 * sum(recv_counts), dtype=torch.int64, device=send.device)
    dist.all_to_all_single(recv, send[: 2 * sum(off)], output_split_sizes=[2 * c for c in recv_counts],
                           input_split_sizes=[2 * c for c in off], group=group)
    return recv, recv_counts


def slab_offsets(nnz_local: int, device, group=None) -> Tuple[int, int]:
    """(entries owned by lower ranks, total entries): the shift that turns a slab's colptr into the
    global colptr (8 bytes per rank on the wire)."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    mine = torch.tensor([nnz_local], dtype=torch.int64, device=device)
    allv = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allv, mine, group=group)
    counts = [int(t.item()) for t in allv]
    return sum(counts[:rank]), sum(counts)


class DistExtendableSparseMatrix:
    """ExtendableSparseMatrix sharded by column ownership over the ranks of a process group.

    `backend` is the per-rank slab object; the product backend is capi.Handle in slab mode
    (libxsparse_b200).  It must offer: pending, route_count() -> counts, route_prepare(send, capacity)
    -> counts, route_finish(src, records, count) (ascending src), flush(mode) -> (nnz, changed).
    """

    def __init__(self, m: int, n: int, splits: Sequence[int] | None = None, group=None, device=None, backend=None,
                 idx_type=None, index_base: int = 1):
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.m, self.n = int(m), int(n)
        self.splits = list(splits) if splits is not None else uniform_splits(self.n, self.world)
        assert len(self.splits) == self.world + 1 and self.splits[0] == 0 and self.splits[-1] == self.n
        if backend is None:
            from . import capi

            dev = torch.cuda.current_device() if device is None else int(device)
            backend = capi.Handle(self.m, self.n, capi.I64 if idx_type is None else idx_type, index_base, 1, dev,
                                  slab=(self.world, self.rank, self.splits))
            self.device = torch.device("cuda", dev)
        else:
            self.device = torch.device("cpu") if device is None else device
        self.h = backend
        self.col_begin, self.col_end = self.splits[self.rank], self.splits[self.rank + 1]
        self._nnz_offset = 0
        self._nnz_global = 0
        self._changed_any = False
        self._offsets_pending = None
        self.last_exchange = {"sent_off_rank": 0, "received_off_rank": 0, "kept": 0}
        self._send = None
        self.last_phase_ms = []
        # fixed-capacity exchange (xsb_route_pack / xsb_route_unpack): capacities both sides derive from the last
        # exactly counted step -- what this rank sent to d is what d received from this rank
        self._caps_out = None  # per destination rank
        self._caps_in = None   # per source rank
        self._recv = None
        self._lib_stream = None
        self.fixed_steps = 0
        import os

        self._phase_events = os.environ.get("XSB_DIST_TIMING", "") == "1"
        self.last_device_phase_ms = None
        # transport of the fixed-capacity blocks: "peer" = straight into the receiver's mailbox over NVLink peer
        # memory (xsb_route_pack_peer / xsb_route_unpack_peer; ranks of one node), "nccl" = grouped send / receive
        self._transport_wanted = os.environ.get("XSB_EXCHANGE", "peer").lower()
        self._peer = None  # None: not decided yet; True / False after the first fixed-capacity step
        self._early = False  # exchange_begin() already packed this step
        self.transport_note = ""
        # values-only re-assembly of a stream frozen across the slabs (freeze_pattern / freeze_elements): the sizes of
        # the per-step exchange of values, fixed at freeze time (own rank: 0)
        self._frozen = False
        self._vcounts_out = None  # per destination rank
        self._vcounts_in = None   # per source rank
        self._vsend = None
        self._vrecv = None

    # insertion: global (i,j) on any rank
    def insert_batch(self, I, J, V, flavour=0):
        self.h.insert_batch(I, J, V, flavour)

    def insert_elements(self, dofs, Aloc, flavour=1, col_dofs=None):  # XSB_RAW: the element loop's rawupdateindex!
        self.h.insert_elements(dofs, Aloc, flavour, col_dofs=col_dofs)

    def _send_buffer(self, records: int) -> torch.Tensor:
        words = 2 * max(records, 1)
        if self._send is None or self._send.numel() < words:
            self._send = torch.empty(words, dtype=torch.int64, device=self.device)
        return self._send

    @staticmethod
    def _capacity(count: int) -> int:
        """Block capacity for a bucket that held `count` records in the last counted step.  A pair of ranks that
        exchanged nothing then is left out of the fixed-capacity steps altogether (capacity 0: a record for such a
        rank later on makes the flush fail; `recount()` makes the next step a counted one again)."""
        return 0 if int(count) == 0 else max(1024, 2 * int(count))

    def recount(self):
        """The next flush counts again (exact exchange) and re-derives the block capacities.  Collective."""
        self._caps_out = self._caps_in = None
        self._recv = None
        self._teardown_peer()

    def _setup_peer(self):
        """Collective: every rank allocates its mailbox, the 64-byte IPC handles are all-gathered, every rank maps
        the mailboxes of the ranks it exchanges blocks with.  Any rank failing (GPUs without peer access, ranks on
        different nodes) makes ALL ranks fall back to the NCCL transport."""
        import socket

        self._peer = False
        if self._transport_wanted != "peer" or not hasattr(self.h, "route_pack_peer") or self.device.type != "cuda":
            self.transport_note = "nccl (requested)" if self._transport_wanted != "peer" else "nccl"
            return
        world = self.world
        mine = {"host": socket.gethostname(), "caps_in": [int(c) for c in self._caps_in], "handle": None, "err": None}
        try:
            rows = [None] * world
            dist.all_gather_object(rows, mine["caps_in"], group=self.group)
            caps = [[0 if s == d else int(rows[d][s]) for s in range(world)] for d in range(world)]
            mine["handle"] = self.h.peer_exchange_create(caps)
        except Exception as e:  # noqa: BLE001  (reported to all ranks below)
            mine["err"] = str(e)[:200]
        infos = [None] * world
        dist.all_gather_object(infos, mine, group=self.group)
        ok = all(i["err"] is None and i["handle"] is not None for i in infos) and len({i["host"] for i in infos}) == 1
        err = None
        if ok:
            try:
                self.h.peer_exchange_connect(b"".join(i["handle"] for i in infos))
            except Exception as e:  # noqa: BLE001
                err = str(e)[:200]
        errs = [None] * world
        dist.all_gather_object(errs, err, group=self.group)
        if ok and all(e is None for e in errs):
            self._peer = True
            self.transport_note = "peer memory (mailboxes over NVLink, CUDA IPC)"
            return
        why = next((i["err"] for i in infos if i["err"]), None) or next((e for e in errs if e), None) or "ranks on several nodes"
        self.transport_note = f"nccl (peer exchange unavailable: {why})"
        self._teardown_peer(force=True)

    def _teardown_peer(self, force=False):
        if (self._peer or force) and hasattr(self.h, "peer_exchange_disconnect"):
            self.h.peer_exchange_disconnect()
            dist.barrier(group=self.group)  # nobody frees a mailbox that a peer still has mapped
            self.h.peer_exchange_destroy()
        self._peer = None if not force else False

    def close(self):
        """Collective: releases the peer mailboxes (if any) and the slab handle."""
        self._resolve_offsets()
        self._teardown_peer()
        self.h.close()

    def _flush_fixed(self, mode, wait):
        """The step of an assembly LOOP: same routing, but with the block capacities agreed after the last counted
        step no count visits the host -- pack, ONE all-to-all with host-known split sizes, unpack and the flush are
        stream-ordered on the library's stream (NCCL is chained to it through the current-stream events)."""
        import time

        t0 = time.perf_counter()
        h, world, rank = self.h, self.world, self.rank
        if self._peer is None:
            self._setup_peer()
        if self._peer:
            return self._flush_peer(mode, wait, t0)
        co = [0 if d == rank else self._caps_out[d] for d in range(world)]
        ci = [0 if s == rank else self._caps_in[s] for s in range(world)]
        in_split = [0 if d == rank else 2 * (co[d] + 1) for d in range(world)]
        out_split = [0 if s == rank else 2 * (ci[s] + 1) for s in range(world)]
        if self._send is None or self._send.numel() < max(sum(in_split), 2):
            self._send = torch.empty(max(sum(in_split), 2), dtype=torch.int64, device=self.device)
        if self._recv is None or self._recv.numel() < max(sum(out_split), 2):
            # every block starts with a header {records, magic}; the blocks of ranks that send nothing are never
            # received into and keep the "no records" header written here
            self._recv = torch.zeros(max(sum(out_split), 2), dtype=torch.int64, device=self.device)
            pos = 0
            for s in range(world):
                if s != rank:
                    self._recv[pos + 1] = _ROUTE_MAGIC
                    pos += out_split[s]
        if self._lib_stream is None:
            self._lib_stream = torch.cuda.ExternalStream(h.stream, device=self.device)
        cnt = int(h.pending)
        ev = None
        if self._phase_events:  # device-side phase times (XSB_DIST_TIMING=1): events on the library's stream
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
            ev[0].record(self._lib_stream)
        h.route_pack(self._send, co, sum(in_split) // 2)
        if ev:
            ev[1].record(self._lib_stream)
        # point-to-point with the ranks this rank actually exchanges records with (an interface plane: the
        # neighbours), grouped into one NCCL launch; no collective couples ranks that share nothing
        ops, spos, rpos = [], 0, 0
        for p in range(world):
            if p == rank:
                continue
            if co[p] > 0:
                ops.append(dist.P2POp(dist.isend, self._send[spos: spos + in_split[p]], p, group=self.group))
            if ci[p] > 0:
                ops.append(dist.P2POp(dist.irecv, self._recv[rpos: rpos + out_split[p]], p, group=self.group))
            spos += in_split[p]
            rpos += out_split[p]
        if ops:
            with torch.cuda.stream(self._lib_stream):
                for w in dist.batch_isend_irecv(ops):
                    w.wait()  # stream-level: the library's stream waits for the transfers, the host does not
        if ev:
            ev[2].record(self._lib_stream)
        h.route_unpack(self._recv, ci)
        if ev:
            ev[3].record(self._lib_stream)
        nnz, changed = h.flush(mode)
        if ev:
            ev[4].record(self._lib_stream)
            ev[4].synchronize()
            self.last_device_phase_ms = {"pack": ev[0].elapsed_time(ev[1]), "p2p": ev[1].elapsed_time(ev[2]),
                                         "unpack": ev[2].elapsed_time(ev[3]), "flush": ev[3].elapsed_time(ev[4])}
        mine = torch.tensor([nnz, int(changed)], dtype=torch.int64, device=self.device)
        allv = torch.empty(2 * world, dtype=torch.int64, device=self.device)
        work = dist.all_gather_into_tensor(allv, mine, group=self.group, async_op=True)
        self._offsets_pending = (work, allv, mine)
        self.last_exchange = {"sent_off_rank": None, "received_off_rank": None, "kept": None, "staged": cnt,
                              "transport": self.transport_note, "fixed_capacity_blocks": {"out": co, "in": ci}}
        if wait:
            self._resolve_offsets()
        self.fixed_steps += 1
        self.last_phase_ms = [0.0, 0.0, 0.0, 0.0, 1e3 * (time.perf_counter() - t0), 0.0]
        return nnz, (self._changed_any if wait else bool(changed))

    def exchange_begin(self):
        """Optional, between insertions: everything staged SO FAR that other ranks own leaves now (peer transport:
        xsb_route_pack_peer stores it into the receivers' mailboxes while this rank goes on inserting); what is
        inserted afterwards in this step must be owned by this rank -- `flush` fails otherwise.  An assembly loop
        that visits its interface elements first hides the whole exchange behind the interior.  Without the peer
        transport (counted steps, NCCL) the call does nothing and `flush` exchanges everything."""
        if self._peer is None and self._caps_out is not None and hasattr(self.h, "route_pack"):
            self._setup_peer()
        if self._peer and not self._early:
            self.h.route_pack_peer()
            self._early = True

    def _flush_peer(self, mode, wait, t0):
        """The fixed-capacity step over peer memory: the copy-out kernel of xsb_route_pack_peer stores every block
        into its receiver's mailbox and raises the receiver's flag; xsb_route_unpack_peer waits for this step's
        flags on the library's stream, takes the blocks and frees them for the senders.  No NCCL call, no host
        synchronisation before the flush."""
        import time

        h, world = self.h, self.world
        cnt = int(h.pending)
        ev = None
        if self._phase_events:
            if self._lib_stream is None:
                self._lib_stream = torch.cuda.ExternalStream(h.stream, device=self.device)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            ev[0].record(self._lib_stream)
        if not self._early:
            h.route_pack_peer()
        self._early = False
        if ev:
            ev[1].record(self._lib_stream)
        h.route_unpack_peer()
        if ev:
            ev[2].record(self._lib_stream)
        nnz, changed = h.flush(mode)
        if ev:
            ev[3].record(self._lib_stream)
            ev[3].synchronize()
            self.last_device_phase_ms = {"pack": ev[0].elapsed_time(ev[1]), "p2p": 0.0,
                                         "unpack": ev[1].elapsed_time(ev[2]), "flush": ev[2].elapsed_time(ev[3])}
        mine = torch.tensor([nnz, int(changed)], dtype=torch.int64, device=self.device)
        allv = torch.empty(2 * world, dtype=torch.int64, device=self.device)
        work = dist.all_gather_into_tensor(allv, mine, group=self.group, async_op=True)
        self._offsets_pending = (work, allv, mine)
        self.last_exchange = {"sent_off_rank": None, "received_off_rank": None, "kept": None, "staged": cnt,
                              "transport": self.transport_note,
                              "fixed_capacity_blocks": {"out": [0 if d == self.rank else self._caps_out[d] for d in range(world)],
                                                        "in": [0 if s == self.rank else self._caps_in[s] for s in range(world)]}}
        if wait:
            self._resolve_offsets()
        self.fixed_steps += 1
        self.last_phase_ms = [0.0, 0.0, 0.0, 0.0, 1e3 * (time.perf_counter() - t0), 0.0]
        return nnz, (self._changed_any if wait else bool(changed))

    def flush(self, mode=0, wait=True, fixed=None):
        """Route, exchange, merge.  Returns (local nnz, pattern changed on any rank); with wait=False the
        second value is the LOCAL flag and the global one is `changed_any` (read on demand).

        fixed: None = the fixed-capacity exchange once a counted step has set the capacities (product backend
        only; every rank takes the same decision: the counted step is collective); False = always count."""
        import time

        can_fix = hasattr(self.h, "route_pack") and self.device.type == "cuda"
        if fixed is None:
            fixed = can_fix and self._caps_out is not None
        if fixed:
            if not can_fix or self._caps_out is None:
                raise RuntimeError("fixed-capacity exchange needs a counted step first")
            return self._flush_fixed(mode, wait)

        t = [time.perf_counter()]

        def lap():
            t.append(time.perf_counter())

        cnt = int(self.h.pending)
        counts = self.h.route_count()
        lap()
        leaving = sum(c for r, c in enumerate(counts) if r != self.rank)
        send = self._send_buffer(leaving)
        self.h.route_prepare(send, leaving)
        lap()
        recv, rcounts = exchange_off_rank(send, counts, self.rank, self.group)
        if self.device.type == "cuda":
            torch.cuda.current_stream(self.device).synchronize()
        lap()
        pos = 0
        for src in range(self.world):  # ascending source rank; the own records stayed where they were
            if src != self.rank:
                self.h.route_finish(src, recv[2 * pos: 2 * (pos + rcounts[src])], rcounts[src])
                pos += rcounts[src]
        lap()
        nnz, changed = self.h.flush(mode)
        lap()
        # one 16-byte all-gather: entries per slab (-> global colptr offsets) and "pattern changed".  With
        # wait=False it is only LAUNCHED here (stream-ordered behind the flush); nnz_offset / nnz_global /
        # changed_any read it when they are first asked for, so an assembly loop that does not look at
        # the global offsets every step does not stop for them.
        mine = torch.tensor([nnz, int(changed)], dtype=torch.int64, device=self.device)
        allv = torch.empty(2 * self.world, dtype=torch.int64, device=self.device)
        work = dist.all_gather_into_tensor(allv, mine, group=self.group, async_op=True)
        self._offsets_pending = (work, allv, mine)
        self.last_exchange = {"sent_off_rank": cnt - counts[self.rank], "received_off_rank": sum(rcounts),
                              "kept": counts[self.rank]}
        self._caps_out = [self._capacity(c) for c in counts]
        self._caps_in = [self._capacity(c) for c in rcounts]
        if wait:
            self._resolve_offsets()
        lap()
        # host wall time of the phases (ms): count, copy-out, all-to-all, append, flush, offsets
        self.last_phase_ms = [1e3 * (b - a) for a, b in zip(t[:-1], t[1:])]
        return nnz, (self._changed_any if wait else bool(changed))

    def _resolve_offsets(self):
        if self._offsets_pending is not None:
            work, allv, _ = self._offsets_pending
            work.wait()
            vals = allv.cpu().tolist()
            per_rank, flags = vals[0::2], vals[1::2]
            self._nnz_offset, self._nnz_global = sum(per_rank[: self.rank]), sum(per_rank)
            self._changed_any = any(flags)
            self._offsets_pending = None
            if self._changed_any and self._frozen:
                # the pattern changed on some rank: the values its frozen stream sends elsewhere no longer fit the
                # owners' maps, so every rank drops its map (the rank whose pattern changed already has)
                self.unfreeze()

    # ---- values-only re-assembly of a stream frozen across the slabs ----
    def _fail_everywhere(self, err):
        """Collective: every rank learns whether any rank failed; if one did, every rank is left unfrozen and raises
        (the failing rank its own error)."""
        codes = torch.zeros(self.world, dtype=torch.int64, device=self.device)
        if err is not None:
            # any failure counts, also one that carries no library status (a bad argument caught in Python): the MAX
            # reduction only sees positive entries
            code = getattr(err, "code", None)
            codes[self.rank] = code if isinstance(code, int) and code > 0 else _FAILED_WITHOUT_STATUS
        dist.all_reduce(codes, op=dist.ReduceOp.MAX, group=self.group)
        bad = [(r, c) for r, c in enumerate(codes.cpu().tolist()) if c != 0]
        if not bad:
            return
        self.unfreeze()
        if err is not None:
            raise err
        r, c = bad[0]
        why = "an error without a library status" if c == _FAILED_WITHOUT_STATUS else f"status {c}"
        raise RuntimeError(f"freezing the slab stream failed on rank {r} ({why}); every rank is left unfrozen")

    def _freeze(self, first):
        """The collective freeze: `first()` resolves the own positions and returns the positions per owner; the counts
        and then the foreign positions (8 bytes each) travel all-to-all; finish resolves what arrived."""
        self.unfreeze()
        self._resolve_offsets()
        counts, err = None, None
        try:
            counts = first()
        except Exception as e:  # noqa: BLE001  (reported to every rank)
            err = e
        self._fail_everywhere(err)
        world, rank = self.world, self.rank
        off = [0 if r == rank else int(c) for r, c in enumerate(counts)]
        send = torch.empty(max(sum(off), 1), dtype=torch.int64, device=self.device)
        err = None
        try:
            self.h.freeze_slab_prepare(send, sum(off))
        except Exception as e:  # noqa: BLE001
            err = e
        self._fail_everywhere(err)
        if self.device.type == "cuda":
            torch.cuda.current_stream(self.device).synchronize()
        sc = torch.tensor(off, dtype=torch.int64, device=self.device)
        rc = torch.empty(world, dtype=torch.int64, device=self.device)
        dist.all_to_all_single(rc, sc, group=self.group)
        rcounts = [0 if r == rank else int(c) for r, c in enumerate(rc.cpu().tolist())]
        recv = torch.empty(max(sum(rcounts), 1), dtype=torch.int64, device=self.device)
        dist.all_to_all_single(recv[: sum(rcounts)], send[: sum(off)], output_split_sizes=rcounts,
                               input_split_sizes=off, group=self.group)
        if self.device.type == "cuda":
            torch.cuda.current_stream(self.device).synchronize()
        err = None
        try:
            self.h.freeze_slab_finish(recv, rcounts)
        except Exception as e:  # noqa: BLE001
            err = e
        self._fail_everywhere(err)
        self._vcounts_out, self._vcounts_in = off, rcounts
        self._vsend = torch.empty(max(sum(off), 1), dtype=torch.float64, device=self.device)
        self._vrecv = torch.empty(max(sum(rcounts), 1), dtype=torch.float64, device=self.device)
        self._frozen = True

    def freeze_pattern(self, I, J):
        """Collective: freezes this rank's stream of GLOBAL positions (I[k], J[k]) -- any owner -- for values-only
        re-assembly.  Every position must already be an entry of its owner's slab.  One rank's error (a position
        outside the matrix or absent from the pattern) fails the freeze on every rank and leaves every rank unfrozen."""
        self._freeze(lambda: self.h.freeze_slab(I, J))

    def freeze_elements(self, dofs, col_dofs=None):
        """freeze_pattern for the stream insert_elements(dofs, ., col_dofs=col_dofs) stages: reassemble_values then
        takes the element matrices ((ncells, k, k), or (ncells, kc, kr) with col_dofs) as they are."""
        self._freeze(lambda: self.h.freeze_slab_elements(dofs, col_dofs))

    def unfreeze(self):
        self.h.unfreeze()
        self._frozen = False
        self._vcounts_out = self._vcounts_in = None

    def reassemble_values(self, V, mode=0, zero_first=True):
        """One values-only step: V holds a value per position of this rank's frozen stream.  The values of positions
        other ranks own go to them with one grouped point-to-point exchange whose sizes were fixed at freeze time, and
        every slab entry folds its resident value (+0.0 with zero_first) followed by the values of rank 0, 1, ... in
        each rank's stream order -- the same bits as one matrix re-assembling the rank-ordered concatenation of the
        streams.  Stream-ordered on the library's stream; the host does not wait for the device."""
        self._resolve_offsets()
        if not self._frozen:
            raise RuntimeError("no frozen stream: freeze_pattern / freeze_elements first")
        h, world, rank = self.h, self.world, self.rank
        co, ci = self._vcounts_out, self._vcounts_in
        if self.device.type == "cuda":
            if self._lib_stream is None:
                self._lib_stream = torch.cuda.ExternalStream(h.stream, device=self.device)
            self._lib_stream.wait_stream(torch.cuda.current_stream(self.device))  # V may come from the current stream
        h.reassemble_slab_pack(V, self._vsend)
        ops, spos, rpos = [], 0, 0
        for p in range(world):
            if p == rank:
                continue
            if co[p] > 0:
                ops.append(dist.P2POp(dist.isend, self._vsend[spos: spos + co[p]], p, group=self.group))
            if ci[p] > 0:
                ops.append(dist.P2POp(dist.irecv, self._vrecv[rpos: rpos + ci[p]], p, group=self.group))
            spos += co[p]
            rpos += ci[p]
        if ops:
            if self.device.type == "cuda":
                with torch.cuda.stream(self._lib_stream):
                    for w in dist.batch_isend_irecv(ops):
                        w.wait()  # stream-level: the library's stream waits for the transfers, the host does not
            else:
                for w in dist.batch_isend_irecv(ops):
                    w.wait()
        h.reassemble_slab_values(V, self._vrecv, mode, zero_first)
        if self.device.type == "cuda" and isinstance(V, torch.Tensor) and V.is_cuda:
            # the pack and the fold read V on the library's stream, which the host does not wait for: keep V's memory
            # from being handed to new work on other streams before they are done
            V.record_stream(self._lib_stream)

    def dropzeros(self):
        """Collective dropzeros!: every rank removes the stored +-0.0 of its own slab (no entries move between ranks),
        then one all-gather refreshes nnz_offset / nnz_global and whether any rank's pattern changed; if one did,
        every rank unfreezes, as after a flush.  Returns (local nnz, pattern changed on any rank)."""
        self._resolve_offsets()
        nnz, changed = self.h.dropzeros()
        mine = torch.tensor([nnz, int(changed)], dtype=torch.int64, device=self.device)
        allv = torch.empty(2 * self.world, dtype=torch.int64, device=self.device)
        work = dist.all_gather_into_tensor(allv, mine, group=self.group, async_op=True)
        self._offsets_pending = (work, allv, mine)
        self._resolve_offsets()
        return nnz, self._changed_any

    @property
    def nnz_offset(self) -> int:
        """Entries owned by lower ranks: the shift from the slab's colptr to the global one."""
        self._resolve_offsets()
        return self._nnz_offset

    @property
    def nnz_global(self) -> int:
        self._resolve_offsets()
        return self._nnz_global

    @property
    def changed_any(self) -> bool:
        """The last flush changed the pattern on some rank."""
        self._resolve_offsets()
        return self._changed_any

    def mul(self, x_local, out=None):
        """y = A * x for the matrix sharded by column slabs: rank r holds x[col_begin:col_end] and computes its slab's
        contribution A[:, slab] * x[slab] with the column-order kernel (xsb_mul: every y_i a left fold over the slab's
        columns, separately rounded products); the contributions are then summed over the ranks in RANK ORDER,
        y = ((y_0 + y_1) + y_2) + ..., on every rank, from one all-gather -- so all ranks hold the same bits and the
        result does not depend on the collective's internal reduction tree.  Reference: the partition loop of
        mul!(r, ext::GenericMTExtendableSparseMatrixCSC, x) (genericmtextendablesparsematrixcsc.jl:124-143), whose
        row partitions write disjoint parts of r; with column slabs the parts overlap and are added in slab order.
        Against the single-process column-order sum this re-associates the additions at the slab boundaries only
        (|error| <= (ranks-1) ulps of the partial sums); patterns whose rows never span two slabs give identical bits."""
        y = torch.empty(self.m, dtype=torch.float64, device=self.device) if self.device.type == "cuda" else None
        if y is None:
            import numpy as np

            y = torch.from_numpy(self.h.mul(np.ascontiguousarray(x_local)))
        else:
            self.h.mul(x_local, y)
        parts = torch.empty((self.world, self.m), dtype=torch.float64, device=y.device)
        dist.all_gather_into_tensor(parts.view(-1), y, group=self.group)
        acc = parts[0].clone() if out is None else out.copy_(parts[0])
        for r in range(1, self.world):
            acc += parts[r]
        return acc

    def global_colptr(self, local_colptr):
        """Slab colptr (slab_width+1 entries) shifted to index the global rowval/nzval arrays."""
        return local_colptr + self.nnz_offset
