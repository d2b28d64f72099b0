#!/usr/bin/env python
"""Values-only re-assembly of fdrand n^3 (cfg 5 at the default n = 400) on column slabs, one GPU per rank.

    torchrun --nproc-per-node N tools/exp_values_dist.py [n] [steps]

Every rank generates the calls of its node range (xsb_emit_fdrand_range), builds its slab with the routed flush and
freezes its stream of global positions across the ranks (DistExtendableSparseMatrix.freeze_pattern).  A step is
reassemble_values(V, zero_first=True): pack, grouped point-to-point of the interface values, fold.  It is timed with
CUDA events on the library's stream; the reported time is the largest over the ranks.  With N = 1 the same global
stream runs through a plain handle (xsb_reassemble_values_zeroed).  Rank 0 prints one JSON line per mode with the
time per step, B_vo per rank (SURVEY.md section 8d: 8 B per value read, 4 B per map entry, 8 B per nzval written)
over the device copy rate measured in the same run, the bytes exchanged per step, the card, its power limit, and
whether the SHA-256 of every rank's nzval equals the same slice of a plain handle that re-assembled the rank-ordered
concatenation of the streams (checked for N > 1 against a plain handle on rank 0's GPU)."""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import __graft_entry__ as ge  # noqa: E402

ge.build()
import xsparse_b200 as xsb  # noqa: E402
from xsparse_b200 import capi  # noqa: E402
from xsparse_b200.dist import DistExtendableSparseMatrix  # noqa: E402

SEED = 20240717


def node_stream(nx, lo, hi, dev):
    """(I, J, V) of the calls of fdrand nodes [lo, hi) in call order, on the device."""
    n = nx ** 3
    g = xsb.Handle(n, n, device=dev)
    g.set_precount(False)  # keep the staged records in call order
    g.emit_fdrand(nx, nx, nx, seed=SEED, l_range=(lo, hi))
    cnt = g.pending
    I = torch.empty(max(cnt, 1), dtype=torch.int64, device=f"cuda:{dev}")
    J, V = torch.empty_like(I), torch.empty(max(cnt, 1), dtype=torch.float64, device=f"cuda:{dev}")
    got = C.c_int64(0)
    capi.check(capi.lib().xsb_debug_fetch_staged(g._h, 0, I.data_ptr(), J.data_ptr(), V.data_ptr(), None, cnt,
                                                  C.byref(got)), g._h)
    g.close()
    return I[:cnt], J[:cnt], V[:cnt]


def copy_rate(dev):
    x = torch.empty(1 << 28, dtype=torch.float64, device=f"cuda:{dev}")
    y = torch.empty_like(x)
    y.copy_(x)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(10):
        y.copy_(x)
    b.record()
    b.synchronize()
    return 2 * 8 * x.numel() * 10 / (a.elapsed_time(b) * 1e-3) / 1e9  # GB/s, read + write


def timed(stream, fn, steps):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record(stream)
    for _ in range(steps):
        fn()
    b.record(stream)
    b.synchronize()
    return a.elapsed_time(b) / steps


def main():
    nx = int(sys.argv[1]) if len(sys.argv) > 1 else 400
    steps = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(dev)
    n = nx ** 3
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                          "-i", str(dev)], capture_output=True, text=True).stdout.strip()
    rate = copy_rate(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))
    lo, hi = (n * rank) // world, (n * (rank + 1)) // world
    I, J, V = node_stream(nx, lo, hi, dev)
    out = {}
    if world == 1:
        h = xsb.Handle(n, n, device=dev)
        h.emit_fdrand(nx, nx, nx, seed=SEED)
        h.flush()
        h.freeze_pattern(I, J, count=len(I))
        stream = torch.cuda.ExternalStream(h.stream, device=f"cuda:{dev}")
        for name, mode in (("deterministic", capi.DETERMINISTIC), ("fast", capi.FAST)):
            ms = timed(stream, lambda: h.reassemble_values(V, mode, count=len(V), zero_first=True), steps)
            h.synchronize()
            nz = h.fetch_csc_numpy()[2]
            b_vo = 12 * len(V) + 8 * h.nnz
            out[name] = {"ms": ms, "b_vo_per_rank": [b_vo], "share_of_copy_rate": b_vo / (ms * 1e-3) / (rate * 1e9),
                         "exchanged_bytes_per_step": 0, "sha256": [hashlib.sha256(nz.tobytes()).hexdigest()],
                         "slab_matches_single": True}
    else:
        D = DistExtendableSparseMatrix(n, n, device=dev)
        D.h.emit_fdrand(nx, nx, nx, seed=SEED, l_range=(lo, hi))
        D.flush()
        D.freeze_pattern(I, J)
        sc, rc = D.h.frozen_slab_counts()
        stream = torch.cuda.ExternalStream(D.h.stream, device=f"cuda:{dev}")
        for name, mode in (("deterministic", capi.DETERMINISTIC), ("fast", capi.FAST)):
            ms = timed(stream, lambda: D.reassemble_values(V, mode, zero_first=True), steps)
            D.h.synchronize()
            msall = [None] * world
            dist.all_gather_object(msall, ms)
            nz = D.h.fetch_csc_numpy()[2]
            total = len(V) + sum(rc)
            b_vo = 12 * total + 8 * D.h.nnz + 8 * sum(c for d, c in enumerate(sc) if d != rank)
            info = [None] * world
            dist.all_gather_object(info, (b_vo, 8 * sum(c for d, c in enumerate(sc) if d != rank),
                                          hashlib.sha256(nz.tobytes()).hexdigest(), D.h.nnz))
            out[name] = {"ms": max(msall), "ms_per_rank": msall, "b_vo_per_rank": [x[0] for x in info],
                         "share_of_copy_rate": max(x[0] for x in info) / (max(msall) * 1e-3) / (rate * 1e9),
                         "exchanged_bytes_per_step": sum(x[1] for x in info), "sha256": [x[2] for x in info],
                         "nnz": [x[3] for x in info]}
        # the single-handle reference: rank 0 alone receives every rank's stream, releases its slab and re-assembles
        # the rank-ordered concatenation on one plain handle
        allIJV = [None] * world if rank == 0 else None
        dist.gather_object((I.cpu().numpy(), J.cpu().numpy(), V.cpu().numpy()), allIJV, dst=0)
        del I, J, V
        D.close()
        if rank == 0:
            torch.cuda.empty_cache()
            P = xsb.Handle(n, n, device=dev)
            P.emit_fdrand(nx, nx, nx, seed=SEED)
            P.flush()
            Ic = np.concatenate([x[0] for x in allIJV])
            Jc = np.concatenate([x[1] for x in allIJV])
            Vc = np.concatenate([x[2] for x in allIJV])
            P.freeze_pattern(Ic, Jc)
            for name, mode in (("deterministic", capi.DETERMINISTIC), ("fast", capi.FAST)):
                if mode == capi.FAST:
                    continue  # atomics: the bits depend on the order the hardware takes
                P.reassemble_values(Vc, mode, zero_first=True)
                nz = P.fetch_csc_numpy()[2]
                off, ok = 0, True
                for r in range(world):
                    cnt = out[name]["nnz"][r]
                    ok &= hashlib.sha256(nz[off: off + cnt].tobytes()).hexdigest() == out[name]["sha256"][r]
                    off += cnt
                out[name]["slab_matches_single"] = ok
            P.close()
    if rank == 0:
        for name, r in out.items():
            r.pop("sha256", None)
            print(json.dumps({"cfg": f"fdrand {nx}^3", "ranks": world, "mode": name, "gpu": gpu,
                              "copy_rate_GBps": rate, **r}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
