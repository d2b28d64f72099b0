#!/usr/bin/env python
"""Flushes forced onto the column-sort fallback (column_path 2: grouping off, a stable sort by column, then the
thread-per-column fold) for FEM 128^3, fdrand 200^3 and block RD 96^3 x 4 (development tool, not a bench line).

  python tools/exp_thread_fold.py [--root TREE] [--reps N] [--warmup W] [fem128] [fd200] [rd96]

--root imports the library of another checkout (for example the parent commit) so that two versions can be timed
on the same card, alternating processes.  One JSON line per workload: the flush times (host clock around flush!,
which ends in a device synchronise; the emit is not timed), their median, the column path and whether the one-pass
(direct) fold ran, and the SHA-256 of colptr|rowval|nzval; then one line with the card's name and power limit.
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--reps", type=int, default=7)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("workloads", nargs="*", default=["fem128", "fd200", "rd96"])
args = ap.parse_args()
if args.reps < 5:
    raise SystemExit("--reps: at least 5 timed flushes")

sys.path.insert(0, os.path.abspath(args.root))
import __graft_entry__ as ge  # noqa: E402

ge.build()
import xsparse_b200 as xsb  # noqa: E402


def emitter(name):
    kind = name.rstrip("0123456789")
    size = int(name[len(kind):])
    if kind == "fem":
        return size ** 3, lambda h: h.emit_p1fem(size, size, size, flavour=xsb.RAW)
    if kind == "fd":
        return size ** 3, lambda h: h.emit_fdrand(size, size, size, seed=7)
    if kind == "rd":
        return 4 * size ** 3, lambda h: h.emit_blockrd(size, size, size, 4, seed=7)
    raise SystemExit(f"unknown workload {name}")


def run(name):
    n, emit = emitter(name)
    h = xsb.Handle(n, n)
    h.set_grouping(xsb.capi.GROUPING_OFF)
    times = []
    for r in range(args.warmup + args.reps):
        h.reset()
        emit(h)
        t0 = time.perf_counter()
        h.flush()
        t1 = time.perf_counter()
        if r >= args.warmup:
            times.append((t1 - t0) * 1e3)
    st = h.flush_stats()
    if st["column_path"] != 2:
        raise SystemExit(f"{name}: column_path {st['column_path']}, not the column-sort fallback")
    cp, rv, nz = h.fetch_csc_numpy()
    dig = hashlib.sha256()
    for a in (cp, rv, nz):
        dig.update(a.tobytes())
    h.close()
    print(json.dumps({"root": os.path.abspath(args.root), "workload": name, "ms": [round(t, 4) for t in times],
                      "median_ms": round(statistics.median(times), 4), "column_path": st["column_path"],
                      "direct_fold": st["direct_fold"], "nnz": int(st["nnz_new"]), "csc_sha256": dig.hexdigest()}),
          flush=True)


for w in args.workloads:
    run(w)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                      text=True).stdout.strip()
print(json.dumps({"card": card}), flush=True)
