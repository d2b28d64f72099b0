#!/usr/bin/env python
"""Element-by-element insertion against the generic insertion paths (development tool).

Input: FEM mesh^3 (default 128^3: 12,290,298 tetrahedra, k = 4, 196,644,768 calls) in element form, resident in HBM:
cellnodes[t, jl] = J[20 t + 1 + jl], Aloc[il, jl, t] = V[20 t + 5 il + 1 + jl] of the emitter's stream (the mass
terms are dropped).  The same calls go in four ways, alternating, after one warm-up round:
    elements/i32   xsb_insert_elements, Int32 dofs (Int32 handle)
    elements/i64   xsb_insert_elements, Int64 dofs
    triplets       xsb_insert_triplets of the expanded stream on the device (16 B per call)
    ijv/i64        xsb_insert_batch of device (I, J, V) arrays, Int64 indices (24 B per call)
Per path: insert and flush time (CUDA events on the handle's stream; the insert includes its bounds read-back), the
flush's column path and precounted share, G insertions/s, the insert's algorithmic bytes (what it must read and the
16-byte records it writes) and their share of the device-to-device copy rate measured in the same run.  The card's
name and power limit are read in the same run.  All paths must give the same CSC bits.
Usage: exp_elements.py [mesh] [reps]"""
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import __graft_entry__ as ge  # noqa: E402

ge.build()
import xsparse_b200 as xsb  # noqa: E402

mesh = int(sys.argv[1]) if len(sys.argv) > 1 else 128
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
n = mesh ** 3


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return {"name": name, "nvidia_smi": q[0] if q else None}
    except (OSError, subprocess.SubprocessError):
        return {"name": name, "nvidia_smi": None}


def copy_peak_gbs(nbytes=1 << 32, rounds=10):
    """Device-to-device copy rate (read + write bytes over time), best of `rounds`."""
    a = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda").fill_(1.0)
    b = torch.empty_like(a)
    best = 1e30
    for _ in range(rounds + 2):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        b.copy_(a)
        e1.record()
        e1.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2 * nbytes / (best * 1e-3) / 1e9


def element_form():
    """FEM mesh^3 from the emitter, staged in call order, turned into (dofs[t, jl], Aloc[t, jl, il]) on the device."""
    g = xsb.Handle(n, n)
    g.set_precount(False)
    g.emit_p1fem(mesh, mesh, mesh, flavour=xsb.RAW)
    cnt = g.pending
    dI = torch.empty(cnt, dtype=torch.int64, device="cuda")
    dJ = torch.empty_like(dI)
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
    torch.cuda.synchronize()
    return dofs, A


peak = copy_peak_gbs()
dofs64, A = element_form()
ncells, k = dofs64.shape
calls = ncells * k * k
dofs32 = dofs64.to(torch.int32)
I = dofs64[:, None, :].expand(ncells, k, k).reshape(-1).contiguous()  # row of call k^2 c + k jl + il: dofs[c, il]
J = dofs64[:, :, None].expand(ncells, k, k).reshape(-1).contiguous()  # column: dofs[c, jl]
V = A.view(-1)
T = torch.empty((calls, 2), dtype=torch.int64, device="cuda")
T[:, 0] = I | (J << 32)
T[:, 1] = V.view(torch.int64)
torch.cuda.synchronize()

PATHS = {
    # name: (index type of the handle, insert call, algorithmic bytes of the insert)
    "elements/i32": (xsb.I32, lambda h: h.insert_elements(dofs32, A, xsb.RAW), ncells * (4 * k + 8 * k * k) + 16 * calls),
    "elements/i64": (xsb.I64, lambda h: h.insert_elements(dofs64, A, xsb.RAW), ncells * (8 * k + 8 * k * k) + 16 * calls),
    "triplets": (xsb.I64, lambda h: h.insert_triplets(T, xsb.RAW, 0, calls), 32 * calls),
    "ijv/i64": (xsb.I64, lambda h: h.insert_batch(I, J, V, xsb.RAW), 40 * calls),
}
handles = {p: xsb.Handle(n, n, idx_type=PATHS[p][0]) for p in PATHS}
for h in handles.values():
    h.set_profiling(True)
times = {p: {"insert": [], "flush": []} for p in PATHS}
stats = {}
for rep in range(reps + 1):  # round 0 warms up every shape
    for p, (_, ins, _) in PATHS.items():
        h = handles[p]
        h.reset()
        h.timer_start()
        ins(h)
        ms = h.timer_stop()
        h.flush()
        st = h.flush_stats()
        if rep > 0:
            times[p]["insert"].append(ms)
            times[p]["flush"].append(st["ms_total"])
        stats[p] = st


def device_csc(h):
    nnz = h.nnz
    cp = torch.empty(h.n + 1, dtype=torch.int64, device="cuda")
    rv = torch.empty(nnz, dtype=torch.int64, device="cuda")
    nz = torch.empty(nnz, dtype=torch.float64, device="cuda")
    if h.idx_type == xsb.I32:
        cp32, rv32 = cp.to(torch.int32), rv.to(torch.int32)
        h.fetch_csc(cp32, rv32, nz)
        h.synchronize()
        cp, rv = cp32.to(torch.int64), rv32.to(torch.int64)
    else:
        h.fetch_csc(cp, rv, nz)
        h.synchronize()
    return cp, rv, nz.view(torch.int64)


ref = device_csc(handles["triplets"])
same = {p: all(torch.equal(x, y) for x, y in zip(device_csc(handles[p]), ref)) for p in PATHS}
out = {"mesh": mesh, "cells": ncells, "k": k, "calls": calls, "nnz": int(handles["triplets"].nnz), "reps": reps,
       "card": card(), "copy_peak_gbs": round(peak, 1), "same_csc_bits": same, "paths": {}}
for p, (_, _, nbytes) in PATHS.items():
    ins = sorted(times[p]["insert"])
    fl = sorted(times[p]["flush"])
    med = ins[len(ins) // 2]
    out["paths"][p] = {
        "insert_ms_min": round(ins[0], 4), "insert_ms_median": round(med, 4),
        "flush_ms_median": round(fl[len(fl) // 2], 4),
        "column_path": stats[p]["column_path"], "precounted": round(stats[p]["precounted"], 4),
        "G_insertions_per_s_insert": round(calls / (med * 1e-3) / 1e9, 1),
        "insert_bytes_GB": round(nbytes / 1e9, 3),
        "insert_GBs": round(nbytes / (med * 1e-3) / 1e9, 1),
        "insert_share_of_copy_peak": round(nbytes / (med * 1e-3) / 1e9 / peak, 3),
    }
    r = out["paths"][p]
    print(f"{p:13s} insert {r['insert_ms_median']:.3f} ms (min {r['insert_ms_min']:.3f})  flush {r['flush_ms_median']:.3f} ms"
          f"  path {r['column_path']} precounted {r['precounted']:.3f}  {r['G_insertions_per_s_insert']} G ins/s"
          f"  {r['insert_bytes_GB']} GB -> {r['insert_share_of_copy_peak']:.2f} of copy peak  same bits: {same[p]}")
print(f"card: {out['card']}  copy peak {peak:.0f} GB/s")
print(json.dumps(out))
for h in handles.values():
    h.close()
sys.exit(0 if all(same.values()) else 1)
