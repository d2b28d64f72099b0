#!/usr/bin/env python
"""Rectangular element matrices against the generic insertion paths (development tool).

Input: the Kuhn mesh^3 of the FEM emitter (default 128^3: 12,290,298 tetrahedra, 2,097,152 nodes), resident in HBM.
Three element loops whose rows and columns come from different connectivities:
    p0xp1   m = cells,     n = nodes, kr = 1,  kc = 4   (row: the cell, columns: its nodes)
    p1xp0   m = nodes,     n = cells, kr = 4,  kc = 1   (the transposed shape)
    vp1xp1  m = 3 nodes,   n = nodes, kr = 12, kc = 4   (vector P1 rows 3 node + component, scalar P1 columns)
Values: Gaussian, fixed seed.  Per workload the same calls go in four ways, alternating, after one warm-up round:
    elements/i32   xsb_insert_elements_rect, Int32 dofs (Int32 handle)
    elements/i64   xsb_insert_elements_rect, Int64 dofs
    triplets       xsb_insert_triplets of the expanded stream on the device (16 B per call)
    ijv/i64        xsb_insert_batch of device (I, J, V) arrays, Int64 indices (24 B per call)
Per path: insert and flush medians (CUDA events on the handle's stream), the flush's column path and precounted
share, G insertions/s, the insert's algorithmic bytes (what it must read and the 16-byte records it writes) and their
share of the device-to-device copy rate measured in the same run.  The card's name and power limit are read in the
same run.  Exits non-zero unless every path gives the same CSC bits.
Usage: exp_elements_rect.py [mesh] [reps]"""
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
nnodes = mesh ** 3


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


def mesh_cells():
    """cellnodes[t, jl] (1-based) of the emitter's Kuhn mesh: node jl of tetrahedron t is the column of its stream's
    calls 20 t + 1 + jl."""
    g = xsb.Handle(nnodes, nnodes)
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
    del dI, dV
    cells = dJ.view(-1, 4, 5)[:, 0, 1:5].contiguous()
    del dJ
    torch.cuda.synchronize()
    return cells


def workloads(cells):
    ncells = cells.shape[0]
    own = torch.arange(1, ncells + 1, dtype=torch.int64, device="cuda")[:, None]
    vec = (3 * (cells[:, :, None] - 1) + torch.arange(3, device="cuda") + 1).reshape(ncells, 12)
    return {
        "p0xp1": (ncells, nnodes, own, cells),
        "p1xp0": (nnodes, ncells, cells, own),
        "vp1xp1": (3 * nnodes, nnodes, vec, cells),
    }


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


def run(name, m, n, rdofs, cdofs, peak):
    ncells, kr = rdofs.shape
    kc = cdofs.shape[1]
    calls = ncells * kr * kc
    gen = torch.Generator(device="cuda")
    gen.manual_seed(20261021)
    A = torch.randn((ncells, kc, kr), dtype=torch.float64, device="cuda", generator=gen)
    r32, c32 = rdofs.to(torch.int32), cdofs.to(torch.int32)
    I = rdofs[:, None, :].expand(ncells, kc, kr).reshape(-1).contiguous()  # row of call p: rdofs[c, il]
    J = cdofs[:, :, None].expand(ncells, kc, kr).reshape(-1).contiguous()  # column: cdofs[c, jl]
    V = A.view(-1)
    T = torch.empty((calls, 2), dtype=torch.int64, device="cuda")
    T[:, 0] = I | (J << 32)
    T[:, 1] = V.view(torch.int64)
    torch.cuda.synchronize()
    paths = {
        # name: (index type of the handle, insert call, algorithmic bytes of the insert)
        "elements/i32": (xsb.I32, lambda h: h.insert_elements(r32, A, xsb.RAW, col_dofs=c32),
                         ncells * (4 * (kr + kc) + 8 * kr * kc) + 16 * calls),
        "elements/i64": (xsb.I64, lambda h: h.insert_elements(rdofs, A, xsb.RAW, col_dofs=cdofs),
                         ncells * (8 * (kr + kc) + 8 * kr * kc) + 16 * calls),
        "triplets": (xsb.I64, lambda h: h.insert_triplets(T, xsb.RAW, 0, calls), 32 * calls),
        "ijv/i64": (xsb.I64, lambda h: h.insert_batch(I, J, V, xsb.RAW), 40 * calls),
    }
    handles = {p: xsb.Handle(m, n, idx_type=paths[p][0]) for p in paths}
    for h in handles.values():
        h.set_profiling(True)
    times = {p: {"insert": [], "flush": []} for p in paths}
    stats = {}
    for rep in range(reps + 1):  # round 0 warms up every shape
        for p, (_, ins, _) in paths.items():
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
    ref = device_csc(handles["triplets"])
    same = {p: all(torch.equal(x, y) for x, y in zip(device_csc(handles[p]), ref)) for p in paths}
    out = {"m": m, "n": n, "cells": ncells, "kr": kr, "kc": kc, "calls": calls, "nnz": int(handles["triplets"].nnz),
           "same_csc_bits": same, "paths": {}}
    for p, (_, _, nbytes) in paths.items():
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
        print(f"{name:7s} {p:13s} insert {r['insert_ms_median']:.3f} ms (min {r['insert_ms_min']:.3f})"
              f"  flush {r['flush_ms_median']:.3f} ms  path {r['column_path']} precounted {r['precounted']:.3f}"
              f"  {r['G_insertions_per_s_insert']} G ins/s  {r['insert_bytes_GB']} GB ->"
              f" {r['insert_share_of_copy_peak']:.2f} of copy peak  same bits: {same[p]}", flush=True)
    for h in handles.values():
        h.close()
    return out


peak = copy_peak_gbs()
cells = mesh_cells()
result = {"mesh": mesh, "reps": reps, "card": card(), "copy_peak_gbs": round(peak, 1), "workloads": {}}
for name, (m, n, rdofs, cdofs) in workloads(cells).items():
    result["workloads"][name] = run(name, m, n, rdofs, cdofs, peak)
    torch.cuda.empty_cache()
print(f"card: {result['card']}  copy peak {peak:.0f} GB/s")
print(json.dumps(result))
sys.exit(0 if all(all(w["same_csc_bits"].values()) for w in result["workloads"].values()) else 1)
