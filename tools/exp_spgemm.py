#!/usr/bin/env python
"""A * B of resident matrices (xsb_matmul) against expand-then-assemble through the library's own flush
(development tool).

Workloads (Int64 indices, base 1, resident in HBM; a mesh N^3 has N^3 nodes, as in tools/exp_csc_algebra.py):
    fem/AA      FEM 128^3 (p1fem emitter, RAW: its explicit zeros stay stored) squared, a is b
    fem*fd      FEM 128^3 times fdrand 128^3 (seed 20240717)
    rd/AA       block RD 64^3 x 4 species squared (28 entries per column, f(j) up to 784: the 1024-slot tables)
    rd8/AA      block RD 32^3 x 8 species squared (56 entries per column, f(j) up to 3136: the 4096-slot tables)
    rd12/AA     block RD 24^3 x 12 species squared (84 entries per column, f(j) up to 7056: the row tiles)
    rect/D1D2   p0xp1 times p1xp0 of the Kuhn mesh 128^3 (cell-to-cell coupling through shared nodes)
    rect/D2D1   p1xp0 times p0xp1 (node-to-node)
The p0xp1 (cells x nodes, row the cell, columns its four nodes) and p1xp0 operators are built from the FEM emitter's
connectivity with xsb_insert_elements_rect and Gaussian element values, as tools/exp_elements_rect.py builds them.
Per workload:
    matmul      xsb_matmul; host clock ending in a device synchronise, one warm-up call, median of `reps`
    baseline    the same product expanded: (I, J, V) of every product in (j, B position, A position) order, built
                with torch on the device (untimed), then xsb_insert_batch RAW followed by a DETERMINISTIC xsb_flush
                (timed the same way).  Its CSC must equal the product's except possibly the sign of a zero, because
                the flush seeds a new entry with +0.0 and spmatmul assigns the first product; those entries are counted.
Reported: products, nnz(C), the columns per path (f(j) = products of column j; a column goes to the first warp table
whose size holds f(j), to the row tiles above 4096, nowhere when f(j) = 0), the time of each kernel family from one
separate torch.profiler run of the call, products/s, algorithmic bytes (16 B per entry of A, B and C plus 8 B per colptr entry)
over the call time and as a share of the device-to-device copy rate measured in the same run, the card's name and
power limit.  The RD and rect workloads are also checked bit for bit against tests/spgemm_ref.py at a reduced mesh.
Exits non-zero when a result differs.
Usage: exp_spgemm.py [reps]"""
import ctypes as C
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import __graft_entry__ as ge  # noqa: E402

ge.build()
import xsparse_b200 as xsb  # noqa: E402
from tests import spgemm_ref as ref  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
TABLE_SIZES = (256, 1024, 4096)  # the warp-table bins of csrc/xsb_spgemm.cu; f(j) above the last: row tiles


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


def device_csc(h):
    nnz = h.nnz
    cp = torch.empty(h.n + 1, dtype=torch.int64, device="cuda")
    rv = torch.empty(max(nnz, 1), dtype=torch.int64, device="cuda")
    nz = torch.empty(max(nnz, 1), dtype=torch.float64, device="cuda")
    h.fetch_csc(cp, rv, nz)
    h.synchronize()
    return cp, rv[:nnz], nz[:nnz]


def timed(fn):
    """Median of `reps` calls after one warm-up call; fn returns something to close (or None)."""
    ts = []
    out = None
    for r in range(reps + 1):
        if out is not None:
            out.close()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        if r:
            ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts)), out


def expand_products(A, B):
    """(I, J, V) of every product in (j, B position, A position) order, 1-based, on the device."""
    cpa, rva, nza = A
    cpb, rvb, nzb = B
    k = rvb - 1
    lens = cpa[k + 1] - cpa[k]
    total = int(lens.sum())
    pidx = torch.repeat_interleave(torch.arange(len(rvb), device="cuda"), lens, output_size=total)
    first = torch.cumsum(lens, 0) - lens
    q = (cpa[k] - 1)[pidx] + torch.arange(total, device="cuda") - first[pidx]
    del first
    bcol = torch.repeat_interleave(torch.arange(1, len(cpb), device="cuda"), cpb[1:] - cpb[:-1], output_size=len(rvb))
    J = bcol[pidx]
    V = nza[q] * nzb[pidx]
    I = rva[q]
    del q, pidx, bcol
    return I, J, V


def path_histogram(A, B):
    """Columns of B per path of xsb_matmul, from f(j) = sum of nnz(A[:, k]) over the k stored in B[:, j]."""
    cpa, _, _ = A
    cpb, rvb, _ = B
    k = rvb - 1
    n = len(cpb) - 1
    bcol = torch.repeat_interleave(torch.arange(n, device="cuda"), cpb[1:] - cpb[:-1], output_size=len(rvb))
    f = torch.zeros(n, dtype=torch.int64, device="cuda").index_add_(0, bcol, cpa[k + 1] - cpa[k])
    edges = torch.tensor(TABLE_SIZES, dtype=torch.int64, device="cuda")
    where = torch.bucketize(f, edges)  # 0: f <= 256, 1: <= 1024, 2: <= 4096, 3: row tiles
    where[f == 0] = 4
    cnt = torch.bincount(where, minlength=5).tolist()
    out = {f"table{t}": cnt[i] for i, t in enumerate(TABLE_SIZES)}
    out.update({"tiles": cnt[3], "no_products": cnt[4], "f_min_nonzero": int(f[f > 0].min()) if cnt[4] < n else 0,
                "f_max": int(f.max()) if n else 0})
    return out


def kernel_split(a, b):
    """ms per kernel family of one xsb_matmul call, from a torch.profiler run of its own."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        a.matmul(b).close()
        torch.cuda.synchronize()
    fam = {}
    for ev in prof.key_averages():
        m = re.search(r"(spgemm_\w+|scan_\w+)_kernel(<[^,>]+(?:, (true|false))?(?:, (\d+))?)?", ev.key)
        if not m:
            continue
        key = m.group(1)
        if m.group(3):
            key += ("/write" if m.group(3) == "true" else "/count")
        if m.group(4):
            key += "/" + m.group(4)
        us = getattr(ev, "device_time_total", None)
        fam[key] = fam.get(key, 0.0) + (us if us is not None else ev.cuda_time_total) / 1e3
    return {k: round(v, 3) for k, v in sorted(fam.items())}


def mesh_cells(mesh):
    """(ncells, 4) 1-based nodes of the FEM emitter's Kuhn mesh on mesh^3 nodes (see tools/exp_elements_rect.py)."""
    nn = mesh ** 3
    g = xsb.Handle(nn, nn)
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
    return cells, nn


def rect_operators(mesh):
    cells, nn = mesh_cells(mesh)
    nc = cells.shape[0]
    gen = torch.Generator(device="cuda")
    gen.manual_seed(20261022)
    own = torch.arange(1, nc + 1, dtype=torch.int64, device="cuda")[:, None]
    d1 = xsb.Handle(nc, nn)
    d1.insert_elements(own, torch.randn((nc, 4, 1), dtype=torch.float64, device="cuda", generator=gen), xsb.RAW,
                       col_dofs=cells)
    d1.flush()
    d2 = xsb.Handle(nn, nc)
    d2.insert_elements(cells, torch.randn((nc, 1, 4), dtype=torch.float64, device="cuda", generator=gen), xsb.RAW,
                       col_dofs=own)
    d2.flush()
    return d1, d2


def fem(mesh):
    n = mesh ** 3
    h = xsb.Handle(n, n)
    h.emit_p1fem(mesh, mesh, mesh, flavour=xsb.RAW)
    h.flush()
    return h


def fdrand(nx):
    n = nx ** 3
    h = xsb.Handle(n, n)
    h.emit_fdrand(nx, nx, nx, seed=20240717)
    h.flush()
    return h


def blockrd(nx, ns=4):
    n = nx ** 3 * ns
    h = xsb.Handle(n, n)
    h.emit_blockrd(nx, nx, nx, ns)
    h.flush()
    return h


def matches_reference(a, b):
    """a * b on the device against tests/spgemm_ref.py, bit for bit."""
    hc = a.matmul(b)
    got = hc.fetch_csc_numpy()
    want = ref.spmatmul(a.m, b.n, a.fetch_csc_numpy(), b.fetch_csc_numpy())
    hc.close()
    return bool(np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and
                np.array_equal(got[2].view(np.uint64), want[2].view(np.uint64)))


def run(name, a, b, peak):
    ms, hc = timed(lambda: a.matmul(b))
    A, B = device_csc(a), device_csc(b)
    paths = path_histogram(A, B)
    split = kernel_split(a, b)
    Cd = device_csc(hc)
    I, J, V = expand_products(A, B)
    products = len(V)
    base_h = xsb.Handle(a.m, b.n)

    def baseline():
        base_h.reset()
        base_h.insert_batch(I, J, V, xsb.RAW)
        base_h.flush(xsb.DETERMINISTIC)

    bms, _ = timed(baseline)
    del I, J, V
    Bd = device_csc(base_h)
    base_h.close()
    same_pattern = all(torch.equal(x, y) for x, y in zip(Cd[:2], Bd[:2]))
    vc, vb = Cd[2].view(torch.int64), Bd[2].view(torch.int64)
    differ = vc != vb
    zero_sign = int((differ & (Cd[2] == 0) & (Bd[2] == 0)).sum())
    same = bool(same_pattern and int(differ.sum()) == zero_sign)
    nbytes = 16 * (a.nnz + b.nnz + hc.nnz) + 8 * ((a.n + 1) + (b.n + 1) + (hc.n + 1))
    gbs = nbytes / (ms * 1e-3) / 1e9
    r = {"case": name, "m": a.m, "k": a.n, "n": b.n, "nnz_a": a.nnz, "nnz_b": b.nnz, "nnz_c": hc.nnz,
         "products": products, "ms": round(ms, 3), "G_products_per_s": round(products / (ms * 1e-3) / 1e9, 2),
         "alg_bytes": int(nbytes), "alg_gbs": round(gbs, 1), "of_copy": round(gbs / peak, 3),
         "baseline_ms": round(bms, 3), "speedup_over_baseline": round(bms / ms, 2),
         "matches_baseline": same, "zero_sign_differences": zero_sign, "columns_per_path": paths,
         "kernel_ms": split}
    hc.close()
    del A, B, Cd, Bd, vc, vb, differ
    torch.cuda.empty_cache()
    print(json.dumps(r), flush=True)
    return r


def main():
    info = card()
    peak = copy_peak_gbs()
    res = {"card": info, "copy_gbs": round(peak, 1), "reps": reps, "rows": [], "reference": {}}
    ok = True

    hf = fem(128)
    res["rows"].append(run("fem/AA", hf, hf, peak))
    hd = fdrand(128)
    res["rows"].append(run("fem*fd", hf, hd, peak))
    hf.close()
    hd.close()
    for name, nx, ns in (("rd/AA", 64, 4), ("rd8/AA", 32, 8), ("rd12/AA", 24, 12)):
        hr = blockrd(nx, ns)
        res["rows"].append(run(name, hr, hr, peak))
        hr.close()
    d1, d2 = rect_operators(128)
    res["rows"].append(run("rect/D1D2", d1, d2, peak))
    res["rows"].append(run("rect/D2D1", d2, d1, peak))
    d1.close()
    d2.close()
    ok &= all(r["matches_baseline"] for r in res["rows"])

    # the same kinds of product at a reduced mesh, bit for bit against the numpy restatement
    hr = blockrd(12)
    res["reference"]["rd/AA@12"] = matches_reference(hr, hr)
    hr.close()
    for nx, ns in ((6, 8), (5, 12)):
        hr = blockrd(nx, ns)
        res["reference"][f"rd{ns}/AA@{nx}"] = matches_reference(hr, hr)
        hr.close()
    d1, d2 = rect_operators(10)
    res["reference"]["rect/D1D2@10"] = matches_reference(d1, d2)
    res["reference"]["rect/D2D1@10"] = matches_reference(d2, d1)
    d1.close()
    d2.close()
    ok &= all(res["reference"].values())
    res["ok"] = bool(ok)
    print(json.dumps(res))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
