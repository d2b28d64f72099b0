#!/usr/bin/env python
"""A + B, A - B and dropzeros! on resident matrices (development tool).

Workloads (Int64 indices, base 1, resident in HBM):
    add/same      FEM 128^3 (p1fem emitter, RAW: its explicit zeros stay stored) + the same pattern with other
                  values (x 1.5 - 0.25)
    add/differ    FEM 128^3 + fdrand 128^3 (seed 20240717): two different patterns of the same n
    sub/differ    FEM 128^3 - fdrand 128^3
    drop/rd       dropzeros! after eliminate_dirichlet! on block RD 96^3 x 4 species (every 7th unknown marked)
    drop/noop     dropzeros! on FEM 128^3 once a first, untimed dropzeros! has removed its stored zeros: the timed
                  calls drop nothing
    host/rd       the former host dropzeros (download the CSC, filter with numpy, upload through xsb_set_csc)
                  on the drop/rd input
Every call is timed with a host clock that ends in a device synchronise (the calls synchronise before they return),
one warm-up round, then the median of `reps`.  Algorithmic bytes: 16 B per input and output entry (Int64 row and
Float64 value) plus 8 B per colptr entry read or written; their rate is given as a share of the device-to-device
copy rate measured in the same run.  The card's name and power limit are read in the same run.  The device results
are compared with numpy on the host; the script exits non-zero when one differs.
Usage: exp_csc_algebra.py [reps]"""
import json
import os
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
from tests import csc_algebra_ref as alg  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7


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
    return cp, rv[:nnz], nz[:nnz]


def timed(fn, setup=None):
    ts = []
    for r in range(reps + 1):
        if setup:
            setup()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        if r:
            ts.append(1e3 * (time.perf_counter() - t0))
        if hasattr(out, "close") and r < reps:
            out.close()
    return float(np.median(ts)), out


def bits_equal(a, b):
    return all(np.array_equal(np.asarray(x), np.asarray(y)) for x, y in zip(a[:2], b[:2])) and np.array_equal(
        np.asarray(a[2]).view(np.uint64), np.asarray(b[2]).view(np.uint64))


def main():
    info = card()
    peak = copy_peak_gbs()
    mesh = 128
    n = mesh ** 3
    res = {"card": info, "copy_gbs": round(peak, 1), "reps": reps, "rows": []}
    ok = True

    def row(name, ms, nbytes, extra):
        gbs = nbytes / (ms * 1e-3) / 1e9
        r = {"case": name, "ms": round(ms, 3), "alg_bytes": int(nbytes), "alg_gbs": round(gbs, 1),
             "of_copy": round(gbs / peak, 3), **extra}
        res["rows"].append(r)
        print(json.dumps(r), flush=True)

    hf = xsb.Handle(n, n)
    hf.emit_p1fem(mesh, mesh, mesh, flavour=xsb.RAW)
    hf.flush()
    cp, rv, nz = device_csc(hf)
    hs = xsb.Handle(n, n)
    hs.set_csc(cp, rv, (nz * 1.5 - 0.25).contiguous())
    hd = xsb.Handle(n, n)
    hd.emit_fdrand(mesh, mesh, mesh, seed=20240717)
    hd.flush()
    F = hf.fetch_csc_numpy()
    for name, a, b, op, sym in (("add/same", hf, hs, xsb.OP_ADD, "+"), ("add/differ", hf, hd, xsb.OP_ADD, "+"),
                                ("sub/differ", hf, hd, xsb.OP_SUB, "-")):
        ms, hc = timed(lambda: a.add(b, op))
        nbytes = 16 * (a.nnz + b.nnz + hc.nnz) + 8 * 3 * (n + 1)
        same = bits_equal(hc.fetch_csc_numpy(), alg.map_zeropres(sym, n, n, F, b.fetch_csc_numpy()))
        ok &= same
        row(name, ms, nbytes, {"nnz_a": a.nnz, "nnz_b": b.nnz, "nnz_c": hc.nnz, "matches_numpy": same})
        hc.close()
    for h in (hs, hd):
        h.close()
    del cp, rv, nz

    nnz_fem = hf.nnz
    hf.dropzeros()
    ms, _ = timed(lambda: hf.dropzeros())
    row("drop/noop", ms, 16 * hf.nnz + 8 * (n + 1), {"nnz_emitted": nnz_fem, "nnz": hf.nnz,
                                                     "changed": hf.dropzeros()[1]})
    hf.close()

    rd, ns = 96, 4
    nrd = rd ** 3 * ns
    hr = xsb.Handle(nrd, nrd)
    hr.emit_blockrd(rd, rd, rd, ns)
    hr.flush()
    rcp, rrv, rnz = device_csc(hr)
    marker = np.zeros(nrd, np.uint8)
    marker[::7] = 1

    def restore():
        hr.set_csc(rcp, rrv, rnz)
        hr.eliminate_dirichlet(marker)

    restore()
    before = hr.fetch_csc_numpy()
    nnz_in = hr.nnz
    ms, _ = timed(lambda: hr.dropzeros(), restore)
    got = hr.fetch_csc_numpy()
    same = bits_equal(got, alg.fkeep_nonzero(nrd, before))
    ok &= same
    row("drop/rd", ms, 16 * (nnz_in + hr.nnz) + 8 * 2 * (nrd + 1),
        {"nnz_in": nnz_in, "nnz_out": hr.nnz, "matches_numpy": same})

    def host_dropzeros():
        c, r, v = hr.fetch_csc_numpy()
        keep = v != 0
        cols = np.repeat(np.arange(nrd), np.diff(c))
        c2 = np.concatenate([[1], 1 + np.cumsum(np.bincount(cols[keep], minlength=nrd))]).astype(np.int64)
        hr.set_csc(c2, np.ascontiguousarray(r[keep]), np.ascontiguousarray(v[keep]))

    ms, _ = timed(host_dropzeros, restore)
    same = bits_equal(hr.fetch_csc_numpy(), got)
    ok &= same
    row("host/rd", ms, 16 * (nnz_in + hr.nnz) + 8 * 2 * (nrd + 1), {"nnz_out": hr.nnz, "matches_device": same})
    hr.close()
    res["ok"] = bool(ok)
    print(json.dumps(res))
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
