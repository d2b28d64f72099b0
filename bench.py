#!/usr/bin/env python
"""bench.py -- assembled entries/s of insert + flush! on B200, with roofline and CPU baseline.

Contract (see DESIGN.md "Measurement"):
  python bench.py --gpus N --steps K --warmup W            our arm (libxsparse_b200 through the C ABI)
  python bench.py --impl reference --gpus N ...            the reference's CPU algorithm (oracle port)
  python bench.py --gpus 1 ... --dump-outputs DIR          also writes the CSC of the last timed step to DIR/*.npy

A step = one full assembly of the workload: reset!, insertion of the whole (i,j,v) stream,
flush! into a fresh CSC.  N=1 workload: BASELINE.json configs[1], the 3-D P1-FEM Laplacian on
a 128^3-node Kuhn mesh (245 805 960 rawupdateindex! calls, 31 065 598 nnz, Float64/Int64).
N>1: weak scaling -- every rank assembles its own 128x128x128-node slab of a 128x128x(127N+1)
mesh; columns are owned by z-slab and the interface plane is routed with an NCCL all-to-all.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "assembled entries/sec (insert+flush!)"
UNIT = "entries/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[3 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.samples[0][1]), "reasons": reasons,
                "samples": len(sm), "power_w_max": max(float(s[2]) for s in self.samples)}


# ---------------------------------------------------------------------------------- workloads
def workload(args):
    n = args.mesh
    return {"workload": f"P1-FEM Laplacian+mass, {n}^3-node Kuhn 6-tet mesh, rawupdateindex! stream + flush! "
                        f"(BASELINE.json configs[1])",
            "nodes": n ** 3, "mesh": n, "Tv": "Float64", "Ti": "Int64", "mode": args.mode,
            "l2_policy": "inputs (3.9 GB of records) far exceed the 126 MB L2; no explicit flush"}


def flush_bytes(n_ins, nnz_old, nnz_new, ncols):
    """Algorithmic bytes of one flush!, SURVEY.md 8(d): 16 B per triplet (packed key + Float64),
    16 B per CSC entry (Int64 row + Float64), 8 B per colptr entry; old CSC read, new CSC written."""
    return 16 * n_ins + 16 * nnz_old + 8 * (ncols + 1) + 16 * nnz_new + 8 * (ncols + 1)


def values_only_bytes(n_ins, nnz):
    """SURVEY.md 8(d): B_vo = 8 N_ins (values) + 4 N_ins (int32 entry -> nzval map) + 8 nnz (nzval written)."""
    return 12 * n_ins + 8 * nnz


FLUSH_KERNELS = ("runfold_kernel", "run_bucket_kernel", "run_totals_kernel", "runpair_scan_kernel", "chunk_sort_kernel")


def ncu_traffic(workload_tag, kernels=FLUSH_KERNELS):
    """dram__bytes_read.sum + dram__bytes_write.sum per flush, summed over the flush's kernels, from the committed
    `ncu --set full` capture of one step of this workload (profiles/r2_ncu_full_<tag>.csv, written by
    tools/ncu_extract.py).  None if no capture of this workload is committed."""
    import csv

    p = os.path.join(ROOT, "profiles", f"r2_ncu_full_{workload_tag}.csv")
    if not os.path.exists(p):
        return None, None
    rows = list(csv.reader(open(p)))
    hdr = rows[0]
    try:
        kn, rd, wr = hdr.index("Kernel Name"), hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
    except ValueError:
        return None, None
    units = rows[1] if len(rows) > 1 else []
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    per_kernel = {}
    for r in rows[2:]:
        k = next((x for x in kernels if x in r[kn]), None)
        if k is None or k in per_kernel:  # one launch of every kernel = one flush
            continue
        try:
            per_kernel[k] = float(r[rd]) * scale.get(units[rd], 1.0) + float(r[wr]) * scale.get(units[wr], 1.0)
        except (ValueError, IndexError):
            pass
    if not per_kernel:
        return None, None
    return sum(per_kernel.values()), per_kernel


def roofline(st, ms, ms_emit, ncols, peak, peak_src, tag):
    """roofline.frac is SURVEY.md 8(d)'s fraction: the flush's ALGORITHMIC bytes (triplets + old CSC read + new
    CSC written) over the device time of the whole flush! (CUDA events on the library's stream around xsb_flush),
    against the measured HBM copy peak.  Per-kernel detail beside it, with each kernel's own algorithmic bytes."""
    n_ins, nnz_old, nnz = st["n_inserted"], st["nnz_old"], st["nnz_new"]
    pairs = st["group_pairs"]
    path = st["column_path"]
    b_flush = flush_bytes(n_ins, nnz_old, nnz, ncols)
    t_flush = ms["ms_total"]
    achieved = b_flush / (t_flush / 1e3) / 1e9
    det = {}
    if path == 4:
        det["runfold_kernel (thread-per-column merge: staged runs + resident column -> new column)"] = (
            ms["ms_fold"], 16 * n_ins + 16 * nnz_old + 16 * nnz + 16 * ncols + 8 * pairs)
        det["run buckets (run_totals + runpair_scan + run_bucket kernels)"] = (ms["ms_pair_sort"], 8 * ncols + 24 * pairs)
        if ms.get("ms_group_count", 0.0) > 0.005:
            det["chunk_sort_kernel (records the producers left in stream order, grouped in place)"] = (
                ms["ms_group_count"], 32 * n_ins * (1.0 - float(st.get("precounted", 0.0))))
    else:
        rec = n_ins + nnz_old
        det["count / histogram"] = (ms["ms_group_count"] + ms.get("ms_histogram", 0.0), 16 * rec)
        det["scatter / sort passes"] = (ms["ms_sort"], 32 * rec * max(1, st["sort_passes"]))
        det["fold"] = (ms["ms_reduce"], 16 * rec + 16 * nnz)
    traffic, per_kernel = ncu_traffic(tag) if (path == 4 and tag) else (None, None)
    name = max(det, key=lambda k: det[k][0])
    out = {"bound": "hbm", "kernel": "xsb_flush (all kernels of one flush!; dominant: " + name.split(" ")[0] + ")",
           "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
           "peak_source": peak_src, "bytes_per_launch": b_flush, "ms_per_launch": t_flush, "launches_per_step": 1,
           "definition": "SURVEY.md 8(d): (16 N_ins + 16 nnz_old + 16 nnz_new + 16 (n+1)) / device time of flush! / peak",
           "traffic_source": f"profiles/r2_ncu_full_{tag}.csv (dram read + write of the flush's kernels)" if traffic else None,
           "traffic_per_kernel": per_kernel,
           "kernels": {k: {"ms": v[0], "GB/s": v[1] / (v[0] / 1e3) / 1e9 if v[0] > 0 else None,
                           "frac": v[1] / (v[0] / 1e3) / 1e9 / peak if v[0] > 0 else None} for k, v in det.items()},
           "column_path": path, "stage_ms_per_step": dict(sorted(ms.items()))}
    if ms_emit is not None:
        span = ms_emit + t_flush
        out["span_emission_to_csc"] = {"ms": span, "achieved": b_flush / (span / 1e3) / 1e9,
                                       "frac": b_flush / (span / 1e3) / 1e9 / peak, "ms_emit": ms_emit,
                                       "note": "8(d)'s time span with the insertion kernels inside: grouping by column "
                                               "happens in the kernels that stage the records"}
    return out


# ---------------------------------------------------------------------------------- CPU legs
def cpu_reference_leg(mesh, steps, warmup):
    """Times the oracle port of the reference's serial path (ExtendableSparseMatrix +
    rawupdateindex! + flush!) on one host core; returns entries/s (best step) and seconds/step."""
    from oracle import oracle as ora

    ora.build()
    I, J, V = ora.fem_stream(mesh, mesh, mesh)
    n = mesh ** 3
    times = []
    digest = None
    for it in range(warmup + steps):
        A = ora.OracleExt(n, n)
        t0 = time.perf_counter()
        A.insert_batch(I, J, V, ora.RAW)
        A.flush()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        if it == warmup + steps - 1:
            digest = csc_digest(*A.csc())
        del A
    ORACLE_DIGEST[mesh] = digest
    return len(V), times


ORACLE_DIGEST = {}  # mesh -> SHA-256 of the oracle's (colptr, rowval, nzval) of the FEM assembly


def csc_digest(colptr, rowval, nzval):
    """SHA-256 over the raw bytes of colptr | rowval | nzval (Int64 / Int64 / Float64, 1-based)."""
    import hashlib

    import numpy as np

    hsh = hashlib.sha256()
    for a, dt in ((colptr, np.int64), (rowval, np.int64), (nzval, np.float64)):
        hsh.update(np.ascontiguousarray(a, dt).tobytes())
    return hsh.hexdigest()


DUMP_SAMPLE = 1 << 20  # rowval / nzval positions --dump-outputs keeps: 3 x 8 MiB beside the 16 MiB colptr of 128^3


def fetch_csc_device(h, torch):
    """The handle's CSC (colptr, rowval, nzval) copied into new tensors on the current CUDA device."""
    nnz = h.nnz
    cp = torch.empty(h.n + 1, dtype=torch.int64, device="cuda")
    rv = torch.empty(nnz, dtype=torch.int64, device="cuda")
    nz = torch.empty(nnz, dtype=torch.float64, device="cuda")
    h.fetch_csc(cp, rv if nnz else None, nz if nnz else None)
    h.synchronize()
    return cp, rv, nz


def csc_outputs(colptr, rowval, nzval, torch):
    """What --dump-outputs writes of a CSC: colptr whole, rowval and nzval at DUMP_SAMPLE positions drawn with a
    fixed seed (the same positions for the same nnz, listed in sample_index), all as float64, which holds every
    index below 2^53 exactly."""
    import numpy as np

    nnz = rowval.numel()
    pos = np.sort(np.random.default_rng(0).choice(nnz, min(nnz, DUMP_SAMPLE), replace=False))
    at = torch.from_numpy(pos).to(rowval.device)
    arrays = {"colptr": colptr, "sample_index": at, "rowval_sample": rowval[at], "nzval_sample": nzval[at]}
    return {name: a.to(torch.float64).cpu().numpy() for name, a in arrays.items()}


def write_outputs(path, arrays):
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def host_threads():
    """Host threads the CPU legs may use: the cores this process is allowed on, capped at 64
    (every partition of the MT path owns a dense column map)."""
    try:
        return max(1, min(64, len(os.sched_getaffinity(0))))
    except AttributeError:
        return max(1, min(64, os.cpu_count() or 1))


def cpu_reference_mt_leg(mesh, steps, warmup, nthreads):
    """Times the oracle port of the reference's PARTITIONED path (MTExtendableSparseMatrixCSC =
    GenericMTExtendableSparseMatrixCSC{SparseMatrixDILNKC}; loop of test/femtools.jl:75-110):
    2*nthreads slab partitions in two colours inserted by `nthreads` host threads, then the
    reference's serial flush! (Base.sum(xmatrices, csc), sparsematrixdilnkc.jl:397-435)."""
    import numpy as np

    from oracle import oracle as ora

    ora.build()
    I, J, V = ora.fem_stream(mesh, mesh, mesh)
    n = mesh ** 3
    nparts = 2 * nthreads
    ncells = len(V) // 20
    pb = 20 * (np.arange(nparts + 1, dtype=np.int64) * ncells // nparts)
    times = []
    for it in range(warmup + steps):
        A = ora.OracleMT(n, n, nparts)
        t0 = time.perf_counter()
        A.insert_partitioned(I, J, V, pb, nthreads, ora.RAW)
        A.flush()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        del A
    return len(V), times


def cpu_baseline_both(mesh, steps, warmup):
    """Serial and partitioned CPU legs on the same sample; the faster one is the baseline."""
    nth = host_threads()
    n_ins, ts = cpu_reference_leg(mesh, steps, warmup)
    serial = n_ins * len(ts) / sum(ts)
    mt = None
    if nth > 1:
        _, tm = cpu_reference_mt_leg(mesh, steps, warmup, nth)
        mt = n_ins * len(tm) / sum(tm)
    use_mt = mt is not None and mt > serial
    times = tm if use_mt else ts
    sample = (f"P1-FEM {mesh}^3-node Kuhn mesh ({n_ins} insertions per assembly), same generator and flavour as "
              f"the GPU workload; C port (gcc -O3) of the reference's algorithm. Serial ExtendableSparseMatrix "
              f"(rawupdateindex! + flush!, 1 thread): {serial / 1e9:.4f} G entries/s. "
              + (f"Partitioned MTExtendableSparseMatrixCSC ({2 * nth} slab partitions, 2 colours, {nth} threads "
                 f"inserting, serial flush! as in the reference): {mt / 1e9:.4f} G entries/s. "
                 if mt is not None else "One host core available: partitioned path not timed. ")
              + f"Reported: the {'partitioned' if use_mt else 'serial'} path")
    cpu = {"value": max(serial, mt or 0.0), "unit": UNIT, "cores": nth if use_mt else 1, "kind": "port",
           "sample": sample, "serial_value": serial, "mt_value": mt, "mt_threads": nth if mt is not None else None}
    return n_ins, times, cpu


def julia_reference(mesh, steps):
    """BASELINE.md 2.1: when a Julia runtime with ExtendableSparse.jl is present on the box (PATH or baseline/_ref),
    the REAL reference is timed (tools/julia_ref.py / .jl).  Returns (seconds per assembly, description) or None."""
    import importlib.util

    spec = importlib.util.spec_from_file_location("julia_ref", os.path.join(ROOT, "tools", "julia_ref.py"))
    jr = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(jr)
    found = jr.probe()
    if found is None:
        return None
    r = jr.run(["time", mesh, max(1, steps)])
    try:
        return float(r.stdout.strip().splitlines()[-1]), f"{found[0]} (ExtendableSparse {found[1]}), julia -t 1"
    except Exception:  # noqa: BLE001
        return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    mesh = args.ref_mesh
    jl = julia_reference(mesh, args.steps)
    n_ins, times, cpu = cpu_baseline_both(mesh, args.steps, args.warmup)
    if jl is not None:  # the package itself, serial; the oracle port's numbers stay in the line beside it
        cpu = dict(cpu, kind="reference", oracle_port_value=cpu["value"], value=max(cpu["value"], n_ins / jl[0]),
                   julia_value=n_ins / jl[0], sample=f"ExtendableSparse.jl itself: {jl[1]}; " + cpu["sample"])
    total = sum(times)
    value = cpu["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload(args),
        "cpu_baseline": cpu,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------- GPU arm
def timed_steps(h, step, steps):
    h.synchronize()
    h.timer_start()
    for _ in range(steps):
        step()
    return h.timer_stop() / steps


def profiled_steps(h, emit, mode, steps):
    """Stage times of `steps` assemblies with CUDA events around every stage of the flush (xsb_set_profiling) and
    around the emission.  Not the headline timing: profiling adds a stream synchronisation per flush."""
    h.set_profiling(True)
    stage, ms_emit = {}, 0.0
    st = None
    for _ in range(steps):
        h.reset()
        h.timer_start()
        emit()
        ms_emit += h.timer_stop()
        h.flush(mode)
        st = h.flush_stats()
        for k, v in st.items():
            if k.startswith("ms_"):
                stage[k] = stage.get(k, 0.0) + v
    h.set_profiling(False)
    return st, {k: v / steps for k, v in stage.items()}, ms_emit / steps


def run_ours(args):
    import numpy as np
    import torch

    import __graft_entry__ as ge

    ge.build()
    import xsparse_b200 as xsb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if args.gpus != 1 and world == 1:
            raise SystemExit("launch N>1 with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    if world > 1:
        import bench_dist

        return bench_dist.run(args, xsb, rank, world, local)

    mesh = args.mesh
    n = mesh ** 3
    mode = xsb.DETERMINISTIC if args.mode == "deterministic" else xsb.FAST
    h = xsb.Handle(n, n, device=local)
    n_ins = xsb.capi.stream_count_p1fem(mesh, mesh, mesh)

    def emit():
        h.emit_p1fem(mesh, mesh, mesh, flavour=xsb.RAW)

    def step():
        h.reset()
        emit()
        return h.flush(mode)

    for _ in range(args.warmup):
        step()
    h.synchronize()
    torch.cuda.synchronize()
    launches0 = h.kernel_launches
    with ClockSampler(local) as clk:
        ms_step = timed_steps(h, step, args.steps)
        launches_timed = h.kernel_launches - launches0
        # the result of the last timed step, taken before the untimed steps below can replace it
        last = fetch_csc_device(h, torch) if args.dump_outputs else None
        # keep the sampler alive for at least a few samples on very short runs
        t_end = time.time() + max(0.0, 0.5 - ms_step * args.steps / 1e3)
        while time.time() < t_end:
            step()
    if last is not None:
        write_outputs(args.dump_outputs, csc_outputs(*last, torch))
        del last
    nnz = h.nnz
    value = n_ins / (ms_step / 1e3)
    peak, peak_src = peaks()
    st, stage_ms, ms_emit = profiled_steps(h, emit, mode, min(args.steps, 3))
    roof = roofline(st, stage_ms, ms_emit, n, peak, peak_src, f"fem{mesh}")
    gpu_digest = csc_digest(*h.fetch_csc_numpy())

    extra = {}
    if not args.no_legs:
        extra["fast"] = measure_fast(args, xsb, h, mesh, n_ins, st, peak)
        extra["splice"] = measure_splice(args, xsb, h, mesh, n, n_ins, mode, peak)
    h.close()
    if not args.no_legs:
        extra["cfg1_small"] = measure_small(args, xsb, local)
        extra["values_only"] = measure_values_only(args, xsb, torch, peak, local)
        extra["cfg5"] = measure_fd(args, xsb, peak, local, args.fd_n)

    # ---- end-to-end through the C ABI with HOST buffers
    e2e = measure_e2e(args, xsb, local, mesh, n, mode, np, torch)

    # ---- CPU baseline (rank 0, N=1): the oracle port on the same workload; its CSC pins the GPU's
    cpu = None
    parity = None
    if not args.no_cpu:
        _, _, cpu = cpu_baseline_both(args.cpu_mesh, 3, 1)  # one warm-up + 3 repetitions of both CPU paths
        if args.cpu_mesh == mesh and ORACLE_DIGEST.get(mesh):
            parity = ORACLE_DIGEST[mesh] == gpu_digest
            if not parity:
                raise SystemExit(f"PARITY FAILURE: SHA-256 of the GPU CSC {gpu_digest} != oracle's {ORACLE_DIGEST[mesh]}")

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload(args),
        "roofline": roof,
        "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches_timed),
        "clocks": clk.summary(), "nnz": int(nnz), "n_inserted": int(n_ins),
        "parity_checked": parity, "csc_sha256": gpu_digest,
        "parity_note": "SHA-256 of colptr|rowval|nzval of the GPU product path == the CPU oracle's on the same 128^3 "
                       "stream (bit-exact CSC)" if parity else None,
    }
    line.update(extra)
    print(json.dumps(line))


def measure_splice(args, xsb, h, mesh, n, n_ins, mode, peak):
    """flush! on top of a RESIDENT matrix (the 3-way merge of sparsematrixlnk.jl:328-378): (i) the same assembly
    once more (every call a CSC hit, extendable.jl:164-166; pattern unchanged), (ii) ~1 % new entries spliced in
    (one off-stencil coupling per column for 1 % of the columns... here: a sparse random stream)."""
    import numpy as np

    out = {}
    # (i) identical second assembly onto the resident CSC
    h.reset()
    h.emit_p1fem(mesh, mesh, mesh, flavour=xsb.RAW)
    h.flush(mode)
    nnz0 = h.nnz

    def again():
        h.emit_p1fem(mesh, mesh, mesh, flavour=xsb.RAW)
        return h.flush(mode)

    for _ in range(3):  # the buffers of a resident assembly are larger: let the handle's buffer rotation settle
        again()
    reps = max(1, min(args.steps, 3))
    ms = timed_steps(h, again, reps)
    nnz1, changed = h.nnz, None
    h.set_profiling(True)
    _, changed = again()
    st = h.flush_stats()
    h.set_profiling(False)
    b = flush_bytes(n_ins, nnz0, nnz1, n)
    out["all_hits"] = {"ms_per_step": ms, "ms_flush": st["ms_total"], "pattern_changed": bool(changed),
                       "nnz": int(nnz1), "entries_per_s": n_ins / (ms / 1e3),
                       "flush_frac_of_hbm_peak": b / (st["ms_total"] / 1e3) / 1e9 / peak,
                       "workload": "the same FEM assembly onto the resident CSC: emit + flush!, nothing new"}
    # (ii) 1 % new entries: random positions, 1 % of nnz of them.  The first splices onto a freshly built matrix
    # allocate CSC stores of a new size class (cudaMallocAsync: ~2.7 ms each, reported as ms_flush_first); from the
    # fourth on the handle's two stores rotate and a flush allocates nothing: that one is timed.
    rng = np.random.default_rng(5)
    k = nnz0 // 100
    first = None
    h.set_profiling(True)
    for it in range(5):
        nnz1 = h.nnz
        I = rng.integers(1, n + 1, k)
        J = rng.integers(1, n + 1, k)
        V = rng.standard_normal(k)
        h.insert_batch(I, J, V, xsb.UPDATE)
        h.timer_start()
        nnz2, ch2 = h.flush(mode)
        ms2 = h.timer_stop()
        st2 = h.flush_stats()
        if first is None:
            first = {"ms_flush": st2["ms_total"], "ms_host_alloc": st2["ms_host_alloc"]}
    h.set_profiling(False)
    out["one_percent_new"] = {"ms_flush": st2["ms_total"], "ms_wall": ms2, "ms_fold": st2["ms_fold"],
                              "ms_host_alloc": st2["ms_host_alloc"], "ms_flush_first": first["ms_flush"],
                              "ms_host_alloc_first": first["ms_host_alloc"], "inserted": int(k), "nnz_old": int(nnz1),
                              "nnz_new": int(nnz2), "pattern_changed": bool(ch2), "column_path": st2["column_path"],
                              "old_entry_traffic_bytes_per_entry": 32,
                              "flush_frac_of_hbm_peak": flush_bytes(k, nnz1, nnz2, n) / (st2["ms_total"] / 1e3) / 1e9 / peak,
                              "workload": "1 % new random entries spliced into the resident 128^3 FEM matrix (fifth splice "
                                          "in a row; the first ones allocate stores of a new size class)"}
    return out


def measure_fast(args, xsb, h, mesh, n_ins, st_det, peak):
    """XSB_FAST (<= 1e-14 relative, pattern bit-exact): same workload, same span."""
    def step():
        h.reset()
        h.emit_p1fem(mesh, mesh, mesh, flavour=xsb.RAW)
        return h.flush(xsb.FAST)

    step()
    ms = timed_steps(h, step, max(1, min(args.steps, 3)))
    return {"ms_per_step": ms, "entries_per_s": n_ins / (ms / 1e3), "mode": "XSB_FAST",
            "workload": "P1-FEM 128^3: emit + flush! in fast mode"}


def measure_small(args, xsb, local):
    """BASELINE.json configs[0]: fdrand 2-D 100x100 (10^4 unknowns, 79 600 updateindex! calls) -- latency-bound:
    device time of reset! + insertion + flush! per assembly, and the number of kernel launches and host
    synchronisations it takes."""
    nx = 100
    h = xsb.Handle(nx * nx, nx * nx, device=local)

    def step():
        h.reset()
        h.emit_fdrand(nx, nx, 1, seed=1, flavour=xsb.UPDATE)
        return h.flush()

    for _ in range(5):
        step()
    l0 = h.kernel_launches
    ms = timed_steps(h, step, 50)
    launches = (h.kernel_launches - l0) / 50
    t0 = time.perf_counter()
    for _ in range(50):
        step()
    h.synchronize()
    wall = (time.perf_counter() - t0) / 50 * 1e3
    nnz = h.nnz
    h.close()
    return {"ms_per_assembly_device": ms, "ms_per_assembly_wall": wall, "kernel_launches_per_assembly": launches,
            "host_syncs_in_flush": 2, "n_inserted": 79600, "nnz": int(nnz),
            "workload": "fdrand 100x100 via updateindex! + flush! (BASELINE.json configs[0]); latency-bound"}


def measure_values_only(args, xsb, torch, peak, local):
    """BASELINE.json configs[2]: fdrand 200^3 built once, then 10 values-only re-assemblies into the frozen pattern
    (Newton loop; values device-resident).  Roofline: B_vo = 12 N_ins + 8 nnz (SURVEY.md 8d)."""
    import ctypes as C

    nx = args.vo_n
    n = nx ** 3
    g = xsb.Handle(n, n, device=local)
    g.set_precount(False)  # staged in stream order: the user's (I, J, V) stream
    g.emit_fdrand(nx, nx, nx, seed=100)
    cnt = g.pending
    dI = torch.empty(cnt, dtype=torch.int64, device="cuda")
    dJ = torch.empty(cnt, dtype=torch.int64, device="cuda")
    dV = torch.empty(cnt, dtype=torch.float64, device="cuda")
    got = C.c_int64(0)
    c = xsb.capi
    c.check(c.lib().xsb_debug_fetch_staged(g._h, 0, dI.data_ptr(), dJ.data_ptr(), dV.data_ptr(), None, cnt, C.byref(got)), g._h)
    g.set_precount(True)
    g.synchronize()
    nnz, _ = g.flush()
    g.timer_start()
    g.freeze_pattern(dI, dJ, count=cnt)
    ms_freeze = g.timer_stop()
    out = {"n_inserted": int(cnt), "nnz": int(nnz), "ms_freeze_once": ms_freeze,
           "workload": f"fdrand {nx}^3 (BASELINE.json configs[2]): 10 values-only re-assemblies into the frozen pattern, "
                       f"nonzeros .= 0 + xsb_reassemble_values, values resident in HBM"}
    b_vo = values_only_bytes(cnt, nnz)
    for name, m in (("deterministic", xsb.DETERMINISTIC), ("fast", xsb.FAST)):
        def re():
            g.reassemble_values(dV, m, count=cnt, zero_first=True)  # nonzeros(A) .= 0 fused into the re-assembly

        re()
        ms = timed_steps(g, re, 10)
        out[name] = {"ms_per_reassembly": ms, "entries_per_s": cnt / (ms / 1e3),
                     "roofline": {"bound": "hbm", "algorithmic_bytes": b_vo, "achieved": b_vo / (ms / 1e3) / 1e9,
                                  "peak": peak, "unit": "GB/s", "frac": b_vo / (ms / 1e3) / 1e9 / peak}}
    g.close()
    return out


def measure_fd(args, xsb, peak, local, n1):
    """BASELINE.json configs[4] on ONE GPU (the base of the strong-scaling curve): fdrand n1^3 via updateindex!."""
    N = n1 ** 3
    h = xsb.Handle(N, N, device=local)
    n_ins = xsb.capi.stream_count_fdrand(n1, n1, n1)

    def emit():
        h.emit_fdrand(n1, n1, n1, seed=20240717, flavour=xsb.UPDATE)

    def step():
        h.reset()
        emit()
        return h.flush()

    step()
    step()
    ms = timed_steps(h, step, max(1, min(args.steps, 3)))
    st, stage_ms, ms_emit = profiled_steps(h, emit, xsb.DETERMINISTIC, 1)
    b = flush_bytes(n_ins, 0, st["nnz_new"], N)
    out = {"ms_per_step": ms, "entries_per_s": n_ins / (ms / 1e3), "n_gpus": 1, "n_inserted": int(n_ins),
           "nnz": int(st["nnz_new"]), "ms_emit": ms_emit, "ms_flush": stage_ms["ms_total"],
           "flush_frac_of_hbm_peak": b / (stage_ms["ms_total"] / 1e3) / 1e9 / peak, "column_path": st["column_path"],
           "workload": f"fdrand 3-D {n1}^3 (BASELINE.json configs[4]) on one GPU: the base of the strong-scaling curve "
                       f"(bench.py --gpus N prints the same key for N ranks)"}
    h.close()
    return out


def measure_e2e(args, xsb, local, mesh, n, mode, np, torch):
    """Same metric through the drop-in boundary with HOST buffers, the call sequence of the Julia glue's
    Base.sum(exts, csc) (julia/ExtendableSparseB200.jl; mirrored by extendablesparse.jl_b200/dropin.py):
        xsb_set_csc (old CSC host -> device) -> xsb_insert_triplets (the partition's 16-byte triplets, pinned host
        memory -> device) -> xsb_flush -> xsb_fetch_csc (new CSC device -> pinned host)
    on ONE cached handle.  Headline: the build from an empty matrix.  Beside it: a SPLICE step (resident CSC of
    the first assembly uploaded through xsb_set_csc, 1 % new entries) and the stream as three Int64/Int64/Float64
    arrays (xsb_insert_batch: 24 B per insertion)."""
    import ctypes as C

    from xsparse_b200 import dropin

    emesh = args.e2e_mesh
    en = emesh ** 3
    c = xsb.capi
    g = xsb.Handle(en, en, device=local)
    g.set_precount(False)  # the host arrays hold the stream in call order, as user code would produce it
    g.emit_p1fem(emesh, emesh, emesh, flavour=xsb.RAW)
    cnt = g.pending
    dI = torch.empty(cnt, dtype=torch.int64, device="cuda")
    dJ = torch.empty(cnt, dtype=torch.int64, device="cuda")
    dV = torch.empty(cnt, dtype=torch.float64, device="cuda")
    got = C.c_int64(0)
    c.check(c.lib().xsb_debug_fetch_staged(g._h, 0, dI.data_ptr(), dJ.data_ptr(), dV.data_ptr(), None, cnt,
                                           C.byref(got)), g._h)
    hI = torch.empty(cnt, dtype=torch.int64, pin_memory=True)
    hJ = torch.empty(cnt, dtype=torch.int64, pin_memory=True)
    hV = torch.empty(cnt, dtype=torch.float64, pin_memory=True)
    hI.copy_(dI)
    hJ.copy_(dJ)
    hV.copy_(dV)
    # the same stream as xsb_triplet {u32 row, u32 col, f64 val}: two 64-bit words per insertion
    dT = torch.empty((cnt, 2), dtype=torch.int64, device="cuda")
    dT[:, 0] = dI | (dJ << 32)
    dT[:, 1] = dV.view(torch.int64)
    hT = torch.empty((cnt, 2), dtype=torch.int64, pin_memory=True)
    hT.copy_(dT)
    torch.cuda.synchronize()
    del dI, dJ, dV
    g.reset()
    g.set_precount(True)

    # the generic insertion path with the stream RESIDENT in HBM (what a CUDA.jl kernel that wrote its triplets to a
    # device array would call): xsb_insert_triplets on a device pointer + xsb_flush, nothing crosses PCIe
    def step_dev():
        g.reset()
        g.insert_triplets(dT, xsb.RAW, 0, cnt)
        return g.flush(mode)

    for _ in range(2):
        step_dev()
    g.synchronize()
    g.timer_start()
    for _ in range(3):
        step_dev()
    ms_dev = g.timer_stop() / 3
    g.set_profiling(True)
    step_dev()
    ms_dev_flush = g.flush_stats()["ms_total"]
    g.set_profiling(False)
    del dT
    g.reset()

    # the extension object of the glue, its triplet buffer living in pinned host memory
    ext = dropin.SparseMatrixB200(en, en, buffer=hT.numpy().view(c.TRIPLET_DTYPE).reshape(-1))
    ext.fill = cnt
    ext.runs = [(0, xsb.RAW)]
    empty = (np.ones(en + 1, np.int64), np.empty(0, np.int64), np.empty(0, np.float64))
    (cp0, rv0, nz0), _ = dropin.sum_extensions([ext], en, en, empty, mode, handle=g)
    nnz = len(rv0)
    ocp = torch.empty(en + 1, dtype=torch.int64, pin_memory=True)
    orv = torch.empty(nnz + nnz // 50 + 16, dtype=torch.int64, pin_memory=True)
    onz = torch.empty(nnz + nnz // 50 + 16, dtype=torch.float64, pin_memory=True)
    outb = (ocp.numpy(), orv.numpy(), onz.numpy())

    def step_build():
        return dropin.sum_extensions([ext], en, en, empty, mode, out=outb, handle=g)

    def timed(step, reps):
        step()
        g.synchronize()
        g.timer_start()
        for _ in range(reps):
            step()
        return g.timer_stop() / reps

    reps = max(1, min(args.steps, 3))
    ms = timed(step_build, reps)
    check_a = (int(orv[:1000].sum()), float(onz[:1000].sum()))

    def step_ijv():
        g.set_csc(*[torch.from_numpy(a) for a in empty[:1]] + [None, None])
        g.insert_batch(hI, hJ, hV, xsb.RAW, count=cnt)
        g.flush(mode)
        g.fetch_csc(ocp, orv, onz)

    ms_ijv = timed(step_ijv, reps)
    assert check_a == (int(orv[:1000].sum()), float(onz[:1000].sum())), "triplet and (I,J,V) assemblies differ"

    # splice: the matrix of the first assembly is the wrapper's host CSC; 1 % new entries arrive
    pcp = torch.empty(en + 1, dtype=torch.int64, pin_memory=True).copy_(torch.from_numpy(cp0))
    prv = torch.empty(nnz, dtype=torch.int64, pin_memory=True).copy_(torch.from_numpy(rv0))
    pnz = torch.empty(nnz, dtype=torch.float64, pin_memory=True).copy_(torch.from_numpy(nz0))
    rng = np.random.default_rng(11)
    k = max(1, nnz // 100)
    hS = torch.empty((k, 2), dtype=torch.int64, pin_memory=True)
    sv = hS.numpy().view(c.TRIPLET_DTYPE).reshape(-1)
    sv["row"], sv["col"], sv["val"] = rng.integers(1, en + 1, k), rng.integers(1, en + 1, k), rng.standard_normal(k)
    sext = dropin.SparseMatrixB200(en, en, buffer=sv)
    sext.fill = k
    sext.runs = [(0, xsb.UPDATE)]
    resident = (pcp.numpy(), prv.numpy(), pnz.numpy())

    def step_splice():
        return dropin.sum_extensions([sext], en, en, resident, mode, out=outb, handle=g)

    (_, srv, _), _ = step_splice()
    ms_splice = timed(step_splice, reps)
    nnz_s = len(srv)
    g.close()
    d2h = 8 * (en + 1) + 16 * int(nnz)
    return {"value": cnt / (ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": 16 * cnt + 8 * (en + 1),
            "d2h_bytes_per_step": d2h, "ms_per_step": ms,
            "workload": f"P1-FEM {emesh}^3-node mesh through the drop-in sequence of Base.sum(exts, csc): xsb_set_csc (empty "
                        f"CSC) + {cnt} insertions from a pinned host buffer of 16-byte triplets (xsb_insert_triplets) + "
                        f"xsb_flush + xsb_fetch_csc into pinned host arrays",
            "splice": {"ms_per_step": ms_splice, "inserted": int(k), "nnz_old": int(nnz), "nnz_new": int(nnz_s),
                       "h2d_bytes_per_step": 16 * k + 16 * int(nnz) + 8 * (en + 1),
                       "d2h_bytes_per_step": 8 * (en + 1) + 16 * int(nnz_s),
                       "workload": "flush! with a resident matrix: old CSC uploaded through xsb_set_csc, 1 % new entries "
                                   "(xsb_insert_triplets), merged CSC read back"},
            "device_triplets": {"value": cnt / (ms_dev / 1e3), "unit": UNIT, "ms_per_step": ms_dev,
                                "ms_insert": ms_dev - ms_dev_flush, "ms_flush": ms_dev_flush,
                                "workload": "same stream as 16-byte triplets resident in HBM: xsb_insert_triplets on a "
                                            "device pointer (pack_grouped2_kernel) + xsb_flush; no PCIe"},
            "ijv": {"value": cnt / (ms_ijv / 1e3), "unit": UNIT, "h2d_bytes_per_step": 24 * cnt + 8 * (en + 1),
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_ijv,
                    "workload": "same stream as three pinned host arrays Int64 I, Int64 J, Float64 V "
                                "(xsb_insert_batch)"}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mesh", type=int, default=128, help="nodes per direction of the FEM mesh (128 = configs[1])")
    ap.add_argument("--e2e-mesh", type=int, default=128)
    ap.add_argument("--cpu-mesh", type=int, default=128, help="mesh of the cpu_baseline sample")
    ap.add_argument("--ref-mesh", type=int, default=128, help="mesh of one --impl reference step (128 = the GPU arm's workload)")
    ap.add_argument("--mode", default="deterministic", choices=["deterministic", "fast"])
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--verify", action="store_true",
                    help="N > 1: compare every rank's slab (SHA-256) with the same global assembly done on one GPU")
    ap.add_argument("--no-legs", action="store_true", help="skip the splice / fast / values_only / cfg5 legs")
    ap.add_argument("--vo-n", type=int, default=200, help="grid of the values_only leg (200 = configs[2])")
    ap.add_argument("--workload", default="fem", choices=["fem", "fd400"],
                    help="N>1 only: fem = weak scaling of configs[1] (default, the bench line); fd400 = configs[4], "
                         "fdrand 400^3 sharded by node slab over the ranks (strong scaling, no e2e leg)")
    ap.add_argument("--fd-n", type=int, default=400, help="grid points per direction of --workload fd400")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="one GPU: write the CSC of the last timed step to DIR/*.npy (float64; colptr whole, rowval and "
                         "nzval at a fixed seeded sample of positions) to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs needs the single-GPU arm (--impl ours --gpus 1)")
    args.warmup = max(3, args.warmup) if args.impl == "ours" else max(0, args.warmup)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
