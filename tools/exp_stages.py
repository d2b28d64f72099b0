#!/usr/bin/env python
"""Stage timings of one flush! per workload (development tool, not a bench line).

  python tools/exp_stages.py [fem128] [fd200] [rd96] [fem64] ...   (default: fem128 fd200 rd96)
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

ge.build()
import xsparse_b200 as xsb  # noqa: E402


def run(name, reps=4, mode=None):
    kind = name.rstrip("0123456789")
    size = int(name[len(kind):])
    if kind == "fem":
        n = size ** 3
        emit = lambda h: h.emit_p1fem(size, size, size, flavour=xsb.RAW)
    elif kind == "fd":
        n = size ** 3
        emit = lambda h: h.emit_fdrand(size, size, size, seed=7)
    elif kind == "rd":
        n = 4 * size ** 3
        emit = lambda h: h.emit_blockrd(size, size, size, 4, seed=7)
    else:
        raise SystemExit(f"unknown workload {name}")
    h = xsb.Handle(n, n)
    h.set_profiling(True)
    mode = xsb.DETERMINISTIC if mode is None else mode
    best = None
    emits = []
    for r in range(reps):
        h.reset()
        h.timer_start()
        emit(h)
        ms_emit = h.timer_stop()
        h.flush(mode)
        st = h.flush_stats()
        st["ms_emit"] = ms_emit
        emits.append(ms_emit)
        if best is None or st["ms_total"] < best["ms_total"]:
            best = st
    best["ms_emit"] = min(emits)
    print("   emit per rep: " + " ".join(f"{e:.3f}" for e in emits))
    rec = best["n_inserted"]
    keys = ["ms_emit", "ms_total", "ms_preagg", "ms_group_count", "ms_pair_sort", "ms_group_scatter", "ms_fold", "ms_compact",
            "ms_colptr", "ms_histogram", "ms_sort", "ms_reduce", "ms_other"]
    print(f"{name}: n_ins={rec} nnz={best['nnz_new']} path={best['column_path']} pairs={best['group_pairs']} "
          f"passes={best['sort_passes']} launches={best['kernel_launches']} direct={best['direct_fold']} "
          f"preagg={best['preagg_records']}")
    print("   " + "  ".join(f"{k[3:]}={best[k]:.3f}" for k in keys))
    gbs = lambda b, ms: b / ms / 1e6 if ms > 0 else 0
    print(f"   GB/s: count={gbs(16 * rec, best['ms_group_count']):.0f} scatter={gbs(32 * rec, best['ms_group_scatter']):.0f} "
          f"fold={gbs(16 * rec + 16 * best['nnz_new'], best['ms_fold']):.0f} "
          f"compact={gbs(32 * best['nnz_new'], best['ms_compact']):.0f} emit={gbs(16 * rec, best['ms_emit']):.0f}  "
          f"G entries/s (emit+flush)={rec / (best['ms_emit'] + best['ms_total']) / 1e6:.2f}")
    h.close()


if __name__ == "__main__":
    names = [a for a in sys.argv[1:] if not a.startswith("-")] or ["fem128", "fd200", "rd96"]
    mode = xsb.FAST if "--fast" in sys.argv else None
    for nm in names:
        run(nm, mode=mode)
