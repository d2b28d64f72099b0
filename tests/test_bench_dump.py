"""bench.py --dump-outputs: the CSC of the last timed step as float64 .npy files (colptr whole, rowval / nzval at a
fixed seeded sample of positions), bounded in size and the same from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def oracle_fem_csc(oracle, mesh):
    I, J, V = oracle.fem_stream(mesh, mesh, mesh)
    A = oracle.OracleExt(mesh ** 3, mesh ** 3)
    A.insert_batch(I, J, V, oracle.RAW)
    return A.csc()


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def test_dump_sample_is_seeded_bounded_and_exact(oracle, monkeypatch, tmp_path):
    import torch

    import bench

    cp, rv, nz = (torch.from_numpy(a) for a in oracle_fem_csc(oracle, 8))
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    out = bench.csc_outputs(cp, rv, nz, torch)
    assert sorted(out) == ["colptr", "nzval_sample", "rowval_sample", "sample_index"]
    assert all(a.dtype == np.float64 for a in out.values())
    pos = out["sample_index"].astype(np.int64)
    assert len(pos) == 1000 and np.all(np.diff(pos) > 0) and pos[0] >= 0 and pos[-1] < len(rv)
    assert np.array_equal(out["colptr"], cp.numpy())
    assert np.array_equal(out["rowval_sample"], rv.numpy()[pos])
    assert np.array_equal(bits(out["nzval_sample"]), bits(nz.numpy()[pos]))
    again = bench.csc_outputs(cp, rv, nz, torch)
    assert all(np.array_equal(bits(out[k]), bits(again[k])) for k in out)
    bench.write_outputs(str(tmp_path / "d"), out)
    for k, a in out.items():
        assert np.array_equal(bits(np.load(tmp_path / "d" / f"{k}.npy")), bits(a))
    # a CSC smaller than the sample is kept whole
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1 << 20)
    whole = bench.csc_outputs(cp, rv, nz, torch)
    assert np.array_equal(whole["sample_index"], np.arange(len(rv)))
    # the flagship (FEM 128^3: 2^21 + 1 columns, 31 065 598 nnz) stays far below 64 MiB
    assert 8 * ((128 ** 3 + 1) + 3 * bench.DUMP_SAMPLE) < 64 << 20


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"],
                                   ["--gpus", "2", "--dump-outputs", "x"]])
def test_bench_rejects_arguments_it_cannot_honour(extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "error" in out.stderr


@pytest.mark.gpu
def test_bench_dump_equals_oracle(oracle, tmp_path):
    """The dump of a FEM 48^3 bench run (1.6 M nnz: a real sample) against the oracle's CSC at the same positions."""
    import torch

    import bench

    mesh = 48
    d = tmp_path / "out"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3",
                          "--mesh", str(mesh), "--e2e-mesh", "12", "--no-cpu", "--no-legs", "--dump-outputs", str(d)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    got = {f[:-4]: np.load(d / f) for f in os.listdir(d)}
    want = bench.csc_outputs(*(torch.from_numpy(a) for a in oracle_fem_csc(oracle, mesh)), torch)
    assert sorted(got) == sorted(want) and len(want["sample_index"]) == bench.DUMP_SAMPLE
    for k in want:
        assert got[k].dtype == np.float64 and np.array_equal(bits(got[k]), bits(want[k])), k
