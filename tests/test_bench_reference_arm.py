"""`bench.py --impl reference` (the CPU arm the driver runs beside the CUDA arm) on a small workload: one JSON line with
the contract's keys, the reference arm's own additions, and the same `config` dict the CUDA arm prints for the
workload (the driver compares the two).  Runs on CPU: the arm executes the oracle port, never the CUDA library."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    rec = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in rec, key
    assert rec["impl"] == "reference" and rec["steps"] == 2 and rec["warmup"] == 1 and rec["higher_is_better"] is True
    assert rec["value"] > 0 and rec["unit"] == "complex samples/s" and rec["vs_baseline"] is None
    cb = rec["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == rec["value"] and "transforms of N=1024" in cb["sample"]
    assert rec["e2e"] == {"value": rec["value"], "unit": rec["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    sys.path.insert(0, ROOT)
    import bench
    n, batch, real, desc = bench.WORKLOADS["c1"]
    assert rec["config"] == bench.workload_config(desc, n, batch, 1, real)


def test_reference_arm_dumps_its_last_step(tmp_path):
    """--dump-outputs: the transforms of the last timed step as float32 (real, imaginary) pairs, and their indices."""
    import numpy as np
    sys.path.insert(0, ROOT)
    from oracle import oracle as O
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1",
                        "--steps", "1", "--warmup", "0", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    rec = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert rec["dump"]["files"] == ["output.npy", "output_rows.npy"]
    y, rows = np.load(out / "output.npy"), np.load(out / "output_rows.npy")
    assert y.dtype == np.float32 and rows.dtype == np.float64 and y.shape[1:] == (1024, 2)
    assert y.shape[0] == rows.shape[0] == rec["dump"]["rows"] and y.nbytes + rows.nbytes <= 64 << 20
    assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < rec["dump"]["of_rows"]
    got = y[..., 0] + 1j * y[..., 1]
    x = np.concatenate([O.fill_input(1, 1024, np.complex64, first_transform=int(row)) for row in rows])
    want = O.transform(x, O.FFT)
    assert np.abs(got - want).max() / np.abs(want).max() < 1e-5
