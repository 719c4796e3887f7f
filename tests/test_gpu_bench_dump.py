"""bench.py --dump-outputs on the CUDA path: the files hold what the last timed step computed, are the same from run
to run (and for any number of steps), and stay within 64 MB; --steps is the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle as O
from helpers import rel_err

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--also", "none", "--no-e2e",
                        "--no-cpu-baseline", "--dump-outputs", str(out_dir), *args],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    rec = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    y, rows = np.load(out_dir / "output.npy"), np.load(out_dir / "output_rows.npy")
    assert y.dtype == np.float32 and rows.dtype == np.float64
    assert sum(os.path.getsize(out_dir / f) for f in os.listdir(out_dir)) <= 64 << 20
    return rec, y[..., 0] + 1j * y[..., 1], rows


def test_batched_dump_is_a_seeded_sample_of_the_last_step(tmp_path):
    n = 1 << 20
    first, y, rows = _bench(tmp_path / "a", "--workload", "c2", "--batch", "8", "--steps", "3", "--warmup", "1")
    assert first["steps"] == 3 and first["gpu_launches"] % 3 == 0
    assert y.shape == (6, n) and list(rows) == sorted(set(rows)) and 0 <= rows[0] and rows[-1] < 8   # 48 MB of 64
    for i, r in enumerate(rows):
        want = O.transform(O.fill_input(1, n, np.complex64, first_transform=int(r))[0], O.FFT)
        assert rel_err(y[i], want) < 1e-5, r
    second, y2, rows2 = _bench(tmp_path / "b", "--workload", "c2", "--batch", "8", "--steps", "2", "--warmup", "1")
    assert second["steps"] == 2 and second["gpu_launches"] * 3 == first["gpu_launches"] * 2
    assert np.array_equal(rows, rows2) and np.array_equal(y, y2)


def test_distributed_dump_is_the_last_step(tmp_path):
    """c5 on one GPU: each step transforms the previous result, so after 3 warm-up steps and 1 timed step the output
    is the fourth forward transform of the input, N^2 x."""
    n = 1 << 20
    rec, y, rows = _bench(tmp_path / "c5", "--workload", "c5", "--log2n", "20", "--steps", "1", "--warmup", "0")
    assert rec["steps"] == 1 and rec["warmup"] == 3
    assert list(rows) == list(range(y.shape[0])) and y.size == n
    x = O.fill_input(1, n, np.complex64)[0].astype(np.complex128)
    assert rel_err(y.reshape(-1), float(n) ** 2 * x) < 1e-5
