"""Throughput table over transform sizes (one B200): path, kernel, samples/s, fraction of the measured HBM peak, launches
per transform call, rel. error of one transform vs the oracle.
    PYTHONPATH=. python tools/size_table.py f32 243 729 2187 65536 ...     (sizes; 2^k may be written as 2^k)
Environment knobs of the library (FOURIER_B200_FUSED, _TWOPASS, _RING, _LAG) apply and are echoed."""
import json
import os
import sys

import numpy as np
import torch

import fourier_b200 as fb
from oracle import oracle as O


def peak():
    try:
        return float(json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0


def bench(real, n, total=1 << 28, steps=5):
    batch = max(1, total // n // (1 if real == "f32" else 2))
    p = fb.create_fft_f32(n) if real == "f32" else fb.create_fft_f64(n)
    dt = torch.complex64 if real == "f32" else torch.complex128
    x = torch.empty((batch, n), dtype=dt, device="cuda")
    fb.fill_input(x)
    y = torch.empty_like(x)
    for _ in range(3):
        p.transform(x, y, fb.Transform.Fft)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        p.transform(x, y, fb.Transform.Fft)
    b.record()
    torch.cuda.synchronize()
    sps = batch * n / (a.elapsed_time(b) / steps) * 1e3
    pick = min(5, batch - 1)
    npdt = np.complex64 if real == "f32" else np.complex128
    want = O.transform(O.fill_input(1, n, npdt, first_transform=pick)[0], O.FFT)
    err = float(np.abs(y[pick].cpu().numpy() - want).max() / np.abs(want).max())
    bps = 16 if real == "f32" else 32
    print(f"{real} N={n:8d} batch={batch:8d} {p.info()['path_name']:16s} {p.kernel_name()[:44]:44s} {sps:.3e} samples/s "
          f"{100 * sps * bps / 1e9 / peak():5.1f} % of HBM peak  launches {p.info()['last_launches']:4d}  rel err {err:.1e}", flush=True)
    p.close()


if __name__ == "__main__":
    real = sys.argv[1]
    knobs = {k: v for k, v in os.environ.items() if k.startswith("FOURIER_B200")}
    if knobs:
        print(knobs)
    for s in sys.argv[2:]:
        bench(real, (1 << int(s[2:])) if s.startswith("2^") else int(s))
