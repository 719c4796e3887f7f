"""The FOURIER_B200_* tuning knobs are read once, when a plan is created (csrc/plan.h, Tuning): a plan and its exec
calls never run with two configurations.  And the kernel attributes a plan needs are set on every device a process
uses, not only on the first."""
import ctypes

import numpy as np
import pytest

import fourier_b200 as fb
from oracle import oracle as O
from helpers import rel_err

pytestmark = pytest.mark.gpu

TOL = {"f32": 1e-5, "f64": 1e-12}


def test_rows_exchange_keeps_the_chunking_of_plan_creation(monkeypatch):
    import torch
    from fourier_b200.distributed import CudaBackend
    for knob in ("CHUNK_MB", "DIST_CHUNK_MB", "DIST_LANES", "DIST_OVERLAP"):
        monkeypatch.delenv("FOURIER_B200_" + knob, raising=False)
    n, rows = 1 << 14, 96
    torch.manual_seed(5)
    src = torch.randn(rows * n, dtype=torch.complex64, device="cuda")
    be = CudaBackend("f32")

    def run():
        out = torch.zeros(rows * n, dtype=torch.complex64, device="cuda")
        table = (ctypes.c_void_p * 1)(out.data_ptr())
        be.launches = 0   # counts info()["last_launches"] of the call
        be.fft_rows_exchange(src, table, 1, 0, rows, n, True, (True, 7, 1 << 30))
        torch.cuda.synchronize()
        return be.launches, out

    launches, want = run()    # creates the plan: 64 MB chunks, all 96 rows in one chunk
    assert launches == 2
    monkeypatch.setenv("FOURIER_B200_DIST_CHUNK_MB", "2")    # 16 rows per chunk, on one stream
    monkeypatch.setenv("FOURIER_B200_DIST_OVERLAP", "0")
    got_launches, got = run()  # same backend, so the same plan
    assert got_launches == launches
    assert torch.equal(got, want)


def test_trace_knob_set_after_plan_creation_is_ignored(monkeypatch, tmp_path):
    monkeypatch.delenv("FOURIER_B200_TRACE", raising=False)
    n = 1 << 20
    p = fb.create_fft_f32(n)
    assert p.kernel_name() == "fused::fused_twopass_kernel"
    trace = tmp_path / "trace.txt"
    monkeypatch.setenv("FOURIER_B200_TRACE", str(trace))
    x = O.fill_input(2, n, np.complex64)
    out = np.empty_like(x)
    p.transform(x, out, fb.Transform.Fft)
    assert not trace.exists()
    assert rel_err(out, O.transform(x, O.FFT)) < TOL["f32"]


def test_cta_plans_on_two_devices():
    """The CTA kernel needs more than 48 KB of dynamic shared memory, a per-device kernel attribute."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    cases = [("f32", 729, "onchip_cta"), ("f64", 1009, "bluestein_fused")]   # 1009: chirp-z on the CTA kernel
    try:
        for dev in (0, 1):
            fb.set_device(dev)
            for real, n, path in cases:
                p = fb.create_fft_f32(n) if real == "f32" else fb.create_fft_f64(n)
                assert p.info()["device"] == dev and p.info()["path_name"] == path
                assert p.kernel_name().startswith("cta::cta_fft_kernel")
                x = O.fill_input(3, n, np.complex64 if real == "f32" else np.complex128)
                xd = torch.from_numpy(x).to(f"cuda:{dev}")
                for code in (fb.Transform.Fft, fb.Transform.Ifft):
                    yd = torch.empty_like(xd)
                    p.transform(xd, yd, code)
                    torch.cuda.synchronize(dev)
                    e = rel_err(yd.cpu().numpy(), O.transform(x, int(code)))
                    assert e < TOL[real], (dev, real, n, code, e)
                p.close()
    finally:
        fb.set_device(0)
