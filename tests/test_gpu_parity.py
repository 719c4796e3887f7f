"""GPU parity tests: the CUDA path, called through the C ABI (libfourier.so via fourier_b200), against
the CPU oracle (oracle/, the plain-C restatement of the reference) on the same inputs.

Tolerances (BASELINE.json north_star / SURVEY.md 8c):
    max|X_gpu - X_ref| / max|X_ref| < 1e-5 (f32), < 1e-12 (f64), X_ref = oracle in the same precision;
the sweep 1..=255 additionally uses the reference test-suite's own rule (1e-4 | 8 ulp, 1e-11 | 8 ulp,
fourier/tests/integrity.rs:89-143) against the reference's naive DFT.
"""
import os
import subprocess

import numpy as np
import pytest

import fourier_b200 as fb
from fourier_b200 import _lib
from oracle import oracle as O
from helpers import assert_near_reference_rule, golden_10pt, rel_err, sweep_input, truth_f64

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL = {"f32": 1e-5, "f64": 1e-12}
NP = {"f32": np.complex64, "f64": np.complex128}
T = fb.Transform


def create(real, n, general=False):
    return fb.create_fft_f32(n, general) if real == "f32" else fb.create_fft_f64(n, general)


def gpu_transform(plan, x, code):
    out = np.empty_like(x)
    plan.transform(x, out, code)
    return out


# ---- reference test-suite cases ------------------------------------------------------------------------

@pytest.mark.parametrize("real", ["f32", "f64"])
def test_golden_10pt(real):
    # fourier/tests/integrity.rs:48-72 (committed as tests/golden/integrity_10pt.json)
    x, y = golden_10pt()
    p = create(real, 10)
    assert p.info()["path_name"].startswith("bluestein")
    assert_near_reference_rule(gpu_transform(p, x.astype(NP[real]), T.Fft), y)
    assert_near_reference_rule(gpu_transform(p, y.astype(NP[real]), T.Ifft), x)


@pytest.mark.parametrize("real", ["f32", "f64"])
@pytest.mark.parametrize("forward", [True, False])
def test_sweep_1_to_255(real, forward):
    # integrity.rs:145-192 through the single-transform reference ABI with host buffers
    data = sweep_input(256, NP[real], forward)
    code = T.Fft if forward else T.Ifft
    worst = 0.0
    for size in range(1, 256):
        x = np.ascontiguousarray(data[:size])
        p = create(real, size)
        out = np.empty_like(x)
        p.c_transform(x, out, code)
        assert_near_reference_rule(out, O.naive_dft(x, inverse=not forward))
        e = rel_err(out, O.transform(x, int(code)))
        worst = max(worst, e)
        assert e < TOL[real], (size, e)
        p.close()
    print(f"sweep {real} forward={forward}: worst rel err vs oracle {worst:.3e}")


@pytest.mark.parametrize("real", ["f32", "f64"])
@pytest.mark.parametrize("size", [64, 73, 128])
def test_static_sizes(real, size):
    # integrity.rs:234-254 and the fourier-macros doc-test size
    for forward in (True, False):
        x = np.ascontiguousarray(sweep_input(256, NP[real], forward)[:size])
        got = gpu_transform(create(real, size), x, T.Fft if forward else T.Ifft)
        assert_near_reference_rule(got, O.naive_dft(x, inverse=not forward))


# ---- every Transform code, BASELINE sizes and edge sizes vs the oracle ----------------------------------

SIZES = [1, 2, 3, 4, 5, 6, 8, 9, 12, 16, 17, 27, 32, 48, 64, 81, 96, 100, 128, 243, 256, 384, 512, 729, 1000,
         1009, 1024, 1536, 2048, 4096, 6561, 8192, 12288, 16384, 32768, 65536]


@pytest.mark.parametrize("real", ["f32", "f64"])
@pytest.mark.parametrize("code", [0, 1, 2, 3, 4])
def test_all_codes_vs_oracle(real, code):
    rng = np.random.default_rng(100 + code)
    for n in SIZES:
        x = (rng.standard_normal((3, n)) + 1j * rng.standard_normal((3, n))).astype(NP[real])
        got = gpu_transform(create(real, n), x, T(code))
        want = O.transform(x, code)
        assert rel_err(got, want) < TOL[real], (n, code, rel_err(got, want))
        assert rel_err(got, truth_f64(x, code)) < 3 * TOL[real], (n, code)


@pytest.mark.parametrize("real,n", [("f32", 1 << 20), ("f64", 1 << 16), ("f32", 1 << 16), ("f64", 1 << 20),
                                    ("f32", 1 << 18), ("f32", 3 << 18), ("f64", 1 << 14), ("f32", 1 << 22),
                                    ("f32", 1 << 13), ("f32", 1 << 15), ("f32", 1 << 17), ("f32", 1 << 19),
                                    ("f64", 1 << 13), ("f64", 1 << 15)])
def test_large_sizes_vs_oracle(real, n):
    x = O.fill_input(3, n, NP[real], first_transform=11)
    p = create(real, n)
    for code in (T.Fft, T.Ifft):
        got = gpu_transform(p, x, code)
        want = O.transform(x, int(code))
        e = rel_err(got, want)
        print(f"N={n} {real} {code.name} path={p.info()['path_name']} rel err {e:.3e}")
        assert e < TOL[real], (n, code, e)


@pytest.mark.parametrize("real,n", [("f32", 1 << 21), ("f32", 1 << 23), ("f32", 1 << 25), ("f64", 1 << 17),
                                    ("f64", 1 << 19), ("f64", 1 << 21)])
def test_three_pass_path_above_the_two_pass_sizes(real, n):
    """Power-of-two N beyond the two-pass kernels: outer column pass + two-pass rows with a transposed store
    (csrc/bigpow2.cu).  Every Transform code against the oracle, in place == out of place, batch == loop, the
    independent per-stage path, and one launch count: 1 + 2 per chunk of rows."""
    import torch
    x = O.fill_input(2, n, NP[real], first_transform=5)
    p = create(real, n)
    assert p.info()["path_name"] == "threepass" and p.info()["n1"] * p.info()["n2"] == n
    assert "column_kernel" in p.kernel_name()
    first = None
    for code in (T.Fft, T.Ifft, T.UnscaledIfft, T.SqrtScaledFft, T.SqrtScaledIfft):
        got = gpu_transform(p, x, code)
        e = rel_err(got, O.transform(x, int(code)))
        print(f"N=2^{n.bit_length() - 1} {real} {code.name}: rel err {e:.3e}")
        assert e < TOL[real], (n, code, e)
        if code == T.Fft:
            first = got
    assert p.info()["last_launches"] <= 2 * (1 + 2 * 8)
    xd = torch.from_numpy(x).cuda()
    p.transform_in_place(xd, T.Fft)                       # in place, device pointers, batch of 2
    assert np.array_equal(xd.cpu().numpy(), first)
    single = np.empty_like(x[1])
    p.c_transform(np.ascontiguousarray(x[1]), single, T.Fft)
    assert np.array_equal(single, first[1])
    if n <= 1 << 23:
        gen = create(real, n, general=True)
        assert gen.info()["path_name"] == "global_stages"
        assert rel_err(first, gpu_transform(gen, x, T.Fft)) < TOL[real]


@pytest.mark.parametrize("real,n", [("f32", 3 << 13), ("f32", 9 << 14), ("f32", 27 << 11), ("f32", 3 << 18), ("f32", 27 << 16),
                                    ("f64", 3 << 12), ("f64", 9 << 13), ("f64", 27 << 10)])
def test_three_pass_path_with_an_outer_radix3_pass(real, n):
    """N = 3^b * 2^k (b <= 3) above the CTA kernel's shared memory: outer radix-3 / 9 / 27 pass + two-pass rows with the
    transposed store (csrc/bigpow2.cu).  3 / 9 / 27 rows per transform pad the 32-row tiles of the row kernel: batches of
    1, 2 and 5 transforms; every Transform code against the oracle; in place; the independent per-stage path."""
    import torch
    p = create(real, n)
    assert p.info()["path_name"] == "threepass" and p.info()["n1"] in (3, 9, 27) and p.info()["n1"] * p.info()["n2"] == n
    assert "radix3_column_kernel" in p.kernel_name()
    x = O.fill_input(5, n, NP[real], first_transform=9)
    want = {int(c): O.transform(x, int(c)) for c in (T.Fft, T.Ifft, T.UnscaledIfft, T.SqrtScaledFft, T.SqrtScaledIfft)}
    for code, w in want.items():
        got = gpu_transform(p, x, T(code))
        e = rel_err(got, w)
        assert e < TOL[real], (n, code, e)
    first = gpu_transform(p, x, T.Fft)
    for b in (1, 2):
        assert np.array_equal(gpu_transform(p, np.ascontiguousarray(x[:b]), T.Fft), first[:b])
    xd = torch.from_numpy(x).cuda()
    p.transform_in_place(xd, T.Fft)
    assert np.array_equal(xd.cpu().numpy(), first)
    gen = create(real, n, general=True)
    assert gen.info()["path_name"] == "global_stages"
    assert rel_err(first, gpu_transform(gen, x, T.Fft)) < TOL[real]


@pytest.mark.parametrize("real,n", [("f32", 1_500_001), ("f64", 100_003)])
def test_bluestein_around_a_three_pass_inner_plan(real, n):
    """Bluestein sizes whose inner power of two (2^22 f32, 2^18 f64) lies above the two-pass kernels."""
    x = O.fill_input(1, n, NP[real], first_transform=2)
    p = create(real, n)
    assert p.info()["path_name"] == "bluestein" and p.info()["inner_path_name"] == "threepass"
    got = gpu_transform(p, x, T.Fft)
    assert rel_err(got, truth_f64(x, int(T.Fft))) < TOL[real]


@pytest.mark.parametrize("real", ["f32", "f64"])
def test_random_sizes_all_paths(real):
    """60 pseudo-random sizes up to 40000 (primes, prime powers, {2,3}-smooth, odd composites): every path
    (on-chip, two-pass tiles, general stages, fused and unfused Bluestein) against the oracle."""
    rng = np.random.default_rng(2026)
    sizes = set(int(v) for v in rng.integers(2, 6000, 30)) | set(int(v) for v in rng.integers(6000, 40000, 12))
    sizes |= {997, 1021, 1031, 2047, 2048, 2049, 3 * 1024, 5 * 1024, 9 * 512, 2 * 3 ** 7, 7 ** 4, 4093, 8191, 10007, 3 ** 9}
    seen = {}
    for n in sorted(sizes):
        x = (rng.standard_normal((2, n)) + 1j * rng.standard_normal((2, n))).astype(NP[real])
        p = create(real, n)
        seen[p.info()["path_name"]] = seen.get(p.info()["path_name"], 0) + 1
        for code in (T.Fft, T.SqrtScaledIfft):
            got, want = gpu_transform(p, x, code), O.transform(x, int(code))
            e = rel_err(got, want)
            if e >= TOL[real]:
                # The reference forms the Bluestein chirp angle pi*i^2/N in f64 WITHOUT reducing i^2 mod 2N
                # (bluesteins.rs:31,33,57), so for N in the thousands its own f64 result is only good to
                # ~1e-12; the GPU plan reduces the index exactly.  Accept a discrepancy only if it is the
                # oracle's distance from the f64 truth and the GPU result is an order of magnitude closer.
                truth = truth_f64(x, int(code))
                assert p.info()["path_name"].startswith("bluestein"), (n, code, e)
                # (measured on B200, f64: N=2804 gpu-vs-truth 7e-16, oracle-vs-truth 1.1e-12; N=30011: 1e-15 vs 1.3e-11)
                assert rel_err(got, truth) < TOL[real] / 10 and rel_err(want, truth) > e / 2, (n, code, e)
                continue
            assert e < TOL[real], (n, code, p.info()["path_name"], e)
        p.close()
    print(real, "paths exercised:", seen)
    assert {"global_stages", "bluestein", "bluestein_fused", "onchip_cta"} <= set(seen)


def test_smooth_sizes_run_in_one_launch():
    """No {2,3}-smooth N <= 4096 falls to the one-kernel-per-stage path, and the reference's own bench sizes
    (fourier-bench/benches/fft_bench.rs:153-159: 243/729/2187 radix-3, 1418/3125/1013 Bluestein) are ONE launch."""
    n = 2
    smooth = []
    for a in range(13):
        for b in range(8):
            v = (2 ** a) * (3 ** b)
            if 2 <= v <= 4096:
                smooth.append(v)
    for real in ("f32", "f64"):
        for v in sorted(smooth):
            p = create(real, v)
            assert p.info()["path_name"] != "global_stages", (real, v, p.info()["path_name"])
            p.close()
        for v in (243, 729, 2187, 96, 384, 1536, 1418, 3125, 1013, 222, 722):
            x = O.fill_input(5, v, NP[real], first_transform=3)
            p = create(real, v)
            for code in (T.Fft, T.Ifft, T.SqrtScaledFft):
                got = gpu_transform(p, x, code)
                e = rel_err(got, O.transform(x, int(code)))
                if e >= TOL[real] and p.info()["path_name"].startswith("bluestein"):
                    # f64 Bluestein sizes in the thousands: the reference's own chirp is only good to ~1e-12
                    # (INTEGRATION.md section 6); the GPU result must then be far closer to the f64 truth
                    assert rel_err(got, truth_f64(x, int(code))) < TOL[real] / 10, (real, v, code, e)
                    continue
                assert e < TOL[real], (real, v, code, p.info()["path_name"], e)
            # f64 N=3125 needs M=8192 on chip: two 128 KB buffers do not fit an SM, it stays on the unfused path
            if not (real == "f64" and v == 3125):
                assert p.info()["last_launches"] == 1, (real, v, p.info()["path_name"], p.info()["last_launches"])
            p.close()


@pytest.mark.parametrize("real", ["f32", "f64"])
def test_cta_kernel_batches_and_in_place(real):
    """The CTA-level kernel with batches that are not a multiple of its group size, in place and out of place."""
    import torch
    for n in (6, 9, 48, 243, 2187, 3000 if real == "f32" else 1500, 4374, 12288 if real == "f32" else 6144):
        p = create(real, n)
        if n not in (3000, 1500):
            assert p.info()["path_name"] == "onchip_cta", (n, p.info()["path_name"])
        for batch in (1, 7, 100):
            x = O.fill_input(batch, n, NP[real], first_transform=batch)
            want = O.transform(x, O.FFT)
            assert rel_err(gpu_transform(p, x, T.Fft), want) < TOL[real], (n, batch)
            d = torch.from_numpy(x.copy()).cuda()
            p.transform_in_place(d, T.Fft)
            assert rel_err(d.cpu().numpy(), want) < TOL[real], (n, batch, "in place")
        p.close()


def test_config1_single_1024_via_reference_abi():
    # BASELINE.json configs[0]: one 1024-point c-f32 forward FFT through fourier_create_float +
    # fourier_transform_float with host buffers
    x = O.fill_input(1, 1024, np.complex64)[0]
    p = fb.create_fft_f32(1024)
    out = np.empty_like(x)
    p.c_transform(x, out, T.Fft)
    e = rel_err(out, O.transform(x, O.FFT))
    print(f"config 1: rel err vs oracle {e:.3e}, vs f64 truth {rel_err(out, truth_f64(x, 0)):.3e}")
    assert e < 1e-5


@pytest.mark.parametrize("real", ["f32", "f64"])
def test_config4_bluestein_1009(real):
    x = O.fill_input(64, 1009, NP[real])
    p = create(real, 1009)
    assert p.info()["inner_size"] == 2048
    for code in T:
        assert rel_err(gpu_transform(p, x, code), O.transform(x, int(code))) < TOL[real], code


# ---- interface semantics ------------------------------------------------------------------------------------

@pytest.mark.parametrize("real", ["f32", "f64"])
@pytest.mark.parametrize("n", [1, 6, 8, 96, 1009, 4096, 1 << 16])
def test_in_place_equals_out_of_place_and_batch_equals_loop(real, n):
    x = O.fill_input(5, n, NP[real], first_transform=3)
    p = create(real, n)
    out = gpu_transform(p, x, T.Fft)
    y = x.copy()
    p.transform_in_place(y, T.Fft)
    assert np.array_equal(out, y)
    for b in range(5):
        single = np.empty_like(x[b])
        p.c_transform(np.ascontiguousarray(x[b]), single, T.Fft)
        assert np.array_equal(single, out[b])
        z = x[b].copy()
        p.c_transform_in_place(z, T.Fft)
        assert np.array_equal(z, out[b])
    assert np.array_equal(x, O.fill_input(5, n, NP[real], first_transform=3)), "transform() must not touch its input"


@pytest.mark.parametrize("real", ["f32", "f64"])
@pytest.mark.parametrize("n", [96, 1009, 4096, 1 << 16, 1 << 20])
def test_device_pointer_path_equals_host_path(real, n):
    import torch
    x = O.fill_input(4, n, NP[real])
    p = create(real, n)
    host = gpu_transform(p, x, T.Fft)
    xd = torch.from_numpy(x).cuda()
    yd = torch.empty_like(xd)
    p.transform(xd, yd, T.Fft)
    assert np.array_equal(yd.cpu().numpy(), host)
    assert np.array_equal(xd.cpu().numpy(), x)
    p.transform_in_place(xd, T.Fft)
    assert np.array_equal(xd.cpu().numpy(), host)


@pytest.mark.parametrize("real", ["f32", "f64"])
def test_device_input_generator_matches_oracle(real):
    import torch
    dt = torch.complex64 if real == "f32" else torch.complex128
    t = torch.empty((7, 1009), dtype=dt, device="cuda")
    fb.fill_input(t, first_transform=5)
    want = O.fill_input(7, 1009, NP[real], first_transform=5)
    assert np.array_equal(t.cpu().numpy().view(np.uint8), want.view(np.uint8))


@pytest.mark.parametrize("real", ["f32", "f64"])
@pytest.mark.parametrize("n", [64, 128, 512, 1024, 4096, 1 << 13, 1 << 14, 1 << 15, 1 << 16, 1 << 17, 1 << 19, 1 << 20])
def test_fused_paths_agree_with_general_path(real, n):
    # the one-kernel-per-stage path is an independent implementation of the same transform
    x = O.fill_input(3, n, NP[real], first_transform=1)
    fast, gen = create(real, n), create(real, n, general=True)
    assert gen.info()["path_name"] == "global_stages"
    for code in (T.Fft, T.SqrtScaledIfft):
        assert rel_err(gpu_transform(fast, x, code), gpu_transform(gen, x, code)) < TOL[real]


def test_misaligned_device_pointer_is_refused():
    """ADVICE r1: the kernels use 16-byte vector accesses / TMA on device buffers; a slice that starts at an odd f32
    sample is only 8-byte aligned and must be refused up front (no launch, no sticky CUDA error)."""
    import torch
    p = create("f32", 1 << 20)
    big = torch.zeros(2 * (1 << 20) + 2, dtype=torch.complex64, device="cuda")
    x, y = big[1:1 + (1 << 20)], torch.empty(1 << 20, dtype=torch.complex64, device="cuda")
    assert x.data_ptr() % 16 == 8
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        p.transform(x, y, T.Fft)
    with pytest.raises(RuntimeError, match="16-byte aligned"):
        p.transform(y, x, T.Fft)
    torch.cuda.synchronize()                      # the context is still healthy
    ok = torch.empty(1 << 20, dtype=torch.complex64, device="cuda")
    fb.fill_input(ok.view(1, -1))
    p.transform(ok, y, T.Fft)
    torch.cuda.synchronize()
    want = O.transform(O.fill_input(1, 1 << 20, np.complex64)[0], O.FFT)
    assert rel_err(y.cpu().numpy(), want) < TOL["f32"]


def test_kernel_names_follow_the_path():
    names = {(r, n): create(r, n).kernel_name() for r, n in
             [("f32", 1 << 20), ("f64", 1 << 16), ("f32", 1 << 16), ("f32", 1024), ("f32", 1009), ("f32", 729),
              ("f64", 1009), ("f64", 1 << 15), ("f32", 3 ** 9), ("f32", 1 << 15)]}
    assert "fused_twopass_kernel" in names[("f32", 1 << 20)] and "fused_twopass_kernel" in names[("f64", 1 << 16)]
    assert "fused_twopass_kernel" in names[("f32", 1 << 16)]
    assert "onchip_fft_kernel" in names[("f32", 1024)] and "bluestein_fused_kernel" in names[("f32", 1009)]
    assert "cta_fft_kernel" in names[("f32", 729)] and "chirp" in names[("f64", 1009)]
    assert "tile_kernel" in names[("f64", 1 << 15)] and "stockham_stage_kernel" in names[("f32", 3 ** 9)]
    assert "fused_twopass_kernel" in names[("f32", 1 << 15)]


def test_error_conventions():
    L = _lib.load()
    assert not L.fourier_create_float(0)          # reference hangs on 0 (autosort/mod.rs:112): refused
    p = fb.create_fft_f32(8)
    x = O.fill_input(1, 8, np.complex64)[0]
    y = x.copy()
    p.c_transform_in_place(y, 99)                 # unknown code: silent no-op (ffi lib.rs:10,37)
    assert np.array_equal(x, y)
    with pytest.raises(ValueError):
        p.transform(np.zeros(7, np.complex64), np.zeros(7, np.complex64), T.Fft)  # assert_eq!, fft.rs:57-58
    with pytest.raises(TypeError):
        p.transform(np.zeros(8, np.complex128), np.zeros(8, np.complex128), T.Fft)
    L.fourier_destroy_float(None)


# ---- size-independent properties at BASELINE.json's full transform sizes ---------------------------------

def _device_batch(real, n, batch, first=0):
    import torch
    dt = torch.complex64 if real == "f32" else torch.complex128
    t = torch.empty((batch, n), dtype=dt, device="cuda")
    return fb.fill_input(t, first_transform=first)


@pytest.mark.parametrize("real,n,batch", [("f32", 1 << 20, 96), ("f64", 1 << 16, 512), ("f32", 1009, 8192)])
def test_properties_at_baseline_sizes(real, n, batch):
    import torch
    p = create(real, n)
    x = _device_batch(real, n, batch)
    X = torch.empty_like(x)
    p.transform(x, X, T.Fft)
    # Parseval: sum|X|^2 = N sum|x|^2 per transform
    ex = (x.abs() ** 2).sum(dim=1).double()
    eX = (X.abs() ** 2).sum(dim=1).double()
    assert float(((eX / (n * ex)) - 1).abs().max()) < (1e-4 if real == "f32" else 1e-11)
    # DC bin = sum of the input
    dc = x.sum(dim=1)
    assert float((X[:, 0] - dc).abs().max() / dc.abs().max()) < (2e-3 if real == "f32" else 1e-10)
    # round trip FFT -> IFFT
    y = torch.empty_like(x)
    p.transform(X, y, T.Ifft)
    assert float((y - x).abs().max()) < (2e-5 if real == "f32" else 1e-12)
    # linearity: F(a x0 + b x1) = a F(x0) + b F(x1)
    a, b = 0.75, -1.25
    z = (a * x[0::2] + b * x[1::2]).contiguous()
    Z = torch.empty_like(z)
    p.transform(z, Z, T.Fft)
    lin = a * X[0::2] + b * X[1::2]
    assert float((Z - lin).abs().max() / lin.abs().max()) < (1e-5 if real == "f32" else 1e-12)
    # sqrt-scaled pair is unitary
    U = torch.empty_like(x)
    p.transform(x, U, T.SqrtScaledFft)
    eU = (U.abs() ** 2).sum(dim=1).double()
    assert float((eU / ex - 1).abs().max()) < (1e-4 if real == "f32" else 1e-11)
    # sampled transforms of the batch against the oracle on the identical (hash-generated) input
    for b_idx in (0, 1, batch // 2, batch - 1):
        want = O.transform(O.fill_input(1, n, NP[real], first_transform=b_idx)[0], O.FFT)
        assert rel_err(X[b_idx].cpu().numpy(), want) < TOL[real], b_idx


# ---- the drop-in programs, run against libfourier.so on the GPU box ------------------------------------------

@pytest.mark.parametrize("src,cc,flags", [("dropin_test.c", "gcc", ["-std=c11"]),
                                          ("dropin_test.cpp", "g++", ["-std=c++11"]),
                                          ("trait_mirror_test.cpp", "g++", ["-std=c++11"])])
def test_dropin_programs_run(tmp_path, src, cc, flags):
    libdir = os.path.join(ROOT, "fourier_b200", "lib")
    exe = tmp_path / "dropin"
    subprocess.run([cc, *flags, "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "ffi", src), "-o", str(exe), "-L", libdir, "-lfourier", "-lm",
                    f"-Wl,-rpath,{libdir}"], check=True, capture_output=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "passed" in r.stdout
