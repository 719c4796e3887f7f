"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/fourier.h and include/fourier_b200.h declare, the drop-in programs compile and link against
it, and the host-side mirror of the reference interface behaves.  No compute calls (no GPU here)."""
import json
import os
import re
import shutil
import subprocess

import pytest

import fourier_b200 as fb
from fourier_b200 import _lib, build as fbuild

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INCLUDE = os.path.join(ROOT, "include")
LIBDIR = os.path.join(ROOT, "fourier_b200", "lib")
FFI = os.path.join(ROOT, "tests", "ffi")


@pytest.fixture(scope="module")
def libfourier():
    fbuild.build()
    return _lib.load()


def _declared(header):
    text = open(os.path.join(INCLUDE, header)).read()
    names = set(re.findall(r"\b(fourier_b200_[a-z_0-9]+)\s*\(", text))
    names.discard("fourier_b200_plan_info")  # the struct
    for t in ("float", "double"):
        if "FOURIER_B200_DECLARE(" + t in text:
            names |= {f"fourier_{op}_{t}" for op in ("create", "destroy", "transform_in_place", "transform")}
    return names


def test_library_exports_every_declared_symbol(libfourier):
    declared = _declared("fourier.h") | _declared("fourier_b200.h")
    assert set(_lib.REFERENCE_SYMBOLS) <= declared
    assert set(_lib.EXTENSION_SYMBOLS) <= declared
    for name in sorted(declared):
        assert hasattr(libfourier, name), f"libfourier.so does not export {name}"


def test_exactly_the_reference_symbols_plus_prefixed_extension(libfourier):
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True)
    exported = {l.split()[-1] for l in out.stdout.splitlines() if " T " in l}
    assert set(_lib.REFERENCE_SYMBOLS) <= exported
    extra = {s for s in exported if not s.startswith("fourier_b200_")} - set(_lib.REFERENCE_SYMBOLS)
    assert not extra, f"unexpected exported symbols: {sorted(extra)}"


def test_soname_matches_reference_packaging():
    # fourier-ffi/CMakeLists.txt:15-19,55-65: libfourier.so.0.1.0 with SONAME libfourier.so.0
    out = subprocess.run(["readelf", "-d", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert "libfourier.so.0" in out
    assert not re.search(r"NEEDED.*(torch|cufft|c10)", out), "product library must not depend on torch or cuFFT"


@pytest.mark.parametrize("src,cc,flags", [
    ("dropin_test.c", "gcc", ["-std=c11"]),
    ("dropin_test.cpp", "g++", ["-std=c++11"]),
    ("trait_mirror_test.cpp", "g++", ["-std=c++11"]),
])
def test_dropin_programs_compile_and_link(tmp_path, libfourier, src, cc, flags):
    exe = tmp_path / "a.out"
    cmd = [cc, *flags, "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", INCLUDE, os.path.join(FFI, src),
           "-o", str(exe), "-L", LIBDIR, "-lfourier", "-lm", f"-Wl,-rpath,{LIBDIR}"]
    subprocess.run(cmd, check=True, capture_output=True)
    assert exe.exists()


@pytest.mark.parametrize("src,cc,hdr", [
    ("test.c", "gcc", "ours"), ("test.cpp", "g++", "ours"), ("test.c", "gcc", "reference"),
    ("test.cpp", "g++", "reference")])
def test_reference_ffi_tests_link_unmodified(tmp_path, libfourier, src, cc, hdr):
    """The reference's own FFI test programs (fourier-ffi/test.c, test.cpp), compiled with the
    reference's warning flags (CMakeLists.txt:9-13) against either header, link against libfourier.so
    with no undefined symbols.  tests/golden/reference_ffi_symbols.json holds the library symbols each
    compiled program references; a program of the same language that references exactly those symbols
    is linked here, and the symbols compiled against our header must be ones include/fourier.h declares.
    (The equivalent programs in tests/ffi/ are run by tests/test_gpu_parity.py.)"""
    with open(os.path.join(ROOT, "tests", "golden", "reference_ffi_symbols.json")) as f:
        symbols = json.load(f)["programs"][src][hdr]
    assert set(_lib.REFERENCE_SYMBOLS) == set(symbols)
    if hdr == "ours":
        assert set(symbols) <= _declared("fourier.h")
    prog = tmp_path / ("refs.c" if cc == "gcc" else "refs.cpp")
    prog.write_text("#ifdef __cplusplus\nextern \"C\" {\n#endif\n"
                    + "".join(f"void {s}(void);\n" for s in symbols)
                    + "#ifdef __cplusplus\n}\n#endif\n"
                    + "int main(void) {\n  void (*volatile refs[])(void) = {" + ", ".join(symbols) + "};\n"
                    + "  return refs[0] == 0;\n}\n")
    exe = tmp_path / "ref_test"
    cmd = [cc, "-Wall", "-Wextra", "-pedantic", "-Werror", str(prog), "-o", str(exe), "-L", LIBDIR, "-lfourier", "-lm"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


def test_transform_enum_mirrors_reference():
    # fourier-algorithms/src/fft.rs:5-36 and fourier-ffi/src/lib.rs:3-12
    T = fb.Transform
    assert [int(t) for t in (T.Fft, T.Ifft, T.UnscaledIfft, T.SqrtScaledFft, T.SqrtScaledIfft)] == [0, 1, 2, 3, 4]
    assert T.Fft.is_forward() and T.SqrtScaledFft.is_forward()
    assert not (T.Ifft.is_forward() or T.UnscaledIfft.is_forward() or T.SqrtScaledIfft.is_forward())
    assert T.Fft.inverse() is T.Ifft and T.Ifft.inverse() is T.Fft
    assert T.SqrtScaledFft.inverse() is T.SqrtScaledIfft and T.UnscaledIfft.inverse() is None


def test_no_cpu_fallback_without_a_gpu(libfourier):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert libfourier.fourier_b200_device_count() == 0
    with pytest.raises(RuntimeError, match="no usable CUDA device"):
        fb.create_fft_f32(1024)
    assert not libfourier.fourier_create_double(8)


def test_distributed_building_blocks_reject_bad_arguments(libfourier):
    """Argument validation of the exchange / pack / peer-memory entry points happens before any CUDA call, so it
    can be checked without a GPU: nonzero return code and a message in fourier_b200_last_error()."""
    import ctypes
    L = _lib.load()
    outs = (ctypes.c_void_p * 2)(None, None)
    assert L.fourier_b200_exchange_float(None, outs, 2, 0, 8, 8, 16, 16, 0, 0, 0, 0, None) != 0
    assert "exchange" in _lib.last_error()
    buf = ctypes.create_string_buffer(64)
    assert L.fourier_b200_exchange_double(buf, outs, 0, 0, 8, 8, 16, 16, 0, 0, 0, 0, None) != 0      # no ranks
    assert L.fourier_b200_exchange_double(buf, outs, 2, 2, 8, 8, 16, 16, 0, 0, 0, 0, None) != 0      # rank out of range
    assert L.fourier_b200_exchange_double(buf, outs, 2, 0, 8, 8, 16, 16, 0, 3, 0, 64, None) != 0     # twiddle mode
    assert L.fourier_b200_pack_float(buf, buf, 1, 8, 8, 8, 8, 64, 7, 0, 0, 64, None) != 0            # twiddle mode
    ptr, handle = ctypes.c_void_p(), ctypes.create_string_buffer(64)
    assert L.fourier_b200_peer_alloc(0, ctypes.byref(ptr), handle) != 0                              # empty buffer
    assert L.fourier_b200_peer_open(None, ctypes.byref(ptr)) != 0
    assert L.fourier_b200_peer_close(None) == 0 and L.fourier_b200_peer_free(None) == 0              # no-ops


def test_product_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under fourier_b200/ may include, import, link or dlopen it
    (comments may mention it)."""
    pkg = os.path.join(ROOT, "fourier_b200")
    bad = re.compile(r"#\s*include[^\n]*oracle|^\s*(from|import)\s+[^\n]*oracle|libfourier_oracle|dlopen", re.M)
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert not bad.search(text), f
    out = subprocess.run(["readelf", "-d", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert "oracle" not in out


@pytest.mark.skipif(shutil.which("cmake") is None or (shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc")),
                    reason="cmake / nvcc not available")
def test_cmake_package_configures(tmp_path):
    """CMakeLists.txt (the packaging that mirrors fourier-ffi/CMakeLists.txt: shared + static `fourier`, the four
    C / C++ test programs, find_package config) must at least configure; the full build takes minutes and is not
    part of the CPU suite."""
    env = dict(os.environ)
    env.setdefault("CUDACXX", shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc")
    r = subprocess.run(["cmake", "-S", ROOT, "-B", str(tmp_path / "b"), "-DCMAKE_BUILD_TYPE=Release"],
                       capture_output=True, text=True, env=env)
    assert r.returncode == 0, r.stdout + r.stderr
    targets = subprocess.run(["cmake", "--build", str(tmp_path / "b"), "--target", "help"], capture_output=True, text=True).stdout
    for t in ("fourier_shared", "fourier_static", "test_c_static", "test_c_shared", "test_cpp_static", "test_cpp_shared"):
        assert t in targets, targets
