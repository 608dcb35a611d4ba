"""Host-side facts of the correlation function that need no GPU: the library's r tables equal astrild_b200/tables.py
(and so the oracle's) bit for bit; corr.cu's kernels keep everything in registers (no spills under -Xptxas -v, no local
memory in the SASS) and the 1-D binning kernel builds r^2 from DADDs of the squared tables, with no squaring on the
device; and the CPU-fiber suite of corr.cu is clean under AddressSanitizer."""
import ctypes as ct
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from tests.test_abi import _tables_lib
from tests.test_sass_bispec import count, one, sass  # noqa: F401  (the cuobjdump fixture)
from tests.test_simt_asan import _libasan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("N", [8, 33, 128, 512, 1024])
@pytest.mark.parametrize("L", [1000.0, 500.0, 7.3])
def test_library_r_tables_bit_identical_to_the_numpy_tables(built_lib, N, L):
    from astrild_b200 import tables
    lib = _tables_lib(built_lib)
    d, i, vp = ct.c_double, ct.c_int, ct.c_void_p
    lib.apk_tables_r_axis.argtypes = [i, d, vp]
    lib.apk_tables_r_edges.argtypes = [i, d, d, d, d, vp, i, ct.POINTER(i)]
    r = np.empty(N)
    assert lib.apk_tables_r_axis(N, L, r.ctypes.data) == 0
    np.testing.assert_array_equal(r, tables.r_axis(N, L))
    for rmin, dr, rmax in ((0.0, 0.0, 0.0), (L / N, 0.0, 0.0), (0.013 * L, 0.0071 * L, 0.9 * L)):
        want = tables.r_edges(N, L, rmin, dr or None, rmax or None)
        n = ct.c_int()
        assert lib.apk_tables_r_edges(N, L, rmin, dr, rmax, None, 0, ct.byref(n)) == 0
        assert n.value == len(want)
        e = np.empty(n.value)
        assert lib.apk_tables_r_edges(N, L, rmin, dr, rmax, e.ctypes.data, len(e), ct.byref(n)) == 0
        np.testing.assert_array_equal(e, want)


def test_no_spills_under_ptxas_verbose(tmp_path):
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    csrc = os.path.join(ROOT, "astrild_b200", "csrc")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v",
                          "-I", os.path.join(ROOT, "include"), "-I", csrc, "-c", os.path.join(csrc, "corr.cu"),
                          "-o", str(tmp_path / "corr.o")], capture_output=True, text=True, check=True)
    blocks = re.findall(r"Function properties for (\S*xi_\w+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, "
                        r"(\d+) bytes spill loads", out.stderr)
    assert len(blocks) >= 13                                 # 8 fills, 4 binnings, the fold
    for name, frame, st, ld in blocks:
        assert (int(frame), int(st), int(ld)) == (0, 0, 0), name


def test_binning_sass(sass):  # noqa: F811
    for inst in ("xi_bin_kernelILb0ELb0E", "xi_bin_kernelILb1ELb0E", "xi_bin_kernelILb0ELb1E", "xi_bin_kernelILb1ELb1E"):
        ops = one(sass, inst)
        assert count(ops, "LDL") + count(ops, "STL") == 0, inst
    ops = one(sass, "xi_bin_kernelILb0ELb0E")                # the per-call 1-D binning
    assert count(ops, "DADD") >= 2                           # r^2 = (ra^2 + rb^2) + rz^2
    assert count(ops, "DMUL") == 0, "the 1-D binning squares on the device"
    assert count(ops, "LDG") >= 1


@pytest.mark.skipif(os.environ.get("APK_SIMT_ASAN", "0") not in ("", "0"), reason="already inside the sanitized run")
def test_corr_kernels_clean_under_address_sanitizer():
    lib = _libasan()
    if lib is None or shutil.which("g++") is None:
        pytest.skip("libasan or g++ not found")
    env = dict(os.environ, APK_SIMT_ASAN="1", LD_PRELOAD=lib, ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0")
    out = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider", "tests/test_simt_corr.py"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    tail = (out.stdout + out.stderr)[-4000:]
    assert "AddressSanitizer" not in tail, tail
    assert out.returncode == 0, tail
