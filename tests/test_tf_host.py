"""Machine-level facts of the Taylor-Fourier kernels (tf.cu) that need no GPU: no spills under -Xptxas -v; in the SASS
of the moment tile kernel no local memory, one native integer ATOMS.ADD per moment and no CAS loop; the combine kernel
has no local memory; and the CPU-fiber suite of tf.cu is clean under AddressSanitizer."""
import os
import re
import shutil
import subprocess
import sys
from math import comb

import pytest

from tests.test_sass_bispec import count, one, sass  # noqa: F401  (the cuobjdump fixture)
from tests.test_simt_asan import _libasan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_no_spills_under_ptxas_verbose(tmp_path):
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not found")
    csrc = os.path.join(ROOT, "astrild_b200", "csrc")
    out = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
                          "-Xptxas", "-v", "-I", os.path.join(ROOT, "include"), "-I", csrc, "-c", os.path.join(csrc, "tf.cu"),
                          "-o", str(tmp_path / "tf.o")], capture_output=True, text=True, check=True)
    blocks = re.findall(r"Function properties for (\S*tf_\w+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, "
                        r"(\d+) bytes spill loads", out.stderr)
    assert len([b for b in blocks if "wrap_index_slow" not in b[0]]) == 11   # 5 orders x (unit, mass) tile kernels, combine
    for name, frame, st, ld in blocks:
        assert (int(frame), int(st), int(ld)) == (0, 0, 0), name


@pytest.mark.parametrize("order", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("mass", [0, 1])
def test_moment_tile_kernel_sass(sass, order, mass):  # noqa: F811
    ops = one(sass, rf"tf_moment_tile_kernelILi{order}ELb{mass}E")
    assert count(ops, "LDL") + count(ops, "STL") == 0
    assert count(ops, "ATOMS.ADD") == comb(order + 3, 3), "one integer shared-memory atomic per moment"
    assert not any("CAS" in op for op in ops), "a CAS loop in the moment tile kernel"
    assert count(ops, "REDG.E.ADD.F32.FTZ.RN.STRONG.GPU") + count(ops, "RED.E.ADD.F32.FTZ.RN.STRONG.GPU") >= 1


def test_combine_kernel_sass(sass):  # noqa: F811
    ops = one(sass, r"tf_combine_kernel")
    assert count(ops, "LDL") + count(ops, "STL") == 0
    assert count(ops, "FFMA") >= 2


@pytest.mark.skipif(os.environ.get("APK_SIMT_ASAN", "0") not in ("", "0"), reason="already inside the sanitized run")
def test_tf_kernels_clean_under_address_sanitizer():
    lib = _libasan()
    if lib is None or shutil.which("g++") is None:
        pytest.skip("libasan or g++ not found")
    env = dict(os.environ, APK_SIMT_ASAN="1", LD_PRELOAD=lib, ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0")
    out = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider", "tests/test_simt_tf.py"],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    tail = (out.stdout + out.stderr)[-4000:]
    assert "AddressSanitizer" not in tail, tail
    assert out.returncode == 0, tail
