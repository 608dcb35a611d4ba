"""Machine-level facts of the bispectrum's triple-product reduction (bispec.cu), read with cuobjdump (no GPU needed):
the float32 instantiation keeps its register tile in registers (no local memory), reads its operands with shared-memory
loads (no shared-memory atomics) and multiplies with FFMA; the float64 instantiation (the triangle counts) uses DFMA."""
import re
import shutil
import subprocess

import pytest


@pytest.fixture(scope="module")
def sass(built_lib):
    if shutil.which("cuobjdump") is None:
        pytest.skip("cuobjdump not on PATH")
    text = subprocess.run(["cuobjdump", "-sass", built_lib], capture_output=True, text=True, check=True).stdout
    kernels, name = {}, None
    for line in text.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            kernels[name] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*(?:\.[A-Z0-9_]+)*)", line)
        if m and name:
            kernels[name].append(m.group(1))
    return kernels


def one(kernels, pattern):
    hits = [k for k in kernels if re.search(pattern, k)]
    assert len(hits) == 1, (pattern, hits)
    return kernels[hits[0]]


def count(ops, prefix):
    return sum(op == prefix or op.startswith(prefix + ".") for op in ops)


def test_float_reduction_is_ffma_on_shared_memory_operands(sass):
    ops = one(sass, r"bk_reduce_kernelIfE")
    assert count(ops, "LDL") + count(ops, "STL") == 0, "the float32 reduction spills to local memory"
    assert not any(op.startswith("ATOMS") for op in ops)
    assert count(ops, "FFMA") >= 32                   # 8 x 4 register tile per point (the point loop is unrolled)
    assert count(ops, "LDS") >= 4                     # F_i, the j-run and the l-run from shared memory
    assert any(op.startswith("LDS.128") for op in ops), "the j- and l-runs are read with vector loads"
    assert any(op.startswith("LDGSTS") for op in ops), "chunks are staged with asynchronous copies"


def test_double_reduction_uses_dfma(sass):
    ops = one(sass, r"bk_reduce_kernelIdE")
    assert count(ops, "DFMA") >= 16                   # 4 x 4 register tile
    assert count(ops, "LDL") + count(ops, "STL") == 0
    assert not any(op.startswith("ATOMS") for op in ops)
