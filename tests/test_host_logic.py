"""Host-side logic that needs no GPU: tables, error paths, the product never touching the oracle."""
import os
import re

import numpy as np
import pytest
import torch

from astrild_b200 import tables
from oracle import pk_oracle as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("N", [8, 33, 128, 512])
@pytest.mark.parametrize("L", [1.0, 500.0, 1000.0])
def test_tables_bit_identical_to_oracle(N, L):
    kx, _, kz = o.k_tables(N, L)
    np.testing.assert_array_equal(tables.k_axis(N, L), kx)
    np.testing.assert_array_equal(tables.k_axis(N, L)[: N // 2 + 1], kz)
    np.testing.assert_array_equal(tables.k_edges(N, L, 2 * np.pi / L), o.k_edges(N, L, 2 * np.pi / L))
    np.testing.assert_array_equal(tables.k_edges(N, L), o.k_edges(N, L))
    np.testing.assert_array_equal(tables.hermitian_weights(N), o.hermitian_weights(N))
    for rs in ("cic", "tsc"):
        for il in (False, True):
            np.testing.assert_array_equal(tables.compensation_axis(rs, il, N), o.compensation_1d(rs, il, N))


def test_edges_count_matches_survey():
    for N in (128, 512, 1024):
        assert len(tables.k_edges(N, 1000.0, 2 * np.pi / 1000.0)) == N // 2      # N/2 edges, N/2-1 bins


def test_interlace_phase_is_pi_n_over_N():
    N, L = 16, 300.0
    np.testing.assert_allclose(tables.interlace_phase_axis(N, L), np.pi * tables.freq_index(N) / N, rtol=1e-15)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "astrild_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", text, flags=re.M), f
                assert "pk_oracle" not in text, f


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_fails_loudly_without_gpu(built_lib):
    import astrild_b200
    from astrild_b200._lib import AstrildPkError
    with pytest.raises(AstrildPkError):
        astrild_b200.ArrayMesh(np.zeros((8, 8, 8)), BoxSize=100.0)
    with pytest.raises(AstrildPkError):
        astrild_b200.ParticleMesh(Nmesh=[8] * 3, BoxSize=100.0)


def test_missing_library_is_an_error(monkeypatch, tmp_path):
    from astrild_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.AstrildPkError):
        _lib.load()


def test_bench_dump_outputs_writes_every_result_array(tmp_path):
    import bench
    res = {"k": np.array([0.1, np.nan]), "power": np.array([2.0 + 1.0j, 3.0 + 0.0j]), "modes": np.array([6, 0]),
           "edges": np.array([0.0, 0.2, 0.4]), "Nsum": np.array([1, 6, 0, 2], dtype=np.int64)}
    bench.dump_outputs(res, str(tmp_path / "out"))
    got = {p.stem: np.load(p) for p in (tmp_path / "out").iterdir()}
    assert set(got) == {"k", "power_real", "power_imag", "modes", "edges", "Nsum"}
    assert all(a.dtype == np.float64 for a in got.values())
    np.testing.assert_array_equal(got["k"], res["k"])
    np.testing.assert_array_equal(got["power_real"] + 1j * got["power_imag"], res["power"])
    np.testing.assert_array_equal(got["Nsum"], res["Nsum"])


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_arguments_it_cannot_honour(argv):
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True)
    assert out.returncode == 2 and "bench.py: error" in out.stderr


def test_recorded_bench_lines_carry_the_contract_keys():
    """The JSON lines bench.py printed on the GPU box at the end of the round (committed under profiles/) have every key the
    measurement contract names -- a guard against a bench change that drops one (the bench itself needs a GPU)."""
    import json
    here = os.path.dirname(os.path.abspath(__file__))
    rec = os.path.join(here, "..", "profiles", "r02_call32")
    line = json.loads(open(os.path.join(rec, "bench_default.json")).read().strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline", "check"):
        assert key in line, key
    assert "workload" in line["config"] and line["n_gpus"] == 1 and line["gpu_launches"] > 0
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
    assert line["e2e"]["h2d_bytes_per_step"] == 12 * line["config"]["particles"]          # x, y, z float32 columns
    roof = line["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(roof)
    assert abs(roof["frac"] - roof["achieved"] / roof["peak"]) < 1e-12 and roof["traffic"] >= roof["algorithmic_bytes_per_launch"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"]) and line["cpu_baseline"]["kind"] == "port"
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(line["clocks"])
    assert line["check"]["ok"] and line["check"]["modes_equal"] and line["check"]["max_rel_P"] <= 1e-4
    # the stage split adds up to the step (CUDA events on one stream)
    ms = line["stages"]["ms"]
    assert abs(ms["deposit_stage"] + ms["fft"] + ms["bin_stage"] - line["ms_per_step"]) < 0.05 * line["ms_per_step"]
    ref = json.loads(open(os.path.join(rec, "bench_reference.json")).read().strip().splitlines()[-1])
    assert ref["impl"] == "reference" and ref["metric"] == line["metric"] and ref["unit"] == line["unit"]
    assert ref["e2e"]["h2d_bytes_per_step"] == 0 and ref["cpu_baseline"]["kind"] == "port"
    assert {k: v for k, v in ref["config"].items() if k in ("workload", "particles", "mesh", "resampler", "interlaced", "compensated")} == \
           {k: v for k, v in line["config"].items() if k in ("workload", "particles", "mesh", "resampler", "interlaced", "compensated")}
