"""Bispectrum measurements on one GPU (FFTBispectrum, astrild_b200/csrc/bispec.cu).  One run does everything:

  BK0  128^3 mesh, 128^3 Zel'dovich particles, TSC interlaced compensated, dk = 2 k_f: parity against the float64 oracle
       with the tolerance of tests/test_gpu_bispectrum.py (|B - B_oracle| <= TAU A);
  BK1  256^3 mesh from 256^3 particles, dk = 2 k_f, default kmax (42 shells);
  BK2  512^3 mesh from 512^3 particles, dk = 4 k_f, default kmax (42 shells).

For BK1 / BK2 it prints ms per stage (fill, c2r, reduction, fold: apk_bispec_last_ms, CUDA events, mean over the timed
calls after warm-up), the one-off time of the triangle counts and the time per call; the useful FLOP 2 (triples kept) N^3
and the reduction's rate over the FP32 FMA bound SMs x 128 x 2 x SM clock (clock read in the same run), and checks the
timed outputs: repeated calls agree bit for bit, and T_F of a sample of triples matches a float64 torch recomputation
from the same complex field within TAU A.  The card's name and power limit are read with queries only.

    python tools/bispec_bench.py [--out profiles/bispec_b200.json] [--only BK0,BK1,BK2] [--iters 5]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import astrild_b200 as ab  # noqa: E402
from astrild_b200 import synthetic, tables  # noqa: E402

TAU = 2e-4            # tests/test_gpu_bispectrum.py
L = 1000.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    name, plim, sm, smmax = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    props = torch.cuda.get_device_properties(0)
    return {"name": name, "power_limit_W": float(plim), "sm_clock_MHz_now": float(sm), "sm_clock_MHz_max": float(smmax),
            "sms": props.multi_processor_count}


def mesh_of(N, seed=7):
    cols = synthetic.zeldovich_particles(N, L, seed, torch.device("cuda"), rms_cells=1.0)
    return cols, ab.CatalogMesh(cols, L, N, resampler="tsc", interlaced=True, compensated=True, normalize=True, pos_scale=1.0)


def bk0():
    from oracle import bk_oracle as bo
    N, dk = 128, 2 * 2 * np.pi / L
    cols, mesh = mesh_of(N)
    r = ab.FFTBispectrum(mesh, dk=dk).bispectrum
    pos = torch.stack(list(cols), 1).double().cpu().numpy() * L
    c = bo.delta_k_from_particles(pos, None, N, L, "tsc", interlaced=True, compensated=True, normalize=True)
    o = bo.bispectrum_fft(c, N, L, bo.default_edges(N, L, dk=dk), with_abs=True)
    keep = o["ntri"] > 0
    worst = float(np.max(np.abs(r["B"] - o["B"][keep]) / o["A"][keep]))
    ok = bool(np.array_equal(r["triangles"], o["ntri"][keep]) and worst <= TAU)
    return {"config": "BK0", "N": N, "particles": N ** 3, "dk_kf": 2, "shells": len(o["edges"]) - 1,
            "triples": int(keep.sum()), "counts_equal": bool(np.array_equal(r["triangles"], o["ntri"][keep])),
            "max_err_over_A": worst, "tau": TAU, "parity_ok": ok}


def reference_check(eng, bk, c, cs, tsum, nsample=24, seed=0):
    """T_F of a sample of triples recomputed in float64 with torch from the same complex field."""
    N = eng.N
    k = torch.as_tensor(tables.k_axis(N, L), device="cuda")
    k2 = (k[:, None, None] ** 2 + k[None, :, None] ** 2) + k[None, None, :N // 2 + 1] ** 2
    e2 = torch.as_tensor(bk.edges ** 2, device="cuda")
    shell = torch.bucketize(k2, e2, right=True) - 1
    shell[0, 0, 0] = -1
    ph = torch.as_tensor(tables.interlace_phase_axis(N, L), device="cuda")
    phase = torch.exp(1j * ((ph[:, None, None] + ph[None, :, None]) + ph[None, None, :N // 2 + 1]))
    comp = torch.as_tensor(tables.compensation_axis("tsc", True, N), device="cuda")
    cf = (0.5 * (c.to(torch.complex128) + cs.to(torch.complex128) * phase)
          / (comp[:, None, None] * comp[None, :, None] * comp[None, None, :N // 2 + 1]))
    del phase
    rng = np.random.default_rng(seed)
    pick = rng.choice(len(bk.triples), size=min(nsample, len(bk.triples)), replace=False)
    need = sorted({int(b) for t in bk.triples[pick] for b in t})
    F = {}
    for b in need:
        F[b] = torch.fft.irfftn(torch.where(shell == b, cf, 0), s=(N, N, N)) * float(N) ** 3
    worst = 0.0
    for t in pick:
        i, j, l = (int(v) for v in bk.triples[t])
        prod = F[i] * F[j] * F[l]
        ref, A = float(prod.sum()), float(prod.abs().sum())
        if A > 0:
            worst = max(worst, abs(float(tsum[t]) - ref) / A)
    return {"sampled_triples": int(len(pick)), "max_err_over_A": worst, "ok": worst <= TAU}


def timed(config, N, dk_f, iters):
    dk = dk_f * 2 * np.pi / L
    cols, mesh = mesh_of(N)
    eng = mesh._eng
    (c, cs), s, comp = mesh._complex_fields()
    del cols
    bk = eng.bispec_binning(0.0, dk, None, comp, True)
    scratch = torch.empty(bk.scratch_bytes, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    eng.bispec_counts(bk, scratch)
    torch.cuda.synchronize()
    count_ms = (time.perf_counter() - t0) * 1e3
    eng.enable_timing(True)
    first = eng.bispec_raw(bk, scratch, c, cs).clone()          # warm-up
    eng.bispec_raw(bk, scratch, c, cs)
    torch.cuda.synchronize()
    stages = []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    last = None
    for _ in range(iters):
        last = eng.bispec_raw(bk, scratch, c, cs)
        stages.append(eng.last_bispec_ms(bk))
    ev1.record()
    torch.cuda.synchronize()
    call_ms = ev0.elapsed_time(ev1) / iters
    eng.enable_timing(False)
    same = bool(torch.equal(first, last))
    tsum = last.cpu().numpy()
    del scratch
    torch.cuda.empty_cache()
    check = reference_check(eng, bk, c, cs, tsum)
    ms = {key: float(np.mean([st[key] for st in stages])) for key in stages[0]}
    kept = len(bk.triples)
    flop = 2.0 * kept * float(N) ** 3
    nb = len(bk.edges) - 1
    return {"config": config, "N": N, "particles": N ** 3, "dk_kf": dk_f, "shells": nb,
            "triples_all": nb * (nb + 1) * (nb + 2) // 6, "triples_kept": kept,
            "scratch_GB": bk.scratch_bytes / 1e9, "f32_fields_GB": 4.0 * nb * N * N * (N + 2) / 1e9,
            "f64_fields_GB": 8.0 * nb * N * N * (N + 2) / 1e9, "stage_ms": ms, "call_ms": call_ms,
            "count_once_ms": count_ms, "iters": iters, "useful_TFLOP": flop / 1e12,
            "reduce_TFLOPs": flop / (ms["reduce"] * 1e-3) / 1e12, "deterministic": same, "reference": check,
            "count_residual": bk.residual}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default="BK0,BK1,BK2")
    ap.add_argument("--iters", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bispec_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    info = card()
    out = {"card": info, "runs": []}
    want = a.only.split(",")
    if "BK0" in want:
        out["runs"].append(bk0())
        print(json.dumps(out["runs"][-1]), flush=True)
    for cfg, N, dkf in (("BK1", 256, 2), ("BK2", 512, 4)):
        if cfg in want:
            r = timed(cfg, N, dkf, a.iters)
            info2 = card()
            fma_bound = info["sms"] * 128 * 2 * info2["sm_clock_MHz_max"] * 1e6 / 1e12
            r["sm_clock_MHz_after"] = info2["sm_clock_MHz_now"]
            r["fp32_fma_bound_TFLOPs"] = fma_bound
            r["reduce_fraction_of_fma_bound"] = r["reduce_TFLOPs"] / fma_bound
            out["runs"].append(r)
            print(json.dumps(r), flush=True)
            ab.engine.clear_engines()
            torch.cuda.empty_cache()
    print(json.dumps({"card": info}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
