"""Taylor-Fourier mesh measurements on one GPU (TaylorFourierMesh, astrild_b200/csrc/tf.cu).  One run does everything:

  TF1  512^3 Zel'dovich particles on a 512^3 mesh, order 3;
  TF2  bench.py's config-3 set (1024^3 Zel'dovich particles) on a 512^3 mesh, order 3, at fold 0 and fold 3 (POWMES'
       grid).

For each: the TF field's stages (partition, moment tiles, r2c, combine: apk_tf_last_ms, CUDA events, mean over the
timed calls after warm-up), the combine's fraction of the 6535.4 GB/s HBM copy bandwidth (BASELINE.md) on algorithmic
bytes (it reads the pass's transformed moments, 8 N^2 (N/2 + 1) bytes each, and writes the output once, reading it
too on later passes), and two end-to-end times with CUDA events around the whole call: FFTPower(TaylorFourierMesh) and
FFTPower(CatalogMesh(TSC, interlaced, compensated)) on the same particles, with their ratio.  The two spectra are
compared below half the Nyquist frequency as a sanity figure.  The card's name, power limit and SM clock are read with
queries only, in the same run.

    python tools/tf_bench.py [--out profiles/r06_tf_b200.json] [--only TF1,TF2] [--iters 5]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import astrild_b200 as ab  # noqa: E402
from astrild_b200 import synthetic  # noqa: E402

HBM_GBs = 6535.4      # BASELINE.md: HBM copy bandwidth measured on a B200
L = 1000.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    name, plim, sm, smmax = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit_W": float(plim), "sm_clock_MHz_now": float(sm), "sm_clock_MHz_max": float(smmax)}


def event_ms(fn, iters):
    """mean ms of fn() between CUDA events (fn's own host synchronisations included), after one warm-up call"""
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = []
    for _ in range(iters):
        a.record()
        res = fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return float(np.mean(out)), float(np.min(out)), res


def measure(cols, N, fold, iters, name, nparticles):
    tfm = ab.TaylorFourierMesh(cols, L, N, order=3, fold=fold, pos_scale=1.0)
    eng = tfm._eng
    tp = eng.tf_plan(3)
    pos_scale = 2.0 ** fold
    out = eng.new_mesh()
    group = tp.nmom
    scratch = torch.empty(eng.tf_scratch_bytes(tp, group), dtype=torch.uint8, device="cuda")
    eng.enable_timing(True)
    for _ in range(2):
        eng.tf_field(tp, cols, None, pos_scale, group=group, out=out, scratch=scratch)
    torch.cuda.synchronize()
    stages = []
    for _ in range(iters):
        eng.tf_field(tp, cols, None, pos_scale, group=group, out=out, scratch=scratch)
        stages.append(eng.last_tf_ms(tp))
    eng.enable_timing(False)
    torch.cuda.synchronize()
    del scratch, out
    ms = {k: float(np.mean([s[k] for s in stages])) for k in stages[0]}
    # passes of `group` moments (the last one may be shorter); each pass walks the payload once per 8 moment tiles,
    # and its combine reads the pass's transformed moments and writes the output (reading it too after the first pass)
    half = 8.0 * N * N * (N // 2 + 1)
    sizes = [min(group, tp.nmom - k0) for k0 in range(0, tp.nmom, group)]
    npass = len(sizes)
    comb_bytes = tp.nmom * half + npass * half + (npass - 1) * half
    r = {"config": name, "N": N, "particles": nparticles, "order": 3, "fold": fold, "moments": tp.nmom, "group": group,
         "tile_walks": sum(-(-g // 8) for g in sizes), "stage_ms": ms, "field_ms": sum(ms.values()), "iters": iters,
         "combine_GB": comb_bytes / 1e9, "combine_fraction_of_hbm": comb_bytes / (ms["combine"] * 1e-3) / 1e9 / HBM_GBs,
         "r2c_ms_each": ms["r2c"] / tp.nmom}
    t_tf, t_tf_min, p_tf = event_ms(lambda: ab.FFTPower(tfm, mode="1d"), iters)
    tsc = ab.CatalogMesh(cols, L, N, resampler="tsc", interlaced=True, compensated=True, normalize=True, pos_scale=1.0,
                         fold=fold)
    t_tsc, t_tsc_min, p_tsc = event_ms(lambda: ab.FFTPower(tsc, mode="1d"), iters)
    k = p_tf.power["k"]
    sel = (p_tf.power["modes"] > 0) & (k > 0) & (k < 0.5 * np.pi * N / (L / 2 ** fold))
    rel = np.abs(p_tf.power["power"].real[sel] / p_tsc.power["power"].real[sel] - 1.0)
    r.update({"fftpower_tf_ms": t_tf, "fftpower_tf_ms_min": t_tf_min, "fftpower_tsc_ms": t_tsc,
              "fftpower_tsc_ms_min": t_tsc_min, "tf_over_tsc": t_tf / t_tsc,
              "tf_vs_tsc_max_rel_diff_below_half_nyquist": float(rel.max()) if rel.size else None,
              "shotnoise": p_tf.attrs["shotnoise"]})
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default="TF1,TF2")
    ap.add_argument("--iters", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tf_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = {"card": card(), "runs": []}
    want = a.only.split(",")
    runs = []
    if "TF1" in want:
        runs.append(("TF1", 512, 7, (0,)))
    if "TF2" in want:
        runs.append(("TF2", 1024, 31337, (0, 3)))
    for name, nside, seed, folds in runs:
        cols = synthetic.zeldovich_particles(nside, L, seed, torch.device("cuda"), rms_cells=1.0)
        for fold in folds:
            r = measure(cols, 512, fold, a.iters, name if len(folds) == 1 else f"{name}-fold{fold}", nside ** 3)
            r["sm_clock_MHz_after"] = card()["sm_clock_MHz_now"]
            out["runs"].append(r)
            print(json.dumps(r), flush=True)
            ab.engine.clear_engines()
            torch.cuda.empty_cache()
        del cols
        torch.cuda.empty_cache()
    print(json.dumps({"card": out["card"]}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
