"""Correlation-function measurements on one GPU (FFTCorr, astrild_b200/csrc/corr.cu).  One run does everything:

  XI1  512^3 mesh, 512^3 Zel'dovich particles, TSC interlaced compensated, 1-D auto; the timed output grid is checked
       against the float64 oracle (oracle/xi_oracle.py) from the same complex fields, with the tolerance of
       tests/test_gpu_corr.py (|xi - xi_oracle| <= TAU S, S = sum_stored w |p|);
  XI2  1024^3, bench.py's config-3 set (1024^3 particles, TSC interlaced compensated): 1-D, then 2d with poles (0, 2, 4);
  XI3  halo x matter at 1024^3: 10^6 mass-weighted halos (synthetic.halo_subset) crossed with the config-3 matter, 1-D.

For each it prints ms per stage (fill, c2r, bin: apk_xi_last_ms, CUDA events, mean over the timed calls after warm-up)
and the fraction of the 6535.4 GB/s HBM copy bandwidth (BASELINE.md) reached on algorithmic bytes: the fill reads
8 N^2 (N/2 + 1) bytes per input grid and writes that once; the binning reads 4 N^3.  The binning does not read the
points beyond rmax (the corners of the cube, ~48 % at the default rmax = L/2 + dr/2), so its figure is an effective
rate.  The card's name, power limit and SM clock are read with queries only, in the same run.

    python tools/corr_bench.py [--out profiles/r05_corr_b200.json] [--only XI1,XI2,XI3] [--iters 10]
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

TAU = 1e-4            # tests/test_gpu_corr.py
HBM_GBs = 6535.4      # BASELINE.md: HBM copy bandwidth measured on a B200
L = 1000.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True)
    name, plim, sm, smmax = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit_W": float(plim), "sm_clock_MHz_now": float(sm), "sm_clock_MHz_max": float(smmax)}


def catalog(N, seed):
    cols = synthetic.zeldovich_particles(N, L, seed, torch.device("cuda"), rms_cells=1.0)
    return cols, ab.CatalogMesh(cols, L, N, resampler="tsc", interlaced=True, compensated=True, normalize=True,
                                pos_scale=1.0)


def timed(eng, xb, fields, iters):
    c1, c1s, c2, c2s = fields
    grid = eng.new_mesh()
    scratch = torch.empty(max(xb.scratch_bytes, 1), dtype=torch.uint8, device="cuda")
    eng.enable_timing(True)
    for _ in range(2):                                          # warm-up (and the once-per-binning geometry pass)
        eng.xi_raw(xb, c1, c1s, c2, c2s, grid=grid, scratch=scratch)
    torch.cuda.synchronize()
    stages = []
    sums = None
    for _ in range(iters):
        _, sums = eng.xi_raw(xb, c1, c1s, c2, c2s, grid=grid, scratch=scratch)
        stages.append(eng.last_xi_ms(xb))
    eng.enable_timing(False)
    torch.cuda.synchronize()
    ms = {k: float(np.mean([s[k] for s in stages])) for k in stages[0]}
    N = eng.N
    ngrids = 1 + (c1s is not None) + (c2 is not None) + (c2s is not None)
    half = 8.0 * N * N * (N // 2 + 1)
    fill_bytes, bin_bytes = (ngrids + 1) * half, 4.0 * N ** 3
    out = {"stage_ms": ms, "call_ms": sum(ms.values()), "iters": iters, "fill_GB": fill_bytes / 1e9,
           "bin_GB": bin_bytes / 1e9, "fill_fraction_of_hbm": fill_bytes / (ms["fill"] * 1e-3) / 1e9 / HBM_GBs,
           "bin_fraction_of_hbm": bin_bytes / (ms["bin"] * 1e-3) / 1e9 / HBM_GBs,
           "nedges": len(xb.edges), "Nmu": xb.nmu, "ells": list(xb.ells), "scratch_MB": xb.scratch_bytes / 1e6}
    return out, grid, sums


def xi1(iters):
    from oracle import pk_oracle as po
    from oracle import xi_oracle as xo
    N = 512
    _, mesh = catalog(N, 7)
    eng = mesh._eng
    (c, cs), s, comp = mesh._complex_fields()
    xb = eng.xi_binning(compensation=comp, interlaced=True)
    r, grid, _ = timed(eng, xb, (c, cs, None, None), iters)
    # the oracle from the same complex fields (normalised), in float64 on the host
    k1 = po.compensate(po.interlace_combine(c.cpu().numpy().astype(np.complex128) * (s / N ** 3),
                                            cs.cpu().numpy().astype(np.complex128) * (s / N ** 3), N, L), "tsc", True, N)
    p = np.abs(xo.product(k1, None))
    S = float((p * po.hermitian_weights(N)[None, None, :]).sum())
    del p
    want = xo.xi_grid(k1, None, N)
    del k1
    got = grid[..., :N].double().cpu().numpy() / xb.grid_scale * s * s / float(N) ** 6
    err = float(np.abs(got - want).max()) / S
    r.update({"config": "XI1", "N": N, "particles": N ** 3, "max_err_over_S": err, "tau": TAU, "parity_ok": err <= TAU})
    return r


def xi2(iters):
    N = 1024
    _, mesh = catalog(N, 31337)
    eng = mesh._eng
    (c, cs), s, comp = mesh._complex_fields()
    runs = []
    for Nmu, poles in ((1, ()), (5, (0, 2, 4))):
        xb = eng.xi_binning(Nmu=Nmu, poles=poles, compensation=comp, interlaced=True)
        r, _, _ = timed(eng, xb, (c, cs, None, None), iters)
        r.update({"config": "XI2" + ("" if Nmu == 1 else "-poles"), "N": N, "particles": N ** 3})
        runs.append(r)
    return runs


def xi3(iters):
    N = 1024
    cols, matter = catalog(N, 31337)
    hx, hy, hz, hm = synthetic.halo_subset(cols, 10 ** 6, 7)
    halos = ab.CatalogMesh((hx, hy, hz), L, N, weight=hm, resampler="tsc", interlaced=True, compensated=True,
                           normalize=True, pos_scale=1.0)
    eng = matter._eng
    (h, hs), _, comp = halos._complex_fields()
    (c, cs), _, _ = matter._complex_fields()
    xb = eng.xi_binning(compensation=comp, interlaced=True)
    r, _, _ = timed(eng, xb, (h, hs, c, cs), iters)
    r.update({"config": "XI3", "N": N, "particles": N ** 3, "halos": 10 ** 6})
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--only", default="XI1,XI2,XI3")
    ap.add_argument("--iters", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("corr_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    out = {"card": card(), "runs": []}
    want = a.only.split(",")
    for name, fn in (("XI1", xi1), ("XI2", xi2), ("XI3", xi3)):
        if name in want:
            res = fn(a.iters)
            for r in (res if isinstance(res, list) else [res]):
                r["sm_clock_MHz_after"] = card()["sm_clock_MHz_now"]
                out["runs"].append(r)
                print(json.dumps(r), flush=True)
            ab.engine.clear_engines()
            torch.cuda.empty_cache()
    print(json.dumps({"card": out["card"]}))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
