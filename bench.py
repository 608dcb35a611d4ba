#!/usr/bin/env python
"""bench.py -- P(k) pipeline throughput (deposit + r2c FFT + shell binning) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3] [--impl ours|reference]
                    [--dump-outputs DIR]

One "step" = one complete P(k) of one synthetic particle set: deposit (sort + tiled deposit;
twice when interlaced), r2c FFT(s), fused binning, result on the host.  Prints ONE JSON line.
--dump-outputs DIR writes the result of the last timed step as DIR/<name>.npy (float64; complex
arrays as <name>_real and <name>_imag).  The inputs are generated from fixed seeds, so two builds
run with the same arguments can be compared output for output.

Workloads (BASELINE.json configs):
  c3  1024^3 Zel'dovich particles, TSC + interlacing + window compensation, 1024^3 mesh  -- the
      configuration the metric is quoted on; the default
  c2  512^3 Zel'dovich particles, CIC, 512^3 mesh
  c1  128^3 uniform particles, CIC, 128^3 mesh (the reference's CPU-runnable case)
Inputs are far larger than L2 (126 MB), so no explicit L2 flush is needed between steps.
"""
from __future__ import annotations

import argparse
import datetime
import json
import math
import os
import signal
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    "c1": dict(n=128, mesh=128, box=1000.0, resampler="cic", interlaced=False, compensated=False, seed=12345,
               kind="uniform", name="c1: 128^3 uniform particles, CIC, 128^3 mesh"),
    "c2": dict(n=512, mesh=512, box=1000.0, resampler="cic", interlaced=False, compensated=False, seed=2024,
               kind="zeldovich", name="c2: 512^3 Zel'dovich particles, CIC, 512^3 mesh"),
    "c3": dict(n=1024, mesh=1024, box=1000.0, resampler="tsc", interlaced=True, compensated=True, seed=31337,
               kind="zeldovich", name="c3: 1024^3 Zel'dovich particles, TSC + interlacing + compensation, 1024^3 mesh"),
}
WORKLOADS["c4"] = dict(WORKLOADS["c3"], halos=10 ** 6, halo_seed=7,
                       name="c4: cross P(k) of 10^6 mass-weighted halos (log-normal masses, drawn from the particles) x 1024^3 "
                            "Zel'dovich particles, TSC + interlacing + compensation, one 1024^3 mesh geometry")
WORKLOADS["c5"] = dict(n=2048, mesh=2048, box=1000.0, resampler="cic", interlaced=False, compensated=False, seed=4242,
                       kind="sine", name="c5: 2048^3 particles (lattice + smooth analytic displacement), CIC, 2048^3 mesh, 8 GPUs")
# diagnostics only (not BASELINE configs): a half-size c3 for profiling, and an incoherent-order c2
WORKLOADS["c3s"] = dict(WORKLOADS["c3"], n=512, mesh=512, name="c3s: 512^3 particles, TSC + interlacing + compensation, 512^3 mesh (profiling)")
WORKLOADS["c4s"] = dict(WORKLOADS["c4"], n=512, mesh=512, halos=125000,
                        name="c4s: cross P(k) of 125000 mass-weighted halos x 512^3 particles, TSC + interlacing + compensation, 512^3 mesh")
WORKLOADS["c2u"] = dict(WORKLOADS["c2"], kind="uniform", name="c2u: 512^3 uniform-random particles (incoherent order), CIC, 512^3 mesh")
METRIC = "P(k) pipeline Mparticles/s (deposit+FFT+binning)"
UNIT = "Mparticles/s"
HBM_PEAK_GBS = 6535.4       # denominator of the roofline fractions: HBM copy bandwidth measured on a B200 (BASELINE.md)


def make_particles(wl: dict, dev, x_planes=None, rank: int = 0, world: int = 1):
    """-> (pos, halos): the workload's particle columns x, y, z (float32, box units [0,1)) on `dev` -- all of them, or
    the lattice planes [a, b) of a slab rank -- and, for the cross-spectrum workloads, (x, y, z, mass) of the halos."""
    from astrild_b200 import synthetic
    n, L = wl["n"], wl["box"]
    if wl["kind"] == "zeldovich":
        pos = synthetic.zeldovich_particles(n, L, wl["seed"], dev, x_planes=x_planes)
    elif wl["kind"] == "sine":
        pos = synthetic.sine_displaced_particles(n, wl["seed"], dev, x_planes=x_planes)
    else:
        pos = synthetic.uniform_particles(n, wl["seed"], dev)
        if world > 1:
            pos = tuple(c[rank::world].contiguous() for c in pos)
    halos = None
    if wl.get("halos"):
        assert x_planes is None, "the halo workloads run on one GPU"
        halos = synthetic.halo_subset(pos, wl["halos"], wl["halo_seed"])
    return pos, halos


def golden_check(wl_key: str, res: dict, rtol: float = 1e-4):
    """Compares a result with tests/golden/<workload>_pk.npz (the ORACLE's P(k) of the same particle set, made by
    tools/make_fixtures.py): mode counts must be equal, <k> within 1e-12, P(k) within rtol per bin.  -> dict or None."""
    path = os.path.join(ROOT, "tests", "golden", f"{wl_key}_pk.npz")
    if not os.path.exists(path):
        return None
    g = np.load(path)
    ok = np.isfinite(g["power"]) & (g["modes"] > 0)
    modes_equal = bool(np.array_equal(np.asarray(res["modes"]), g["modes"]))
    rel = np.abs(np.asarray(res["power"]).real[ok] / g["power"][ok] - 1.0)
    relk = np.abs(np.asarray(res["k"])[ok] / g["k"][ok] - 1.0)
    out = {"fixture": os.path.relpath(path, ROOT), "modes_equal": modes_equal, "max_rel_P": float(rel.max()),
           "max_rel_k": float(relk.max()), "rtol": rtol, "bins": int(ok.sum())}
    out["ok"] = bool(modes_equal and out["max_rel_P"] <= rtol and out["max_rel_k"] <= 1e-12)
    return out


def dump_outputs(res: dict, out_dir: str) -> None:
    """Writes every numeric array of a step's result (k, power, modes, edges, Nsum; the slab path adds total_mass) as
    <out_dir>/<name>.npy in float64, complex arrays as <name>_real and <name>_imag.  A few kB per workload: the result
    has one entry per k shell."""
    os.makedirs(out_dir, exist_ok=True)
    for name, value in res.items():
        a = np.asarray(value)
        if a.dtype.kind not in "biufc":
            continue
        parts = {name + "_real": a.real, name + "_imag": a.imag} if a.dtype.kind == "c" else {name: a}
        for part, arr in parts.items():
            np.save(os.path.join(out_dir, part + ".npy"), arr.astype(np.float64))


# ------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm (oracle restating pmesh/nbodykit) on host cores
# ------------------------------------------------------------------------------------------
def cpu_step(wl: dict, threads: int, sample_particles: int, sample_planes: int, state: dict) -> dict:
    """One bounded sample of the CPU path, scaled to the full workload.  Returns seconds."""
    from oracle import pk_oracle as o, pk_oracle_fast as f
    import scipy.fft as sfft

    n, N, L = wl["n"], wl["mesh"], wl["box"]
    Np = n ** 3
    ns = min(sample_particles, Np)
    if "canvas" not in state:
        state["canvas"] = np.zeros((N, N, N), dtype=np.float64)
    if "pos" not in state:
        state["pos"] = lattice_sample(wl, ns)
    passes = 2 if wl["interlaced"] else 1
    t0 = time.perf_counter()
    for i in range(passes):
        f.paint(state["pos"], None, N, L, wl["resampler"], 0.5 * i, out=state["canvas"], threads=threads)
    t_dep = (time.perf_counter() - t0) * (Np / ns)
    # FFT sample: the 3-D r2c is N planes of 2-D r2c over (y,z) + N*Nk pencils of 1-D c2c along x.
    sp = min(sample_planes, N)
    Nk = N // 2 + 1
    t0 = time.perf_counter()
    c = sfft.rfft2(state["canvas"][:sp], axes=(1, 2), workers=threads)
    t_2d = (time.perf_counter() - t0) * (N / sp)
    pencils = np.ascontiguousarray(np.broadcast_to(c[:1, :sp, :], (N, sp, Nk)))
    t0 = time.perf_counter()
    sfft.fft(pencils, axis=0, workers=threads, overwrite_x=True)
    t_1d = (time.perf_counter() - t0) * (N / sp)
    t_fft = (t_2d + t_1d) * passes
    # binning sample: sp x-planes of the k-grid
    t0 = time.perf_counter()
    if wl["interlaced"]:
        kx, ky, kz = o.k_tables(N, L)
        ph = np.exp(0.5j * (kx[:sp, None, None] + ky[None, :, None] + kz[None, None, :]) * (L / N))
        c = 0.5 * c + 0.5 * c * ph
    if wl["compensated"]:
        w = o.compensation_1d(wl["resampler"], wl["interlaced"], N)
        c = c / (w[:sp, None, None] * w[None, :, None] * w[None, None, :Nk])
    kxs, kys, kzs = o.k_tables(N, L)
    edges = o.k_edges(N, L, 2 * np.pi / L)
    e2 = edges ** 2
    nb = len(edges) + 1
    cc = np.ascontiguousarray(c)

    def work(rng_):
        xs, yr, yi = np.zeros(nb), np.zeros(nb), np.zeros(nb)
        nsum = np.zeros(nb, dtype=np.int64)
        f.lib().orc_bin_power(f._ptr(cc), None, N, f._ptr(kxs), f._ptr(kys), f._ptr(kzs), f._ptr(e2), len(edges),
                              L ** 3, f._ptr(xs), f._ptr(yr), f._ptr(yi), f._ptr(nsum), int(rng_[0]), int(rng_[1]))
        return nsum.sum()

    b = np.linspace(0, sp, max(1, min(threads, sp)) + 1).astype(int)
    if threads == 1:
        work((0, sp))
    else:
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(work, zip(b[:-1], b[1:])))
    t_bin = (time.perf_counter() - t0) * (N / sp)
    return {"deposit": t_dep, "fft": t_fft, "bin": t_bin, "total": t_dep + t_fft + t_bin}


def lattice_sample(wl: dict, ns: int) -> np.ndarray:
    """First ns particles of a lattice-ordered set with rms 1-cell Gaussian displacements: the same
    memory-access coherence as the Zel'dovich workload (uniform sets: uniform random)."""
    n, L = wl["n"], wl["box"]
    rng = np.random.default_rng(wl["seed"])
    if wl["kind"] == "uniform":
        return (rng.random((ns, 3)) * L).astype(np.float32)
    idx = np.arange(ns, dtype=np.int64)
    q = np.stack([idx // (n * n), (idx // n) % n, idx % n], axis=1).astype(np.float64)
    pos = (q + 0.5 + rng.normal(0.0, 1.0, (ns, 3))) / n
    return ((pos - np.floor(pos)) * L).astype(np.float32)


def cpu_sample_desc(wl, sample_particles, sample_planes, threads):
    return (f"deposit of the first {min(sample_particles, wl['n'] ** 3)} particles (lattice order) onto the full {wl['mesh']}^3 f64 mesh "
            f"({threads} thread{'s, x-planes dealt round-robin' if threads > 1 else ''}, scaled to Np); {min(sample_planes, wl['mesh'])} of {wl['mesh']} planes of 2-D r2c + as many "
            f"x-pencil blocks of 1-D c2c (scipy pocketfft f64, {threads} threads, scaled); binning of "
            f"{min(sample_planes, wl['mesh'])} x-planes ({threads} threads, scaled)")


def run_reference(args, wl_key: str) -> None:
    """--impl reference: the reference's own CPU path.  nbodykit/pmesh/pfft are not installable
    here (no MPI/FFTW, no network), so this times the oracle port that restates them."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import pk_oracle_fast as f
    f.build()
    wl = WORKLOADS[wl_key]
    threads = os.cpu_count() or 1
    sp, spl = (1 << 24 if threads >= 4 else 1 << 22), 32
    state: dict = {}
    for _ in range(args.warmup):
        cpu_step(wl, threads, sp, spl, state)
    t0 = time.perf_counter()
    times = [cpu_step(wl, threads, sp, spl, state) for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    tot = sum(t["total"] for t in times)
    Np = wl["n"] ** 3
    N = wl["mesh"]
    value = Np * args.steps / tot / 1e6
    cfg = {"workload": wl["name"], "particles": Np, "mesh": N, "boxsize": wl["box"], "resampler": wl["resampler"],
           "interlaced": wl["interlaced"], "compensated": wl["compensated"],
           "parallelism": "single GPU" if args.gpus == 1 else f"x-slab decomposition over {args.gpus} GPUs",
           "l2": "inputs >> L2 (126 MB): no flush needed"}
    if wl.get("halos"):
        cfg["halos"] = wl["halos"]
    frac = {"particles": min(sp, Np) / Np, "planes": min(spl, N) / N}
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup,
           # one step = one bounded SAMPLE of the workload (wall time below); `value` is the whole workload's
           # throughput extrapolated from it stage by stage (deposit ~ particles, FFT and binning ~ planes)
           "ms_per_step": 1e3 * wall / args.steps, "extrapolated": True, "sample_fraction": frac,
           "ms_per_step_full_workload_extrapolated": 1e3 * tot / args.steps,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
           "data": "synthetic", "config": cfg,
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "extrapolated": True,
                            "sample_fraction": frac, "sample": cpu_sample_desc(wl, sp, spl, threads)},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "stages_s": {k: statistics.mean(t[k] for t in times) for k in ("deposit", "fft", "bin")}}
    print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc = gpu_index, None
        self.path = os.path.join(tempfile.gettempdir(), f"apk_clocks_{os.getpid()}.csv")

    def start(self):
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=self.fh, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict | None:
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.remove(self.path)
        except OSError:
            pass
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
def run_ours(args, wl_key: str) -> None:
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the P(k) path has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cpus = None
    if world > 1:
        # a stuck collective aborts after 3 minutes instead of holding the box (NCCL watchdog)
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
        if os.environ.get("APK_BENCH_NUMA", "1") != "0":
            from astrild_b200.distributed import bind_host_to_gpu
            numa_cpus = bind_host_to_gpu(local_rank)      # before any pinned host buffer exists (host-buffer leg)

    import astrild_b200 as ab

    wl = WORKLOADS[wl_key]
    n, N, L = wl["n"], wl["mesh"], wl["box"]
    Np = n ** 3
    kmin = 2 * np.pi / L
    cross = bool(wl.get("halos"))
    if cross and world > 1:
        raise SystemExit("bench.py: the cross-spectrum workloads (c4) run on one GPU")
    Nh = wl.get("halos", 0)
    n_meshes = 2 if wl["interlaced"] else 1
    halos = None

    if world > 1:
        from astrild_b200 import distributed
        runner = distributed.SlabPk(N, L, resampler=wl["resampler"], interlaced=wl["interlaced"],
                                    compensated=wl["compensated"], device=dev)
        pos, _ = make_particles(wl, dev, x_planes=runner.lattice_planes(n), rank=rank, world=world)
        torch.cuda.empty_cache()

        def step():
            return runner.power(pos, pos_scale=1.0, kmin=kmin, normalize=True)

        def e2e_step(host_pos, host_halos=None):
            return runner.power(tuple(host_pos), pos_scale=1.0, kmin=kmin, normalize=True)
        eng = runner.eng
        binning = None
        runner.profile = True
    else:
        pos, halos = make_particles(wl, dev)
        if args.order != "input":
            if args.order == "cell":
                key = (pos[0] * N).long().clamp_(0, N - 1)
                key = (key * N + (pos[1] * N).long().clamp_(0, N - 1)) * N + (pos[2] * N).long().clamp_(0, N - 1)
                perm = torch.argsort(key)
                del key
            else:
                perm = torch.randperm(pos[0].numel(), device=dev, generator=torch.Generator(device=dev).manual_seed(5))
            pos = tuple(c[perm].contiguous() for c in pos)
            del perm
        torch.cuda.empty_cache()
        eng = ab.get_engine(N, L, dev)
        comp = (wl["resampler"], wl["interlaced"]) if wl["compensated"] else None
        binning = eng.binning(kmin=kmin, compensation=comp, interlaced=wl["interlaced"])
        mesh1 = eng.new_mesh()
        mesh2 = eng.new_mesh() if wl["interlaced"] else None
        hmesh1 = eng.new_mesh() if cross else None
        hmesh2 = eng.new_mesh() if (cross and wl["interlaced"]) else None
        eng.ensure_workspace(Np, False, wl["interlaced"])
        s_matter = N ** 3 / Np                                        # normalize=True, unit masses: W = Np
        stage_ev = []

        def deposit_field(p, m, out1, out2, method):
            if out2 is not None:       # interlaced twins: one shared partition, two tile passes
                eng.deposit_pair(p, m, wl["resampler"], 1.0, method, out=(out1, out2))
            else:
                eng.deposit(p, m, wl["resampler"], 0.0, 1.0, method, out=out1)

        def step(record=None):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if record is not None else None
            if ev: ev[0].record()
            deposit_field(pos, None, mesh1, mesh2, "sorted")
            d1 = eng.last_deposit_ms() if record is not None else None
            s_first = s_matter
            if cross:                  # the halo catalogue: mass-weighted, small -> the library picks the direct-atomic path
                hm, hfac = eng.pow2_scaled(halos[3])
                deposit_field(halos[:3], hm, hmesh1, hmesh2, "auto")
                s_first = N ** 3 / eng.mesh_sum(hmesh1)           # 1 + delta = mesh / mean: the power-of-two mass unit cancels
            if ev: ev[1].record()
            c1 = eng.r2c(mesh1)
            c1s = eng.r2c(mesh2) if mesh2 is not None else None
            h1 = eng.r2c(hmesh1) if cross else None
            h1s = eng.r2c(hmesh2) if hmesh2 is not None else None
            if ev: ev[2].record()
            raw = eng.bin_power_raw(binning, h1, h1s, c1, c1s) if cross else eng.bin_power_raw(binning, c1, c1s)
            if ev: ev[3].record()
            scale = L ** 3 * s_first * s_matter / float(N) ** 6
            res = eng.finish(raw, binning, scale)                    # D2H of the shell sums: the result
            if record is not None:
                b = eng.last_bin_ms(binning)
                rec = {"deposit_stage": ev[0].elapsed_time(ev[1]), "fft": ev[1].elapsed_time(ev[2]),
                       "bin_stage": ev[2].elapsed_time(ev[3]), "bin_kernel": b["bin"], "bin_fold": b["fold"]}
                for k in d1:
                    rec["dep_" + k] = d1[k]
                record.append(rec)
            return res

        def e2e_step(host_pos, host_halos=None):
            kw = dict(resampler=wl["resampler"], interlaced=wl["interlaced"], compensated=wl["compensated"], normalize=True,
                      pos_scale=1.0, device=dev)
            matter = ab.CatalogMesh(tuple(host_pos), L, N, method="sorted", **kw)
            if host_halos is None:
                return ab.FFTPower(matter, mode="1d", kmin=kmin).power
            hal = ab.CatalogMesh(tuple(host_halos[:3]), L, N, weight=host_halos[3], **kw)
            return ab.FFTPower(hal, mode="1d", second=matter, kmin=kmin).power

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---------------- device-resident throughput --------------------------------------------
    eng.enable_timing(True)
    for _ in range(args.warmup):
        res = step()
    sampler = ClockSampler(local_rank)
    records: list = []
    barrier()
    sampler.start()
    t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
    torch.cuda.cudart().cudaProfilerStart()          # `ncu --profile-from-start off` then sees the timed steps only
    t_start.record()
    for _ in range(args.steps):
        res = step(records) if world == 1 else step()
    t_end.record()
    barrier()
    torch.cuda.cudart().cudaProfilerStop()
    ms = t_start.elapsed_time(t_end)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    dep_ms_rank0 = None
    if world > 1:
        try:
            dep_ms_rank0 = eng.last_deposit_ms()                    # own-particle deposit of the last timed step
        except Exception:
            dep_ms_rank0 = None
    # one nvidia-smi query takes 0.2-0.4 s: a few samples need ~1.5 s of load.  If the timed region was shorter,
    # the same step keeps running (untimed) under the sampler.  The count comes from the all-reduced time, so
    # every rank runs the same number of (collective) steps.
    extra_steps = 0
    if ms < 1500.0:
        extra_steps = min(400, int(math.ceil((1500.0 - ms) / max(ms / args.steps, 1e-3))))
    for _ in range(extra_steps):
        step()
    barrier()
    clocks = sampler.stop()
    if clocks is not None:
        clocks["untimed_steps_under_sampler"] = extra_steps
    slab_profile = dict(runner.last_profile) if world > 1 else None
    slab_info = dict(getattr(runner, "last_info", {})) if world > 1 else None
    ms_per_step = ms / args.steps
    value = Np / (ms_per_step * 1e-3) / 1e6
    check = golden_check(wl_key, res)            # the timed path's own result against the oracle's fixture

    # ---------------- routing at its design load (N > 1, after the timed region) ---------------
    routing_stress = None
    if world > 1 and not args.no_routing_stress and hasattr(runner, "routing_stress"):
        routing_stress = runner.routing_stress(pos, pos_scale=1.0, kmin=kmin, seed=1234 + rank)

    # ---------------- end to end through the public API, host buffers ------------------------
    host_pos = [] if args.no_e2e else [torch.empty(c.shape, dtype=c.dtype, pin_memory=True) for c in pos]
    for h, c in zip(host_pos, pos):
        h.copy_(c)
    host_halos = None
    if cross and not args.no_e2e:
        host_halos = [torch.empty(c.shape, dtype=c.dtype, pin_memory=True) for c in halos]
        for h, c in zip(host_halos, halos):
            h.copy_(c)
    h2d = sum(h.numel() * h.element_size() for h in host_pos + (host_halos or []))
    cpu_sp, cpu_planes = 1 << 23, 64
    if world == 1:
        del pos
        torch.cuda.empty_cache()
    e2e_steps = max(1, min(args.steps, 5))
    e2e_s = float("nan")
    e2e_check = None
    if not args.no_e2e:
        e2e_step(host_pos, host_halos)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            pw = e2e_step(host_pos, host_halos)
        barrier()
        e2e_s = (time.perf_counter() - t0) / e2e_steps
        e2e_check = golden_check(wl_key, pw if isinstance(pw, dict) else pw.data)
    # row N2 (one GPU): the same host buffers as a BATCH of snapshots through one plan (astrild_b200.PkBatch) -- results are
    # fetched later, so snapshot i + 1's upload runs under snapshot i's transforms and binning
    e2e_batch = None
    if not args.no_e2e and world == 1 and not cross:
        nsnap = 4
        batch = ab.PkBatch(N, L, resampler=wl["resampler"], interlaced=wl["interlaced"], compensated=wl["compensated"],
                           normalize=True, pos_scale=1.0, kmin=kmin, device=dev, method="sorted")
        batch.run([(0, tuple(host_pos))])
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = batch.run([(i, tuple(host_pos)) for i in range(nsnap)])
        torch.cuda.synchronize()
        bs = (time.perf_counter() - t0) / nsnap
        last = "snap_%d" % (nsnap - 1)
        bcheck = golden_check(wl_key, {"k": got["k"][last], "power": got["P"][last] + got["shotnoise"][last], "modes": got["modes"][last]})
        e2e_batch = {"snapshots": nsnap, "ms_per_snapshot": 1e3 * bs, "value": Np / bs / 1e6, "unit": UNIT,
                     "api": "astrild_b200.PkBatch.run([(snap_nr, host x,y,z pinned), ...])", "check": bcheck}
        del batch
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    nb1 = len(res["edges"]) + 1
    d2h = 4 * nb1 * 8 + 16
    e2e = None if args.no_e2e else {"value": Np / e2e_s / 1e6, "unit": UNIT, "h2d_bytes_per_step": int(h2d * world) if world > 1 else int(h2d),
           "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_s,
           "api": ("astrild_b200.CatalogMesh(host x,y,z pinned) -> FFTPower(mode='1d', kmin=2pi/L)" if world == 1 else
                   "astrild_b200.distributed.SlabPk.power(host x,y,z pinned per rank)"),
           "check": e2e_check}
    if e2e is not None and e2e_batch is not None:
        e2e["batch"] = e2e_batch

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant hand-written kernel ---------------------------
    peak = HBM_PEAK_GBS
    peak_src = "measured HBM copy bandwidth of a B200 (BASELINE.md)"
    traffic = {}
    try:                                            # DRAM bytes per launch from the committed ncu --set full capture
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(wl_key, {})
    except Exception:
        pass
    roofline, stages = None, None
    n_fields = 2 if cross else 1
    if records:
        avg = {k: statistics.mean(r[k] for r in records) for k in records[0]}
        dep_bytes = Np * 12 + 4 * N ** 3                               # per tile-kernel launch
        part_bytes = Np * 12                                           # the partition reads every particle once
        bin_bytes = 8 * N * N * (N // 2 + 1) * n_meshes * n_fields
        fft_bytes = (4 * N ** 3 + 8 * N * N * (N // 2 + 1)) * n_meshes * n_fields
        dep_kernel_ms = avg["dep_deposit"] / n_meshes
        cand = {
            "brick_tile_kernel": (dep_bytes, dep_kernel_ms, dep_kernel_ms * n_meshes),
            "brick_scatter_kernel": (part_bytes, avg["dep_scatter"], avg["dep_scatter"]),
            "bin_power_kernel": (bin_bytes, avg["bin_kernel"], avg["bin_kernel"]),
        }
        if avg.get("dep_count", 0.0) > 0.0:
            cand["brick_count_kernel"] = (part_bytes, avg["dep_count"], avg["dep_count"])
        name = max(cand, key=lambda k: cand[k][2])                     # the kernel with the largest share of the step
        by, t, _ = cand[name]
        roofline = {"bound": "hbm", "kernel": name, "achieved": by / (t * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                    "frac": by / (t * 1e-3) / 1e9 / peak, "traffic": traffic.get(name), "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": by, "ms_per_launch": t,
                    "launches_per_step": n_meshes if name == "brick_tile_kernel" else 1}
        stage_bytes = Np * 12 + 4 * N ** 3 * n_meshes                  # SURVEY 8(d) B_dep of the matter field
        stages = {
            "ms": {k: round(v, 4) for k, v in avg.items()},
            "deposit_stage_GBps": stage_bytes / (avg["deposit_stage"] * 1e-3) / 1e9,
            "deposit_stage_frac": stage_bytes / (avg["deposit_stage"] * 1e-3) / 1e9 / peak,
            "fft_GBps_algorithmic": fft_bytes / (avg["fft"] * 1e-3) / 1e9,
            "bin_kernel_GBps": bin_bytes / (avg["bin_kernel"] * 1e-3) / 1e9,
            "bin_kernel_frac": bin_bytes / (avg["bin_kernel"] * 1e-3) / 1e9 / peak,
            "tile_kernel_GBps": dep_bytes / (dep_kernel_ms * 1e-3) / 1e9,
            "tile_kernel_frac": dep_bytes / (dep_kernel_ms * 1e-3) / 1e9 / peak,
            "kernel_fracs": {k: round(v[0] / (v[1] * 1e-3) / 1e9 / peak, 4) for k, v in cand.items()},
        }

    # ---------------- CPU baseline beside it (rank 0, N = 1 only) ----------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import pk_oracle_fast as f
        f.build()
        t = cpu_step(wl, 1, cpu_sp, cpu_planes, {})     # same sample generator (and prefix) as --impl reference
        cpu = {"value": Np / t["total"] / 1e6, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": cpu_sample_desc(wl, cpu_sp, cpu_planes, 1), "extrapolated": True,
               "sample_fraction": {"particles": min(cpu_sp, Np) / Np, "planes": min(cpu_planes, N) / N},
               "seconds_scaled": {k: round(v, 2) for k, v in t.items()}}

    roofline_nvlink = None
    if world > 1 and dep_ms_rank0 is not None:
        # rank 0's share: its particles and its n0 planes per launch; the tile kernel shares the SMs with the first
        # mesh's FFT / transpose (side stream), so this is its time inside the step, not alone
        np_rank, planes = pos[0].numel(), N // world
        dep_bytes = np_rank * 12 + 4 * planes * N * N
        t = dep_ms_rank0["deposit"] / n_meshes
        roofline = {"bound": "hbm", "kernel": "brick_tile_kernel", "achieved": dep_bytes / (t * 1e-3) / 1e9, "peak": peak,
                    "unit": "GB/s", "frac": dep_bytes / (t * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": dep_bytes, "ms_per_launch": t, "rank": 0,
                    "deposit_kernels_ms_rank0": {k: round(v, 4) for k, v in dep_ms_rank0.items()}}
        # NVLink: bytes this rank sends to its peers per step in the x<->y transposes, over the time of the
        # peer-store kernels (CUDA events on their stream), against 900 GB/s per direction (NVLink 5)
        if slab_info and slab_info.get("transpose_ms"):
            out_bytes = 8 * (N // world) * N * (N // 2 + 1) * (world - 1) / world * n_meshes
            tms = slab_info["transpose_ms"]
            roofline_nvlink = {"bound": "nvlink", "kernel": "transpose_p2p_kernel" if slab_info.get("transpose") == "p2p-store" else "nccl all-to-all",
                               "bytes_out_per_gpu_per_step": out_bytes, "ms_per_step": tms,
                               "achieved": out_bytes / (tms * 1e-3) / 1e9, "peak": 900.0, "unit": "GB/s",
                               "frac": out_bytes / (tms * 1e-3) / 1e9 / 900.0, "peak_source": "NVLink 5 nominal, per direction"}
    # hand-written kernels per step and rank.  1 GPU: partition (scatter), scan x2, one tile kernel per mesh, bin, fold
    # (+ count when the two-pass partition is selected).  Slab path: route (stage, scan, group) + those + the received
    # particles (one RED kernel per mesh) + 2 ghost-plane adds per mesh + one peer-store transpose per mesh.
    kernels_per_step = (4 + n_meshes + 2) if world == 1 else (3 + 4 + n_meshes + 2 + n_meshes + 2 * n_meshes + n_meshes)
    if cross:
        kernels_per_step += n_meshes + 1             # halo catalogue: one direct-atomic kernel per mesh + the mass sum
    config = {"workload": wl["name"], "particles": Np, "mesh": N, "boxsize": L, "resampler": wl["resampler"],
              "interlaced": wl["interlaced"], "compensated": wl["compensated"],
              "parallelism": "single GPU" if world == 1 else f"x-slab decomposition over {world} GPUs",
              "l2": "inputs >> L2 (126 MB): no flush needed"}
    if cross:
        config["halos"] = Nh
    if numa_cpus is not None:
        config["host_cpus_bound_per_rank"] = numa_cpus
    if getattr(args, "order", "input") != "input":
        config["particle_order"] = args.order + " (diagnostic reordering of the set)"
    if world > 1 and slab_info:
        config["transpose"] = slab_info.get("transpose")
        config["critical_path"] = slab_info.get("critical_path")
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32 mesh/FFT, f64 index + shell sums", "data": "synthetic",
           "config": config,
           "clocks": clocks, "e2e": e2e,
           "gpu_launches": kernels_per_step * args.steps * world,
           "gpu_launches_note": "hand-written kernels in the timed region, all ranks: per step and rank brick partition + segment sums + scan "
                                "(shared by the interlaced twins), one tile kernel per mesh, bin + fold"
                                + ("" if world == 1 else "; plus route stage/scan/group, one RED deposit per mesh for the received "
                                   "particles, ghost-plane adds and one peer-store transpose per mesh") +
                                "; cuFFT, NCCL and torch kernels are not counted",
           "roofline": roofline, "stages": stages if world == 1 else {"ms_rank0_last_step": {k: round(v, 3) for k, v in slab_profile.items()}},
           "cpu_baseline": cpu,
           "check": dict(check or {"fixture": None, "ok": None},
                         first_bins_P=[float(x) for x in res["power"].real[:3]], modes0=int(res["modes"][0]))}
    if roofline_nvlink is not None:
        out["roofline_nvlink"] = roofline_nvlink
    if routing_stress is not None:
        out["routing_stress"] = routing_stress
    print(json.dumps(out), flush=True)
    if args.dump_outputs:
        dump_outputs(res, args.dump_outputs)
    if world > 1:
        dist.destroy_process_group()
    bad = [c for c in (check, e2e_check) if c is not None and not c["ok"]]
    if bad:
        sys.stderr.write(f"bench.py: result differs from the oracle fixture: {bad}\n")
        sys.exit(3)


def pick_workload(args) -> str:
    """The workload follows from the arguments alone (not from the device's free memory), so the same arguments always
    run, and --dump-outputs writes, the same computation."""
    if args.workload:
        return args.workload
    if args.impl == "reference":
        return os.environ.get("APK_BENCH_WORKLOAD", "c3")
    return "c3"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (diagnostic runs only)")
    ap.add_argument("--order", default="input", choices=["input", "cell", "random"],
                    help="diagnostic (N = 1): reorder the particle set on the device before the run -- 'cell' = sorted by mesh "
                         "cell (z fastest), 'random' = shuffled; the golden check still applies (P(k) does not depend on order)")
    ap.add_argument("--no-routing-stress", action="store_true", help="N > 1: skip the unsorted-input run after the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm times a sample of the workload, not a whole P(k)")
    # whole-run watchdog: a dead-lock (collectives, device-side barriers) must not hold the GPUs for long
    limit = int(os.environ.get("APK_BENCH_TIME_LIMIT_S", "1500"))
    if limit > 0 and hasattr(signal, "SIGALRM"):
        def _expired(signum, frame):
            sys.stderr.write(f"bench.py: no result after {limit} s -- giving up (rank {os.environ.get('RANK', '0')})\n")
            sys.stderr.flush()
            os._exit(124)
        signal.signal(signal.SIGALRM, _expired)
        signal.alarm(limit)
    wl = pick_workload(args)
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    sys.dont_write_bytecode = True      # the bench writes nothing into the tree it runs from (it may be read-only)
    main()
