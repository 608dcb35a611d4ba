"""PkEngine: one mesh geometry on one CUDA device, driving libastrild_pk.so.

PyTorch is used for device memory, streams and host<->device copies only; every number is
produced by the CUDA library.  Reference call sites this engine serves:
  pm.paint / ArrayMesh / FFTPower in
  /root/reference/src/astrild/particles/hutils/stats_subfind.py:125-150 and
  /root/reference/src/astrild/power_spectra/power_spectrum_3d.py:164-226.
"""
from __future__ import annotations

import ctypes as ct
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib, tables
from ._lib import AstrildPkError

_ENGINES: dict = {}


def get_engine(Nmesh: int, BoxSize: float, device=None) -> "PkEngine":
    """Cached engine per (Nmesh, BoxSize, device): plans and buffers are reused across snapshots."""
    dev = _resolve_device(device)
    key = (int(Nmesh), float(BoxSize), dev.index)
    eng = _ENGINES.get(key)
    if eng is None:
        eng = _ENGINES[key] = PkEngine(Nmesh, BoxSize, dev)
    return eng


def clear_engines() -> None:
    for eng in list(_ENGINES.values()):
        eng.close()
    _ENGINES.clear()


def _resolve_device(device) -> torch.device:
    if not torch.cuda.is_available():
        raise AstrildPkError("astrild_b200 needs a CUDA device: there is no CPU fallback for the P(k) path")
    if device is None:
        return torch.device("cuda", torch.cuda.current_device())
    dev = torch.device(device)
    if dev.type != "cuda":
        raise AstrildPkError(f"astrild_b200 runs on CUDA devices only, got {dev}")
    return torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())


def _ptr(t):
    return None if t is None else ct.c_void_p(t.data_ptr())


@dataclass
class Binning:
    handle: ct.c_void_p
    edges: np.ndarray
    key: tuple


@dataclass
class BispecBinning:
    handle: ct.c_void_p
    edges: np.ndarray
    triples: np.ndarray          # (ntriples, 3) int32: the kept (i, j, l), i <= j <= l
    scratch_bytes: int
    key: tuple
    dk: float
    kmax: float
    ntri: np.ndarray | None = None
    residual: float | None = None


@dataclass
class XiBinning:
    handle: ct.c_void_p
    edges: np.ndarray
    muedges: np.ndarray
    ells: tuple
    nmu: int
    scratch_bytes: int
    grid_scale: float            # the output grid holds grid_scale * sum w p e^{ikr} of the un-normalised fields
    key: tuple


@dataclass
class TfPlan:
    handle: ct.c_void_p
    order: int
    nmom: int                    # C(order + 3, 3) moment grids
    key: tuple


@dataclass
class KmuBinning:
    handle: ct.c_void_p
    edges: np.ndarray
    muedges: np.ndarray
    ells: tuple
    key: tuple


class PkEngine:
    def __init__(self, Nmesh: int, BoxSize: float, device=None, x0: int = 0, n0: int | None = None):
        self.lib = _lib.load()
        self.device = _resolve_device(device)
        self.N = int(Nmesh)
        self.L = float(BoxSize)
        self.Nk = self.N // 2 + 1
        self.ldz = 2 * self.Nk
        self.x0 = int(x0)
        self.n0 = self.N if n0 is None else int(n0)
        self._plan = ct.c_void_p()
        with torch.cuda.device(self.device):
            _lib.call("apk_plan_create", ct.byref(self._plan), self.N, self.L, self.x0, self.n0, self.device.index)
        lo, hi = ct.c_int(), ct.c_int()
        _lib.call("apk_plan_ghost_planes", self._plan, ct.byref(lo), ct.byref(hi))
        self.ghost_lo, self.ghost_hi = lo.value, hi.value
        self._workspace = None
        self._binnings: dict = {}
        self._scratch = torch.zeros(8, dtype=torch.float64, device=self.device)
        self.ensure_workspace(0, False)

    # ------------------------------------------------------------------ lifetime
    def close(self) -> None:
        if self._plan:
            for b in self._binnings.values():
                if isinstance(b, BispecBinning):
                    self.lib.apk_bispec_destroy(b.handle)
                elif isinstance(b, XiBinning):
                    self.lib.apk_xi_destroy(b.handle)
                elif isinstance(b, TfPlan):
                    self.lib.apk_tf_destroy(b.handle)
                else:
                    (self.lib.apk_kmu_destroy if isinstance(b, KmuBinning) else self.lib.apk_binning_destroy)(b.handle)
            self._binnings.clear()
            self.lib.apk_plan_destroy(self._plan)
            self._plan = ct.c_void_p()
            self._workspace = None
            self._staging = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream(self):
        return ct.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ buffers
    def new_mesh(self, ghosts: bool = False) -> torch.Tensor:
        """float32 [planes][N][2*(N/2+1)]: the in-place r2c layout (ghost planes for slab deposits)."""
        planes = self.n0 + (self.ghost_lo + self.ghost_hi if ghosts else 0)
        return torch.empty((planes, self.N, self.ldz), dtype=torch.float32, device=self.device)

    def ensure_workspace(self, max_particles: int, with_mass: bool, interlaced: bool = False) -> None:
        need = ct.c_size_t()
        _lib.call("apk_plan_workspace_bytes", self._plan, int(max_particles), int(with_mass), int(interlaced),
                  ct.byref(need))
        if self._workspace is None or self._workspace.numel() < need.value:
            if self._workspace is not None:
                torch.cuda.synchronize(self.device)      # another stream may still be working in the old one
            self._workspace = None
            self._workspace = torch.empty(need.value, dtype=torch.uint8, device=self.device)
            _lib.call("apk_plan_set_workspace", self._plan, _ptr(self._workspace), self._workspace.numel())

    # ------------------------------------------------------------------ per-kernel timing
    timing = False

    def enable_timing(self, on: bool = True) -> None:
        _lib.call("apk_plan_enable_timing", self._plan, int(on))
        self.timing = bool(on)

    def last_deposit_ms(self) -> dict:
        ms = (ct.c_float * 4)()
        _lib.call("apk_plan_last_deposit_ms", self._plan, ms)
        return {"count": ms[0], "scan": ms[1], "scatter": ms[2], "deposit": ms[3]}

    def last_bin_ms(self, binning: "Binning") -> dict:
        ms = (ct.c_float * 2)()
        _lib.call("apk_binning_last_ms", binning.handle, ms)
        return {"bin": ms[0], "fold": ms[1]}

    # ------------------------------------------------------------------ stage 1: deposit
    def _positions(self, pos):
        """-> (p0, p1, p2, layout, dtype, np, keepalive) on this device."""
        if isinstance(pos, (tuple, list)) and len(pos) == 3 and not np.isscalar(pos[0]):
            cols = [self._to_device(c).contiguous() for c in pos]
            if not (cols[0].dtype == cols[1].dtype == cols[2].dtype):
                raise AstrildPkError("SoA position columns must share one dtype")
            if not (cols[0].ndim == 1 and cols[0].shape == cols[1].shape == cols[2].shape):
                raise AstrildPkError("SoA position columns must be 1-D and equally long")
            return cols[0], cols[1], cols[2], _lib.APK_SOA, cols[0].dtype, cols[0].shape[0], cols
        t = self._to_device(pos)
        if t.ndim != 2 or t.shape[1] != 3:
            raise AstrildPkError(f"positions must be (Np, 3) or three (Np,) columns, got shape {tuple(t.shape)}")
        t = t.contiguous()
        return t, None, None, _lib.APK_AOS, t.dtype, t.shape[0], [t]

    def _to_device(self, a) -> torch.Tensor:
        t = a if isinstance(a, torch.Tensor) else torch.as_tensor(np.ascontiguousarray(a))
        if t.dtype not in (torch.float32, torch.float64):
            t = t.to(torch.float64)
        if t.device != self.device:
            t = t.to(self.device, non_blocking=True)
        return t

    def deposit(self, pos, mass=None, resampler: str = "tsc", shift: float = 0.0,
                pos_scale: float | None = None, method: str = "auto", out: torch.Tensor | None = None,
                zero: bool = True) -> torch.Tensor:
        """pm.paint(pos, mass=mass, resampler=resampler) into a float32 mesh (mass per cell).

        pos_scale: grid coordinate g = pos * pos_scale * N; default 1/BoxSize (positions in the
        units of BoxSize); pass 1.0 for Ramses-style [0,1) coordinates.
        """
        rs = _lib.RESAMPLERS.get(str(resampler).lower())
        if rs is None:
            raise AstrildPkError(f"unknown resampler {resampler!r}")
        p0, p1, p2, layout, dt, npart, keep = self._positions(pos)
        m = None
        if mass is not None and not np.isscalar(mass):
            m = self._to_device(mass).contiguous()
            if m.ndim != 1 or m.shape[0] != npart:
                raise AstrildPkError("mass must be a scalar or have one entry per particle")
        slab = self.n0 < self.N
        if out is None:
            out = self.new_mesh(ghosts=slab)
        scalar = float(mass) if (mass is not None and np.isscalar(mass)) else 1.0
        # a scalar weight multiplies what THIS call deposits: when accumulating into a mesh that already holds
        # something, deposit into a scratch mesh first (scaling `out` would rescale its previous content)
        target = out if (zero or scalar == 1.0) else torch.empty_like(out)
        self.ensure_workspace(npart, m is not None)
        _lib.call("apk_deposit", self._plan, _ptr(p0), _ptr(p1), _ptr(p2), layout,
                  _lib.APK_F32 if dt == torch.float32 else _lib.APK_F64,
                  float(1.0 / self.L if pos_scale is None else pos_scale), _ptr(m),
                  _lib.APK_F32 if (m is None or m.dtype == torch.float32) else _lib.APK_F64,
                  int(npart), rs, float(shift), _lib.DEPOSIT_METHODS[method], int(bool(zero) or target is not out),
                  _ptr(target), self.stream)
        if target is not out:
            out.add_(target, alpha=scalar)
        elif scalar != 1.0:
            out.mul_(scalar)
        del keep
        return out

    def deposit_pair(self, pos, mass=None, resampler: str = "tsc", pos_scale: float | None = None,
                     method: str = "auto", out: tuple | None = None, zero: bool = True) -> tuple:
        """The interlaced twins (shift 0 and 0.5) in one call: one brick partition serves both meshes."""
        rs = _lib.RESAMPLERS.get(str(resampler).lower())
        if rs is None:
            raise AstrildPkError(f"unknown resampler {resampler!r}")
        p0, p1, p2, layout, dt, npart, keep = self._positions(pos)
        m = None
        if mass is not None and not np.isscalar(mass):
            m = self._to_device(mass).contiguous()
            if m.ndim != 1 or m.shape[0] != npart:
                raise AstrildPkError("mass must be a scalar or have one entry per particle")
        slab = self.n0 < self.N
        m0, m1 = out if out is not None else (self.new_mesh(ghosts=slab), self.new_mesh(ghosts=slab))
        scalar = float(mass) if (mass is not None and np.isscalar(mass)) else 1.0
        scratch = not zero and scalar != 1.0          # see deposit(): never rescale what the meshes already hold
        t0, t1 = (torch.empty_like(m0), torch.empty_like(m1)) if scratch else (m0, m1)
        self.ensure_workspace(npart, m is not None, True)
        _lib.call("apk_deposit_interlaced", self._plan, _ptr(p0), _ptr(p1), _ptr(p2), layout,
                  _lib.APK_F32 if dt == torch.float32 else _lib.APK_F64,
                  float(1.0 / self.L if pos_scale is None else pos_scale), _ptr(m),
                  _lib.APK_F32 if (m is None or m.dtype == torch.float32) else _lib.APK_F64,
                  int(npart), rs, _lib.DEPOSIT_METHODS[method], int(bool(zero) or scratch), _ptr(t0), _ptr(t1), self.stream)
        if scratch:
            m0.add_(t0, alpha=scalar); m1.add_(t1, alpha=scalar)
        elif scalar != 1.0:
            m0.mul_(scalar); m1.mul_(scalar)
        del keep
        return m0, m1

    def pow2_scaled(self, mass) -> tuple:
        """(mass / 2^e, 2^e) with 2^e the power of two nearest to max |mass| (exact scaling).  Masses in physical
        units (1e10..1e15) would put |field(k)|^2 near the float32 range in the binning kernel; the factor is
        folded back into the host-side scale, or cancels when the field is divided by its mean."""
        m = self._to_device(mass)
        top = float(m.abs().max().item()) if m.numel() else 1.0
        if not np.isfinite(top) or top <= 0.0:
            return m, 1.0
        fac = 2.0 ** round(float(np.log2(top)))
        return (m * (1.0 / fac)).contiguous(), fac

    def _deposit_shifts(self, pos, mass, resampler, shifts, pos_scale, method, meshes, zero):
        if tuple(shifts) == (0.0, 0.5):
            self.deposit_pair(pos, mass, resampler, pos_scale, method, out=(meshes[0], meshes[1]), zero=zero)
        else:
            for mesh, sh in zip(meshes, shifts):
                self.deposit(pos, mass, resampler, sh, pos_scale, method, out=mesh, zero=zero)

    def deposit_many(self, pos, mass=None, resampler: str = "tsc", shifts=(0.0,), pos_scale: float | None = None,
                     method: str = "auto", chunk_rows: int = 1 << 25, out: list | None = None) -> list:
        """One mesh per entry of ``shifts`` (interlacing: (0, 0.5)) from the same particles.

        Device inputs: plain deposits.  HOST inputs (NumPy / CPU tensors): the particles are uploaded
        ONCE, in chunks, on a copy stream, and each chunk is deposited into every mesh while the next
        chunk is in flight -- the end-to-end rate is then the PCIe rate, not PCIe + compute.
        Pinned host memory gives asynchronous copies; pageable memory works but copies synchronously.
        out: meshes to (zero and) fill instead of new ones.  Nothing here waits for the device: a caller that queues
        several sets back to back (catalog.PkBatch) has set i + 1's first chunks in flight under set i's transforms.
        """
        cols = pos if (isinstance(pos, (tuple, list)) and len(pos) == 3 and not np.isscalar(pos[0])) else None
        first = cols[0] if cols is not None else pos
        on_host = not (isinstance(first, torch.Tensor) and first.is_cuda)
        npart = int(first.shape[0])
        meshes = list(out) if out is not None else [self.new_mesh(ghosts=self.n0 < self.N) for _ in shifts]
        if not on_host or npart <= chunk_rows:
            dev = self._positions(pos)           # one upload shared by all shifts
            dpos = (dev[0], dev[1], dev[2]) if dev[3] == _lib.APK_SOA else dev[0]
            dmass = None if (mass is None or np.isscalar(mass)) else self._to_device(mass)
            self._deposit_shifts(dpos, dmass if dmass is not None else mass, resampler, shifts, pos_scale, method,
                                 meshes, True)
            return meshes

        def as_host_tensor(a):
            t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
            return t if t.dtype in (torch.float32, torch.float64) else t.to(torch.float64)

        hcols = [as_host_tensor(c) for c in cols] if cols is not None else [as_host_tensor(pos)]
        hmass = None if (mass is None or np.isscalar(mass)) else as_host_tensor(mass)
        scalar = float(mass) if (mass is not None and np.isscalar(mass)) else 1.0
        srcs = hcols + ([hmass] if hmass is not None else [])
        cur = torch.cuda.current_stream(self.device)
        # Staging buffers, their "free again" events and the copy stream live as long as the engine: a later call (the
        # next snapshot of a batch) starts copying as soon as a buffer's last deposit is done, not when everything
        # queued on `cur` -- the previous snapshot's transforms and binning -- has finished.
        sig = (chunk_rows, tuple((t.dtype, tuple(t.shape[1:])) for t in srcs))
        st = getattr(self, "_staging", None)
        if st is None or st["sig"] != sig:
            copy_stream = torch.cuda.Stream(self.device)
            bufs = [[torch.empty((chunk_rows,) + tuple(t.shape[1:]), dtype=t.dtype, device=self.device) for t in srcs]
                    for _ in range(2)]
            # the allocator may hand out blocks whose last use is still queued on `cur`: order the first copy after
            # it, and tell the allocator that the copy stream uses these blocks
            copy_stream.wait_stream(cur)
            for pair in bufs:
                for buf in pair:
                    buf.record_stream(copy_stream)
            st = self._staging = {"sig": sig, "stream": copy_stream, "bufs": bufs, "free": [None, None],
                                  "ready": [torch.cuda.Event() for _ in range(2)]}
        copy_stream, bufs, ready, free = st["stream"], st["bufs"], st["ready"], st["free"]
        self.ensure_workspace(chunk_rows, hmass is not None, len(shifts) == 2)
        for c, a in enumerate(range(0, npart, chunk_rows)):
            b = min(a + chunk_rows, npart)
            s = c & 1
            with torch.cuda.stream(copy_stream):
                if free[s] is not None:
                    copy_stream.wait_event(free[s])
                for buf, src in zip(bufs[s], srcs):
                    buf[: b - a].copy_(src[a:b], non_blocking=True)
                ready[s].record(copy_stream)
            cur.wait_event(ready[s])
            part = [buf[: b - a] for buf in bufs[s]]
            ppos = tuple(part[:3]) if cols is not None else part[0]
            pm = part[-1] if hmass is not None else None         # a scalar weight is applied once, after the loop
            self._deposit_shifts(ppos, pm, resampler, shifts, pos_scale, method, meshes, c == 0)
            free[s] = torch.cuda.Event()
            free[s].record(cur)
        cur.wait_stream(copy_stream)
        if scalar != 1.0:
            for mesh in meshes:
                mesh.mul_(scalar)
        return meshes

    # ------------------------------------------------------------------ stage 1': ArrayMesh
    def load_mesh(self, array, subtract_mean: bool = True, out: torch.Tensor | None = None) -> torch.Tensor:
        """Gridded field [n0][N][N] (float32/float64, host or device) -> float32 mesh.

        The mean is removed in float64 before the cast: it only feeds the k = 0 mode, which
        FFTPower zeroes, and removing it keeps the single-precision FFT clean of DC leakage.
        """
        t = self._to_device(array).contiguous()
        if tuple(t.shape) != (self.n0, self.N, self.N):
            raise AstrildPkError(f"value_map must have shape {(self.n0, self.N, self.N)}, got {tuple(t.shape)}")
        dt = _lib.APK_F32 if t.dtype == torch.float32 else _lib.APK_F64
        if out is None:
            out = self.new_mesh()
        mean = 0.0
        if subtract_mean:
            _lib.call("apk_mesh_sum", self._plan, _ptr(t), dt, _ptr(self._scratch), self.stream)
            mean = float(self._scratch[0].item()) / (self.n0 * self.N * self.N)
        _lib.call("apk_load_mesh", self._plan, _ptr(t), dt, mean, _ptr(out), self.stream)
        return out

    def mesh_sum(self, mesh: torch.Tensor, out: torch.Tensor | None = None):
        """float64 sum over the real cells of a mesh (sum of deposited mass).  out: a float64 device tensor whose first
        element receives the sum WITHOUT a host synchronisation (returned as is); default: the Python float."""
        view = mesh[self.ghost_lo:self.ghost_lo + self.n0] if mesh.shape[0] != self.n0 else mesh
        _lib.call("apk_padded_mesh_sum", self._plan, _ptr(view), _ptr(self._scratch if out is None else out), self.stream)
        return float(self._scratch[0].item()) if out is None else out

    def store_mesh(self, mesh: torch.Tensor, scale: float = 1.0) -> torch.Tensor:
        """mesh -> contiguous float64 [n0][N][N] * scale (what paint(...).value holds)."""
        out = torch.empty((self.n0, self.N, self.N), dtype=torch.float64, device=self.device)
        _lib.call("apk_store_mesh", self._plan, _ptr(mesh), float(scale), _ptr(out), self.stream)
        return out

    # ------------------------------------------------------------------ stage 2: r2c
    def r2c(self, mesh: torch.Tensor) -> torch.Tensor:
        """In-place un-normalised r2c; returns the complex64 [N][N][N/2+1] view of the same memory."""
        if self.n0 != self.N:
            raise AstrildPkError("r2c on a slab engine: use astrild_b200.distributed")
        _lib.call("apk_fft_r2c", self._plan, _ptr(mesh), self.stream)
        return torch.view_as_complex(mesh.view(self.N, self.N, self.Nk, 2))

    # ------------------------------------------------------------------ stage 3: binning
    def binning(self, kmin: float = 0.0, dk: float | None = None, kmax: float | None = None,
                compensation: tuple | None = None, interlaced: bool = False, k_dtype=np.float64,
                axes=None) -> Binning:
        """Binning tables for FFTPower(mode='1d', kmin, dk, kmax).

        compensation: None or (resampler, interlaced_flag) selecting nbodykit's Compensate* factor.
        axes: None for the single-GPU [x][y][z] grid, or (a_index_array, b_index_array, dc_a, dc_b,
        n_a, n_b, ka, kb) for a transposed slab (see distributed.py).
        """
        key = (float(kmin), dk, kmax, compensation, bool(interlaced), np.dtype(k_dtype).str,
               None if axes is None else axes["key"])
        b = self._binnings.get(key)
        if b is not None:
            return b
        N, L = self.N, self.L
        kfull = tables.k_axis(N, L, k_dtype)
        edges = tables.k_edges(N, L, kmin, dk, kmax)
        if len(edges) < 2:
            raise AstrildPkError("binning needs at least two k edges")
        kz = np.ascontiguousarray(kfull[: self.Nk])
        wz = np.ascontiguousarray(tables.hermitian_weights(N))
        if axes is None:
            ia = ib = np.arange(N)
        else:
            ia, ib = axes["ia"], axes["ib"]
        ka = np.ascontiguousarray(kfull[ia])
        kb = np.ascontiguousarray(kfull[ib])
        dc_a = int(np.flatnonzero(ia == 0)[0]) if (ia == 0).any() else -1
        dc_b = int(np.flatnonzero(ib == 0)[0]) if (ib == 0).any() else -1
        comp = [None] * 3
        if compensation is not None:
            c = tables.compensation_axis(compensation[0], bool(compensation[1]), N)
            comp = [np.ascontiguousarray(c[ia]), np.ascontiguousarray(c[ib]), np.ascontiguousarray(c[: self.Nk])]
        ph = [None] * 3
        if interlaced:
            p = tables.interlace_phase_axis(N, L)
            ph = [np.ascontiguousarray(p[ia]), np.ascontiguousarray(p[ib]), np.ascontiguousarray(p[: self.Nk])]

        def hp(a):
            return None if a is None else a.ctypes.data_as(ct.c_void_p)

        handle = ct.c_void_p()
        _lib.call("apk_binning_create", ct.byref(handle), self._plan, len(ka), len(kb), len(kz),
                  hp(ka), hp(kb), hp(kz), hp(wz), hp(edges), len(edges),
                  hp(comp[0]), hp(comp[1]), hp(comp[2]), hp(ph[0]), hp(ph[1]), hp(ph[2]), dc_a, dc_b)
        b = Binning(handle, edges, key)
        self._binnings[key] = b
        return b

    # ------------------------------------------------------------------ stage 3': (k, mu) binning and multipoles
    def kmu_binning(self, kmin: float = 0.0, dk: float | None = None, kmax: float | None = None, Nmu: int = 5, poles=(),
                    los=(0.0, 0.0, 1.0), compensation: tuple | None = None, interlaced: bool = False, k_dtype=np.float64,
                    axes=None):
        """Tables for FFTPower(mode='2d', Nmu=, poles=, los=) (row N4) -> KmuBinning.  axes: as in ``binning`` (the
        transposed slab of the multi-GPU path: all x, this rank's y)."""
        ells = tuple(sorted(set([0] + [int(e) for e in poles])))
        key = ("kmu", float(kmin), dk, kmax, int(Nmu), ells, tuple(float(x) for x in los), compensation, bool(interlaced),
               np.dtype(k_dtype).str, None if axes is None else axes["key"])
        got = self._binnings.get(key)
        if got is not None:
            return got
        N, L = self.N, self.L
        kfull = tables.k_axis(N, L, k_dtype)
        edges = tables.k_edges(N, L, kmin, dk, kmax)
        if len(edges) < 2:
            raise AstrildPkError("binning needs at least two k edges")
        ia = np.arange(N) if axes is None else axes["ia"]
        ib = np.arange(N) if axes is None else axes["ib"]
        ka, kb_ = np.ascontiguousarray(kfull[ia]), np.ascontiguousarray(kfull[ib])
        kz = np.ascontiguousarray(kfull[: self.Nk])
        wz = np.ascontiguousarray(tables.hermitian_weights(N))
        dc_a = int(np.flatnonzero(ia == 0)[0]) if (ia == 0).any() else -1
        dc_b = int(np.flatnonzero(ib == 0)[0]) if (ib == 0).any() else -1
        comp, ph = [None] * 3, [None] * 3
        if compensation is not None:
            c = tables.compensation_axis(compensation[0], bool(compensation[1]), N)
            comp = [np.ascontiguousarray(c[ia]), np.ascontiguousarray(c[ib]), np.ascontiguousarray(c[: self.Nk])]
        if interlaced:
            p = tables.interlace_phase_axis(N, L)
            ph = [np.ascontiguousarray(p[ia]), np.ascontiguousarray(p[ib]), np.ascontiguousarray(p[: self.Nk])]
        ea = np.asarray(ells, dtype=np.int32)
        la = np.asarray(los, dtype=np.float64)

        def hp(a):
            return None if a is None else a.ctypes.data_as(ct.c_void_p)

        handle = ct.c_void_p()
        _lib.call("apk_kmu_create", ct.byref(handle), self._plan, len(ka), len(kb_), self.Nk, hp(ka), hp(kb_), hp(kz), hp(wz),
                  hp(edges), len(edges), int(Nmu), hp(ea), len(ells), hp(la), hp(comp[0]), hp(comp[1]), hp(comp[2]),
                  hp(ph[0]), hp(ph[1]), hp(ph[2]), dc_a, dc_b)
        got = KmuBinning(handle, edges, np.linspace(0.0, 1.0, int(Nmu) + 1), ells, key)
        self._binnings[key] = got
        return got

    def bin_kmu_raw(self, kb: "KmuBinning", c1, c1s=None, c2=None, c2s=None) -> torch.Tensor:
        """Raw sums on the device: float64 [3 + 2 nell][(nedges + 1) (Nmu + 2)] = xsum, musum, nsum (int64 bits),
        ysum_re[nell], ysum_im[nell]."""
        nb = (len(kb.edges) + 1) * (len(kb.muedges) + 1)
        nell = len(kb.ells)
        out = torch.empty((3 + 2 * nell, nb), dtype=torch.float64, device=self.device)
        _lib.call("apk_kmu_bin", kb.handle, _ptr(c1), _ptr(c1s), _ptr(c2), _ptr(c2s), _ptr(out[0]), _ptr(out[1]),
                  _ptr(out[3]), _ptr(out[3 + nell]), _ptr(out[2]), self.stream)
        return out

    @staticmethod
    def finish_kmu(host: np.ndarray, nsum: np.ndarray, kb: "KmuBinning", scale: float) -> dict:
        """Sums -> (k, mu) spectrum and multipoles with nbodykit's conventions (project_to_basis tail): ``k``, ``mu``,
        ``power`` (complex), ``modes`` of shape (Nk, Nmu) and ``poles`` = {"k", "modes", "power_<ell>"}.
        host: float64 [3 + 2 nell][nb] (row 2 ignored), nsum: int64 [nb]."""
        nk1, nm2, nell = len(kb.edges) + 1, len(kb.muedges) + 1, len(kb.ells)
        xsum, musum = host[0].reshape(nk1, nm2), host[1].reshape(nk1, nm2)
        nsum = nsum.reshape(nk1, nm2)
        ysum = (host[3:3 + nell] + 1j * host[3 + nell:3 + 2 * nell]).reshape(nell, nk1, nm2) * scale
        sl = slice(1, -1)
        with np.errstate(invalid="ignore", divide="ignore"):
            res = {"k": (xsum / nsum)[sl, sl], "mu": (musum / nsum)[sl, sl], "power": (ysum[0] / nsum)[sl, sl],
                   "modes": nsum[sl, sl].copy(), "edges": kb.edges, "muedges": kb.muedges}
            n1 = nsum[sl, sl].sum(axis=-1)
            pol = {"k": xsum[sl, sl].sum(axis=-1) / n1, "modes": n1}
            for i, ell in enumerate(kb.ells):
                pol["power_%d" % ell] = ysum[i][sl, sl].sum(axis=-1) / n1
            res["poles"] = pol
        return res

    def bin_kmu(self, kb: "KmuBinning", c1, c1s=None, c2=None, c2s=None, scale: float = 1.0) -> dict:
        host = self.bin_kmu_raw(kb, c1, c1s, c2, c2s).cpu().numpy()
        return self.finish_kmu(host, host[2].view(np.int64).copy(), kb, scale)

    def bin_power_raw(self, binning: Binning, c1, c1s=None, c2=None, c2s=None) -> torch.Tensor:
        """Raw shell sums on the device: float64 [4][nedges+1] = ksum, psum_re, psum_im, nmodes(int64 bits)."""
        nb1 = len(binning.edges) + 1
        out = torch.empty((4, nb1), dtype=torch.float64, device=self.device)
        _lib.call("apk_bin_power", binning.handle, _ptr(c1), _ptr(c1s), _ptr(c2), _ptr(c2s),
                  _ptr(out[0]), _ptr(out[1]), _ptr(out[2]), _ptr(out[3]), self.stream)
        return out

    @staticmethod
    def finish(raw: torch.Tensor, binning: Binning, scale: float) -> dict:
        """Device sums -> host arrays with nbodykit's conventions (project_to_basis tail)."""
        host = raw.cpu().numpy()
        nsum = host[3].view(np.int64).copy()
        with np.errstate(invalid="ignore", divide="ignore"):
            k = (host[0] / nsum)[1:-1]
            power = ((host[1] + 1j * host[2]) * scale / nsum)[1:-1]
        return {"k": k, "power": power, "modes": nsum[1:-1].copy(), "edges": binning.edges,
                "Nsum": nsum}

    def bin_power(self, binning: Binning, c1, c1s=None, c2=None, c2s=None, scale: float = 1.0) -> dict:
        return self.finish(self.bin_power_raw(binning, c1, c1s, c2, c2s), binning, scale)

    # ------------------------------------------------------------------ bispectrum (FFT estimator)
    def bispec_binning(self, kmin: float = 0.0, dk: float | None = None, kmax: float | None = None,
                       compensation: tuple | None = None, interlaced: bool = False, k_dtype=np.float64) -> "BispecBinning":
        """Shells and kept triples of a bispectrum (apk_bispec_create): dk defaults to 2 pi / L, kmax to (2/3) pi N / L.
        Cached like the other binnings; it owns the triangle counts once ``bispec_counts`` has computed them."""
        if self.n0 != self.N:
            raise AstrildPkError("the bispectrum runs on single-GPU engines only (no slab path)")
        dk = 2 * np.pi / self.L if dk is None else float(dk)
        kmax = 2.0 / 3.0 * np.pi * self.N / self.L if kmax is None else float(kmax)
        key = ("bispec", float(kmin), dk, kmax, compensation, bool(interlaced), np.dtype(k_dtype).str)
        got = self._binnings.get(key)
        if got is not None:
            return got
        rs = 0 if compensation is None else _lib.RESAMPLERS[str(compensation[0]).lower()]
        handle = ct.c_void_p()
        _lib.call("apk_bispec_create", ct.byref(handle), self._plan, float(kmin), dk, kmax,
                  _lib.APK_F32 if np.dtype(k_dtype) == np.float32 else _lib.APK_F64, rs, int(bool(interlaced)))
        try:
            nt = ct.c_int()
            _lib.call("apk_bispec_triples", handle, None, 0, ct.byref(nt))
            ijl = np.zeros((max(nt.value, 1), 3), dtype=np.int32)
            _lib.call("apk_bispec_triples", handle, ijl.ctypes.data_as(ct.c_void_p), nt.value, ct.byref(nt))
            need = ct.c_size_t()
            _lib.call("apk_bispec_scratch_bytes", handle, ct.byref(need))
        except Exception:
            self.lib.apk_bispec_destroy(handle)
            raise
        got = BispecBinning(handle, tables.k_edges(self.N, self.L, kmin, dk, kmax), ijl[:nt.value].copy(), need.value,
                            key, dk, kmax)
        self._binnings[key] = got
        return got

    def bispec_counts(self, bk: "BispecBinning", scratch: torch.Tensor) -> np.ndarray:
        """N_tri per kept triple (int64, host), computed once per binning in float64 on the device."""
        if bk.ntri is None:
            out = torch.empty(max(len(bk.triples), 1), dtype=torch.int64, device=self.device)
            res = ct.c_double()
            _lib.call("apk_bispec_count", bk.handle, _ptr(scratch), scratch.numel(), _ptr(out), ct.byref(res), self.stream)
            bk.ntri = out[:len(bk.triples)].cpu().numpy().copy()
            bk.residual = res.value
        return bk.ntri

    def bispec_raw(self, bk: "BispecBinning", scratch: torch.Tensor, c1, c1s=None) -> torch.Tensor:
        """T_F = sum_x F_i F_j F_l per kept triple, float64 on the device."""
        out = torch.empty(max(len(bk.triples), 1), dtype=torch.float64, device=self.device)
        _lib.call("apk_bispec_measure", bk.handle, _ptr(c1), _ptr(c1s), _ptr(scratch), scratch.numel(), _ptr(out),
                  self.stream)
        return out[:len(bk.triples)]

    def last_bispec_ms(self, bk: "BispecBinning") -> dict:
        ms = (ct.c_float * 4)()
        _lib.call("apk_bispec_last_ms", bk.handle, ms)
        return {"fill": ms[0], "c2r": ms[1], "reduce": ms[2], "fold": ms[3]}

    def bispectrum(self, bk: "BispecBinning", tsum, power: dict, field_scale: float, shot: float) -> dict:
        """Raw sums (device or host) + the 1-D ``bin_power`` result of the same edges -> host arrays, triples with no
        triangle dropped.  B = (L^6 s^3 / N^9) T_F / (N^3 N_tri); Bshot = shot (P1 + P2 + P3) - 2 shot^2 / mean (passed
        in as ``shot`` = (S, mean) or NaN / 0)."""
        t = tsum.cpu().numpy() if isinstance(tsum, torch.Tensor) else np.asarray(tsum, dtype=np.float64)
        ntri = bk.ntri
        keep = ntri > 0
        ijl = bk.triples[keep]
        N, L = float(self.N), self.L
        B = (L ** 6 * field_scale ** 3 / N ** 9) * t[keep] / (N ** 3 * ntri[keep].astype(np.float64))
        k, P = power["k"], power["power"].real
        P1, P2, P3 = P[ijl[:, 0]], P[ijl[:, 1]], P[ijl[:, 2]]
        if isinstance(shot, tuple):
            S, mean = shot
            Bshot = (S * (P1 + P2 + P3) - 2.0 * S * S) / mean
        else:
            Bshot = np.full(len(ijl), float(shot))
        return {"k1": k[ijl[:, 0]], "k2": k[ijl[:, 1]], "k3": k[ijl[:, 2]], "bins": ijl.astype(np.int64), "B": B,
                "triangles": ntri[keep].copy(), "P1": P1, "P2": P2, "P3": P3, "Bshot": Bshot}

    # ------------------------------------------------------------------ correlation function (FFT estimator)
    def xi_binning(self, rmin: float = 0.0, dr: float | None = None, rmax: float | None = None, Nmu: int = 1, poles=(),
                   los=(0.0, 0.0, 1.0), compensation: tuple | None = None, interlaced: bool = False) -> "XiBinning":
        """Edges, (r, mu) bins and the C2R plan of a correlation function (apk_xi_create): dr defaults to L / N, rmax to
        L / 2 + dr / 2.  Nmu == 1 without poles is the 1-D path.  Cached like the other binnings."""
        if self.n0 != self.N:
            raise AstrildPkError("the correlation function runs on single-GPU engines only (no slab path)")
        ells = tuple(sorted(set([0] + [int(e) for e in poles])))
        key = ("xi", float(rmin), None if dr is None else float(dr), None if rmax is None else float(rmax), int(Nmu), ells,
               tuple(float(x) for x in los), compensation, bool(interlaced))
        got = self._binnings.get(key)
        if got is not None:
            return got
        rs = 0 if compensation is None else _lib.RESAMPLERS[str(compensation[0]).lower()]
        ea = np.asarray(ells, dtype=np.int32)
        la = np.asarray(los, dtype=np.float64)
        handle = ct.c_void_p()
        _lib.call("apk_xi_create", ct.byref(handle), self._plan, float(rmin), 0.0 if dr is None else float(dr),
                  0.0 if rmax is None else float(rmax), int(Nmu), ea.ctypes.data_as(ct.c_void_p), len(ells),
                  la.ctypes.data_as(ct.c_void_p), rs, int(bool(interlaced)))
        try:
            n = ct.c_int()
            _lib.call("apk_xi_edges", handle, None, 0, ct.byref(n))
            edges = np.empty(n.value)
            _lib.call("apk_xi_edges", handle, edges.ctypes.data_as(ct.c_void_p), n.value, ct.byref(n))
            need, gs = ct.c_size_t(), ct.c_double()
            _lib.call("apk_xi_scratch_bytes", handle, ct.byref(need))
            _lib.call("apk_xi_grid_scale", handle, ct.byref(gs))
        except Exception:
            self.lib.apk_xi_destroy(handle)
            raise
        got = XiBinning(handle, edges, np.linspace(0.0, 1.0, int(Nmu) + 1), ells, int(Nmu), need.value, gs.value, key)
        self._binnings[key] = got
        return got

    def xi_raw(self, xb: "XiBinning", c1, c1s=None, c2=None, c2s=None, grid: torch.Tensor | None = None,
               scratch: torch.Tensor | None = None) -> tuple:
        """-> (grid, sums): the padded mesh holding xi on the grid (times xb.grid_scale, un-normalised fields) and the raw
        float64 sums [3 + nell][(nedges + 1) (Nmu + 2)] = rsum, musum, count (int64 bits), ysum[ell].  The complex
        fields are read, never modified."""
        if grid is None:
            grid = self.new_mesh()
        if tuple(grid.shape) != (self.N, self.N, self.ldz) or grid.dtype != torch.float32 or not grid.is_contiguous():
            raise AstrildPkError(f"the output grid must be a contiguous float32 mesh {(self.N, self.N, self.ldz)}")
        if scratch is None and xb.scratch_bytes:
            scratch = torch.empty(xb.scratch_bytes, dtype=torch.uint8, device=self.device)
        nb = (len(xb.edges) + 1) * (xb.nmu + 2)
        sums = torch.empty((3 + len(xb.ells), nb), dtype=torch.float64, device=self.device)
        _lib.call("apk_xi_measure", xb.handle, _ptr(c1), _ptr(c1s), _ptr(c2), _ptr(c2s), _ptr(grid), _ptr(scratch),
                  0 if scratch is None else scratch.numel(), _ptr(sums), self.stream)
        return grid, sums

    @staticmethod
    def finish_xi(host: np.ndarray, xb: "XiBinning", scale: float) -> dict:
        """Raw sums (host float64, row 2 int64 bits) -> ``r``, ``corr``, ``modes`` (and ``mu`` for Nmu > 1) of shape
        (Nr, Nmu) and ``poles`` = {"r", "modes", "corr_<ell>"}; scale = s1 s2 / N^6 (the fields' scales)."""
        nr1, nm2 = len(xb.edges) + 1, xb.nmu + 2
        nsum = host[2].view(np.int64).reshape(nr1, nm2)
        xsum, musum = host[0].reshape(nr1, nm2), host[1].reshape(nr1, nm2)
        ysum = host[3:].reshape(-1, nr1, nm2) * scale
        sl = slice(1, -1)
        with np.errstate(invalid="ignore", divide="ignore"):
            res = {"r": (xsum / nsum)[sl, sl], "mu": (musum / nsum)[sl, sl], "corr": (ysum[0] / nsum)[sl, sl],
                   "modes": nsum[sl, sl].copy(), "edges": xb.edges, "muedges": xb.muedges}
            n1 = nsum[sl, sl].sum(axis=-1)
            pol = {"r": xsum[sl, sl].sum(axis=-1) / n1, "modes": n1}
            for i, ell in enumerate(xb.ells[:ysum.shape[0]]):
                pol["corr_%d" % ell] = ysum[i][sl, sl].sum(axis=-1) / n1
            res["poles"] = pol
        return res

    def last_xi_ms(self, xb: "XiBinning") -> dict:
        ms = (ct.c_float * 3)()
        _lib.call("apk_xi_last_ms", xb.handle, ms)
        return {"fill": ms[0], "c2r": ms[1], "bin": ms[2]}

    # ------------------------------------------------------------------ Taylor-Fourier mesh (window-free delta(k))
    def tf_plan(self, order: int = 3) -> "TfPlan":
        """The Taylor-Fourier object of one order (apk_tf_create): coefficient tables w^a / a!.  Cached like the
        binnings and destroyed with the engine."""
        if self.n0 != self.N:
            raise AstrildPkError("the Taylor-Fourier mesh runs on single-GPU engines only (no slab path)")
        order = int(order)
        key = ("tf", order)
        got = self._binnings.get(key)
        if got is not None:
            return got
        handle = ct.c_void_p()
        _lib.call("apk_tf_create", ct.byref(handle), self._plan, order)
        got = TfPlan(handle, order, (order + 1) * (order + 2) * (order + 3) // 6, key)
        self._binnings[key] = got
        return got

    def tf_scratch_bytes(self, tp: "TfPlan", group: int) -> int:
        need = ct.c_size_t()
        _lib.call("apk_tf_scratch_bytes", tp.handle, int(group), ct.byref(need))
        return need.value

    def tf_field(self, tp: "TfPlan", pos, mass=None, pos_scale: float | None = None, group: int | None = None,
                 out: torch.Tensor | None = None, scratch: torch.Tensor | None = None) -> torch.Tensor:
        """c_TF of the particles (apk_tf_field) as the complex64 [N][N][N/2+1] view of a padded mesh (``out`` or a new
        one), un-normalised like ``r2c``'s output.  Host particles are uploaded once.  group: moment meshes per pass
        (default: all of them if they fit in free device memory, else as many as fit)."""
        p0, p1, p2, layout, dt, npart, keep = self._positions(pos)
        m = None
        if mass is not None:
            m = self._to_device(mass).contiguous()
            if m.ndim != 1 or m.shape[0] != npart:
                raise AstrildPkError("mass must have one entry per particle")
        if out is None:
            out = self.new_mesh()
        if tuple(out.shape) != (self.N, self.N, self.ldz) or out.dtype != torch.float32 or not out.is_contiguous():
            raise AstrildPkError(f"the output must be a contiguous float32 mesh {(self.N, self.N, self.ldz)}")
        mesh_bytes = 4 * self.N * self.N * self.ldz
        if group is None:
            free, _total = torch.cuda.mem_get_info(self.device)
            free += torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
            group = max(1, min(tp.nmom, int(free * 0.9) // mesh_bytes))
        need = self.tf_scratch_bytes(tp, group)
        if scratch is None or scratch.numel() < need:
            scratch = torch.empty(need, dtype=torch.uint8, device=self.device)
        self.ensure_workspace(npart, m is not None)
        _lib.call("apk_tf_field", tp.handle, _ptr(p0), _ptr(p1), _ptr(p2), layout,
                  _lib.APK_F32 if dt == torch.float32 else _lib.APK_F64,
                  float(1.0 / self.L if pos_scale is None else pos_scale), _ptr(m),
                  _lib.APK_F32 if (m is None or m.dtype == torch.float32) else _lib.APK_F64, int(npart), int(group),
                  _ptr(scratch), scratch.numel(), _ptr(out), self.stream)
        # self.stream is torch's current stream on self.device, the stream the caching allocator tied `scratch`, `out`
        # and the uploaded particles to: a block freed here is handed out again only to work queued after this call's
        del keep
        return torch.view_as_complex(out.view(self.N, self.N, self.Nk, 2))

    def last_tf_ms(self, tp: "TfPlan") -> dict:
        ms = (ct.c_float * 4)()
        _lib.call("apk_tf_last_ms", tp.handle, ms)
        return {"partition": ms[0], "tiles": ms[1], "r2c": ms[2], "combine": ms[3]}
