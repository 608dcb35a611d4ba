"""The slice of ``nbodykit.lab`` / ``pmesh.pm`` that astrild's P(k) path uses, on the B200.

astrild does ``from nbodykit.lab import *`` and ``import pmesh`` and then calls exactly
  pmesh.pm.ParticleMesh(Nmesh=[n]*3, BoxSize=L).paint(pos, mass=m, resampler="tsc")
        /root/reference/src/astrild/particles/hutils/stats_subfind.py:130-132
  ArrayMesh(value_map, Nmesh=n, compensated=..., interlaced=..., window=..., BoxSize=L)
        /root/reference/src/astrild/power_spectra/power_spectrum_3d.py:183-188, 197-212
  FFTPower(first, mode="1d", second=..., kmin=2*pi/L) -> r.power["k"|"power"|"modes"], r.power.attrs["shotnoise"]
        /root/reference/src/astrild/power_spectra/power_spectrum_3d.py:189-195, 216-224
Same names, same arguments, same returned arrays; the arithmetic runs in libastrild_pk.so.

Semantics kept from nbodykit (SURVEY.md section 0):
  * ArrayMesh only STORES compensated/interlaced/window in attrs; nothing is deconvolved or
    interlaced for a gridded field, and its shotnoise is 0.
  * CatalogMesh (particles) is where resampler / interlaced / compensated act.
"""
from __future__ import annotations

import numpy as np
import torch

from . import engine as _engine
from ._lib import AstrildPkError


def _box3(BoxSize) -> float:
    b = np.atleast_1d(np.asarray(BoxSize, dtype=np.float64))
    if not np.all(b == b[0]):
        raise AstrildPkError("only cubic boxes are supported (astrild passes a scalar BoxSize)")
    return float(b[0])


def _nmesh(Nmesh) -> int:
    n = np.atleast_1d(np.asarray(Nmesh))
    if not np.all(n == n[0]):
        raise AstrildPkError("only cubic meshes are supported (astrild passes Nmesh=[n]*3 or n)")
    return int(n[0])


class RealField:
    """What ``pm.paint`` returns: ``.value`` is the (N,N,N) float64 array of mass per cell."""

    def __init__(self, eng, mesh, scale: float = 1.0):
        self._eng, self._mesh, self._scale = eng, mesh, scale
        self._value = None

    @property
    def value(self) -> np.ndarray:
        if self._value is None:
            self._value = self._eng.store_mesh(self._mesh, self._scale).cpu().numpy()
        return self._value

    @property
    def device_mesh(self) -> torch.Tensor:
        """The float32 padded device mesh (zero-copy hand-over to ArrayMesh / FFTPower)."""
        return self._mesh

    def __truediv__(self, s):
        return RealField(self._eng, self._mesh, self._scale / float(s))

    def __mul__(self, s):
        return RealField(self._eng, self._mesh, self._scale * float(s))

    __rmul__ = __mul__

    def csum(self) -> float:
        return self._eng.mesh_sum(self._mesh) * self._scale


class ParticleMesh:
    """``pmesh.pm.ParticleMesh(Nmesh=[n]*3, BoxSize=L)`` with ``paint``."""

    def __init__(self, Nmesh, BoxSize=1.0, dtype="f8", resampler="cic", device=None, **_ignored):
        self.Nmesh = np.array([_nmesh(Nmesh)] * 3)
        self.BoxSize = np.array([_box3(BoxSize)] * 3)
        self.resampler = resampler
        self._eng = _engine.get_engine(int(self.Nmesh[0]), float(self.BoxSize[0]), device)

    def paint(self, pos, mass=1.0, resampler=None, hold=False, out=None, shift: float = 0.0,
              method: str = "auto") -> RealField:
        m = None if (np.isscalar(mass) and float(mass) == 1.0) else mass
        mesh = self._eng.deposit(pos, m, resampler or self.resampler, shift=shift, method=method,
                                 out=None if out is None else out.device_mesh, zero=not hold)
        return RealField(self._eng, mesh)


class ArrayMesh:
    """``nbodykit.lab.ArrayMesh(array, BoxSize, **kwargs)``: a gridded field as a mesh source.

    ``array`` may be a NumPy array, a torch tensor, or the RealField that ``paint`` returned
    (possibly divided by dx**3) -- the latter stays on the device.
    """

    def __init__(self, array, BoxSize, comm=None, root=0, device=None, **kwargs):
        self.attrs = dict(kwargs)
        L = _box3(BoxSize)
        self.attrs["BoxSize"] = np.array([L] * 3)
        self._field_scale = 1.0
        if isinstance(array, RealField):
            self._eng = array._eng
            self._real = array
            self._array = None
            N = self._eng.N
            if self._eng.L != L:
                raise AstrildPkError("ArrayMesh BoxSize differs from the ParticleMesh that painted the field")
        else:
            a = array if isinstance(array, torch.Tensor) else np.asarray(array)
            if a.ndim != 3 or not (a.shape[0] == a.shape[1] == a.shape[2]):
                raise AstrildPkError(f"ArrayMesh needs a cubic 3-D array, got shape {tuple(a.shape)}")
            if np.iscomplexobj(a) if not isinstance(a, torch.Tensor) else a.is_complex():
                raise AstrildPkError("complex input to ArrayMesh is not supported on this path")
            N = int(a.shape[0])
            self._eng = _engine.get_engine(N, L, device)
            self._array = a
            self._real = None
        self.attrs["Nmesh"] = np.array([N] * 3)

    # the device mesh ready for the r2c, and the scalar the field must be multiplied by
    def _to_device_mesh(self):
        if self._real is not None:
            # FFT is in place: work on a copy so the painted field stays valid
            return self._real.device_mesh.clone(), self._real._scale
        return self._eng.load_mesh(self._array), 1.0

    def _complex_fields(self):
        mesh, scale = self._to_device_mesh()
        return (self._eng.r2c(mesh), None), scale, None

    shotnoise = 0.0
    N_attr = 0


class CatalogMesh:
    """Particles as a mesh source with nbodykit's CatalogMesh options (SURVEY.md Appendix A.3).

    position: (Np,3) or three (Np,) columns in the units of BoxSize; weight: per-particle mass.
    normalize=True gives 1 + delta (field / mean); normalize=False keeps rho = mass / dx^3,
    which is what astrild's SubFind.power_spectrum feeds to FFTPower.
    """

    def __init__(self, position, BoxSize, Nmesh, weight=None, resampler="cic", interlaced=False,
                 compensated=False, normalize=True, pos_scale=None, device=None, method="auto", fold: int = 0):
        """fold = f > 0: the box is folded f times onto itself, x -> (2^f x) mod L (SURVEY.md 8f row N3; POWMES'
        ``nfoldpow``, /root/reference/configs/powmes.config:8-10, read back at power_spectra/powmes.py:40-61): the mesh
        then covers a box of L / 2^f, the spectrum is sampled at multiples of 2^f k_f up to 2^f times the mesh's
        Nyquist frequency, and its amplitude and shot noise refer to the full volume L^3.  The deposit kernels wrap
        positions any number of (folded) box lengths outside the box, so folding costs nothing extra."""
        self._fold = int(fold)
        if self._fold < 0 or self._fold > 10:
            raise AstrildPkError("fold must be between 0 and 10")
        L = _box3(BoxSize)
        self.attrs = {"BoxSize": np.array([L] * 3), "Nmesh": np.array([_nmesh(Nmesh)] * 3),
                      "resampler": resampler, "interlaced": bool(interlaced), "compensated": bool(compensated),
                      "fold": self._fold}
        self._eng = _engine.get_engine(_nmesh(Nmesh), L / 2 ** self._fold, device)
        self._pos, self._w = position, weight
        # grid coordinate g = pos * pos_scale * N in units of the FOLDED box; an explicit pos_scale is the caller's
        # factor to the full box's [0, 1)
        pos_scale = None if (pos_scale is None and self._fold == 0) else (1.0 / L if pos_scale is None else pos_scale) * 2 ** self._fold
        self._normalize, self._pos_scale, self._method = bool(normalize), pos_scale, method
        if compensated and str(resampler).lower() not in ("cic", "tsc"):
            raise AstrildPkError("compensated=True needs resampler 'cic' or 'tsc'")
        self.shotnoise = 0.0

    def _npart(self) -> int:
        p = self._pos
        first = p[0] if (isinstance(p, (tuple, list)) and len(p) == 3 and not np.isscalar(p[0])) else p
        return int(first.shape[0])

    def _shotnoise(self) -> float:
        """V * W2 / W^2 with W = sum of weights, W2 = sum of squared weights, float64 sums (nbodykit
        CatalogMesh.to_real_field attrs; V / N for unit weights)."""
        V, n, w = float(self.attrs["BoxSize"][0]) ** 3, self._npart(), self._w
        if n == 0:
            return 0.0
        if w is None or np.isscalar(w):
            m = 1.0 if w is None else float(w)
            return V / n if self._normalize else n * m * m / V
        if isinstance(w, torch.Tensor):
            wd = w.double()
            W, W2 = float(wd.sum().item()), float((wd * wd).sum().item())
        else:
            wd = np.asarray(w, dtype=np.float64)
            W, W2 = float(wd.sum()), float((wd * wd).sum())
        if not self._normalize:
            return W2 / V                              # the un-normalised field rho = mass / dx^3: rho_mean^2 times the above
        return V * W2 / (W * W) if W != 0.0 else 0.0

    def _complex_fields(self):
        eng, a = self._eng, self.attrs
        shifts = (0.0, 0.5) if a["interlaced"] else (0.0,)
        w, unit = self._w, 1.0
        if w is not None and not np.isscalar(w) and isinstance(w, torch.Tensor) and w.is_cuda:
            w, unit = eng.pow2_scaled(w)              # device weights: deposit in units of 2^e (exact), see pow2_scaled
        elif w is not None and not np.isscalar(w):
            wa = np.asarray(w)
            top = float(np.abs(wa).max()) if wa.size else 1.0
            if np.isfinite(top) and top > 0.0:
                unit = 2.0 ** round(float(np.log2(top)))
                w = wa * wa.dtype.type(1.0 / unit) if wa.dtype in (np.float32, np.float64) else wa.astype(np.float64) / unit
        meshes = eng.deposit_many(self._pos, w, a["resampler"], shifts, self._pos_scale, self._method)
        mesh, mesh_s = meshes[0], (meshes[1] if a["interlaced"] else None)
        total = eng.mesh_sum(mesh) if self._normalize else None
        if self._normalize:
            scale = eng.N ** 3 / total                # 1 + delta = mesh / mean: the unit cancels
        else:
            scale = unit / (eng.L / eng.N) ** 3 / 8.0 ** self._fold     # rho of the FULL box: 2^3f folded copies overlap
        scale *= 2.0 ** (1.5 * self._fold)            # P refers to the full volume: V = 8^f V_folded (FFTPower uses eng.L^3)
        # nbodykit CatalogMesh attrs (SURVEY.md A.3): shotnoise = V * sum(w^2) / sum(w)^2  (= V / N unweighted)
        self.shotnoise = self._shotnoise()
        c = eng.r2c(mesh)
        cs = eng.r2c(mesh_s) if mesh_s is not None else None
        comp = (str(a["resampler"]).lower(), a["interlaced"]) if a["compensated"] else None
        return (c, cs), scale, comp


class TaylorFourierMesh:
    """Particles as a window-free mesh source: the Taylor-Fourier estimator of Colombi et al. (2009), POWMES' ``norder``.

    ``TaylorFourierMesh(position, BoxSize, Nmesh, weight=None, order=3, normalize=True, fold=0, pos_scale=None,
    device=None)``.  For order n, the moment grids M_alpha[h] = sum_p m_p dx^a dy^b dz^c (h = the particle's nearest grid
    point, d = g - h, |alpha| <= n) are deposited on the device, transformed and combined into
    c_TF(k) = sum_alpha (-i)^|alpha| (wx^a wy^b wz^c / a! b! c!) M^_alpha(k) (w = 2 pi freq_index / N): the DFT of the
    particles themselves up to sum_p |m_p| (|w|_1 / 2)^(n+1) / (n+1)!, with no assignment window to deconvolve and no
    aliasing beyond that.  Order 0 is the NGP paint.  The field has no interlaced twin and no compensation.

    position, weight, normalize, fold and pos_scale are CatalogMesh's: 1 + delta (or rho = mass / dx^3), the box folded
    f times onto itself (x -> 2^f x mod L, the spectrum reaching 2^f times the mesh's Nyquist frequency), amplitude and
    ``shotnoise`` = V sum(w^2) / sum(w)^2 of the full volume.  That Poisson value is what ``attrs`` report; the TF
    estimate's own noise floor differs from it by the factor E|T_n(w.d)|^2 (DESIGN section 10).  Single-GPU meshes only.
    """

    def __init__(self, position, BoxSize, Nmesh, weight=None, order=3, normalize=True, fold: int = 0, pos_scale=None,
                 device=None):
        self._fold = int(fold)
        if self._fold < 0 or self._fold > 10:
            raise AstrildPkError("fold must be between 0 and 10")
        order = int(order)
        if order < 0 or order > 4:
            raise AstrildPkError("order must be between 0 and 4")
        L = _box3(BoxSize)
        self.attrs = {"BoxSize": np.array([L] * 3), "Nmesh": np.array([_nmesh(Nmesh)] * 3), "order": order,
                      "fold": self._fold}
        self._eng = _engine.get_engine(_nmesh(Nmesh), L / 2 ** self._fold, device)
        if self._eng.n0 != self._eng.N:
            raise AstrildPkError("TaylorFourierMesh runs on single-GPU meshes only (no slab path)")
        self._pos, self._w = position, weight
        self._order = order
        self._normalize = bool(normalize)
        self._pos_scale = (1.0 / L if pos_scale is None else pos_scale) * 2 ** self._fold
        self.shotnoise = 0.0

    _npart = CatalogMesh._npart
    _shotnoise = CatalogMesh._shotnoise

    def _complex_fields(self):
        eng = self._eng
        w, unit = self._w, 1.0
        if w is not None and np.isscalar(w):
            unit, w = float(w), None                  # a scalar weight scales the field (it cancels when normalised)
        elif w is not None and isinstance(w, torch.Tensor) and w.is_cuda:
            w, unit = eng.pow2_scaled(w)              # weights in units of 2^e (exact), see PkEngine.pow2_scaled
        elif w is not None:
            wa = np.asarray(w)
            top = float(np.abs(wa).max()) if wa.size else 1.0
            if np.isfinite(top) and top > 0.0:
                unit = 2.0 ** round(float(np.log2(top)))
                w = wa * wa.dtype.type(1.0 / unit) if wa.dtype in (np.float32, np.float64) else wa.astype(np.float64) / unit
        tp = eng.tf_plan(self._order)
        c = eng.tf_field(tp, self._pos, w, self._pos_scale)
        if self._normalize:
            # the k = 0 mode of c_TF is the sum of the moment-0 grid: the deposited mass (in units of `unit`)
            total = float(c[0, 0, 0].real.item())
            scale = eng.N ** 3 / total
        else:
            scale = unit / (eng.L / eng.N) ** 3 / 8.0 ** self._fold
        scale *= 2.0 ** (1.5 * self._fold)
        self.shotnoise = self._shotnoise()
        return (c, None), scale, None


class BinnedStatistic:
    """Minimal stand-in for nbodykit's BinnedStatistic: ``obj["k"]``, ``.attrs``, ``.edges``."""

    def __init__(self, dims, edges, data: dict, attrs: dict):
        self.dims = list(dims)
        self.edges = dict(zip(dims, edges))
        self.data = data
        self.attrs = attrs
        self.shape = tuple(len(e) - 1 for e in edges)
        self.variables = list(data)

    def __getitem__(self, key):
        return self.data[key]

    def __contains__(self, key):
        return key in self.data

    def __iter__(self):
        return iter(self.data)


class FFTPower:
    """``FFTPower(first, mode='1d' | '2d', second=None, Nmu=, poles=, los=, kmin=0., dk=None, kmax=None)``.

    Result in ``self.power`` with variables ``k`` (mean |k| of the modes in the bin, NaN if
    empty), ``power`` (complex; real part is P(k)), ``modes`` (int64) and attrs including
    ``shotnoise``: 0 for ArrayMesh input (astrild's case, SURVEY.md section 0 item 3) and for cross
    spectra, V*sum(w^2)/sum(w)^2 for the auto spectrum of a CatalogMesh (nbodykit semantics).
    """

    def __init__(self, first, mode="1d", Nmesh=None, BoxSize=None, second=None, los=(0, 0, 1),
                 Nmu=None, dk=None, kmin=0.0, kmax=None, poles=None, k_dtype=np.float64):
        if mode not in ("1d", "2d"):
            raise AstrildPkError("mode must be '1d' or '2d'")
        poles = [] if poles is None else [int(e) for e in poles]
        if mode == "1d":
            Nmu = 1                                  # nbodykit: one mu bin over [0, 1]
        elif Nmu is None:
            Nmu = 5
        eng = first._eng
        if second is not None and second is not first and second._eng is not eng:
            raise AstrildPkError("first and second must share Nmesh, BoxSize and device")
        self.first, self.second = first, first if second is None else second
        N, L = eng.N, eng.L
        (c1, c1s), s1, comp1 = first._complex_fields()
        if second is None or second is first:
            c2 = c2s = None
            s2, comp2 = s1, comp1
        else:
            (c2, c2s), s2, comp2 = second._complex_fields()
            if (c1s is None) != (c2s is None):
                raise AstrildPkError("first and second must both be interlaced or both not")
            if comp1 != comp2:
                raise AstrildPkError("first and second must use the same window compensation")
        scale = L ** 3 * s1 * s2 / float(N) ** 6
        res2d = None
        if mode == "2d" or poles:
            # (k, mu) wedges and multipoles (row N4): nbodykit's project_to_basis with Nmu bins of |mu| in [0, 1]
            kb = eng.kmu_binning(kmin, dk, kmax, Nmu, poles, tuple(float(x) for x in los), comp1, c1s is not None, k_dtype)
            res2d = eng.bin_kmu(kb, c1, c1s, c2, c2s, scale)
            edges = kb.edges
            res = {"k": res2d["poles"]["k"], "power": res2d["poles"]["power_0"], "modes": res2d["poles"]["modes"],
                   "Nsum": None}
        else:
            binning = eng.binning(kmin, dk, kmax, comp1, c1s is not None, k_dtype)
            res = eng.bin_power(binning, c1, c1s, c2, c2s, scale)
            edges = binning.edges
        # nbodykit FFTBase._compute_3d_power: shotnoise = first.attrs.get('shotnoise', 0) for an AUTO spectrum, 0 for a
        # cross spectrum; an ArrayMesh carries none (astrild's case: the subtraction at power_spectrum_3d.py:224 is - 0)
        auto = second is None or second is first
        shot = float(getattr(first, "shotnoise", 0.0)) if auto else 0.0
        self.attrs = {"mode": mode, "Nmesh": np.array([N] * 3), "BoxSize": np.array([L] * 3),
                      "dk": 2 * np.pi / L if dk is None else dk, "kmin": kmin, "kmax": kmax,
                      "Nmu": 1, "los": list(los), "poles": [], "volume": L ** 3,
                      "shotnoise": shot, "N1": 0, "N2": 0}
        self.attrs["Nmu"], self.attrs["poles"] = int(Nmu), list(poles)
        if mode == "2d":
            self.power = BinnedStatistic(["k", "mu"], [edges, res2d["muedges"]],
                                         {"k": res2d["k"], "mu": res2d["mu"], "power": res2d["power"],
                                          "modes": res2d["modes"]}, dict(self.attrs))
        else:
            self.power = BinnedStatistic(["k"], [edges], {"k": res["k"], "power": res["power"],
                                                          "modes": res["modes"]}, dict(self.attrs))
        self.poles = None
        if poles:
            data = {"k": res2d["poles"]["k"], "modes": res2d["poles"]["modes"]}
            data.update({"power_%d" % e: res2d["poles"]["power_%d" % e] for e in poles})
            self.poles = BinnedStatistic(["k"], [edges], data, dict(self.attrs))
        self._Nsum = res["Nsum"]

    def run(self):
        return self.power, self.poles


def _free_device_bytes(device) -> int:
    """Bytes a new allocation can get on ``device``: free device memory plus what torch's allocator holds unused."""
    free, _total = torch.cuda.mem_get_info(device)
    return int(free) + int(torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device))


class FFTBispectrum:
    """Bispectrum B(k1, k2, k3) of one field: ``FFTBispectrum(first, kmin=0., dk=None, kmax=None)``.

    ``first`` is a CatalogMesh or an ArrayMesh, as for FFTPower.  Shells are the 1-D bins of the same edges
    (dk = 2 pi / L and kmax = (2/3) pi N / L by default: no triangle is aliased then; kmax may go up to the Nyquist
    wavenumber, and the estimator then also counts triangles that close modulo the grid).  The FFT estimator runs on the
    device: shell fields F_b = c2r of the field masked to shell b, B = V^2 <delta delta delta> =
    (L^6 s^3 / N^9) sum_x F_i F_j F_l / (N^3 N_tri), with N_tri the exact number of ordered triangles (q1, q2, q3) of
    the three shells, computed once in float64 and cached.

    ``self.bispectrum`` is a BinnedStatistic over one ``triangle`` dimension (triples i <= j <= l with at least one
    triangle) with variables ``k1 k2 k3`` (mean |k| of each shell), ``bins`` (i, j, l), ``B``, ``triangles`` (N_tri),
    ``P1 P2 P3`` (the shells' P(k), shot noise not subtracted) and ``Bshot`` = S (P1 + P2 + P3) - 2 S^2 for the
    Poisson shot noise S of the field's P(k) (divided by the mean density for an un-normalised field).  Bshot holds
    for unit or scalar weights; it is 0 for an ArrayMesh and NaN for per-particle weights.  It is reported, never
    subtracted.  Auto-bispectra of single-GPU meshes only; the scratch (the shell fields) must fit in free device
    memory.
    """

    def __init__(self, first, kmin=0.0, dk=None, kmax=None, k_dtype=np.float64, second=None, third=None):
        if (second is not None and second is not first) or (third is not None and third is not first):
            raise AstrildPkError("FFTBispectrum computes auto-bispectra only: cross bispectra are not supported")
        if getattr(first, "_fold", 0):
            raise AstrildPkError("FFTBispectrum does not support folded boxes (fold > 0)")
        eng = first._eng
        if eng.n0 != eng.N:
            raise AstrildPkError("FFTBispectrum runs on single-GPU meshes only (no slab path)")
        N, L = eng.N, eng.L
        (c1, c1s), s, comp = first._complex_fields()
        bk = eng.bispec_binning(kmin, dk, kmax, comp, c1s is not None, k_dtype)
        free = _free_device_bytes(eng.device)
        if bk.scratch_bytes > free:
            raise AstrildPkError(
                f"FFTBispectrum needs {bk.scratch_bytes} bytes of device scratch for {len(bk.edges) - 1} shell fields, "
                f"{free} are free: use a larger dk (fewer shells) or a smaller kmax")
        scratch = torch.empty(bk.scratch_bytes, dtype=torch.uint8, device=eng.device)
        eng.bispec_counts(bk, scratch)
        tsum = eng.bispec_raw(bk, scratch, c1, c1s)
        binning = eng.binning(kmin, bk.dk, bk.kmax, comp, c1s is not None, k_dtype)
        power = eng.bin_power(binning, c1, c1s, None, None, L ** 3 * s * s / float(N) ** 6)
        del scratch
        if isinstance(first, (CatalogMesh, TaylorFourierMesh)):
            w = first._w
            S = float(first.shotnoise)
            if w is not None and not np.isscalar(w):
                shot = float("nan")
            else:
                m = 1.0 if w is None else float(w)
                mean = 1.0 if first._normalize else first._npart() * m / L ** 3
                shot = (S, mean)
        else:
            S, shot = 0.0, 0.0
        res = eng.bispectrum(bk, tsum, power, s, shot)
        self.first = first
        self.attrs = {"edges": bk.edges, "Nmesh": np.array([N] * 3), "BoxSize": np.array([L] * 3), "shotnoise": S,
                      "kmin": kmin, "dk": bk.dk, "kmax": bk.kmax, "volume": L ** 3,
                      "count_residual": bk.residual}
        ntr = len(res["B"])
        self.bispectrum = BinnedStatistic(["triangle"], [np.arange(ntr + 1)], res, dict(self.attrs))

    def run(self):
        return self.bispectrum


class FFTCorr:
    """Two-point correlation function: ``FFTCorr(first, mode='1d' | '2d', Nmesh=None, BoxSize=None, second=None,
    los=[0, 0, 1], Nmu=5, dr=None, rmin=0., rmax=None, poles=[])`` (nbodykit's signature).

    The FFT estimator, the configuration-space twin of FFTPower on the same fields: with p = c1 conj(c2) (k = 0 zeroed)
    xi(r) = Re sum_k w(k) p(k) e^{i k.r} over the stored half grid with FFTPower's Hermitian weights, i.e.
    <delta1(x + r) delta2(x)> for normalised fields (rho_mean^2 xi for un-normalised ones); r = x1 - x2.  Binned on the
    real grid with nbodykit's project_to_basis conventions: every grid point has weight 1, edges
    ``arange(rmin, rmax, dr)`` with dr = L / N and rmax = L / 2 + dr / 2 by default, mu = (r . los) / |r|, wedges of |mu|
    and multipoles (2 ell + 1) L_ell(mu) xi of the signed mu (odd ell carry the asymmetry of a cross correlation).

    ``self.corr`` has ``r`` (mean |r| of the bin's grid points), ``corr``, ``modes`` (grid points) and, in 2d, ``mu``
    with dims (r, mu); ``self.poles`` has ``r``, ``modes`` and ``corr_<ell>``.  This is a mesh estimator: good for r of a
    few cells and up.  r = 0 is an ordinary grid point, so with rmin = 0 the first bin carries the shot-noise spike;
    ``attrs["shotnoise"]`` is FFTPower's value and is reported, never subtracted.  Single-GPU meshes without folding;
    the output grid and the C2R's work area must fit in free device memory.
    """

    def __init__(self, first, mode="1d", Nmesh=None, BoxSize=None, second=None, los=(0, 0, 1), Nmu=5, dr=None, rmin=0.0,
                 rmax=None, poles=()):
        if mode not in ("1d", "2d"):
            raise AstrildPkError("mode must be '1d' or '2d'")
        poles = [] if poles is None else [int(e) for e in poles]
        Nmu = 1 if mode == "1d" else int(Nmu)
        for m in (first, second):
            if m is not None and getattr(m, "_fold", 0):
                raise AstrildPkError("FFTCorr does not support folded boxes (fold > 0)")
        eng = first._eng
        if eng.n0 != eng.N:
            raise AstrildPkError("FFTCorr runs on single-GPU meshes only (no slab path)")
        if second is not None and second is not first and second._eng is not eng:
            raise AstrildPkError("first and second must share Nmesh, BoxSize and device")
        self.first, self.second = first, first if second is None else second
        N, L = eng.N, eng.L
        (c1, c1s), s1, comp1 = first._complex_fields()
        if second is None or second is first:
            c2 = c2s = None
            s2 = s1
        else:
            (c2, c2s), s2, comp2 = second._complex_fields()
            if (c1s is None) != (c2s is None):
                raise AstrildPkError("first and second must both be interlaced or both not")
            if comp1 != comp2:
                raise AstrildPkError("first and second must use the same window compensation")
        xb = eng.xi_binning(rmin, dr, rmax, Nmu, poles, tuple(float(x) for x in los), comp1, c1s is not None)
        need = 4 * N * N * eng.ldz + xb.scratch_bytes
        free = _free_device_bytes(eng.device)
        if need > free:
            raise AstrildPkError(f"FFTCorr needs {need} bytes of device memory for its output grid and the C2R's work "
                                 f"area, {free} are free")
        grid, sums = eng.xi_raw(xb, c1, c1s, c2, c2s)
        del grid
        res = eng.finish_xi(sums.cpu().numpy(), xb, s1 * s2 / float(N) ** 6)
        auto = second is None or second is first
        shot = float(getattr(first, "shotnoise", 0.0)) if auto else 0.0
        dr_used = float(xb.edges[1] - xb.edges[0]) if len(xb.edges) > 1 else float("nan")
        self.attrs = {"mode": mode, "Nmesh": np.array([N] * 3), "BoxSize": np.array([L] * 3), "edges": xb.edges,
                      "dr": L / N if dr is None else dr, "rmin": rmin, "rmax": L / 2 + dr_used / 2 if rmax is None else rmax,
                      "Nmu": Nmu, "poles": list(poles), "los": list(los), "volume": L ** 3, "shotnoise": shot}
        if mode == "2d":
            self.corr = BinnedStatistic(["r", "mu"], [xb.edges, xb.muedges],
                                        {"r": res["r"], "mu": res["mu"], "corr": res["corr"], "modes": res["modes"]},
                                        dict(self.attrs))
        else:
            self.corr = BinnedStatistic(["r"], [xb.edges], {"r": res["r"][:, 0], "corr": res["corr"][:, 0],
                                                            "modes": res["modes"][:, 0]}, dict(self.attrs))
        self.poles = None
        if poles:
            data = {"r": res["poles"]["r"], "modes": res["poles"]["modes"]}
            data.update({"corr_%d" % e: res["poles"]["corr_%d" % e] for e in poles})
            self.poles = BinnedStatistic(["r"], [xb.edges], data, dict(self.attrs))

    def run(self):
        return self.corr, self.poles
