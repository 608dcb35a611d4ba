"""Host-built tables of the binning stage (the host side of the C-ABI boundary).

These mirror the set-up code of the reference stack that astrild calls into -- pmesh's
``ParticleMesh.__init__`` k tables and nbodykit's ``FFTPower`` edges / ``Compensate*`` factors
(call sites: /root/reference/src/astrild/power_spectra/power_spectrum_3d.py:181-195,
/root/reference/src/astrild/particles/hutils/stats_subfind.py:142-148; semantics SURVEY.md
Appendix A.3-A.6).  They are uploaded to the device verbatim: the CUDA kernel never
re-derives a wavenumber, so which float ends up on which side of a bin edge is decided
here, in float64 NumPy, exactly as the reference decides it.
"""
from __future__ import annotations

import numpy as np


def freq_index(N: int) -> np.ndarray:
    """Lattice frequency of storage index i (Nyquist of an even N is -N/2, as in pmesh)."""
    i = np.arange(N, dtype=np.int64)
    return np.where(2 * i < N, i, i - N)


def k_axis(N: int, L: float, k_dtype=np.float64) -> np.ndarray:
    """pmesh: ``w = n * (2 pi / N)``; ``k = w * N / L`` -- this expression order."""
    n = freq_index(N).astype(k_dtype)
    w = n * k_dtype(2 * np.pi / N)
    return (w * k_dtype(N) / k_dtype(L)).astype(np.float64)


def k_edges(N: int, L: float, kmin: float = 0.0, dk: float | None = None,
            kmax: float | None = None) -> np.ndarray:
    """nbodykit FFTPower: ``dk = 2 pi / L``, ``kmax = pi N / L + dk/2``, ``arange(kmin, kmax, dk)``."""
    if dk is None:
        dk = 2 * np.pi / L
    if kmax is None:
        kmax = np.pi * N / L + dk / 2
    return np.arange(kmin, kmax, dk)


def r_axis(N: int, L: float) -> np.ndarray:
    """Displacement of storage index n of the real grid along one axis: ``freq_index(N) * (L / N)`` (minimum image;
    -L/2 kept for even N, as in the k tables)."""
    return freq_index(N) * (L / N)


def r_edges(N: int, L: float, rmin: float = 0.0, dr: float | None = None,
            rmax: float | None = None) -> np.ndarray:
    """FFTCorr's edges: ``dr = L / N``, ``rmax = L / 2 + dr / 2``, ``arange(rmin, rmax, dr)`` (the arange of k_edges)."""
    if dr is None:
        dr = L / N
    if rmax is None:
        rmax = L / 2 + dr / 2
    return np.arange(rmin, rmax, dr)


def hermitian_weights(N: int) -> np.ndarray:
    """2 for stored modes with k_z > 0 (their conjugates are not stored), 1 for k_z = 0 / Nyquist."""
    nz = freq_index(N)[: N // 2 + 1]
    return np.where(nz > 0, 2.0, 1.0)


def compensation_axis(resampler: str, interlaced: bool, N: int) -> np.ndarray:
    """Factor the complex field is divided by along one axis (nbodykit Compensate{CIC,TSC}[Shotnoise])."""
    w = freq_index(N).astype(np.float64) * (2 * np.pi / N)
    r = resampler.lower()
    if r not in ("cic", "tsc"):
        raise ValueError(f"no window compensation defined for resampler {resampler!r}")
    p = 2 if r == "cic" else 3
    if interlaced:
        return np.sinc(w / (2 * np.pi)) ** p
    s = np.sin(0.5 * w) ** 2
    if r == "cic":
        return (1 - 2.0 / 3 * s) ** 0.5
    return (1 - s + 2.0 / 15 * s * s) ** 0.5


def interlace_phase_axis(N: int, L: float) -> np.ndarray:
    """0.5 * k_i * H with H = L / N: the interlaced twin is multiplied by exp(1j * sum of these)."""
    return 0.5 * k_axis(N, L) * (L / N)
