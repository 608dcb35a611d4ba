"""Float64 NumPy oracle of the bispectrum (astrild_b200.FFTBispectrum, astrild_b200/csrc/bispec.cu).

Definition (the one the library implements):
  * shells: bin b holds the modes q of the full N^3 grid with numpy.digitize(k^2, edges^2) == b + 1,
    k^2 = (kx^2 + ky^2) + kz^2 from pk_oracle.k_tables; the k = 0 mode is in no shell;
  * kept triples: i <= j <= l, minus those with lo_l >= hi_i + hi_j and hi_i + hi_j + hi_l <= 2 k_Nyquist
    (no triangle can close, directly or modulo the grid);
  * F_b(x) = sum_{q in b} delta(q) e^{i q.x},  T_F = sum_x F_i F_j F_l,  T_D = the same with delta == 1 = N^3 N_tri;
  * B = V^2 T_F / T_D = V^2 <delta(q1) delta(q2) delta(q3)> over the N_tri ordered triangles q1 + q2 + q3 = 0 (mod N).
delta(q) is pmesh's normalised r2c (pk_oracle.r2c), interlace-combined and compensated as for FFTPower.
"""
from __future__ import annotations

import numpy as np

from . import pk_oracle as po


def default_edges(N: int, L: float, kmin: float = 0.0, dk: float | None = None, kmax: float | None = None):
    """apk_tables_k_edges with the bispectrum's defaults: dk = 2 pi / L, kmax = (2/3) pi N / L."""
    dk = 2 * np.pi / L if dk is None else dk
    kmax = 2.0 / 3.0 * np.pi * N / L if kmax is None else kmax
    return np.arange(kmin, kmax, dk)


def kept_triples(edges: np.ndarray, N: int, L: float) -> np.ndarray:
    """(ntriples, 3) int: i <= j <= l after the skip rule, in the library's order."""
    knyq = np.pi * N / L
    nb = len(edges) - 1
    out = []
    for i in range(nb):
        for j in range(i, nb):
            for l in range(j, nb):
                hij = edges[i + 1] + edges[j + 1]
                if edges[l] >= hij and hij + edges[l + 1] <= 2.0 * knyq:
                    continue
                out.append((i, j, l))
    return np.array(out, dtype=np.int64).reshape(-1, 3)


def shell_index_half(N: int, L: float, edges: np.ndarray, k_dtype=np.float64) -> np.ndarray:
    """Shell (0 .. nb-1, or -1) of every stored mode of the half grid [N][N][N/2+1]."""
    kx, ky, kz = po.k_tables(N, L, k_dtype)
    k2 = (kx[:, None, None] ** 2 + ky[None, :, None] ** 2) + kz[None, None, :] ** 2
    dig = np.digitize(k2, edges ** 2) - 1
    dig[(dig < 0) | (dig >= len(edges) - 1)] = -1
    dig[0, 0, 0] = -1
    return dig


def shell_index_full(N: int, L: float, edges: np.ndarray, k_dtype=np.float64) -> np.ndarray:
    kx, ky, _ = po.k_tables(N, L, k_dtype)
    k2 = (kx[:, None, None] ** 2 + ky[None, :, None] ** 2) + kx[None, None, :] ** 2
    dig = np.digitize(k2, edges ** 2) - 1
    dig[(dig < 0) | (dig >= len(edges) - 1)] = -1
    dig[0, 0, 0] = -1
    return dig


def shell_fields(c: np.ndarray, N: int, L: float, edges: np.ndarray, k_dtype=np.float64) -> np.ndarray:
    """F_b(x) for every shell: (nb, N^3) float64.  c: the half-complex field (None: the indicators D_b)."""
    sh = shell_index_half(N, L, edges, k_dtype)
    nb = len(edges) - 1
    out = np.empty((nb, N ** 3))
    for b in range(nb):
        m = np.where(sh == b, 1.0 if c is None else c, 0.0).astype(np.complex128)
        out[b] = np.fft.irfftn(m, s=(N, N, N), axes=(0, 1, 2)).ravel() * float(N) ** 3
    return out


def triple_sums(F: np.ndarray, triples: np.ndarray, absolute: bool = False) -> np.ndarray:
    """sum_x F_i F_j F_l (or sum_x |F_i F_j F_l|) per triple, float64."""
    nb = F.shape[0]
    out = np.zeros(len(triples))
    want = {}
    for t, (i, j, l) in enumerate(triples):
        want.setdefault(i, []).append((t, j, l))
    Fa = np.abs(F) if absolute else F
    for i, items in want.items():
        G = Fa[i][None, :] * Fa                        # (nb, P): F_i F_j for all j
        C = G @ Fa.T                                   # (nb, nb): sum_x F_i F_j F_l
        for t, j, l in items:
            out[t] = C[j, l]
    del nb
    return out


def bispectrum_fft(delta_k: np.ndarray, N: int, L: float, edges: np.ndarray, k_dtype=np.float64,
                   with_abs: bool = False) -> dict:
    """The FFT estimator in float64.  delta_k: normalised half-complex field (pk_oracle.r2c, interlaced / compensated as
    wanted).  Returns triples, T_F, T_D, N_tri (rounded), B (V^2 T_F / T_D, NaN where N_tri = 0) and, with_abs, A (the
    same with |F_i F_j F_l|: the scale of the terms, for error bounds)."""
    triples = kept_triples(edges, N, L)
    D = shell_fields(None, N, L, edges, k_dtype)
    TD = triple_sums(D, triples)
    ntri = np.rint(TD / float(N) ** 3).astype(np.int64)
    F = shell_fields(delta_k, N, L, edges, k_dtype)
    TF = triple_sums(F, triples)
    V = float(L) ** 3
    with np.errstate(invalid="ignore", divide="ignore"):
        B = V * V * TF / np.where(ntri > 0, TD, np.nan)
    out = {"triples": triples, "TF": TF, "TD": TD, "ntri": ntri, "B": B, "edges": edges,
           "residual": float(np.max(np.abs(TD / float(N) ** 3 - ntri))) if len(TD) else 0.0}
    if with_abs:
        with np.errstate(invalid="ignore", divide="ignore"):
            out["A"] = V * V * triple_sums(F, triples, absolute=True) / np.where(ntri > 0, TD, np.nan)
    return out


def bispectrum_bruteforce(delta: np.ndarray, L: float, edges: np.ndarray, k_dtype=np.float64) -> dict:
    """Direct sum over all mode pairs (q1, q2) of the full complex grid, q3 = -q1 - q2 (mod N).  For N <= 24.

    delta: real (N, N, N) field.  Returns count[i, j, l] (ordered triangles, all nb^3 shell triples), the sum of
    Re delta(q1) delta(q2) delta(q3) per shell triple and B = V^2 sum / count for the kept triples."""
    delta = np.asarray(delta, dtype=np.float64)
    N = delta.shape[0]
    nb = len(edges) - 1
    dk = np.fft.fftn(delta) / float(N) ** 3
    sh = shell_index_full(N, L, edges, k_dtype).ravel()
    idx = np.flatnonzero(sh >= 0)
    n = np.stack(np.unravel_index(idx, (N, N, N)), axis=1)            # storage indices of the in-shell modes
    b = sh[idx]
    v = dk.ravel()[idx]
    count = np.zeros(nb ** 3, dtype=np.int64)
    ssum = np.zeros(nb ** 3)
    dflat = dk.ravel()
    for a in range(len(idx)):
        q3 = np.mod(-(n[a][None, :] + n), N)
        f3 = (q3[:, 0] * N + q3[:, 1]) * N + q3[:, 2]
        b3 = sh[f3]
        ok = b3 >= 0
        key = (b[a] * nb + b[ok]) * nb + b3[ok]
        count += np.bincount(key, minlength=nb ** 3)
        ssum += np.bincount(key, weights=(v[a] * v[ok] * dflat[f3[ok]]).real, minlength=nb ** 3)
    count = count.reshape(nb, nb, nb)
    ssum = ssum.reshape(nb, nb, nb)
    triples = kept_triples(edges, N, L)
    c = count[triples[:, 0], triples[:, 1], triples[:, 2]]
    s = ssum[triples[:, 0], triples[:, 1], triples[:, 2]]
    V = float(L) ** 3
    with np.errstate(invalid="ignore", divide="ignore"):
        B = V * V * s / np.where(c > 0, c, np.nan)
    return {"count": count, "sum": ssum, "triples": triples, "ntri": c, "B": B}


def delta_k_from_particles(pos, mass, N: int, L: float, resampler: str = "tsc", interlaced: bool = False,
                           compensated: bool = False, normalize: bool = True):
    """The oracle's deposit -> normalised half-complex field (pk_oracle.power_from_particles' field())."""
    dx = L / N
    m = 1.0 if mass is None else mass
    real = po.paint(pos, m, N, L, resampler)
    scale = (N ** 3 / real.sum()) if normalize else 1.0 / dx ** 3
    c = po.r2c(real) * scale
    if interlaced:
        real2 = po.paint(pos, m, N, L, resampler, shift=0.5)
        c = po.interlace_combine(c, po.r2c(real2) * scale, N, L)
    if compensated:
        c = po.compensate(c, resampler, interlaced, N)
    return c
