"""Float64 NumPy oracle of the correlation function (astrild_b200.FFTCorr, astrild_b200/csrc/corr.cu).

Definition (the one the library implements; nbodykit 0.3.14's FFTCorr / project_to_basis restated from recollection,
unpinned):
  * input: the normalised half-complex fields FFTPower sees (pk_oracle.r2c, interlace-combined and compensated for a
    CatalogMesh); p(k) = c1(k) conj(c2(k)), the k = 0 mode zeroed; c2 = c1 for an auto correlation;
  * xi(r_n) = Re sum_{stored k} w(k) p(k) e^{i k.r_n} with FFTPower's Hermitian weights w (2 on the non-singular z
    planes, 1 on iz = 0 and, for even N, iz = N/2) = (1/N^3) sum_y d1(y + r_n) d2(y) for plain fields; displacement
    index n is freq_index(n) * L / N per axis (r = x1 - x2);
  * evaluated as irfftn of the half grid whose self-paired planes hold the Hermitian part H = (p(k) + conj p(k')) / 2,
    k' = (-ia, -ib, iz) mod N: on those planes interlacing makes p non-Hermitian, and this is what the half-grid sum
    means there;
  * binning: every grid point has weight 1; r^2 = (ra^2 + rb^2) + rz^2 with ra = freq_index(N) * (L / N);
    digitize(r^2, edges^2), edges = arange(rmin, rmax, dr) (dr = L / N, rmax = L / 2 + dr / 2); mu = (r . los) / |r|
    with r . los = (rx l0 + ry l1) + rz l2 (0 at r = 0), digitize(|mu|, linspace(0, 1, Nmu + 1)) with the mu = 1 column
    folded into the last one; multipoles (2 ell + 1) L_ell(mu) xi with signed mu, summed over mu and divided by the
    count of the r bin.
"""
from __future__ import annotations

import numpy as np

from . import pk_oracle as po


def r_axis(N: int, L: float) -> np.ndarray:
    return po.freq_index(N) * (L / N)


def r_edges(N: int, L: float, rmin: float = 0.0, dr: float | None = None, rmax: float | None = None) -> np.ndarray:
    dr = L / N if dr is None else dr
    rmax = L / 2 + dr / 2 if rmax is None else rmax
    return np.arange(rmin, rmax, dr)


def product(c1: np.ndarray, c2: np.ndarray | None) -> np.ndarray:
    """p = c1 conj(c2) on the half grid, k = 0 zeroed."""
    p = c1 * np.conj(c1 if c2 is None else c2)
    p[0, 0, 0] = 0.0
    return p


def plane_symmetrised(p: np.ndarray, N: int) -> np.ndarray:
    """The half grid with the Hermitian part (p(k) + conj p(k')) / 2 on iz = 0 and (even N) iz = N/2."""
    out = np.array(p, dtype=np.complex128)
    mirror = (-np.arange(N)) % N
    for iz in ([0, N // 2] if N % 2 == 0 else [0]):
        plane = p[:, :, iz]
        out[:, :, iz] = 0.5 * (plane + np.conj(plane[mirror][:, mirror]))
    return out


def xi_grid(c1: np.ndarray, c2: np.ndarray | None, N: int) -> np.ndarray:
    """xi on the N^3 grid (float64), index n = displacement freq_index(n) L / N."""
    H = plane_symmetrised(product(c1, c2), N)
    return np.fft.irfftn(H, s=(N, N, N), axes=(0, 1, 2)) * float(N) ** 3


def xi_explicit(p: np.ndarray, N: int) -> np.ndarray:
    """Re sum_{stored k} w(k) p(k) e^{i k.r_n}, evaluated term by term (O(N^6): small N only)."""
    w = po.hermitian_weights(N)
    n = np.arange(N)
    kz = np.arange(N // 2 + 1)
    ex = np.exp(2j * np.pi * np.outer(n, n) / N)              # [k index][r index]
    ez = np.exp(2j * np.pi * np.outer(kz, n) / N)
    t = np.einsum("abz,ax,by,zr->xyr", p * w[None, None, :], ex, ex, ez)
    return t.real


def xi_direct(d1: np.ndarray, d2: np.ndarray | None) -> np.ndarray:
    """(1/N^3) sum_y d1(y + r_n) d2(y) of plain real fields by direct circular shifts (O(N^6))."""
    d2 = d1 if d2 is None else d2
    N = d1.shape[0]
    out = np.empty((N, N, N))
    for a in range(N):
        for b in range(N):
            for c in range(N):
                out[a, b, c] = np.sum(np.roll(d1, (-a, -b, -c), axis=(0, 1, 2)) * d2)
    return out / float(N) ** 3


def bin_xi(xi: np.ndarray, N: int, L: float, edges: np.ndarray, Nmu: int = 1, poles=(), los=(0.0, 0.0, 1.0)) -> dict:
    """Full sums (digitize indices: under/overflow kept) over the N^3 grid points: rsum, musum, Nsum [Nr+2][Nmu+2],
    ysum [nell][Nr+2][Nmu+2], the mu = 1 column folded into column Nmu; ells = [0] + poles, sorted."""
    r = r_axis(N, L)
    r2 = r * r
    R2 = (r2[:, None, None] + r2[None, :, None]) + r2[None, None, :]
    rdl = (r[:, None, None] * los[0] + (r * los[1])[None, :, None]) + (r * los[2])[None, None, :]
    rn = np.sqrt(R2)
    with np.errstate(invalid="ignore", divide="ignore"):
        mu = np.where(rn > 0.0, rdl / np.where(rn > 0.0, rn, 1.0), 0.0)
    muedges = np.linspace(0.0, 1.0, Nmu + 1)
    dig_r = np.digitize(R2.ravel(), edges ** 2)
    dig_mu = np.digitize(np.abs(mu).ravel(), muedges)
    shape = (len(edges) + 1, Nmu + 2)
    multi = np.ravel_multi_index([dig_r, dig_mu], shape)
    size = shape[0] * shape[1]
    ells = sorted(set([0] + [int(e) for e in poles]))
    rsum = np.bincount(multi, weights=rn.ravel(), minlength=size).reshape(shape)
    musum = np.bincount(multi, weights=np.abs(mu).ravel(), minlength=size).reshape(shape)
    nsum = np.bincount(multi, minlength=size).astype(np.int64).reshape(shape)
    ysum = np.stack([np.bincount(multi, weights=((2 * ell + 1) * po.legendre(ell, mu) * xi).ravel(),
                                 minlength=size).reshape(shape) for ell in ells])
    for a in (rsum, musum, nsum):
        a[:, -2] += a[:, -1]
        a[:, -1] = 0
    ysum[..., -2] += ysum[..., -1]
    ysum[..., -1] = 0.0
    return {"rsum": rsum, "musum": musum, "nsum": nsum, "ysum": ysum, "ells": ells, "edges": edges, "muedges": muedges}


def finish(sums: dict, poles=()) -> dict:
    """nbodykit's tail: r, mu, corr, modes of shape (Nr, Nmu) and poles {"r", "modes", "corr_<ell>"}."""
    sl = slice(1, -1)
    n = sums["nsum"]
    with np.errstate(invalid="ignore", divide="ignore"):
        out = {"r": (sums["rsum"] / n)[sl, sl], "mu": (sums["musum"] / n)[sl, sl], "corr": (sums["ysum"][0] / n)[sl, sl],
               "modes": n[sl, sl].copy()}
        n1 = n[sl, sl].sum(axis=-1)
        pol = {"r": sums["rsum"][sl, sl].sum(axis=-1) / n1, "modes": n1}
        for ell in poles:
            pol["corr_%d" % ell] = sums["ysum"][sums["ells"].index(int(ell))][sl, sl].sum(axis=-1) / n1
        out["poles"] = pol
    return out


def fftcorr(c1: np.ndarray, c2: np.ndarray | None, N: int, L: float, Nmu: int = 1, poles=(), los=(0.0, 0.0, 1.0),
            rmin: float = 0.0, dr: float | None = None, rmax: float | None = None) -> dict:
    """FFTCorr on normalised complex fields -> finish() of the binned grid, plus the grid ``xi`` and the ``sums``."""
    xi = xi_grid(c1, c2, N)
    sums = bin_xi(xi, N, L, r_edges(N, L, rmin, dr, rmax), Nmu, poles, los)
    out = finish(sums, poles)
    out["xi"], out["sums"] = xi, sums
    return out
