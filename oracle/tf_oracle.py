"""Float64 NumPy restatement of the Taylor-Fourier (TF) mesh of Colombi et al. (2009)  --  TEST INFRASTRUCTURE ONLY.

Grid coordinate g = pos * pos_scale * N (wrapped modulo N), home cell h = rint(g) mod N, d = g - rint(g) in
[-1/2, 1/2]^3.  For order n and every multi-index alpha = (a, b, c) with |alpha| <= n (graded order, as tf.cu):

    M_alpha[h] = sum_{p with home h} m_p dx^a dy^b dz^c
    c_TF(k)    = sum_alpha (-i)^|alpha| (wx^a wy^b wz^c / (a! b! c!)) rfftn(M_alpha)(k),   w = 2 pi freq_index / N
               = sum_h e^{-i w.h} sum_p m_p T_n(w.d_p)     (T_n: degree-n Taylor polynomial of e^{-i theta})

Facts the tests use: |c_TF - F| <= sum_p |m_p| (|w|_1 / 2)^{n+1} / (n+1)! against the exact DFT F(k) = sum_p m_p
e^{-i w.g_p}; order 0 is the NGP paint; for uniform random particles E|c_TF(k)|^2 = sum_p m_p^2 E_d |T_n(w.d)|^2 (k != 0).
"""
from __future__ import annotations

from math import factorial

import numpy as np

from .pk_oracle import freq_index


def multi_indices(order: int) -> list:
    """(a, b, c) with a + b + c <= order: total degree ascending, then a, then b descending (tf.cu's order)."""
    out = []
    for t in range(order + 1):
        for a in range(t, -1, -1):
            for b in range(t - a, -1, -1):
                out.append((a, b, t - a - b))
    return out


def grid_offsets(pos, N: int, pos_scale: float):
    """-> (home cells int64 (Np, 3) in [0, N), d float64 (Np, 3) in [-1/2, 1/2])."""
    g = np.asarray(pos, dtype=np.float64) * (pos_scale * N)
    r = np.rint(g)
    return np.mod(r, N).astype(np.int64), g - r


def moments(pos, mass, N: int, order: int, pos_scale: float) -> np.ndarray:
    """M_alpha for every multi-index: float64 (n_mom, N, N, N)."""
    h, d = grid_offsets(pos, N, pos_scale)
    m = np.broadcast_to(np.asarray(1.0 if mass is None else mass, dtype=np.float64), (h.shape[0],))
    idx = (h[:, 0] * N + h[:, 1]) * N + h[:, 2]
    out = []
    for a, b, c in multi_indices(order):
        out.append(np.bincount(idx, weights=m * d[:, 0] ** a * d[:, 1] ** b * d[:, 2] ** c, minlength=N ** 3))
    return np.asarray(out).reshape(-1, N, N, N)


def axis_w(N: int) -> np.ndarray:
    return 2.0 * np.pi * freq_index(N).astype(np.float64) / N


def combine(mhat: np.ndarray, N: int, order: int) -> np.ndarray:
    """sum_alpha (-i)^|alpha| (wx^a wy^b wz^c / a! b! c!) mhat_alpha over the rfftn half grid."""
    w = axis_w(N)
    wx, wy, wz = w[:, None, None], w[None, :, None], w[None, None, : N // 2 + 1]
    out = np.zeros(mhat.shape[1:], dtype=np.complex128)
    for k, (a, b, c) in enumerate(multi_indices(order)):
        coef = wx ** a / factorial(a) * wy ** b / factorial(b) * wz ** c / factorial(c)
        out += (-1j) ** (a + b + c) * coef * mhat[k]
    return out


def tf_field(pos, mass, N: int, order: int = 3, pos_scale: float = 1.0) -> np.ndarray:
    """c_TF, complex128 [N][N][N/2+1] (un-normalised, like the device r2c)."""
    mom = moments(pos, mass, N, order, pos_scale)
    return combine(np.fft.rfftn(mom, axes=(1, 2, 3)), N, order)


def exact_dft(pos, mass, N: int, pos_scale: float = 1.0) -> np.ndarray:
    """F(k) = sum_p m_p e^{-i w.g_p} on the half grid (direct sum; small N only)."""
    g = np.asarray(pos, dtype=np.float64) * (pos_scale * N)
    m = np.broadcast_to(np.asarray(1.0 if mass is None else mass, dtype=np.float64), (g.shape[0],))
    w = axis_w(N)
    ex = np.exp(-1j * np.outer(g[:, 0], w))                # (Np, N)
    ey = np.exp(-1j * np.outer(g[:, 1], w))
    ez = np.exp(-1j * np.outer(g[:, 2], w[: N // 2 + 1]))
    return np.einsum("p,pa,pb,pc->abc", m, ex, ey, ez, optimize=True)


def error_bound(mass, npart: int, N: int, order: int) -> np.ndarray:
    """sum_p |m_p| (|w|_1 / 2)^{n+1} / (n+1)! on the half grid."""
    w = np.abs(axis_w(N))
    w1 = w[:, None, None] + w[None, :, None] + w[None, None, : N // 2 + 1]
    msum = float(npart) if mass is None else float(np.abs(np.asarray(mass, dtype=np.float64)).sum())
    return msum * (w1 / 2.0) ** (order + 1) / factorial(order + 1)


def taylor(theta, order: int):
    """T_n(theta) = sum_{t <= n} (-i theta)^t / t!"""
    theta = np.asarray(theta, dtype=np.float64)
    return sum((-1j * theta) ** t / factorial(t) for t in range(order + 1))


def noise_factor(w3, order: int) -> float:
    """E_d |T_n(w.d)|^2 for d uniform on [-1/2, 1/2]^3: Gauss-Legendre with n + 1 nodes per axis (exact: the integrand
    is a polynomial of degree 2n in d)."""
    x, wt = np.polynomial.legendre.leggauss(order + 1)
    x, wt = 0.5 * x, 0.5 * wt
    dx, dy, dz = np.meshgrid(x, x, x, indexing="ij")
    ww = wt[:, None, None] * wt[None, :, None] * wt[None, None, :]
    th = w3[0] * dx + w3[1] * dy + w3[2] * dz
    return float((ww * np.abs(taylor(th, order)) ** 2).sum())


def noise_factor_grid(N: int, order: int) -> np.ndarray:
    """E|T_n(w.d)|^2 for every mode of the half grid (vectorised over the nodes)."""
    x, wt = np.polynomial.legendre.leggauss(order + 1)
    x, wt = 0.5 * x, 0.5 * wt
    w = axis_w(N)
    out = np.zeros((N, N, N // 2 + 1))
    for i, (xi, wi) in enumerate(zip(x, wt)):
        for j, (xj, wj) in enumerate(zip(x, wt)):
            for l, (xl, wl) in enumerate(zip(x, wt)):
                th = w[:, None, None] * xi + w[None, :, None] * xj + w[None, None, : N // 2 + 1] * xl
                out += wi * wj * wl * np.abs(taylor(th, order)) ** 2
    return out
