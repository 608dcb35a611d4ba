"""The correlation-function oracle (oracle/xi_oracle.py) against definitions evaluated directly.

* plain fields: xi_grid equals the O(N^6) circular correlation (1/N^3) sum_y d1(y + r) d2(y) of the mean-subtracted
  fields, auto and cross (this pins the sign r = x1 - x2 and the minimum-image axis);
* interlaced + compensated fields at even and odd N: the irfftn of the plane-symmetrised half grid equals the explicit
  sum Re sum_stored w p e^{ik.r} -- the claim the CUDA fill + C2R relies on;
* the binning: pair counts per bin against an integer-lattice brute force (L = N: r^2 is an exact integer), the
  tie-heavy case dr = L / N at L = 500, counts summing to N^3, and xi summing to 0 (k = 0 is zeroed).
"""
import numpy as np
import pytest

from oracle import pk_oracle as po
from oracle import xi_oracle as xo


def fields(N, seed, cross):
    rng = np.random.default_rng(seed)
    d1 = rng.standard_normal((N, N, N))
    d2 = rng.standard_normal((N, N, N)) + 0.5 * np.roll(d1, (1, -2, 3), axis=(0, 1, 2)) if cross else None
    return d1, d2


@pytest.mark.parametrize("N", [8, 9, 12])
@pytest.mark.parametrize("cross", [False, True])
def test_grid_is_the_circular_correlation(N, cross):
    d1, d2 = fields(N, N, cross)
    c1 = po.r2c(d1)
    c2 = po.r2c(d2) if cross else None
    xi = xo.xi_grid(c1, c2, N)
    want = xo.xi_direct(d1 - d1.mean(), None if d2 is None else d2 - d2.mean())
    np.testing.assert_allclose(xi, want, rtol=0, atol=1e-12 * np.abs(want).max())


def test_displacement_sign_and_axis():
    """d2 = d1 shifted by +s cells: xi peaks at r = x1 - x2 = -s, i.e. at index (-s) mod N."""
    N = 8
    d1, _ = fields(N, 3, False)
    d2 = np.roll(d1, (2, 0, -1), axis=(0, 1, 2))
    xi = xo.xi_grid(po.r2c(d1), po.r2c(d2), N)
    peak = np.unravel_index(np.argmax(xi), xi.shape)
    assert peak == ((-2) % N, 0, 1)
    r = xo.r_axis(N, N)
    assert (r[peak[0]], r[peak[1]], r[peak[2]]) == (-2.0, 0.0, 1.0)


@pytest.mark.parametrize("N", [8, 9])
@pytest.mark.parametrize("cross", [False, True])
def test_interlaced_half_grid_equals_the_explicit_sum(N, cross):
    L = 100.0
    rng = np.random.default_rng(N + 10 * cross)

    def field():
        a, b = rng.standard_normal((N, N, N)), rng.standard_normal((N, N, N))
        c = po.interlace_combine(po.r2c(a), po.r2c(b), N, L)
        return po.compensate(c, "tsc", True, N)

    c1 = field()
    c2 = field() if cross else None
    p = xo.product(c1, c2)
    # interlacing breaks the Hermitian symmetry of the self-paired planes on the modes with a Nyquist index (even N):
    # the symmetrisation is not a no-op there
    mirror = (-np.arange(N)) % N
    if N % 2 == 0:
        assert np.abs(p[:, :, 0] - np.conj(p[:, :, 0][mirror][:, mirror])).max() > 1e-3 * np.abs(p).max()
    np.testing.assert_allclose(xo.xi_grid(c1, c2, N), xo.xi_explicit(p, N), rtol=0, atol=1e-12 * np.abs(p).sum())


@pytest.mark.parametrize("N", [8, 9, 12])
def test_counts_against_integer_lattice(N):
    L = float(N)                                   # r is in cells: r^2 is an exact integer
    edges = xo.r_edges(N, L, rmin=0.0, dr=1.3, rmax=N * 0.9)
    s = xo.bin_xi(np.zeros((N, N, N)), N, L, edges)
    n = np.arange(N)
    f = np.where(2 * n < N, n, n - N)
    R2 = (f[:, None, None] ** 2 + f[None, :, None] ** 2 + f[None, None, :] ** 2).ravel()
    want = np.zeros(len(edges) + 1, dtype=np.int64)
    for v in R2:                                  # by hand: index of the first edge^2 above r^2
        want[int(np.sum(edges ** 2 <= v))] += 1
    np.testing.assert_array_equal(s["nsum"][:, 1], want)
    assert s["nsum"].sum() == N ** 3


def test_ties_on_the_edges_at_dr_equal_to_the_cell():
    N, L = 16, 500.0
    edges = xo.r_edges(N, L)
    s = xo.bin_xi(np.zeros((N, N, N)), N, L, edges)
    r = xo.r_axis(N, L)
    R2 = ((r[:, None, None] ** 2 + r[None, :, None] ** 2) + r[None, None, :] ** 2).ravel()
    e2 = edges ** 2
    assert np.isin(R2, e2).sum() > 0               # grid points lie exactly on edges: digitize decides them
    want = np.bincount(np.searchsorted(e2, R2, side="right"), minlength=len(edges) + 1)
    np.testing.assert_array_equal(s["nsum"].sum(axis=1), want)
    assert s["nsum"].sum() == N ** 3


@pytest.mark.parametrize("N", [8, 9])
def test_xi_sums_to_zero_and_poles_are_consistent(N):
    L = 100.0
    d1, d2 = fields(N, 7, True)
    c1, c2 = po.r2c(d1), po.r2c(d2)
    res = xo.fftcorr(c1, c2, N, L, Nmu=4, poles=[0, 1, 2], los=(0.3, -0.2, 0.9) / np.linalg.norm([0.3, -0.2, 0.9]),
                     rmax=L)
    assert abs(res["xi"].sum()) <= 1e-12 * np.abs(res["xi"]).sum()
    # all points binned (rmax beyond the box diagonal / 2): the monopole sums equal the total of xi
    assert res["sums"]["nsum"].sum() == N ** 3
    np.testing.assert_allclose(res["sums"]["ysum"][0].sum(), res["xi"].sum(), atol=1e-12 * np.abs(res["xi"]).sum())
    # the (r, mu) monopole summed over mu is the 1-D xi
    one = xo.fftcorr(c1, c2, N, L, rmax=L)
    w = res["modes"]
    tol = 1e-12 * np.abs(res["xi"]).max()
    with np.errstate(invalid="ignore"):
        mono = np.where(w > 0, res["corr"] * w, 0.0).sum(axis=1) / w.sum(axis=1)
    np.testing.assert_allclose(mono, one["corr"][:, 0], rtol=0, atol=tol)
    np.testing.assert_allclose(res["poles"]["corr_0"], one["corr"][:, 0], rtol=0, atol=tol)
