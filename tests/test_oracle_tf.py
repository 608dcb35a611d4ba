"""The Taylor-Fourier oracle (oracle/tf_oracle.py) against first principles: a direct float64 DFT of the particles
within the closed-form truncation bound (error falling with the order), order 0 against the NGP paint of pk_oracle,
a single particle against T_n in closed form, and the Gauss-Legendre noise factor E|T_n|^2 against Monte Carlo."""
import numpy as np
import pytest

from oracle import pk_oracle as po
from oracle import tf_oracle as tfo


@pytest.mark.parametrize("N", [8, 9, 12])
@pytest.mark.parametrize("with_mass", [False, True])
def test_oracle_within_the_bound_of_the_exact_dft_and_improving_with_order(N, with_mass):
    rng = np.random.default_rng(N + 100 * with_mass)
    npart = 300
    pos = rng.random((npart, 3)) * 3.0 - 1.0                 # in box units, some outside [0, 1): wrapped
    mass = rng.random(npart) * 2.0 - 0.5 if with_mass else None
    F = tfo.exact_dft(pos, mass, N)
    w = np.abs(tfo.axis_w(N))
    low = (w[:, None, None] + w[None, :, None] + w[None, None, : N // 2 + 1]) <= np.pi    # |w.d| <= pi / 2
    errs = []
    for order in range(5):
        c = tfo.tf_field(pos, mass, N, order)
        err = np.abs(c - F)
        bound = tfo.error_bound(mass, npart, N, order)
        assert np.all(err <= bound * (1 + 1e-9) + 1e-9), order
        errs.append(err[low].max())
    # the series converges everywhere, monotonically where |w.d| <= pi / 2 (near the Nyquist corner, |w.d| <= 3 pi / 2,
    # only the bound above holds order by order)
    assert all(errs[i + 1] < errs[i] for i in range(4)), errs
    assert errs[-1] < 1e-2 * np.abs(F[low]).max()


def test_order_zero_is_the_ngp_paint():
    N, L = 12, 50.0
    rng = np.random.default_rng(3)
    pos = rng.random((500, 3)) * L
    mass = rng.random(500)
    ngp = po.paint(pos, mass, N, L, resampler="nearest")
    np.testing.assert_allclose(tfo.tf_field(pos, mass, N, 0, 1.0 / L), np.fft.rfftn(ngp), rtol=0, atol=1e-11)


@pytest.mark.parametrize("order", [0, 1, 2, 3, 4])
def test_single_particle_is_the_taylor_polynomial(order):
    N = 16
    g = np.array([[3.3, 7.45, 12.91]])                      # grid units
    c = tfo.tf_field(g, None, N, order, pos_scale=1.0 / N)
    w = tfo.axis_w(N)
    h = np.rint(g[0])
    d = g[0] - h
    want = np.zeros_like(c)
    for ia in range(N):
        for ib in range(N):
            for iz in range(N // 2 + 1):
                wv = np.array([w[ia], w[ib], w[iz]])
                want[ia, ib, iz] = np.exp(-1j * wv @ h) * tfo.taylor(wv @ d, order)
    np.testing.assert_allclose(c, want, rtol=0, atol=1e-12)


@pytest.mark.parametrize("order", [1, 2, 3, 4])
def test_noise_factor_gauss_legendre_against_monte_carlo(order):
    rng = np.random.default_rng(order)
    d = rng.random((400000, 3)) - 0.5
    for w3 in ((np.pi, 0.0, 0.0), (0.7, -2.1, 1.3), (np.pi, np.pi, np.pi)):
        v = np.abs(tfo.taylor(d @ np.asarray(w3), order)) ** 2
        gl = tfo.noise_factor(np.asarray(w3), order)
        assert abs(gl - v.mean()) < 5.0 * v.std() / np.sqrt(len(v)), (w3, gl, v.mean())      # 5 sigma of the estimate
    # order 3 in closed form: E|T_3|^2 = E[1 - theta^4 / 12 + theta^6 / 36]
    if order == 3:
        th = d @ np.array([0.7, -2.1, 1.3])
        gl = tfo.noise_factor(np.array([0.7, -2.1, 1.3]), 3)
        exact_poly = np.mean(1 - th ** 4 / 12 + th ** 6 / 36)
        assert abs(gl - exact_poly) < 5e-3
    grid = tfo.noise_factor_grid(6, order)
    w = tfo.axis_w(6)
    assert grid[1, 2, 3] == pytest.approx(tfo.noise_factor(np.array([w[1], w[2], w[3]]), order), rel=1e-12)
