"""TaylorFourierMesh on the device against the float64 oracle (oracle/tf_oracle.py) and first principles.

Float32 tolerance (derived, per mode): the moment grids carry the fixed-point error bounded in test_simt_tf.py (below
2^-22 of sum |m| per cell), each cuFFT r2c of a grid M_alpha errs by at most ~ (3 log2 N + 8) 2^-24 sum_h |M_alpha[h]|
(a float32 FFT's worst-case error relative to the 1-norm of its input, with margin), and the combine adds the float32
rounding of the coefficient tables and of the sum: together
    tol(k) = 2^-24 (3 log2 N + 8 + 4 n_mom) sum_alpha |coef_alpha(k)| sum_h |M_alpha[h]|.
"""
from math import factorial

import numpy as np
import pytest
import torch

import astrild_b200 as ab
from astrild_b200 import _lib
from astrild_b200._lib import AstrildPkError
from astrild_b200.engine import PkEngine
from oracle import pk_oracle as po
from oracle import tf_oracle as tfo

pytestmark = pytest.mark.gpu


def off_ties(pos, N, pos_scale):
    """positions moved by at most 2e-4 cells so that no coordinate is within 1e-4 cells of a rounding tie: the device
    forms the brick-local coordinate in float32 (a few 1e-6 cells), so a particle that close to a tie may be filed under
    either neighbour -- allowed, and covered by the truncation bound, but not by the float32 tolerance below"""
    g = pos.astype(np.float64) * (pos_scale * N)
    f = g - np.floor(g)
    near = np.abs(f - 0.5) < 1e-4
    g = np.where(near, np.floor(g) + 0.5 + np.where(f >= 0.5, 2e-4, -2e-4), g)
    return (g / (pos_scale * N)).astype(pos.dtype)


def tolerance(pos, mass, N, order, pos_scale):
    mom = tfo.moments(pos, mass, N, order, pos_scale)
    w = tfo.axis_w(N)
    tol = np.zeros((N, N, N // 2 + 1))
    for k, (a, b, c) in enumerate(tfo.multi_indices(order)):
        coef = (np.abs(w[:, None, None]) ** a / factorial(a) * np.abs(w[None, :, None]) ** b / factorial(b)
                * np.abs(w[None, None, : N // 2 + 1]) ** c / factorial(c))
        tol += coef * np.abs(mom[k]).sum()
    return 2.0 ** -24 * (3 * np.log2(N) + 8 + 4 * len(mom)) * tol + 2.0 ** -20 * np.abs(mom[0]).sum()


def device_field(pos, mass, N, order, pos_scale, L=1.0, group=None):
    eng = PkEngine(N, L)
    try:
        tp = eng.tf_plan(order)
        c = eng.tf_field(tp, pos, mass, pos_scale, group=group)
        return c.cpu().numpy().astype(np.complex128)
    finally:
        torch.cuda.synchronize()
        eng.close()


@pytest.mark.parametrize("N", [32, 33, 64])
@pytest.mark.parametrize("with_mass", [False, True])
def test_field_against_the_oracle(N, with_mass):
    rng = np.random.default_rng(N + with_mass)
    npart = 40000
    pos = off_ties(rng.random((npart, 3)).astype(np.float32), N, 1.0)
    mass = rng.lognormal(0.0, 1.0, npart).astype(np.float32) if with_mass else None
    for order, group in ((3, None), (3, 7), (1, 1)):
        got = device_field(pos, mass, N, order, 1.0, group=group)
        want = tfo.tf_field(pos, mass, N, order, 1.0)
        tol = tolerance(pos, mass, N, order, 1.0)
        err = np.abs(got - want)
        assert np.all(err <= tol), (order, group, (err / tol).max())


def test_order_zero_is_the_ngp_deposit_and_r2c():
    N, L = 64, 100.0
    rng = np.random.default_rng(5)
    pos = off_ties((rng.random((200000, 3)) * L).astype(np.float32), N, 1.0 / L)
    mass = rng.random(200000).astype(np.float32)
    got = device_field(pos, mass, N, 0, 1.0 / L, L)
    eng = PkEngine(N, L)
    mesh = eng.deposit(pos, mass, resampler="nearest", method="atomic")
    want = eng.r2c(mesh).cpu().numpy().astype(np.complex128)
    eng.close()
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-6 * float(mass.sum()))


@pytest.mark.parametrize("order", [0, 2, 3, 4])
def test_single_particle_in_closed_form(order):
    N = 32
    g = np.array([[3.3, 30.61, 17.08]])
    got = device_field((g / N).astype(np.float64), None, N, order, 1.0)
    w = tfo.axis_w(N)
    h, d = np.rint(g[0]), g[0] - np.rint(g[0])
    th_h = w[:, None, None] * h[0] + w[None, :, None] * h[1] + w[None, None, : N // 2 + 1] * h[2]
    th_d = w[:, None, None] * d[0] + w[None, :, None] * d[1] + w[None, None, : N // 2 + 1] * d[2]
    want = np.exp(-1j * th_h) * tfo.taylor(th_d, order)
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-5)


def test_poisson_known_answer():
    """2^21 uniform particles on 128^3: P(k) of every bin up to Nyquist within 5 sigma of (V / N_p) E|T_3(w.d)|^2
    averaged over the bin's modes (sigma = mean sqrt(2 / modes): k and -k are one independent mode)."""
    N, L, npart, order = 128, 1000.0, 1 << 21, 3
    rng = np.random.default_rng(21)
    pos = (rng.random((npart, 3)) * L).astype(np.float32)
    r = ab.FFTPower(ab.TaylorFourierMesh(pos, L, N, order=order), mode="1d")
    assert r.attrs["shotnoise"] == pytest.approx(L ** 3 / npart)
    fac = tfo.noise_factor_grid(N, order)
    kx, ky, kz = po.k_tables(N, L)
    k2 = (kx[:, None, None] ** 2 + ky[None, :, None] ** 2) + kz[None, None, :] ** 2
    wgt = np.broadcast_to(po.hermitian_weights(N)[None, None, :], k2.shape)
    edges = r.power.edges["k"]
    dig = np.digitize(k2.ravel(), edges ** 2)
    num = np.bincount(dig, weights=(wgt * fac).ravel(), minlength=len(edges) + 1)
    den = np.bincount(dig, weights=wgt.ravel(), minlength=len(edges) + 1)
    with np.errstate(invalid="ignore"):
        expect = (L ** 3 / npart) * (num / den)[1:-1]
    P, modes, k = r.power["power"].real, r.power["modes"], r.power["k"]
    sel = (modes > 0) & (k <= np.pi * N / L)
    sel[0] = False                                           # the bin holding k = 0 (zeroed)
    sigma = expect[sel] * np.sqrt(2.0 / modes[sel])
    z = (P[sel] - expect[sel]) / sigma
    assert np.all(np.abs(z) < 5.0), z[np.argmax(np.abs(z))]
    assert sel.sum() > 50


def test_folding_against_the_oracle_on_explicitly_folded_positions():
    N, L, fold = 32, 500.0, 2
    rng = np.random.default_rng(9)
    pos = off_ties((rng.random((60000, 3)) * L).astype(np.float32), N, 2 ** fold / L)
    mesh = ab.TaylorFourierMesh(pos, L, N, order=3, fold=fold, normalize=False)
    (c, cs), scale, comp = mesh._complex_fields()
    assert cs is None and comp is None
    got = c.cpu().numpy().astype(np.complex128)
    folded = np.mod(pos.astype(np.float64) * 2 ** fold, L)
    want = tfo.tf_field(folded, None, N, 3, 1.0 / L)
    tol = tolerance(folded, None, N, 3, 1.0 / L) + 2e-5 * len(pos)
    assert np.all(np.abs(got - want) <= tol)
    assert scale == pytest.approx(1.0 / (L / 2 ** fold / N) ** 3 / 8.0 ** fold * 2.0 ** (1.5 * fold))
    assert mesh.attrs["fold"] == fold and mesh.attrs["order"] == 3


def test_estimators_on_a_taylor_fourier_mesh():
    N, L = 64, 800.0
    rng = np.random.default_rng(17)
    pos = (rng.random((300000, 3)) * L).astype(np.float32)
    halos = (rng.random((20000, 3)) * L).astype(np.float32)
    hmass = rng.lognormal(30.0, 1.0, 20000)
    pos_copy, hmass_copy = pos.copy(), hmass.copy()
    tm = ab.TaylorFourierMesh(pos, L, N, order=3)
    th = ab.TaylorFourierMesh(halos, L, N, weight=hmass, order=3)
    r1 = ab.FFTPower(tm, mode="1d")
    c = tfo.tf_field(pos, None, N, 3, 1.0 / L) / len(pos)
    want = po.fftpower_1d(c, None, N, L)
    ok = want["modes"] > 0
    np.testing.assert_allclose(r1.power["power"].real[ok], want["power"].real[ok], rtol=2e-3)
    assert np.array_equal(r1.power["modes"], want["modes"])
    r2 = ab.FFTPower(tm, mode="2d", Nmu=4, poles=[0, 2])
    np.testing.assert_allclose(r2.poles["power_0"].real[ok], r1.power["power"].real[ok], rtol=1e-5)
    # halo x matter cross spectrum, both Taylor-Fourier
    rx = ab.FFTPower(th, second=tm, mode="1d")
    ch = tfo.tf_field(halos, hmass, N, 3, 1.0 / L) / hmass.sum()
    wx = po.fftpower_1d(ch, c, N, L)
    scale = np.abs(want["power"].real[ok]).max()
    np.testing.assert_allclose(rx.power["power"].real[ok], wx["power"].real[ok], rtol=0, atol=5e-3 * scale)
    assert rx.attrs["shotnoise"] == 0.0
    xi = ab.FFTCorr(tm, mode="1d")
    assert np.all(np.isfinite(xi.corr["corr"]))
    bk = ab.FFTBispectrum(tm)
    b = bk.bispectrum
    assert len(b["B"]) > 0 and np.all(np.isfinite(b["B"]))
    S = L ** 3 / len(pos)
    np.testing.assert_allclose(b["Bshot"], S * (b["P1"] + b["P2"] + b["P3"]) - 2 * S * S, rtol=1e-12)
    assert np.all(b["Bshot"] != 0.0)
    with pytest.raises(AstrildPkError):
        ab.FFTCorr(ab.TaylorFourierMesh(pos, L, N, fold=1))
    with pytest.raises(AstrildPkError):
        ab.FFTBispectrum(ab.TaylorFourierMesh(pos, L, N, fold=1))
    assert np.array_equal(pos, pos_copy) and np.array_equal(hmass, hmass_copy)
    tpos = torch.as_tensor(pos).cuda()
    tcopy = tpos.clone()
    ab.FFTPower(ab.TaylorFourierMesh(tpos, L, N, order=2), mode="1d")
    assert torch.equal(tpos, tcopy)


def test_error_paths():
    with pytest.raises(AstrildPkError):
        ab.TaylorFourierMesh(np.zeros((4, 3)), 1.0, 16, order=5)
    eng = PkEngine(16, 1.0)
    try:
        h = __import__("ctypes").c_void_p()
        with pytest.raises(AstrildPkError, match="order"):
            _lib.call("apk_tf_create", __import__("ctypes").byref(h), eng._plan, 5)
        tp = eng.tf_plan(3)
        pos = torch.rand((1000, 3), device=eng.device)
        with pytest.raises(AstrildPkError, match="group"):
            eng.tf_field(tp, pos, group=21)
        out = eng.new_mesh()
        small = torch.empty(100, dtype=torch.uint8, device=eng.device)
        with pytest.raises(AstrildPkError, match="scratch"):
            _lib.call("apk_tf_field", tp.handle, _lib._vp(pos.data_ptr()), None, None, _lib.APK_AOS, _lib.APK_F32, 1.0,
                      None, _lib.APK_F32, 1000, 2, _lib._vp(small.data_ptr()), small.numel(), _lib._vp(out.data_ptr()),
                      eng.stream)
    finally:
        eng.close()
    slab = PkEngine(16, 1.0, x0=0, n0=8)
    try:
        with pytest.raises(AstrildPkError):
            slab.tf_plan(3)
        h = __import__("ctypes").c_void_p()
        with pytest.raises(AstrildPkError, match="single-GPU"):
            _lib.call("apk_tf_create", __import__("ctypes").byref(h), slab._plan, 3)
    finally:
        slab.close()
