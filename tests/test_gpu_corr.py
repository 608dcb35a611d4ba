"""FFTCorr on the device (astrild_b200/csrc/corr.cu) against the float64 oracle (oracle/xi_oracle.py).

(a) counts per r bin and per (r, mu) bin bit-identical to the oracle: N = 16, 33, 64; L = N and L = 500; 1d and 2d.
(b) plane waves: delta = A cos(q.x) gives xi = (A^2 / 2) cos(q.r), binned exactly on the host from the grid points; a
    cross pair with a phase shift phi gives (A^2 / 2) cos(q.r - phi), whose odd part is a nonzero dipole.
(c) Zel'dovich particles, TSC, interlaced, compensated, at 64^3 and 128^3, auto and weighted halo x matter, 1d and
    poles (0, 1, 2, 4): |xi_gpu - xi_oracle| <= TAU S (2 ell + 1) with S = sum_stored w |p(k)| (the largest |xi| any
    displacement can have).  Error model of TAU (relative to S, worst case):
      * each field c reaches the fill with a relative error (in the norm the sum weights) of at most ~4e-5: the float32
        deposit (~1e-6), the float32 r2c (~u log2 N^3 ~ 1.3e-6 at 128^3, u = 2^-24 ~ 6e-8) and the interlace /
        compensation products (a few u), with a x10 allowance for the pointwise weighting (as in the bispectrum test);
      * p = c1 conj c2: two fields, 8e-5; the product and the plane symmetrisation: a few u;
      * the C2R: ~u log2 N^3 ~ 1.3e-6 of S; the float64 binning: negligible.
    Sum: ~8.2e-5, so TAU = 1e-4.  Typical errors are one to two orders smaller.
(d) consistency: on the same complex fields the 2d monopole equals the 1d result to 1e-9 of S; xi(0) read from the
    output grid equals sum modes P / V of FFTPower with kmax past sqrt(3) k_Nyquist (every mode binned), within TAU S.
(e) paths: ArrayMesh, CatalogMesh(normalize=False) (rho_mean^2 times the normalised xi), the paint() / dx**3 RealField.
(f) the caller's complex fields are bit-identical after the call.
(g) errors: slab engine, folded box, bad dr, rmax <= rmin, Nmu < 1, more than 8 multipoles, scratch too small,
    output grid overlapping an input, not enough free memory.
"""
import numpy as np
import pytest
import torch

from oracle import bk_oracle as bo
from oracle import pk_oracle as po
from oracle import xi_oracle as xo

pytestmark = pytest.mark.gpu

TAU = 1e-4
L = 500.0


@pytest.fixture(scope="module")
def ab():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import astrild_b200
    return astrild_b200


def S_of(c1, c2=None):
    """sum over the stored half grid of w |p(k)| (normalised fields)."""
    N = c1.shape[0]
    p = np.abs(xo.product(c1, c2))
    return float((p * po.hermitian_weights(N)[None, None, :]).sum())


@pytest.mark.parametrize("N", [16, 33, 64])
@pytest.mark.parametrize("Lbox", ["N", 500.0])
@pytest.mark.parametrize("mode", ["1d", "2d"])
def test_counts_bit_identical(ab, N, Lbox, mode):
    Lb = float(N) if Lbox == "N" else Lbox
    delta = np.random.default_rng(N).standard_normal((N, N, N))
    r = ab.FFTCorr(ab.ArrayMesh(delta, BoxSize=Lb), mode=mode, Nmu=4)
    Nmu = 1 if mode == "1d" else 4
    want = xo.bin_xi(np.zeros((N, N, N)), N, Lb, xo.r_edges(N, Lb), Nmu)["nsum"][1:-1, 1:-1]
    got = r.corr["modes"]
    np.testing.assert_array_equal(got if mode == "2d" else got[:, None], want)
    np.testing.assert_array_equal(r.attrs["edges"], xo.r_edges(N, Lb))


def test_plane_waves(ab):
    N, A, phi = 32, 1.3, 0.7
    n = np.array([0, 0, 3])                         # along the line of sight
    g = np.arange(N) * (2 * np.pi / N)
    x = np.stack(np.meshgrid(g, g, g, indexing="ij"))
    qx = np.tensordot(n, x, axes=1)
    d1, d2 = A * np.cos(qx), A * np.cos(qx + phi)
    r = xo.r_axis(N, L)
    qr = np.tensordot(n * (2 * np.pi / L), np.stack(np.meshgrid(r, r, r, indexing="ij")), axes=1)
    edges = xo.r_edges(N, L)
    auto = ab.FFTCorr(ab.ArrayMesh(d1, BoxSize=L), mode="1d")
    want = xo.finish(xo.bin_xi(0.5 * A * A * np.cos(qr), N, L, edges))["corr"][:, 0]
    np.testing.assert_allclose(auto.corr["corr"], want, rtol=0, atol=1e-5 * A * A)
    cross = ab.FFTCorr(ab.ArrayMesh(d1, BoxSize=L), mode="2d", Nmu=5, poles=[0, 1, 2],
                       second=ab.ArrayMesh(d2, BoxSize=L))
    exact = xo.finish(xo.bin_xi(0.5 * A * A * np.cos(qr - phi), N, L, edges, 5, [0, 1, 2]), [0, 1, 2])["poles"]
    for ell in (0, 1, 2):
        np.testing.assert_allclose(cross.poles["corr_%d" % ell], exact["corr_%d" % ell], rtol=0, atol=1e-5 * A * A * 3)
    assert np.nanmax(np.abs(exact["corr_1"])) > 0.1 * A * A            # the dipole is real information
    assert cross.attrs["shotnoise"] == 0.0


def zeldovich(N, seed=5):
    from astrild_b200 import synthetic
    x, y, z = synthetic.zeldovich_particles(N, L, seed, torch.device("cuda"), rms_cells=1.0)
    return (x, y, z), torch.stack([x, y, z], 1).double().cpu().numpy() * L


@pytest.mark.parametrize("N", [64, 128])
def test_parity_from_particles(ab, N):
    from astrild_b200 import synthetic
    cols, pos = zeldovich(N)
    hx, hy, hz, hm = synthetic.halo_subset(cols, N ** 3 // 8, seed=2)
    hpos = torch.stack([hx, hy, hz], 1).double().cpu().numpy() * L
    kw = dict(resampler="tsc", interlaced=True, compensated=True, normalize=True, pos_scale=1.0)
    matter = ab.CatalogMesh(cols, L, N, **kw)
    halos = ab.CatalogMesh((hx, hy, hz), L, N, weight=hm, **kw)
    cm = bo.delta_k_from_particles(pos, None, N, L, "tsc", interlaced=True, compensated=True, normalize=True)
    ch = bo.delta_k_from_particles(hpos, hm.double().cpu().numpy(), N, L, "tsc", interlaced=True, compensated=True,
                                   normalize=True)
    poles = [0, 1, 2, 4]
    for first, second, c1, c2 in ((matter, None, cm, None), (halos, matter, ch, cm)):
        S = S_of(c1, c2)
        o1 = xo.fftcorr(c1, c2, N, L)
        r1 = ab.FFTCorr(first, mode="1d", second=second)
        assert np.abs(r1.corr["corr"] - o1["corr"][:, 0]).max() <= TAU * S
        o2 = xo.fftcorr(c1, c2, N, L, Nmu=5, poles=poles)
        r2 = ab.FFTCorr(first, mode="2d", Nmu=5, poles=poles, second=second)
        np.testing.assert_array_equal(r2.corr["modes"], o2["modes"])
        for ell in poles:
            err = np.abs(r2.poles["corr_%d" % ell] - o2["poles"]["corr_%d" % ell]).max()
            assert err <= TAU * S * (2 * ell + 1), (ell, err / S)
        np.testing.assert_allclose(r1.corr["r"], o1["r"][:, 0], rtol=1e-12)


def test_xi0_is_parseval_of_fftpower_monopole_is_1d_and_inputs_untouched(ab):
    N = 64
    cols, _ = zeldovich(N, seed=9)
    mesh = ab.CatalogMesh(cols, L, N, resampler="cic", interlaced=True, compensated=True, pos_scale=1.0)
    eng = mesh._eng
    (c1, c1s), s, comp = mesh._complex_fields()
    before = (c1.clone(), c1s.clone())
    xb = eng.xi_binning(compensation=comp, interlaced=True)
    grid, sums = eng.xi_raw(xb, c1, c1s)
    torch.cuda.synchronize()
    assert torch.equal(torch.view_as_real(c1), torch.view_as_real(before[0]))
    assert torch.equal(torch.view_as_real(c1s), torch.view_as_real(before[1]))
    xi0 = float(grid[0, 0, 0]) / xb.grid_scale * s * s / float(N) ** 6
    binning = eng.binning(0.0, None, 2.0 * np.pi * N / L, comp, True)
    p = eng.bin_power(binning, c1, c1s, None, None, L ** 3 * s * s / float(N) ** 6)
    ok = p["modes"] > 0
    parseval = float((p["modes"][ok] * p["power"].real[ok]).sum()) / L ** 3
    assert p["Nsum"][1:-1].sum() == N ** 3                  # every stored mode binned, with its Hermitian weight
    c = c1.cpu().numpy().astype(np.complex128) * (s / N ** 3)
    cs = c1s.cpu().numpy().astype(np.complex128) * (s / N ** 3)
    S = S_of(po.compensate(po.interlace_combine(c, cs, N, L), "cic", True, N))
    assert abs(xi0 - parseval) <= TAU * S
    # on the same fields (a new deposit is not bit-identical) the 2d monopole is the 1d result
    one = eng.finish_xi(sums.cpu().numpy(), xb, s * s / float(N) ** 6)["corr"][:, 0]
    xb2 = eng.xi_binning(Nmu=5, poles=(0, 2), compensation=comp, interlaced=True)
    two = eng.finish_xi(eng.xi_raw(xb2, c1, c1s)[1].cpu().numpy(), xb2, s * s / float(N) ** 6)["poles"]["corr_0"]
    assert np.abs(two - one).max() <= 1e-9 * S


def test_unnormalised_and_realfield_paths(ab):
    N = 64
    cols, pos = zeldovich(N, seed=3)
    norm = ab.FFTCorr(ab.CatalogMesh(cols, L, N, resampler="cic", normalize=True, pos_scale=1.0), poles=[0, 2])
    raw = ab.FFTCorr(ab.CatalogMesh(cols, L, N, resampler="cic", normalize=False, pos_scale=1.0), poles=[0, 2])
    rho = N ** 3 / L ** 3
    big = np.abs(norm.corr["corr"]) > 1e-3 * np.abs(norm.corr["corr"]).max()
    np.testing.assert_allclose(raw.corr["corr"][big], norm.corr["corr"][big] * rho ** 2, rtol=1e-4)
    np.testing.assert_allclose(raw.attrs["shotnoise"], norm.attrs["shotnoise"] * rho ** 2, rtol=1e-12)
    # paint(...) / dx**3 -> ArrayMesh stays on the device; equals the oracle on the same gridded values
    pm = ab.ParticleMesh(Nmesh=[N] * 3, BoxSize=L, resampler="cic")
    field = pm.paint(torch.stack(cols, 1) * L, resampler="cic") / (L / N) ** 3
    r = ab.FFTCorr(ab.ArrayMesh(field, BoxSize=L), mode="2d", Nmu=3, poles=[0, 2])
    c = po.r2c(po.paint(pos, 1.0, N, L, "cic") / (L / N) ** 3)
    o = xo.fftcorr(c, None, N, L, Nmu=3, poles=[0, 2])
    S = S_of(c)
    assert np.nanmax(np.abs(r.corr["corr"] - o["corr"])) <= TAU * S
    assert np.abs(r.poles["corr_2"] - o["poles"]["corr_2"]).max() <= 5 * TAU * S
    assert set(r.corr.variables) == {"r", "mu", "corr", "modes"} and r.corr.dims == ["r", "mu"]
    assert set(r.poles.variables) == {"r", "modes", "corr_0", "corr_2"}
    for key in ("shotnoise", "edges", "dr", "rmin", "rmax", "Nmu", "poles", "los", "volume"):
        assert key in r.attrs
    assert len(r.run()) == 2


def test_error_paths(ab, monkeypatch):
    from astrild_b200 import lab
    from astrild_b200._lib import AstrildPkError
    from astrild_b200.engine import PkEngine
    N = 32
    delta = np.random.default_rng(0).standard_normal((N, N, N))
    slab = PkEngine(N, L, "cuda", x0=0, n0=N // 2)
    try:
        with pytest.raises(AstrildPkError, match="single-GPU"):
            slab.xi_binning()
    finally:
        slab.close()
    cols, _ = zeldovich(16)
    with pytest.raises(AstrildPkError, match="folded"):
        ab.FFTCorr(ab.CatalogMesh(cols, L, 16, pos_scale=1.0, fold=1))
    m = ab.ArrayMesh(delta, BoxSize=L)
    with pytest.raises(AstrildPkError, match="dr must be positive"):
        ab.FFTCorr(m, dr=-1.0)
    with pytest.raises(AstrildPkError, match="must exceed rmin"):
        ab.FFTCorr(m, rmin=100.0, rmax=50.0)
    with pytest.raises(AstrildPkError, match="mu bins"):
        ab.FFTCorr(m, mode="2d", Nmu=0)
    with pytest.raises(AstrildPkError, match="multipoles"):
        ab.FFTCorr(m, poles=list(range(9)))
    eng = m._eng
    (c1, _), _, _ = m._complex_fields()
    xb = eng.xi_binning()
    if xb.scratch_bytes:
        with pytest.raises(AstrildPkError, match="scratch"):
            eng.xi_raw(xb, c1, scratch=torch.empty(1, dtype=torch.uint8, device="cuda"))
    mesh = torch.view_as_real(c1).view(N, N, eng.ldz)
    with pytest.raises(AstrildPkError, match="overlaps"):
        eng.xi_raw(xb, c1, grid=mesh)
    with pytest.raises(AstrildPkError, match="output grid"):
        eng.xi_raw(xb, c1, grid=torch.empty((N, N, N), dtype=torch.float32, device="cuda"))
    monkeypatch.setattr(lab, "_free_device_bytes", lambda device: 1000)
    with pytest.raises(AstrildPkError, match=r"needs \d+ bytes"):
        ab.FFTCorr(ab.ArrayMesh(delta, BoxSize=L))
