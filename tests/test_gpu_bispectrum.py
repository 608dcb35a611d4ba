"""FFTBispectrum on the device (astrild_b200/csrc/bispec.cu) against the float64 oracle (oracle/bk_oracle.py).

(a) triangle counts: bit for bit against the brute force (N = 16, 24) and the oracle's rounded float64 counts (N = 64,
    128); the reported residual of the float64 counts is < 1e-3.
(b) plane waves: delta = sum_a 2 A_a cos(q_a.x + phi_a) with q1 + q2 + q3 = 0 in three shells gives
    B = V^2 2 Re(prod A_a e^{i phi_a}) / N_tri for that triple and nothing above the float32 floor elsewhere.
(c) Zel'dovich particles, TSC, interlaced, compensated: |B_gpu - B_oracle| <= TAU A with A the oracle's absolute-value
    estimator (L^6 s^3 / N^9) sum_x |F_i F_j F_l| / T_D.
    Error model of TAU (relative to A, worst case):
      * each shell field F_b reaches the reduction with a relative error (in the norm that weights the sum) of at most
        ~4e-5: the float32 deposit (per-cell sums of <= 8191-particle chunks in fixed point, ~1e-6), the float32 r2c and
        c2r (~u log2(N^3) ~ 1.3e-6 each at 128^3, u = 2^-24 ~ 6e-8) and the float32 interlace / compensation products
        (a few u), with a x10 allowance for the fields' pointwise (not rms) weighting in the triple sum;
      * three fields: 3 x 4e-5 = 1.2e-4;
      * the reduction: float32 sums over at most 1024 points, then float64: gamma_1024 = 1024 u = 6.1e-5 worst case;
      * the products F_i F_j F_l: 2u.
    Sum: ~1.9e-4, so TAU = 2e-4.  Typical errors (random-walk rounding) are one to two orders smaller.
    k1..k3 and P1..P3 equal FFTPower(mode="1d") of the same edges.
(d) ArrayMesh and CatalogMesh(normalize=False) paths.
(e) errors: slab engine, more shells than the cap, not enough memory (mocked free-memory figure), kmax beyond Nyquist,
    cross bispectra.
"""
import numpy as np
import pytest
import torch

from oracle import bk_oracle as bo
from oracle import pk_oracle as po

pytestmark = pytest.mark.gpu

TAU = 2e-4
L = 500.0


@pytest.fixture(scope="module")
def ab():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import astrild_b200
    return astrild_b200


def ntri_all(res):
    return {tuple(int(v) for v in b): int(n) for b, n in zip(res["bins"], res["triangles"])}


@pytest.mark.parametrize("N", [16, 24])
def test_counts_equal_bruteforce(ab, N):
    edges = bo.default_edges(N, L, kmax=np.pi * N / L)          # up to Nyquist: aliased triangles included
    delta = np.random.default_rng(N).standard_normal((N, N, N))
    r = ab.FFTBispectrum(ab.ArrayMesh(delta, BoxSize=L), kmax=np.pi * N / L)
    bf = bo.bispectrum_bruteforce(delta, L, edges)
    want = {tuple(int(v) for v in t): int(n) for t, n in zip(bf["triples"], bf["ntri"]) if n > 0}
    assert ntri_all(r.bispectrum) == want
    assert r.attrs["count_residual"] < 1e-3
    np.testing.assert_array_equal(r.attrs["edges"], edges)


@pytest.mark.parametrize("N,dk_f", [(64, 1), (128, 4)])
def test_counts_equal_oracle_float64(ab, N, dk_f):
    dk = dk_f * 2 * np.pi / L
    edges = bo.default_edges(N, L, dk=dk)
    delta = np.random.default_rng(1).standard_normal((N, N, N)).astype(np.float32)
    r = ab.FFTBispectrum(ab.ArrayMesh(delta, BoxSize=L), dk=dk)
    triples = bo.kept_triples(edges, N, L)
    TD = bo.triple_sums(bo.shell_fields(None, N, L, edges), triples)
    ntri = np.rint(TD / float(N) ** 3).astype(np.int64)
    want = {tuple(int(v) for v in t): int(n) for t, n in zip(triples, ntri) if n > 0}
    assert ntri_all(r.bispectrum) == want
    assert r.attrs["count_residual"] < 1e-3


def test_plane_waves_known_answer(ab):
    N = 64
    n = np.array([[3, 0, 0], [0, 4, 0], [-3, -4, 0]])
    A = np.array([0.8, 1.1, 0.6])
    phi = np.array([0.3, 1.1, -0.5])
    g = np.arange(N) * (2 * np.pi / N)
    x = np.stack(np.meshgrid(g, g, g, indexing="ij"))
    delta = sum(2 * A[a] * np.cos(np.tensordot(n[a], x, axes=1) + phi[a]) for a in range(3))
    r = ab.FFTBispectrum(ab.ArrayMesh(delta, BoxSize=L))
    res = r.bispectrum
    bins = [tuple(int(v) for v in b) for b in res["bins"]]
    t = bins.index((3, 4, 5))                        # |q| = 3, 4, 5 fundamentals, dk = k_f
    V = L ** 3
    want = V * V * 2 * np.real(np.prod(A * np.exp(1j * phi))) / res["triangles"][t]
    np.testing.assert_allclose(res["B"][t], want, rtol=1e-5)
    # every other triple holds at most one of the waves' modes per side: float32 leakage only
    others = np.delete(res["B"], t)
    assert np.abs(others).max() < 1e-5 * V * V * np.prod(A)
    assert res["Bshot"].tolist() == [0.0] * len(res["B"])


def zeldovich(N, seed=5):
    from astrild_b200 import synthetic
    x, y, z = synthetic.zeldovich_particles(N, L, seed, torch.device("cuda"), rms_cells=1.0)
    return (x, y, z), torch.stack([x, y, z], 1).double().cpu().numpy() * L


@pytest.mark.parametrize("N,dk_f", [(64, 1), (128, 2)])
def test_parity_from_particles(ab, N, dk_f):
    dk = dk_f * 2 * np.pi / L
    cols, pos = zeldovich(N)
    mesh = ab.CatalogMesh(cols, L, N, resampler="tsc", interlaced=True, compensated=True, normalize=True, pos_scale=1.0)
    r = ab.FFTBispectrum(mesh, dk=dk)
    res = r.bispectrum
    edges = bo.default_edges(N, L, dk=dk)
    c = bo.delta_k_from_particles(pos, None, N, L, "tsc", interlaced=True, compensated=True, normalize=True)
    o = bo.bispectrum_fft(c, N, L, edges, with_abs=True)
    keep = o["ntri"] > 0
    assert np.array_equal(res["bins"], o["triples"][keep])
    assert np.array_equal(res["triangles"], o["ntri"][keep])
    err = np.abs(res["B"] - o["B"][keep])
    worst = float(np.max(err / o["A"][keep]))
    assert worst <= TAU, f"largest |B_gpu - B_oracle| / A = {worst:.3g}"
    # the sides' k and P are FFTPower's of the same edges
    p = ab.FFTPower(ab.CatalogMesh(cols, L, N, resampler="tsc", interlaced=True, compensated=True, normalize=True,
                                   pos_scale=1.0), mode="1d", kmin=0.0, dk=dk, kmax=r.attrs["kmax"])
    b = res["bins"]
    for s in range(3):
        np.testing.assert_array_equal(res["k%d" % (s + 1)], p.power["k"][b[:, s]])
        np.testing.assert_allclose(res["P%d" % (s + 1)], p.power["power"].real[b[:, s]], rtol=1e-5)
    S = mesh.shotnoise
    np.testing.assert_allclose(res["Bshot"], S * (res["P1"] + res["P2"] + res["P3"]) - 2 * S * S, rtol=1e-12)


def test_catalog_unnormalised_and_array_paths(ab):
    N = 64
    cols, pos = zeldovich(N, seed=9)
    norm = ab.FFTBispectrum(ab.CatalogMesh(cols, L, N, resampler="cic", normalize=True, pos_scale=1.0)).bispectrum
    raw = ab.FFTBispectrum(ab.CatalogMesh(cols, L, N, resampler="cic", normalize=False, pos_scale=1.0)).bispectrum
    rho = N ** 3 / L ** 3                         # unit masses: mean density
    big = np.abs(norm["B"]) > 1e-2 * np.abs(norm["B"]).max()
    np.testing.assert_allclose(raw["B"][big], norm["B"][big] * rho ** 3, rtol=1e-3)
    np.testing.assert_allclose(raw["Bshot"], norm["Bshot"] * rho ** 3, rtol=1e-6)
    # ArrayMesh of the painted field: the same B as the oracle on the same gridded values
    field = po.paint(pos, 1.0, N, L, "cic")
    r = ab.FFTBispectrum(ab.ArrayMesh(field, BoxSize=L))
    o = bo.bispectrum_fft(po.r2c(field), N, L, bo.default_edges(N, L), with_abs=True)
    keep = o["ntri"] > 0
    assert np.max(np.abs(r.bispectrum["B"] - o["B"][keep]) / o["A"][keep]) <= TAU
    assert set(r.bispectrum.variables) == {"k1", "k2", "k3", "bins", "B", "triangles", "P1", "P2", "P3", "Bshot"}
    for key in ("edges", "Nmesh", "BoxSize", "shotnoise", "kmin", "dk", "kmax"):
        assert key in r.attrs
    # per-particle weights: Bshot is not defined by the Poisson formula
    w = torch.ones(N ** 3, device="cuda", dtype=torch.float32)
    rw = ab.FFTBispectrum(ab.CatalogMesh(cols, L, N, weight=w, resampler="cic", pos_scale=1.0)).bispectrum
    assert np.isnan(rw["Bshot"]).all()


def test_error_paths(ab, monkeypatch):
    from astrild_b200 import lab
    from astrild_b200._lib import AstrildPkError
    from astrild_b200.engine import PkEngine
    N = 32
    delta = np.random.default_rng(0).standard_normal((N, N, N))
    slab = PkEngine(N, L, "cuda", x0=0, n0=N // 2)
    try:
        with pytest.raises(AstrildPkError, match="single-GPU"):
            slab.bispec_binning()
    finally:
        slab.close()
    with pytest.raises(AstrildPkError, match="at most 128"):
        ab.FFTBispectrum(ab.ArrayMesh(delta, BoxSize=L), dk=0.05 * 2 * np.pi / L)
    with pytest.raises(AstrildPkError, match="Nyquist"):
        ab.FFTBispectrum(ab.ArrayMesh(delta, BoxSize=L), kmax=1.01 * np.pi * N / L)
    m = ab.ArrayMesh(delta, BoxSize=L)
    with pytest.raises(AstrildPkError, match="auto-bispectra"):
        ab.FFTBispectrum(m, second=ab.ArrayMesh(delta * 2, BoxSize=L))
    monkeypatch.setattr(lab, "_free_device_bytes", lambda device: 1000)
    with pytest.raises(AstrildPkError, match=r"needs \d+ bytes.*larger dk"):
        ab.FFTBispectrum(ab.ArrayMesh(delta, BoxSize=L))
