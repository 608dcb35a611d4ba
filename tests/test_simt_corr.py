"""corr.cu's device code on CPU fibers (tests/simt): the plane-symmetrising fill against NumPy, and the real-space
binning's counts (bit for bit) and sums against the oracle (oracle/xi_oracle.py).

The fill cases cover even and odd N, auto and cross, plain and interlaced + compensated fields; on the self-paired planes
the two members of every mirrored pair must come out as exact conjugates and the self-paired points with a zero
imaginary part -- the property that makes the C2R's result defined.  The binning cases cover the 1-D path and the
(r, mu) path with multipoles and an oblique line of sight, grids whose padding floats hold huge values (they must never
be read), edges that grid points lie on exactly, several CTAs, and the two private histograms' fold.
"""
import ctypes as ct
import os
import sys

import numpy as np
import pytest

from oracle import pk_oracle as po
from oracle import xi_oracle as xo

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "simt"))


@pytest.fixture(scope="module")
def simt_xi():
    import build_simt_corr
    lib = ct.CDLL(build_simt_corr.build_corr())
    lib.simt_xi_fill.restype = ct.c_int
    lib.simt_xi_fill.argtypes = [ct.c_void_p] * 4 + [ct.c_int, ct.c_void_p, ct.c_void_p, ct.c_float, ct.c_int, ct.c_void_p]
    lib.simt_xi_bin.restype = ct.c_int
    lib.simt_xi_bin.argtypes = [ct.c_void_p, ct.c_int, ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_int, ct.c_void_p, ct.c_int,
                                ct.c_void_p, ct.c_double, ct.c_int, ct.c_int, ct.c_void_p]
    return lib


def hp(a):
    return None if a is None else a.ctypes.data_as(ct.c_void_p)


def cfield(rng, N):
    Nk = N // 2 + 1
    return (rng.standard_normal((N, N, Nk)) + 1j * rng.standard_normal((N, N, Nk))).astype(np.complex64)


@pytest.mark.parametrize("N", [8, 9, 12])
@pytest.mark.parametrize("cross", [False, True])
@pytest.mark.parametrize("interlaced", [False, True])
def test_fill_matches_numpy_and_pairs_are_exact_conjugates(simt_xi, N, cross, interlaced):
    L = 100.0
    rng = np.random.default_rng(N * 4 + 2 * cross + interlaced)
    c1 = cfield(rng, N)
    c1s = cfield(rng, N) if interlaced else None
    c2 = cfield(rng, N) if cross else None
    c2s = cfield(rng, N) if (cross and interlaced) else None
    comp = np.ascontiguousarray(po.compensation_1d("tsc", True, N)) if interlaced else None
    phase = np.ascontiguousarray(0.5 * po.k_tables(N, L)[0] * (L / N)) if interlaced else None
    fac = 2.0 ** -9
    out = np.full(c1.shape, np.nan + 1j * np.nan, dtype=np.complex64)
    assert simt_xi.simt_xi_fill(hp(c1), hp(c1s), hp(c2), hp(c2s), N, hp(comp), hp(phase), fac, 3, hp(out)) == 0

    def combined(c, cs):
        c = c.astype(np.complex128)
        if cs is None:
            return c
        return po.compensate(po.interlace_combine(c, cs.astype(np.complex128), N, L), "tsc", True, N)

    a = combined(c1, c1s)
    b = None if c2 is None else combined(c2, c2s)
    want = xo.plane_symmetrised(xo.product(a, b), N) * fac
    np.testing.assert_allclose(out, want, rtol=0, atol=2e-6 * np.abs(want).max())
    mirror = (-np.arange(N)) % N
    for iz in ([0, N // 2] if N % 2 == 0 else [0]):
        plane = out[:, :, iz]
        assert np.array_equal(plane, np.conj(plane[mirror][:, mirror])), f"plane {iz} is not exactly Hermitian"
        self_paired = [i for i in range(N) if mirror[i] == i]
        for ia in self_paired:
            for ib in self_paired:
                assert plane[ia, ib].imag == 0.0
    assert out[0, 0, 0] == 0


def padded_grid(rng, N):
    g = np.full((N, N, 2 * (N // 2 + 1)), 3e30, dtype=np.float32)      # padding: never read
    g[..., :N] = rng.standard_normal((N, N, N)).astype(np.float32)
    return g


@pytest.mark.parametrize("N,L,dr,rmax", [(16, 16.0, None, None), (9, 500.0, None, None), (12, 500.0, 23.0, 300.0),
                                         (16, 500.0, None, 450.0)])
@pytest.mark.parametrize("Nmu,poles,los", [(1, [], (0.0, 0.0, 1.0)), (4, [0, 2, 4], (0.0, 0.0, 1.0)),
                                           (3, [0, 1, 2, 3], (0.48, -0.6, 0.64))])
def test_binning_counts_bit_for_bit_and_sums(simt_xi, N, L, dr, rmax, Nmu, poles, los):
    rng = np.random.default_rng(N + Nmu)
    g = padded_grid(rng, N)
    xi = g[..., :N].astype(np.float64)
    edges = np.ascontiguousarray(xo.r_edges(N, L, dr=dr, rmax=rmax))
    r = np.ascontiguousarray(xo.r_axis(N, L))
    ells = np.asarray(sorted(set([0] + poles)), dtype=np.int32)
    la = np.asarray(los, dtype=np.float64)
    nb = (len(edges) + 1) * (Nmu + 2)
    geo = np.zeros((3, nb))
    assert simt_xi.simt_xi_bin(hp(g), N, hp(r), hp(edges), len(edges), Nmu, hp(ells), len(ells), hp(la), 1.0, 1, 5, hp(geo)) == 0
    mu_path = not (Nmu == 1 and len(ells) == 1)
    data = np.zeros((len(ells) if mu_path else 1, nb))
    fac = 2.0 ** -7
    assert simt_xi.simt_xi_bin(hp(g), N, hp(r), hp(edges), len(edges), Nmu, hp(ells), len(ells), hp(la), fac, 0, 4, hp(data)) == 0
    want = xo.bin_xi(xi, N, L, edges, Nmu, poles, los)
    shape = (len(edges) + 1, Nmu + 2)
    vis = (slice(1, -1), slice(1, -1))
    counts = geo[2].view(np.int64).reshape(shape)
    np.testing.assert_array_equal(counts[vis], want["nsum"][vis])
    assert counts[0].sum() == 0 and counts[-1].sum() == 0               # under/overflow rows are not accumulated
    np.testing.assert_allclose(geo[0].reshape(shape)[vis], want["rsum"][vis], rtol=1e-12)
    if mu_path:
        np.testing.assert_allclose(geo[1].reshape(shape)[vis], want["musum"][vis], rtol=1e-12, atol=1e-12)
    else:
        assert np.all(geo[1] == 0)
    scale = np.abs(xi).sum() * (2 * max(ells) + 1)
    for i in range(data.shape[0]):
        np.testing.assert_allclose(data[i].reshape(shape)[vis] * fac, want["ysum"][i][vis], rtol=0, atol=1e-12 * scale)
