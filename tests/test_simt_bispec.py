"""bispec.cu's device code on CPU fibers (tests/simt): the shell fill's mode totals against the 1-D binning kernel's
nmodes, and the float32 / float64 triple-product reductions against a float64 NumPy einsum on random fields.

The reduction cases cover chunk edges (N^3 not a multiple of the 64-point chunk, several CTAs splitting the chunks),
the padding columns of the mesh rows (filled with huge values: they must never be read), shell counts that are not a
multiple of the register tile, and tiles that are only partly made of kept triples.
"""
import ctypes as ct
import os
import sys

import numpy as np
import pytest

import tests.test_simt_bin_power as tbp
from oracle import bk_oracle as bo

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "simt"))
L = 100.0


@pytest.fixture(scope="module")
def simt_bk():
    import build_simt_bispec
    lib = ct.CDLL(build_simt_bispec.build_bispec())
    lib.simt_bk_fill.restype = ct.c_int
    lib.simt_bk_fill.argtypes = [ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_void_p, ct.c_void_p, ct.c_int, ct.c_void_p,
                                 ct.c_void_p, ct.c_int, ct.c_int, ct.c_void_p]
    for name in ("simt_bk_reduce_f32", "simt_bk_reduce_f64"):
        fn = getattr(lib, name)
        fn.restype = ct.c_int
        fn.argtypes = [ct.c_void_p, ct.c_int, ct.c_int, ct.c_void_p, ct.c_int, ct.c_int, ct.c_void_p]
    return lib


@pytest.fixture(scope="module")
def simt_bin():
    import build_simt
    lib = ct.CDLL(build_simt.build_bin())
    lib.simt_bin_power.restype = ct.c_int
    lib.simt_bin_power.argtypes = [ct.c_void_p] * 4 + [ct.c_int] * 3 + [ct.c_void_p] * 5 + [ct.c_int] + [ct.c_void_p] * 6 + [
        ct.c_int, ct.c_int, ct.c_int] + [ct.c_void_p] * 4
    return lib


def hp(a):
    return None if a is None else a.ctypes.data_as(ct.c_void_p)


@pytest.mark.parametrize("N,kmin", [(16, 0.0), (15, 2 * np.pi / L), (12, 0.0)])
def test_fill_mode_totals_equal_bin_power_nmodes(simt_bk, simt_bin, N, kmin):
    from astrild_b200 import tables
    k = np.ascontiguousarray(tables.k_axis(N, L))
    edges = np.ascontiguousarray(bo.default_edges(N, L, kmin=kmin, kmax=np.pi * N / L))
    nb, Nk = len(edges) - 1, N // 2 + 1
    rng = np.random.default_rng(N)
    c = (rng.standard_normal((N, N, Nk)) + 1j * rng.standard_normal((N, N, Nk))).astype(np.complex64)
    fields = np.zeros((nb, N, N, Nk), dtype=np.complex128)         # double2: the indicator variant
    assert simt_bk.simt_bk_fill(None, None, N, hp(k), hp(edges), len(edges), None, None, 1, 3, hp(fields)) == 0
    wz = tables.hermitian_weights(N)
    totals = ((fields.real != 0) * wz[None, None, None, :]).reshape(nb, -1).sum(axis=1).astype(np.int64)
    # the 1-D binning's default edges (kmax = pi N / L + dk / 2) start with these: same arange, one more edge
    nmodes = np.asarray(tbp.bin_power(simt_bin, N, L, c, kmin=kmin)["modes"], dtype=np.int64)[:nb].copy()
    if kmin == 0.0:
        nmodes[0] -= 1                                            # the 1-D binning counts k = 0 in its first bin
    np.testing.assert_array_equal(totals, nmodes)
    assert np.all(fields.imag == 0) and np.all((fields.real == 0) | (fields.real == 1))
    # the data fill writes the interlaced, compensated value of each mode into its shell and nowhere else
    cs = (rng.standard_normal((N, N, Nk)) + 1j * rng.standard_normal((N, N, Nk))).astype(np.complex64)
    comp = np.ascontiguousarray(tables.compensation_axis("tsc", True, N))
    ph = np.ascontiguousarray(tables.interlace_phase_axis(N, L))
    ff = np.zeros((nb, N, N, Nk), dtype=np.complex64)
    assert simt_bk.simt_bk_fill(hp(c), hp(cs), N, hp(k), hp(edges), len(edges), hp(comp), hp(ph), 0, 2, hp(ff)) == 0
    want = (0.5 * (c + cs * np.exp(1j * ((ph[:, None, None] + ph[None, :, None]) + ph[None, None, :Nk])))
            / (comp[:, None, None] * comp[None, :, None] * comp[None, None, :Nk]))
    mask = fields.real != 0
    for b in range(nb):
        np.testing.assert_allclose(ff[b][mask[b]], want[mask[b]], rtol=2e-6, atol=2e-6 * np.abs(want).max())
        assert np.all(ff[b][~mask[b]] == 0)


def padded(F, N, fill):
    """(nb, N^3) -> [nb][N][N][2 (N/2+1)] with the two padding floats of every row set to ``fill``."""
    nb = F.shape[0]
    out = np.full((nb, N, N, 2 * (N // 2 + 1)), fill, dtype=F.dtype)
    out[..., :N] = F.reshape(nb, N, N, N)
    return np.ascontiguousarray(out)


@pytest.mark.parametrize("N,nb,ctas", [(10, 11, 3), (16, 13, 1), (9, 5, 4)])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_reduction_matches_einsum(simt_bk, N, nb, ctas, dtype):
    rng = np.random.default_rng(nb * N)
    F = rng.standard_normal((nb, N ** 3)).astype(dtype)
    # kept triples of a uniform shell set (the band l <= i + j + 1), so the tiles are partly skipped
    edges = np.arange(nb + 1) * (2 * np.pi / L)
    triples = np.ascontiguousarray(bo.kept_triples(edges, 4 * nb, L).astype(np.int32))
    assert len(triples) < nb * (nb + 1) * (nb + 2) // 6
    out = np.zeros(len(triples))
    fn = simt_bk.simt_bk_reduce_f32 if dtype == np.float32 else simt_bk.simt_bk_reduce_f64
    big = np.float32(3e38) if dtype == np.float32 else 1e300
    assert fn(hp(padded(F, N, big)), N, nb, hp(triples), len(triples), ctas, hp(out)) == 0
    F64 = F.astype(np.float64)
    want = np.einsum("tp,tp,tp->t", F64[triples[:, 0]], F64[triples[:, 1]], F64[triples[:, 2]])
    scale = np.einsum("tp,tp,tp->t", *(np.abs(F64[triples[:, s]]) for s in range(3)))
    # float32: products rounded (2u) and sums over <= 1024 points in float32 (gamma_1024 = 1024 u) -> 1e-4 of the scale
    tol = 1e-4 if dtype == np.float32 else 1e-12
    assert np.all(np.abs(out - want) <= tol * scale)
