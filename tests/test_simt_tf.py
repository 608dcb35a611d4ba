"""tf.cu's device code on CPU fibers (tests/simt): the moment grids of the NGP brick partition + moment tile kernel per
cell against the float64 oracle (oracle/tf_oracle.py) within the bound the fixed-point accumulation implies, and the
combine kernel against NumPy.

Cases: SoA / AoS, float32 / float64 positions and masses, bricks of several chunks (more than 8191 particles), folded
positions (many box lengths outside the mesh's box), a non-finite row, moment groups split over several tile launches.

The per-cell bound, for moment alpha of degree t = |alpha|, summed over the particles p of the cell:
  * fixed point: the quantum of a chunk is 2^-(s + t) unit with (sum |m| / unit) 2^s >= 2^30 / 1.001, so each
    particle's rounding is at most q_t / 2 = 1.001 * 2^-31 * 2^-t * sum |m| (the chunk's sum, bounded by the total);
  * float32 arithmetic: the payload coordinate (brick-local, < 32 cells) carries a few ulp, dl <= 1e-5 cells, so
    |d^alpha| moves by at most t 2^-(t-1) dl; the mass is rounded to float32 (2^-24) and the product of up to
    ORDER + 1 float32 factors adds (ORDER + 2) 2^-24 |m d^alpha|;
  * the flush converts the cell's integer to float32 and adds it to the mesh once per chunk: 2^-24 |M| per chunk.
Particles within 1e-4 cells of a rounding tie are moved off it (a tie may file a particle under either neighbour).
"""
import ctypes as ct
import os
import sys
from math import comb

import numpy as np
import pytest

from oracle import tf_oracle as tfo

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "simt"))


@pytest.fixture(scope="module")
def simt_tf():
    import build_simt_tf
    lib = ct.CDLL(build_simt_tf.build_tf())
    vp, i = ct.c_void_p, ct.c_int
    lib.simt_tf_moments.restype = i
    lib.simt_tf_moments.argtypes = [vp, vp, vp, i, i, vp, i, ct.c_longlong, i, ct.c_double, i, i, i, vp, i]
    lib.simt_tf_combine.restype = i
    lib.simt_tf_combine.argtypes = [vp, i, i, i, i, i, vp]
    return lib


def hp(a):
    return None if a is None else a.ctypes.data_as(ct.c_void_p)


def off_ties(pos, N, pos_scale):
    """positions moved by at most 2e-4 cells so that no coordinate is within 1e-4 cells of a rounding tie"""
    g = pos.astype(np.float64) * (pos_scale * N)
    f = g - np.floor(g)
    near = np.abs(f - 0.5) < 1e-4
    g = np.where(near, np.floor(g) + 0.5 + np.where(f >= 0.5, 2e-4, -2e-4), g)
    return (g / (pos_scale * N)).astype(pos.dtype)


def run_moments(lib, pos, mass, N, pos_scale, order, k0, G, soa):
    ldz = 2 * (N // 2 + 1)
    meshes = np.zeros((G, N, N, ldz), dtype=np.float32)
    if soa:
        cols = [np.ascontiguousarray(pos[:, d]) for d in range(3)]
        p0, p1, p2 = cols
    else:
        p0, p1, p2 = np.ascontiguousarray(pos), None, None
    assert lib.simt_tf_moments(hp(p0), hp(p1), hp(p2), int(soa), int(pos.dtype == np.float64), hp(mass),
                               int(mass is not None and mass.dtype == np.float64), len(pos), N, pos_scale, order, k0, G,
                               hp(meshes), 2) == 0
    return meshes[..., :N].astype(np.float64)


def cell_bound(pos, mass, N, pos_scale, order):
    """per moment and cell: the bound of the module docstring (float64 (n_mom, N, N, N))"""
    h, d = tfo.grid_offsets(pos, N, pos_scale)
    m = np.abs(np.broadcast_to(np.asarray(1.0 if mass is None else mass, dtype=np.float64), (len(pos),)))
    m = np.where(np.isfinite(m), m, 0.0)
    total = m.sum()
    idx = (h[:, 0] * N + h[:, 1]) * N + h[:, 2]
    chunks = 1 + np.bincount(idx, minlength=N ** 3) // 8191 + 1
    dl = 1e-5
    out = []
    for a, b, c in tfo.multi_indices(order):
        t = a + b + c
        q = 1.001 * 2.0 ** -31 * 2.0 ** -t * total
        ad = np.abs(d[:, 0] ** a * d[:, 1] ** b * d[:, 2] ** c)
        per = q / 2 + m * (t * 2.0 ** -(t - 1) * dl + (order + 2) * 2.0 ** -24 * ad)
        cell = np.bincount(idx, weights=per, minlength=N ** 3)
        absum = np.bincount(idx, weights=m * ad, minlength=N ** 3)
        out.append(cell + chunks * 2.0 ** -24 * absum + 1e-30)
    return np.asarray(out).reshape(-1, N, N, N)


CASES = [
    # N, npart, soa, pos dtype, mass dtype or None, fold, order, k0, G
    (16, 3000, False, np.float32, None, 0, 3, 0, 20),
    (16, 3000, True, np.float64, np.float32, 0, 3, 0, 20),
    (33, 4000, True, np.float32, np.float64, 0, 2, 0, 10),
    (33, 4000, False, np.float64, None, 2, 4, 10, 12),          # folded positions; moments 10 .. 21 in two launches
    (16, 20000, False, np.float32, np.float32, 0, 1, 0, 4),       # one brick, three chunks
]


@pytest.mark.parametrize("N,npart,soa,pdt,mdt,fold,order,k0,G", CASES)
def test_moment_grids_per_cell_within_the_fixed_point_bound(simt_tf, N, npart, soa, pdt, mdt, fold, order, k0, G):
    rng = np.random.default_rng(N * 7 + npart + order)
    if npart > 10000:
        pos = rng.random((npart, 3)) * np.array([0.5, 0.25, 1.0])     # 8 x 4 x 16 cells: one brick
    else:
        pos = rng.random((npart, 3)) * 2.0 ** fold - 0.3
    pos_scale = 2.0 ** fold
    pos = off_ties(pos.astype(pdt), N, pos_scale)
    mass = None if mdt is None else (rng.lognormal(0.0, 1.5, npart) * rng.choice([-1.0, 1.0], npart)).astype(mdt)
    got = run_moments(simt_tf, pos, mass, N, pos_scale, order, k0, G, soa)
    want = tfo.moments(pos, mass, N, order, pos_scale)[k0:k0 + G]
    bound = cell_bound(pos, mass, N, pos_scale, order)[k0:k0 + G]
    err = np.abs(got - want)
    assert np.all(err <= bound), (np.unravel_index(np.argmax(err / bound), err.shape), (err / bound).max())
    assert len(tfo.multi_indices(order)) == comb(order + 3, 3)


def test_non_finite_row_puts_nan_at_its_home_cell_and_leaves_the_others(simt_tf):
    N, npart, order = 16, 2000, 2
    rng = np.random.default_rng(11)
    pos = off_ties(rng.random((npart, 3)).astype(np.float32), N, 1.0)
    mass = rng.random(npart).astype(np.float32)
    bad = 777
    mass[bad] = np.nan
    got = run_moments(simt_tf, pos, mass, N, 1.0, order, 0, 10, False)
    h, _ = tfo.grid_offsets(pos[bad:bad + 1], N, 1.0)
    hx, hy, hz = h[0]
    assert np.all(np.isnan(got[:, hx, hy, hz]))
    keep = np.ones(npart, bool)
    keep[bad] = False
    want = tfo.moments(pos[keep], mass[keep], N, order, 1.0)
    bound = cell_bound(pos[keep], mass[keep], N, 1.0, order)
    ok = np.ones((N, N, N), bool)
    ok[hx, hy, hz] = False
    assert np.all(np.abs(got - want)[:, ok] <= bound[:, ok])


@pytest.mark.parametrize("N,k0,G,accumulate", [(8, 0, 20, 0), (9, 4, 6, 1), (12, 10, 25, 1)])
def test_combine_matches_numpy(simt_tf, N, k0, G, accumulate):
    rng = np.random.default_rng(N + k0)
    Nk = N // 2 + 1
    mom = (rng.standard_normal((G, N, N, Nk)) + 1j * rng.standard_normal((G, N, N, Nk))).astype(np.complex64)
    out = (rng.standard_normal((N, N, Nk)) + 1j * rng.standard_normal((N, N, Nk))).astype(np.complex64)
    before = out.astype(np.complex128)
    assert simt_tf.simt_tf_combine(hp(mom), N, k0, G, accumulate, 3, hp(out)) == 0
    # the oracle's combine of moments k0 .. k0 + G - 1 (the others zero), with float32 coefficient tables
    full = np.zeros((35, N, N, Nk), dtype=np.complex128)
    full[k0:k0 + G] = mom
    w = tfo.axis_w(N)
    want = np.zeros((N, N, Nk), dtype=np.complex128)
    from math import factorial
    for k, (a, b, c) in enumerate(tfo.multi_indices(4)):
        ta = (w ** a / factorial(a)).astype(np.float32).astype(np.float64)
        tb = (w ** b / factorial(b)).astype(np.float32).astype(np.float64)
        coef = ta[:, None, None] * tb[None, :, None] * ((w[:Nk] ** c / factorial(c)).astype(np.float32).astype(np.float64))[None, None, :]
        want += (-1j) ** (a + b + c) * coef * full[k]
    if accumulate:
        want += before
    scale = sum(np.abs(full[k]) * 10.0 for k in range(35)).max() + np.abs(before).max()
    np.testing.assert_allclose(out, want, rtol=0, atol=2e-6 * scale)
