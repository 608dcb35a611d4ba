"""The sorted deposit on the device against the per-cell error bound of oracle/deposit_budget.py (DESIGN §4.1), at
sizes the CPU fibers cannot reach, and the non-finite contract of both methods and of `auto`
(tests/test_simt_deposit_budget.py runs the same device code on CPU fibers)."""
import numpy as np
import pytest
import torch

from oracle import deposit_budget as db
from tests.test_simt_deposit_budget import CASES, check, check_spoiled, clean, make_case, spoil

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ab():
    import astrild_b200
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return astrild_b200


@pytest.mark.parametrize("resampler", ["cic", "tsc"])
@pytest.mark.parametrize("case", CASES)
def test_paint_within_the_budget(ab, oracle_fast, case, resampler):
    rng = np.random.default_rng(CASES.index(case))
    N, L = 32, 100.0
    pos, mass = clean(*make_case(case, N, L, rng), N, L)
    pm = ab.ParticleMesh(Nmesh=[N] * 3, BoxSize=L)
    got = pm.paint(pos, mass=1.0 if mass is None else mass, resampler=resampler, method="sorted").value
    check(got, pos, mass, N, L, resampler)


@pytest.mark.parametrize("resampler", ["cic", "tsc"])
def test_deposit_pair_within_the_budget(ab, oracle_fast, resampler):
    rng = np.random.default_rng(30)
    N, L = 128, 1000.0
    pos = np.concatenate([rng.random((3_000_000, 3)) * L, rng.normal(0.5 * L, 0.02 * L, (1_000_000, 3)) % L])
    pos, _ = clean(pos.astype(np.float32), None, N, L)
    mass = np.exp(rng.normal(0.0, 1.0, len(pos))).astype(np.float32)
    eng = ab.get_engine(N, L)
    for m in (None, mass):
        a, b = (eng.store_mesh(t).cpu().numpy() for t in eng.deposit_pair(pos, m, resampler, method="sorted"))
        check(a, pos, m, N, L, resampler, pair=True)
        check(b, pos, m, N, L, resampler, pair=True, twin=True)


def test_zeldovich_256_pair_within_the_budget(ab, oracle_fast):
    """2^24 Zel'dovich particles on 256^3, TSC, interlaced pair (the shape of config 3, scaled down)."""
    from astrild_b200 import synthetic
    N, L = 256, 1.0
    x, y, z = synthetic.zeldovich_particles(256, 1000.0, 5, "cuda")
    pos = torch.stack([x, y, z], 1).cpu().numpy()
    pos, _ = clean(pos, None, N, L)
    eng = ab.get_engine(N, L)
    a, b = (eng.store_mesh(t).cpu().numpy() for t in eng.deposit_pair(pos, None, "tsc", method="sorted"))
    check(a, pos, None, N, L, "tsc", pair=True)
    check(b, pos, None, N, L, "tsc", pair=True, twin=True)


def test_halo_masses_512_within_the_budget(ab, oracle_fast):
    """10^6 halo-like mass-weighted particles on 512^3 (the shape of config 4)."""
    from astrild_b200 import synthetic
    N, L = 512, 1.0
    cols = synthetic.zeldovich_particles(128, 1000.0, 6, "cuda")
    x, y, z, m = synthetic.halo_subset(cols, 1_000_000, 7)
    pos = torch.stack([x, y, z], 1).cpu().numpy()
    mass = m.cpu().numpy()
    pos, mass = clean(pos, mass, N, L)
    pm = ab.ParticleMesh(Nmesh=[N] * 3, BoxSize=L)
    got = pm.paint(pos, mass=mass, resampler="tsc", method="sorted").value
    check(got, pos, mass, N, L, "tsc")


@pytest.mark.parametrize("method", ["sorted", "atomic", "auto"])
@pytest.mark.parametrize("what", ["nan_mass", "inf_mass", "nan_x", "inf_y"])
def test_a_non_finite_particle_spoils_only_its_own_cells(ab, oracle_fast, what, method):
    rng = np.random.default_rng(2)
    N, L = 64, 100.0
    n = 300_000 if method == "auto" else 20_000          # auto: the sorted path from 2^18 particles on
    pos, _ = clean(rng.random((n, 3)).astype(np.float32) * np.float32(L), None, N, L)
    mass = None if what in ("nan_x", "inf_y") else np.ones(len(pos), np.float32)
    i = 777
    sp, sm = spoil(pos, mass, what, i)
    eng = ab.get_engine(N, L)
    a, b = (eng.store_mesh(t).cpu().numpy() for t in eng.deposit_pair(sp, sm, "tsc", method=method))
    fin = what.endswith("mass")
    if method == "atomic":       # no bound of its own: only the non-finite cells are checked
        for got in (a, b):
            nf = ~np.isfinite(got)
            assert 1 <= nf.sum() <= 27
        return
    check_spoiled(a, pos, mass, i, N, L, "tsc", pair=True, finite_position=fin)
    check_spoiled(b, pos, mass, i, N, L, "tsc", pair=True, twin=True, finite_position=fin)


def test_catalog_mesh_with_a_nan_row_gives_nan_power(ab):
    rng = np.random.default_rng(8)
    N, L = 64, 100.0
    pos = (rng.random((300_000, 3)) * L).astype(np.float32)
    mass = np.ones(len(pos), np.float32)
    mass[12345] = np.nan
    for method in ("sorted", "atomic", "auto"):
        mesh = ab.CatalogMesh(pos, L, N, weight=mass, resampler="tsc", interlaced=True, normalize=False, method=method)
        r = ab.FFTPower(mesh, mode="1d", kmin=2 * np.pi / L)
        assert np.isnan(r.power["power"].real).any(), method


@pytest.mark.parametrize("resampler", ["cic", "tsc"])
def test_masses_near_the_float32_limit(ab, oracle_fast, resampler):
    rng = np.random.default_rng(3)
    N, L = 32, 100.0
    pos, _ = clean(rng.random((20000, 3)).astype(np.float32) * np.float32(L), None, N, L)
    mass = np.full(len(pos), 1e35, np.float32)
    got = ab.ParticleMesh(Nmesh=[N] * 3, BoxSize=L).paint(pos, mass=mass, resampler=resampler, method="sorted").value
    assert np.isfinite(got).all()
    check(got, pos, mass, N, L, resampler)
