"""The sorted deposit's device code on CPU fibers (tests/simt) against a per-cell error bound derived from the oracle
(oracle/deposit_budget.py, DESIGN §4.1), in every cell -- also in the light cells of a clustered or mass-weighted field,
which a tolerance scaled by the heaviest cell does not see -- plus non-finite and very large masses.

The bound holds however the partition splits a brick into chunks; the mutants at the end show that it is tight enough
to catch a wrong rounding mode, a loosened overflow rule and a mis-scaled flush.
"""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "simt"))

from oracle import deposit_budget as db  # noqa: E402
from tests.test_simt_deposit import deposit, load  # noqa: E402

U = 2.0 ** -24


@pytest.fixture(scope="module", params=[0, 1], ids=["rot0", "rot1"])
def simt(request):
    import build_simt
    return load(build_simt.build_rot(request.param))


def make_case(name, N, L, rng, dtype=np.float32):
    """-> (pos, mass or None)"""
    H = L / N
    if name == "uniform":
        pos, mass = rng.random((20000, 3)) * L, None
    elif name == "clump":          # > 8191 particles in one brick: several chunks, plus a uniform background
        pos = np.concatenate([rng.random((12000, 3)) * [10 * H, 5 * H, 12 * H] + 2 * H, rng.random((3000, 3)) * L])
        mass = None
    elif name == "pareto":         # halo-like masses over five decades
        pos = rng.random((15000, 3)) * L
        mass = np.minimum(1.0 / (1.0 - rng.random(len(pos))), 1e5)
    elif name == "heavy_light":    # one particle of mass 1e5 and 4000 of mass 1 in a clump 1.6 cells wide
        pos = np.concatenate([[[10.3 * H, 10.3 * H, 10.3 * H]], 10 * H + rng.random((4000, 3)) * 1.6 * H])
        mass = np.concatenate([[1e5], np.ones(4000)])
    elif name == "negative":
        pos = rng.random((15000, 3)) * L
        mass = rng.normal(0.0, 1.0, len(pos))
    elif name == "pow2":           # masses whose powers of two sit exactly at the chunk's top
        pos = rng.random((12000, 3)) * L
        mass = 2.0 ** rng.integers(-3, 4, len(pos)).astype(np.float64)
        mass[::97] = 8.0
    else:
        raise ValueError(name)
    pos = pos.astype(dtype)
    return pos, (None if mass is None else mass.astype(np.float32))


def clean(pos, mass, N, L):
    """Drops the particles within 1e-3 cells of a tie of a home cell (CIC, TSC, either mesh of the pair)."""
    g = pos.astype(np.float64) * (N / L)
    keep = np.ones(len(pos), bool)
    for off in (0.0, 0.5, 1.0):
        t = g + off
        keep &= (np.abs(t - np.rint(t)) >= 1e-3).all(1)
    return pos[keep], (None if mass is None else mass[keep])


def check(got, pos, mass, N, L, resampler, shift=0.0, pair=False, twin=False, x0=0, n0=None, want=None, spare=0):
    """|got - want| <= bound in every cell, and the total against a random-walk bound; returns (want, bound)."""
    st = {}
    want, bound = db.budget(pos, mass, N, L, resampler, shift, pair, twin=twin, x0=x0, n0=n0, want=want, spare=spare,
                            stats=st)
    err = np.abs(got - want)
    bad = ~(err <= bound)
    assert not bad.any(), (f"{bad.sum()} cells over the bound; worst excess {np.max(err[bad] - bound[bad]):.3g} "
                           f"at {np.argwhere(bad)[:3].tolist()}, bound there {bound[bad][:3]}")
    absm = np.ones(len(pos)) if mass is None else np.abs(np.asarray(mass, np.float64))
    walk = 4 * st["qmax"] * np.sqrt(st["contributions"]) + st["flush"] + 8 * U * absm.sum()
    assert abs(got.sum() - want.sum()) <= walk, (got.sum() - want.sum(), walk)
    return want, bound


CASES = ["uniform", "clump", "pareto", "heavy_light", "negative", "pow2"]


@pytest.mark.parametrize("resampler", ["cic", "tsc"])
@pytest.mark.parametrize("case", CASES)
def test_every_cell_within_the_budget(simt, case, resampler):
    rng = np.random.default_rng(CASES.index(case))
    N, L = 32, 100.0
    pos, mass = clean(*make_case(case, N, L, rng), N, L)
    got, _ = deposit(simt, pos, mass, N, L, resampler)
    check(got, pos, mass, N, L, resampler)


@pytest.mark.parametrize("resampler", ["cic", "tsc"])
@pytest.mark.parametrize("case", ["uniform", "clump", "pareto"])
def test_interlaced_pair_within_the_budget(simt, case, resampler):
    rng = np.random.default_rng(11)
    N, L = 32, 100.0
    pos, mass = clean(*make_case(case, N, L, rng), N, L)
    a, b = deposit(simt, pos, mass, N, L, resampler, pair=True)
    check(a, pos, mass, N, L, resampler, pair=True)
    check(b, pos, mass, N, L, resampler, pair=True, twin=True)


@pytest.mark.parametrize("soa", [False, True], ids=["aos", "soa"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64], ids=["f32", "f64"])
def test_layouts_dtypes_and_odd_mesh(simt, soa, dtype):
    rng = np.random.default_rng(5)
    N, L = 45, 250.0
    pos, mass = clean(*make_case("pareto", N, L, rng, dtype), N, L)
    pos = (pos - 0.2 * L).astype(dtype)      # some outside the box: wrapped
    got, _ = deposit(simt, pos, mass, N, L, "tsc", shift=0.5, soa=soa)
    check(got, pos, mass, N, L, "tsc", shift=0.5)


def test_slab_plan(simt):
    rng = np.random.default_rng(7)
    N, L, x0, n0 = 32, 1000.0, 8, 8
    pos, mass = clean(*make_case("negative", N, L, rng), N, L)
    a, b = deposit(simt, pos, mass, N, L, "tsc", pair=True, x0=x0, n0=n0)
    check(a, pos, mass, N, L, "tsc", pair=True, x0=x0, n0=n0)
    check(b, pos, mass, N, L, "tsc", pair=True, twin=True, x0=x0, n0=n0)


@pytest.mark.parametrize("resampler", ["cic", "tsc"])
def test_faces_of_cells_bricks_and_box(simt, resampler):
    """Particles exactly on cell, brick and box faces (x = 0, L, -0.0, brick edges): filed under either neighbour."""
    rng = np.random.default_rng(9)
    N, L = 32, 32.0
    faces = np.array([0.0, -0.0, L, 8.0, 16.0, 24.0, 29.0, 30.0, 30.5, 0.5, 23.5, 7.5])
    pos = np.concatenate([rng.choice(faces, (3000, 3)), rng.random((3000, 3)) * L]).astype(np.float32)
    mass = np.exp(rng.normal(0, 1, len(pos))).astype(np.float32)
    for m in (None, mass):
        a, b = deposit(simt, pos, m, N, L, resampler, pair=True)
        check(a, pos, m, N, L, resampler, pair=True)
        check(b, pos, m, N, L, resampler, pair=True, twin=True)


def test_budget_is_tight_in_the_light_cells(simt):
    """Heavy + light clump: in the light cells (outside the heavy particle's window) the bound is, at the median, more
    than 10 times tighter than the 5e-6 x max(mesh) that the parity tests allow, and far below it in the sparsest ones.
    It is a worst-case sum of q/2 over the particles covering a cell, and the heavy particle sets q = 2^-13 for its
    whole brick, so it is not 100 times tighter in every light cell; the total-mass check sees a bias there."""
    rng = np.random.default_rng(4)
    N, L = 32, 100.0
    pos, mass = clean(*make_case("heavy_light", N, L, rng), N, L)
    got, _ = deposit(simt, pos, mass, N, L, "tsc")
    want, bound = check(got, pos, mass, N, L, "tsc")
    heavy = db.budget(pos[:1], mass[:1], N, L, "tsc")[0] != 0
    light = (want > 0) & ~heavy
    old = 5e-6 * want.max()
    assert light.sum() > 20
    assert np.median(bound[light]) * 10 <= old, (np.median(bound[light]), old)
    assert bound[light].min() * 1000 <= old


# ------------------------------------------------------------------------------------------- non-finite and large
def spoil(pos, mass, what, i):
    pos, mass = pos.copy(), None if mass is None else mass.copy()
    if what in ("nan_mass", "inf_mass", "-inf_mass"):
        mass[i] = {"nan_mass": np.nan, "inf_mass": np.inf, "-inf_mass": -np.inf}[what]
    elif what == "nan_x":
        pos[i, 0] = np.nan
    elif what == "inf_y":
        pos[i, 1] = np.inf
    return pos, mass


def check_spoiled(got, pos, mass, i, N, L, resampler, pair=False, twin=False, shift=0.0, finite_position=True):
    """One spoiled particle i: every finite cell within the bound of the deposit without it; at least one and at most
    S^3 non-finite cells, inside its window when its position is finite."""
    S = db.SUPPORT[resampler]
    nf = ~np.isfinite(got)
    assert 1 <= nf.sum() <= S ** 3, nf.sum()
    keep = np.arange(len(pos)) != i
    want, bound = db.budget(pos[keep], None if mass is None else mass[keep], N, L, resampler, shift, pair, twin=twin,
                            spare=1)
    err = np.abs(got - want)
    assert (err[~nf] <= bound[~nf]).all(), np.max(err[~nf] - bound[~nf])
    if finite_position:
        window = db.budget(pos[i:i + 1], None, N, L, resampler, shift + (0.5 if twin else 0.0), False)[0] != 0
        assert not (nf & ~window).any()


NONFINITE = ["nan_mass", "inf_mass", "-inf_mass", "nan_x", "inf_y"]


@pytest.mark.parametrize("resampler", ["cic", "tsc"])
@pytest.mark.parametrize("what", NONFINITE)
def test_a_non_finite_particle_spoils_only_its_own_cells(simt, what, resampler):
    rng = np.random.default_rng(2)
    N, L = 32, 100.0
    pos, _ = clean(rng.random((20000, 3)).astype(np.float32) * np.float32(L), None, N, L)
    mass = None if what in ("nan_x", "inf_y") else np.ones(len(pos), np.float32)
    i = 777
    sp, sm = spoil(pos, mass, what, i)
    a, b = deposit(simt, sp, sm, N, L, resampler, pair=True)
    fin = what.endswith("mass")
    check_spoiled(a, pos, mass, i, N, L, resampler, pair=True, finite_position=fin)
    check_spoiled(b, pos, mass, i, N, L, resampler, pair=True, twin=True, finite_position=fin)
    if what == "nan_x":        # the unit-mass path, with masses too
        m1 = np.ones(len(pos), np.float32)
        a, _ = deposit(simt, sp, m1, N, L, resampler)
        check_spoiled(a, pos, m1, i, N, L, resampler, finite_position=False)


@pytest.mark.parametrize("resampler", ["cic", "tsc"])
def test_masses_near_the_float32_limit(simt, resampler):
    """20000 masses of 1e35: each cell (<= 2.4e35) is representable, so the deposit must stay within the bound -- the
    chunk's sum of |m| (~8e38) is not."""
    rng = np.random.default_rng(3)
    N, L = 32, 100.0
    pos, _ = clean(rng.random((20000, 3)).astype(np.float32) * np.float32(L), None, N, L)
    mass = np.full(len(pos), 1e35, np.float32)
    got, _ = deposit(simt, pos, mass, N, L, resampler)
    assert np.isfinite(got).all()
    check(got, pos, mass, N, L, resampler)


# ------------------------------------------------------------------------------------------------------------ mutants
def mutant(tmp_path, old, new):
    import build_simt
    src = build_simt.device_part(os.path.join(build_simt.CSRC, "deposit_sorted.cu"))
    assert src.count(old) == 1, old
    return load(build_simt.compile_kernels(src.replace(old, new), str(tmp_path)))


def fails(fn):
    try:
        fn()
    except AssertionError:
        return True
    return False


def test_mutant_round_toward_zero_is_caught(tmp_path):
    lib = mutant(tmp_path, "(unsigned int)__float2int_rn(wxy * wz[c])", "(unsigned int)(int)(wxy * wz[c])")
    rng = np.random.default_rng(21)
    N, L = 32, 100.0
    pos, mass = clean(*make_case("pareto", N, L, rng), N, L)
    got, _ = deposit(lib, pos, mass, N, L, "tsc")
    assert fails(lambda: check(got, pos, mass, N, L, "tsc"))


def test_mutant_loosened_overflow_rule_is_caught(tmp_path):
    lib = mutant(tmp_path, "constexpr float WMAX = (S == 3) ? 0.43f : 1.001f;\n                const float room",
                 "constexpr float WMAX = (S == 3) ? 0.2f : 1.001f;\n                const float room")
    N, L = 32, 32.0
    pos = np.full((100, 3), 10.0, np.float32)        # one cell: every particle puts 0.75^3 of its mass there
    mass = np.ones(len(pos), np.float32)
    got, _ = deposit(lib, pos, mass, N, L, "tsc")
    assert fails(lambda: check(got, pos, mass, N, L, "tsc"))


def test_mutant_scaled_flush_quantum_is_caught(tmp_path):
    lib = mutant(tmp_path, "const float quantum = __int_as_float((127 - frac_bits) << 23) * unit;",
                 "const float quantum = __int_as_float((127 - frac_bits) << 23) * unit * (1.f + 1.f / 4096.f);")
    rng = np.random.default_rng(22)
    N, L = 32, 100.0
    pos, mass = clean(*make_case("uniform", N, L, rng), N, L)
    got, _ = deposit(lib, pos, mass, N, L, "tsc")
    assert fails(lambda: check(got, pos, mass, N, L, "tsc"))
