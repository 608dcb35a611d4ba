"""The fixed-slot brick partition (deposit_sorted.cu: every brick owns a fixed number of payload slots, at least
TILE_FLUSH = 8191, and there is no count pass) against the two-pass one (count, scan, scatter), on CPU fibers
(tests/simt/deposit_fixed_host.cpp).

A brick of at most 8191 particles is one chunk of the tile kernel in either layout, and the tile's integer adds
commute, so the meshes must be equal BIT FOR BIT.  A larger brick is several chunks whose make-up depends on the order
of the scatter's atomics in either layout: the meshes stay within the deposit's per-cell error budget
(oracle/deposit_budget.py).  A brick of more particles than its slots overflows them: the partition is then filed
again in the two-pass layout on the device.
The whole module runs once more under AddressSanitizer with exactly sized buffers.
"""
import ctypes as ct
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "simt"))

from oracle import deposit_budget as db  # noqa: E402


def build() -> str:
    import build_simt
    out_dir = os.path.join(build_simt.OUT_DIR, "fixed")
    so = os.path.join(out_dir, "libapk_simt_fixed.so")
    srcs = [os.path.join(build_simt.CSRC, f) for f in ("deposit_sorted.cu", "brick_common.cuh", "apk_common.cuh",
                                                         "deposit_common.cuh")]
    srcs += [os.path.join(build_simt.HERE, f) for f in ("simt.h", "deposit_fixed_host.cpp", "build_simt.py")]
    if os.path.exists(so) and all(os.path.getmtime(so) >= os.path.getmtime(s) for s in srcs):
        return so
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "deposit_sorted_kernels.inc"), "w") as f:
        f.write(build_simt.device_part(srcs[0]))
    return build_simt._gxx("deposit_fixed_host.cpp", out_dir, so)


@pytest.fixture(scope="module")
def simt():
    lib = ct.CDLL(build())
    lib.simt_deposit_partition.restype = ct.c_uint
    lib.simt_deposit_partition.argtypes = ([ct.c_void_p] * 3 + [ct.c_int, ct.c_int, ct.c_void_p, ct.c_int, ct.c_longlong,
                                           ct.c_int, ct.c_double, ct.c_double, ct.c_int, ct.c_int, ct.c_int, ct.c_void_p,
                                           ct.c_void_p, ct.c_uint])
    return lib


def deposit(lib, pos, mass, N, L, resampler, slots, pair=False, shift=0.0, soa=False, x0=0, n0=None):
    """-> (mesh, twin or None, overflow word) with the meshes float32 [planes][N][N]; slots = 0: two-pass partition"""
    n0 = N if n0 is None else n0
    planes = N if n0 == N else n0 + 3
    m0 = np.zeros((planes, N, 2 * (N // 2 + 1)), np.float32)
    m1 = np.zeros_like(m0) if pair else None
    if soa:
        cols = [np.ascontiguousarray(pos[:, d]) for d in range(3)]
        ptrs = [c.ctypes.data for c in cols]
    else:
        p = np.ascontiguousarray(pos)
        ptrs = [p.ctypes.data, None, None]
    mp = None if mass is None else np.ascontiguousarray(mass)
    ovf = lib.simt_deposit_partition(ptrs[0], ptrs[1], ptrs[2], int(soa), int(pos.dtype == np.float64),
                                     None if mp is None else mp.ctypes.data, int(mp is not None and mp.dtype == np.float64),
                                     len(pos), N, 1.0 / L, shift, {"cic": 2, "tsc": 3}[resampler], x0, n0, m0.ctypes.data,
                                     None if m1 is None else m1.ctypes.data, int(slots))
    return m0[:, :, :N], (None if m1 is None else m1[:, :, :N]), ovf


def same_bits(a, b):
    assert a.shape == b.shape
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"{np.count_nonzero(a != b)} cells differ"


# (resampler, pair, masses, SoA, float64 positions, N, slab [x0, x0 + n0) or None)
CASES = {
    "cic_single_unit_aos_f32": ("cic", False, False, False, False, 32, None),
    "tsc_single_mass_soa_f32": ("tsc", False, True, True, False, 32, None),
    "tsc_pair_unit_soa_f32": ("tsc", True, False, True, False, 32, None),
    "cic_pair_mass_aos_f64": ("cic", True, True, False, True, 32, None),
    "tsc_pair_mass_aos_f64": ("tsc", True, True, False, True, 32, None),
    "tsc_pair_unit_slab": ("tsc", True, False, False, False, 32, (8, 8)),
    "cic_single_mass_slab_f64": ("cic", False, True, True, True, 32, (16, 8)),
    "tsc_pair_mass_odd_mesh": ("tsc", True, True, True, False, 45, None),
}


@pytest.mark.parametrize("case", list(CASES))
def test_fixed_slots_give_the_two_pass_meshes_bit_for_bit(simt, case):
    resampler, pair, with_mass, soa, f64, N, slab = CASES[case]
    rng = np.random.default_rng(list(CASES).index(case))
    L = 100.0
    pos = (rng.random((15000, 3)) * 1.2 * L - 0.1 * L).astype(np.float64 if f64 else np.float32)   # some out of the box
    mass = np.exp(rng.normal(0, 1, len(pos))).astype(np.float32) if with_mass else None
    x0, n0 = slab if slab else (0, None)
    kw = dict(pair=pair, soa=soa, x0=x0, n0=n0)
    a0, a1, ovf_two = deposit(simt, pos, mass, N, L, resampler, 0, **kw)
    b0, b1, ovf = deposit(simt, pos, mass, N, L, resampler, 8191 + 3000 * (list(CASES).index(case) % 2), **kw)
    assert ovf == 0 and ovf_two == 0
    assert a0.any()
    same_bits(b0, a0)
    if pair:
        same_bits(b1, a1)


def one_brick(n, rng):
    """n particles in brick 0 of a 64^3 mesh (L = 64: positions in cells), away from its faces, and 2000 elsewhere."""
    inside = rng.random((n, 3)) * [20.0, 5.0, 24.0] + 2.0
    rest = rng.random((2000, 3)) * [32.0, 64.0, 64.0] + [30.0, 0.0, 0.0]
    return np.concatenate([inside, rest]).astype(np.float32)


@pytest.mark.parametrize("n,slots,overflows", [(8191, 8191, False), (8192, 8191, True), (9000, 9000, False),
                                               (9001, 9000, True)])
def test_brick_that_fits_its_slots_stays_and_one_more_is_refiled(simt, n, slots, overflows):
    """n particles in brick 0: up to `slots` stay in the fixed-slot layout (8191: one chunk, the two-pass bits; 9000:
    two chunks), one more overflows the slots and the two-pass refiling runs.  Every cell within the budget."""
    rng = np.random.default_rng(n)
    N, L = 64, 64.0
    pos = one_brick(n, rng)
    a0, a1, _ = deposit(simt, pos, None, N, L, "tsc", 0, pair=True)
    b0, b1, ovf = deposit(simt, pos, None, N, L, "tsc", slots, pair=True)
    assert ovf == int(overflows)
    if n <= 8191:
        same_bits(b0, a0)
        same_bits(b1, a1)
    for got, twin in ((b0, False), (b1, True)):
        want, bound = db.budget(pos, None, N, L, "tsc", 0.0, True, twin=twin)
        err = np.abs(got.astype(np.float64) - want)
        assert (err <= bound).all(), np.max(err - bound)


def test_clustered_set_is_refiled_with_masses_cic(simt):
    """A clump of 12000 particles in one cell (rotation ranks up to 31, two chunks) plus a uniform background,
    per-particle masses, CIC: the overflow is seen and the result stays within the budget."""
    rng = np.random.default_rng(9)
    N, L = 32, 100.0
    pos = np.concatenate([rng.random((12000, 3)) * 2.0 + 40.0, rng.random((6000, 3)) * L]).astype(np.float32)
    mass = np.exp(rng.normal(0, 1, len(pos))).astype(np.float32)
    got, _, ovf = deposit(simt, pos, mass, N, L, "cic", 10000)
    assert ovf == 1
    want, bound = db.budget(pos, mass, N, L, "cic", 0.0, False)
    assert (np.abs(got.astype(np.float64) - want) <= bound).all()


@pytest.mark.parametrize("what", ["nan_x", "nan_mass"])
def test_non_finite_particle_keeps_its_nan_home_cell(simt, what):
    rng = np.random.default_rng(11)
    N, L = 32, 100.0
    pos = (rng.random((10000, 3)) * L).astype(np.float32)
    mass = np.ones(len(pos), np.float32)
    i = 4321
    if what == "nan_x":
        pos[i, 0] = np.nan
    else:
        mass[i] = np.nan
    a0, a1, _ = deposit(simt, pos, mass, N, L, "tsc", 0, pair=True)
    b0, b1, ovf = deposit(simt, pos, mass, N, L, "tsc", 8191, pair=True)
    assert ovf == 0
    for a, b in ((a0, b0), (a1, b1)):
        assert 1 <= np.count_nonzero(np.isnan(b)) <= 27
        same_bits(b, a)


def _libasan():
    gcc = shutil.which("gcc")
    if gcc is None:
        return None
    path = subprocess.run([gcc, "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    return path if os.path.isabs(path) and os.path.exists(path) else None


@pytest.mark.skipif(os.environ.get("APK_SIMT_ASAN", "0") not in ("", "0"), reason="already inside the sanitized run")
def test_module_is_clean_under_address_sanitizer():
    lib = _libasan()
    if lib is None:
        pytest.skip("libasan not found")
    env = dict(os.environ, APK_SIMT_ASAN="1", LD_PRELOAD=lib, ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0")
    out = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider", os.path.abspath(__file__)],
                         cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    tail = (out.stdout + out.stderr)[-4000:]
    assert "AddressSanitizer" not in tail, tail
    assert out.returncode == 0, tail
