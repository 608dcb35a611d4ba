"""The fixed-slot brick partition on the device (deposit_sorted.cu): a fixed number of payload slots per brick (twice
the mean occupancy, at least 8191) and no count pass when the plan workspace has room for them (apk_plan_workspace_bytes
reports it for populated meshes), the two-pass partition (count, scan, scatter) when the workspace set is smaller.

Populated sets: both paths give the same meshes (a brick of at most 8191 particles is one chunk of the tile kernel in
either layout, and its integer tile adds commute) up to the order of the float32 REDs with which neighbouring bricks
flush into shared cells -- exact unless their quanta differ and the cell's sum needs more than 24 bits.  A clustered
set overflows its slots: the first call refiles the partition in two passes on the device, later calls on the plan
partition in two passes from the start.  The room for the slots stops at 2 x 8191 records per brick.
"""
import numpy as np
import pytest
import torch

from astrild_b200 import _lib
from astrild_b200.engine import PkEngine
from tests.test_simt_deposit_budget import check, clean

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)


def lattice(n, seed, jitter=2.0):
    """n^3 particles on a lattice (box units [0, 1)) displaced by up to `jitter` cells of an n^3 mesh, lattice order."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    i = torch.arange(n, device=DEV, dtype=torch.float32)
    x, y, z = torch.meshgrid(i, i, i, indexing="ij")
    cols = []
    for c in (x, y, z):
        d = (torch.rand(c.shape, device=DEV, generator=g) * 2 - 1) * jitter
        cols.append(torch.remainder((c + 0.5 + d) / n, 1.0).reshape(-1).contiguous())
    return tuple(cols)


def two_pass_workspace(eng, npart):
    """Sets a workspace with room for `npart` two-pass records only and keeps the engine from growing it."""
    small = ct_size(eng, 1) + 12 * npart + 4096
    eng._workspace = torch.empty(small, dtype=torch.uint8, device=DEV)
    _lib.call("apk_plan_set_workspace", eng._plan, eng._workspace.data_ptr(), small)
    eng.ensure_workspace = lambda *a, **k: None


def ct_size(eng, npart):
    import ctypes as ct
    need = ct.c_size_t()
    _lib.call("apk_plan_workspace_bytes", eng._plan, int(npart), 0, 1, ct.byref(need))
    return need.value


def deposit(eng, pos, resampler, pair):
    eng.enable_timing(True)
    if pair:
        out = eng.deposit_pair(pos, None, resampler, 1.0, "sorted")
    else:
        out = (eng.deposit(pos, None, resampler, 0.0, 1.0, "sorted"),)
    torch.cuda.synchronize()
    return out, eng.last_deposit_ms()


def same(a, b):
    """The lattice sets below keep every brick under 8191 particles: in either layout a brick is one chunk and flushes the
    same float32 value into each cell of its tile.  A cell is covered by the tiles of at most 2 bricks per axis, so it
    is a float32 sum of at most 8 non-negative values, added in whatever order the bricks' REDs arrive: 7 roundings,
    each within 2^-24 of the cell, so two orders differ by at most 14 * 2^-24 of it."""
    tol = 14 * 2.0 ** -24 * torch.maximum(a.abs(), b.abs())
    assert bool(((a - b).abs() <= tol).all()), float(((a - b).abs() - tol).max())
@pytest.mark.parametrize("n,resampler,pair", [(256, "tsc", True), (512, "tsc", True), (512, "cic", False)])
def test_fixed_slots_and_two_pass_meshes_agree(n, resampler, pair):
    pos = lattice(n, 7)
    fixed = PkEngine(n, 1.0, DEV)
    assert ct_size(fixed, n ** 3) > ct_size(fixed, 1) + 12 * n ** 3 + 4096    # room for the fixed slots is reported
    a, ms_a = deposit(fixed, pos, resampler, pair)
    assert ms_a["count"] == 0.0 and ms_a["scatter"] > 0.0            # fixed-slot partition: no count pass
    two = PkEngine(n, 1.0, DEV)
    two_pass_workspace(two, n ** 3)
    b, ms_b = deposit(two, pos, resampler, pair)
    assert ms_b["count"] > 0.0                                        # the smaller workspace: two-pass partition
    for x, y in zip(a, b):
        same(x, y)
    assert abs(float(a[0][:, :, :n].double().sum()) - n ** 3) <= 1e-5 * n ** 3
    fixed.close(); two.close()


def test_clustered_set_falls_back_then_partitions_in_two_passes(oracle_fast):
    """A tenth of the particles in one 16^3-cell corner of a 128^3 mesh: two bricks of ~120 000 particles, far beyond
    their slots.  The first call's fixed-slot scatter overflows and the device refiles the partition; the plan
    remembers it, and the second call partitions in two passes from the start.  Such a brick is ~15 chunks whose make-up
    follows the order of the scatter's atomics, so both meshes are checked cell by cell against the deposit's error
    bound (oracle/deposit_budget.py, which counts every chunk flush reaching a cell)."""
    N, L = 128, 1.0
    rng = np.random.default_rng(12)
    pos = rng.random((2_400_000, 3))
    pos[:240_000] *= 16.0 / N
    pos, _ = clean(pos.astype(np.float32), None, N, L)
    eng = PkEngine(N, L, DEV)
    first, ms1 = deposit(eng, pos, "tsc", True)
    assert ms1["count"] == 0.0                                        # fixed-slot attempt, refiled on the device
    first = [eng.store_mesh(m).cpu().numpy() for m in first]
    second, ms2 = deposit(eng, pos, "tsc", True)
    assert ms2["count"] > 0.0                                         # the plan went straight to two passes
    second = [eng.store_mesh(m).cpu().numpy() for m in second]
    for meshes in (first, second):
        check(meshes[0], pos, None, N, L, "tsc", pair=True)
        check(meshes[1], pos, None, N, L, "tsc", pair=True, twin=True)
    eng.close()


def test_workspace_room_is_capped_and_dense_sets_take_two_passes():
    """64^3 mesh, 72 bricks: 300 000 particles get room for twice their records; 2 000 000 (over 27 000 per brick, more
    than 2 x 8191 on average) get none beyond their own, and deposit with the two-pass partition."""
    eng = PkEngine(64, 1.0, DEV)
    assert abs((ct_size(eng, 300_000) - ct_size(eng, 1)) - 24 * 300_000) <= 512
    assert abs((ct_size(eng, 2_000_000) - ct_size(eng, 1_999_000)) - 12 * 1000) <= 512
    g = torch.Generator(device=DEV).manual_seed(3)
    pos = tuple(torch.rand(2_000_000, device=DEV, generator=g) for _ in range(3))
    (mesh,), ms = deposit(eng, pos, "cic", False)
    assert ms["count"] > 0.0
    assert abs(float(mesh[:, :, :64].double().sum()) - 2_000_000) <= 1.0
    eng.close()
