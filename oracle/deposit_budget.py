"""Per-cell error bound of the sorted deposit (astrild_b200/csrc/deposit_sorted.cu)  --  TEST INFRASTRUCTURE ONLY.

``budget(pos, mass, N, L, resampler, shift, pair)`` returns ``(want, bound)``: ``want`` is the float64 oracle
(``pk_oracle_fast.paint``) and ``bound`` a per-cell bound on |sorted deposit - want| that holds however the partition
orders the particles of a brick into chunks and whichever brick it files a particle at a tie under (DESIGN §4.1):

* quantisation: every particle whose window covers the cell adds ``q_b / 2 + 8 u |m|`` plus the first-order effect of
  the float32 rounding of its brick-local coordinate (``DELTA`` cells per axis) on the product of its three weights.
  ``q_b`` bounds the quantum of every chunk that brick b can form (a chunk is a subset of one brick):
  unit masses ``2^-min(floor(log2(2^32 / (WMAX min(n_b, TILE_FLUSH)))), SMAX)``;
  masses ``max(2 WMAX sum_b|m| 2^-31, 2^ceil(log2 max_b|m|) 2^-30)``;
* flush: ``2 u k_c A_c``, A_c the oracle's deposit of |m| and k_c the number of chunk flushes that reach the cell
  (every chunk of every brick whose tile covers it).

A particle within ``tie`` cells of a tie of its mesh-0 home cell counts in the statistics of every brick it may be
filed under and takes the largest of their quanta.  The brick constants are read from the CUDA sources.
"""
from __future__ import annotations

import os
import re

import numpy as np

from . import pk_oracle_fast

_CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "astrild_b200", "csrc")
U = 2.0 ** -24                    # float32 unit roundoff
DELTA = 2.0 ** -19                # float32 rounding of a brick-local coordinate (|l| < 33) and of its twin (+ 0.5), cells


def _constant(path: str, pattern: str) -> int:
    text = open(os.path.join(_CSRC, path)).read()
    m = re.search(pattern, text)
    assert m, f"{pattern!r} not found in {path}"
    return int(m.group(1))


def brick_constants() -> dict:
    return {"BX": _constant("brick_common.cuh", r"#define APK_BX (\d+)"),
            "BY": _constant("brick_common.cuh", r"#define APK_BY (\d+)"),
            "BZ": _constant("brick_common.cuh", r"constexpr int BZ = (\d+);"),
            "TILE_FLUSH": _constant("deposit_sorted.cu", r"#define APK_TILE_FLUSH (\d+)")}


WMAX = {"cic": 1.001, "tsc": 0.43}
SMAX = {"cic": 23, "tsc": 24}
SUPPORT = {"cic": 2, "tsc": 3}


def _window(S: int, g: np.ndarray, pad: int, tie: float):
    """pmesh's window at grid coordinate g (float64) widened by `pad` cells per side: base index, weights and slopes
    |dw/dg|; the slope is continued for `tie` cells beyond the support (CIC: 1 there, TSC: 0 to first order)."""
    i0 = np.floor(g + (0.5 if S == 3 else 0.0)).astype(np.int64) - (S - 1) // 2 - pad
    dx = g - i0
    w, dw = [], []
    for j in range(S + 2 * pad):
        x = np.abs(dx - j)
        if S == 2:
            w.append(np.where(x < 1.0, 1.0 - x, 0.0)); dw.append(np.where(x < 1.0 + tie, 1.0, 0.0))
        else:
            w.append(np.where(x <= 0.5, 0.75 - x * x, np.where(x < 1.5, 0.5 * (1.5 - x) ** 2, 0.0)))
            dw.append(np.where(x <= 0.5, 2 * x, np.where(x < 1.5, 1.5 - x, 0.0)))
    return i0, np.stack(w, 1), np.stack(dw, 1)


def _add_windows(bound: np.ndarray, S: int, g: np.ndarray, base: np.ndarray, absm: np.ndarray, N: int, pad: int,
                 tie: float):
    """bound[c] += base + DELTA |m| (|w_x'| w_y w_z + w_x |w_y'| w_z + w_x w_y |w_z'|) over each particle's window."""
    if not len(g):
        return
    i0, w, dw = zip(*(_window(S, g[:, d], pad, tie) for d in range(3)))
    n = S + 2 * pad
    for jx in range(n):
        cx = (i0[0] + jx) % N
        for jy in range(n):
            cxy = (cx * N + (i0[1] + jy) % N) * N
            for jz in range(n):
                pw = (dw[0][:, jx] * w[1][:, jy] * w[2][:, jz] + w[0][:, jx] * dw[1][:, jy] * w[2][:, jz] +
                      w[0][:, jx] * w[1][:, jy] * dw[2][:, jz])
                val = base + DELTA * absm * (pw + DELTA)
                ok = np.isfinite(val)
                bound += np.bincount(cxy[ok] + (i0[2][ok] + jz) % N, val[ok], minlength=N ** 3).reshape(N, N, N)


def _wrap_box(mesh: np.ndarray, lo: np.ndarray, ext, value: float, N: int, slab):
    """mesh[lo : lo + ext] += value per axis, periodic (x: local planes for slab plans, not wrapped)."""
    xs = np.arange(lo[0], lo[0] + ext[0])
    xs = xs[(xs >= 0) & (xs < mesh.shape[0])] if slab else xs % N
    ys, zs = np.arange(lo[1], lo[1] + ext[1]) % N, np.arange(lo[2], lo[2] + ext[2]) % N
    mesh[np.ix_(xs, ys, zs)] += value


def budget(pos, mass, N: int, L: float, resampler: str, shift: float = 0.0, pair: bool = False, twin: bool = False,
           x0: int = 0, n0: int | None = None, tie: float = 1e-3, want: np.ndarray | None = None, spare: int = 0,
           stats: dict | None = None):
    """-> (want, bound), float64 [planes][N][N] like the deposit (planes = N, or n0 + 3 for the slab [x0, x0 + n0) with
    ghost planes 1 below and 2 above).  ``shift`` is the deposit's shift; ``twin``: the bound of the interlaced pair's
    second mesh (shift + 0.5; ``pair`` must be set).  Particles of a slab plan that the slab does not own are dropped.
    ``spare``: that many more particles, of mass up to the largest |m|, may be in any brick (a particle with a
    non-finite coordinate is filed under some brick and counts there).  ``stats`` receives ``qmax`` (the largest q_b),
    ``contributions`` (particle-cell pairs) and ``flush`` (the flush term summed over the cells)."""
    assert not twin or pair
    c = brick_constants()
    S = SUPPORT[resampler]
    n0 = N if n0 is None else n0
    slab = n0 < N
    pos = np.asarray(pos)
    g = pos.astype(np.float64) * (N / L) + shift
    m = np.ones(len(pos)) if mass is None else np.asarray(mass, np.float64)
    if slab:
        own = (np.floor(pos[:, 0].astype(np.float64) * (N / L)).astype(np.int64) % N - x0) % N < n0
        pos, g, m = pos[own], g[own], m[own]
        mass = None if mass is None else np.asarray(mass)[own]
    absm = np.abs(m)
    wshift = shift + (0.5 if twin else 0.0)
    if want is None:
        want = pk_oracle_fast.paint(pos, mass, N, L, resampler, wshift)
    absw = want if mass is None else pk_oracle_fast.paint(pos, absm, N, L, resampler, wshift)
    if slab:
        idx = np.arange(x0 - 1, x0 + n0 + 2) % N
        want, absw = want[idx], absw[idx]

    # ---- bricks: of the mesh-0 home cell; at a tie (within `tie` cells) either neighbour
    zc = c["BZ"] - (S - 1) - int(pair)
    edge = np.array([c["BX"], c["BY"], zc])
    planes = n0 + 3 if slab else N
    nb = np.array([-(-planes // edge[0]), -(-N // edge[1]), -(-N // edge[2])])
    a = g - (0.5 if S == 2 else 0.0)
    lo_home = np.floor(a + 0.5 - tie).astype(np.int64)
    hi_home = np.floor(a + 0.5 + tie).astype(np.int64)
    bricks = []                                                  # per axis: [candidate 0, candidate 1] brick index
    for d in range(3):
        cand = []
        for h in (lo_home[:, d], hi_home[:, d]):
            h = h % N
            if d == 0 and slab:
                h = (h - (x0 - 1)) % N
            cand.append(h // edge[d])
        bricks.append(cand)
    finite = np.isfinite(absm) & np.isfinite(g).all(1)
    nbr = int(nb.prod())
    cnt, msum, mtop = np.zeros(nbr), np.zeros(nbr), np.zeros(nbr)
    keys = []
    for ix in (0, 1):
        for iy in (0, 1):
            for iz in (0, 1):
                k = (bricks[0][ix] * nb[1] + bricks[1][iy]) * nb[2] + bricks[2][iz]
                keys.append(k)
    keys = np.stack(keys, 1) if len(pos) else np.zeros((0, 8), np.int64)
    for j in range(keys.shape[1]):
        k = keys[:, j]
        first = np.ones(len(k), bool) if j == 0 else (keys[:, :j] != k[:, None]).all(1)
        cnt += np.bincount(k[first], minlength=nbr)
        msum += np.bincount(k[first & finite], absm[first & finite], minlength=nbr)
        np.maximum.at(mtop, k[first & finite], absm[first & finite])
    cnt += spare
    msum += spare * (absm[finite].max() if finite.any() else 0.0)
    if spare:
        mtop = np.maximum(mtop, absm[finite].max() if finite.any() else 0.0)
    if mass is None:
        s = np.minimum(np.floor(np.log2(2.0 ** 32 / (WMAX[resampler] * np.maximum(np.minimum(cnt, c["TILE_FLUSH"]), 1)))),
                       SMAX[resampler])
        q = 2.0 ** -s
    else:
        with np.errstate(divide="ignore"):
            top = np.maximum(2.0 ** np.ceil(np.log2(mtop)), 2.0 ** -125)
        q = np.maximum(2 * WMAX[resampler] * msum * 2.0 ** -31, top * 2.0 ** -30)
    qp = q[keys].max(1) if len(pos) else np.zeros(0)

    # ---- quantisation: over the particles whose window covers the cell.  Within `tie` of a tie of the window's base,
    # the kernel may take the neighbouring window: such particles cover S + 2 cells per axis, and a cell just outside
    # the support gets a weight of at most the slope there times DELTA.
    bound = np.zeros((N, N, N))
    gw = g + (wshift - shift)
    base = qp / 2 + 8 * U * absm
    _add_windows(bound, S, gw, base, absm, N, 0, 1e-300)
    near = (np.abs(gw + (0.5 if S == 3 else 0.0) - np.rint(gw + (0.5 if S == 3 else 0.0))) < tie).any(1)
    _add_windows(bound, S, gw[near], base[near], absm[near], N, 1, tie)
    if slab:
        bound = bound[np.arange(x0 - 1, x0 + n0 + 2) % N]

    # ---- flush: each chunk of each brick whose tile covers the cell
    off = 1 if S == 3 else 0
    ext = (edge[0] + S - 1 + int(pair), edge[1] + S - 1 + int(pair), c["BZ"])
    k_c = np.zeros_like(bound)
    chunks = np.ceil(cnt / c["TILE_FLUSH"])
    for b in np.nonzero(chunks)[0]:
        bx, by, bz = b // (nb[1] * nb[2]), (b // nb[2]) % nb[1], b % nb[2]
        _wrap_box(k_c, np.array([bx, by, bz]) * edge - off, ext, chunks[b], N, slab)
    flush = 2 * U * k_c * np.abs(absw)
    bound += flush
    if stats is not None:
        stats.update(qmax=float(q[cnt > 0].max()) if (cnt > 0).any() else 0.0,
                     contributions=int(finite.sum()) * S ** 3, flush=float(flush.sum()))
    return want, bound

