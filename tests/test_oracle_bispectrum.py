"""The bispectrum oracle's FFT estimator (oracle/bk_oracle.py) against a brute-force sum over all mode pairs.

N_tri bit for bit and B to 1e-10 relative; N = 12, 16 and 15 (odd); plain fields and interlaced + compensated TSC
deposits; the default kmax ((2/3) pi N / L, no aliasing) and kmax up to Nyquist (triangles that close modulo the grid
are counted by both).  Every triple the skip rule drops has no triangle at all.
"""
import numpy as np
import pytest

from oracle import bk_oracle as bo
from oracle import pk_oracle as po

L = 100.0


def field(N, kind, seed=3):
    rng = np.random.default_rng(seed)
    if kind == "plain":
        d = rng.standard_normal((N, N, N))
        return d - d.mean()
    # interlaced + compensated TSC deposit of random particles: as a real field whose half-complex transform is the
    # oracle's combined field on every mode a shell can hold (no Nyquist-index mode is in a shell)
    pos = rng.random((4 * N ** 3 // 8, 3)) * L
    c = bo.delta_k_from_particles(pos, None, N, L, "tsc", interlaced=True, compensated=True)
    c[0, 0, 0] = 0.0
    return np.fft.irfftn(c, s=(N, N, N), axes=(0, 1, 2)) * float(N) ** 3


@pytest.mark.parametrize("N", [12, 16, 15])
@pytest.mark.parametrize("kind", ["plain", "interlaced_compensated"])
@pytest.mark.parametrize("kmax", ["default", "nyquist"])
def test_fft_estimator_equals_bruteforce(N, kind, kmax):
    edges = bo.default_edges(N, L, kmax=None if kmax == "default" else np.pi * N / L)
    delta = field(N, kind)
    fft = bo.bispectrum_fft(po.r2c(delta), N, L, edges)
    bf = bo.bispectrum_bruteforce(delta, L, edges)
    assert np.array_equal(fft["triples"], bf["triples"])
    assert np.array_equal(fft["ntri"], bf["ntri"]), "triangle counts differ"
    assert fft["residual"] < 1e-6
    ok = bf["ntri"] > 0
    assert ok.sum() > 0
    # B to 1e-10 relative to the scale of its terms (B itself may cancel to ~0)
    scale = np.abs(bf["B"][ok]).max()
    np.testing.assert_allclose(fft["B"][ok], bf["B"][ok], rtol=1e-10, atol=1e-10 * scale)
    # the skip rule only drops triples without a triangle
    nb = len(edges) - 1
    kept = {tuple(t) for t in fft["triples"]}
    for i in range(nb):
        for j in range(i, nb):
            for l in range(j, nb):
                if (i, j, l) not in kept:
                    assert bf["count"][i, j, l] == 0, (i, j, l)
    if kmax == "nyquist":
        # the modular closure is live: some kept triple has shells that reach past 2 k_Nyquist together
        hi, t = edges[1:], fft["triples"]
        assert ((hi[t[:, 0]] + hi[t[:, 1]] + hi[t[:, 2]]) > 2 * np.pi * N / L).any()
