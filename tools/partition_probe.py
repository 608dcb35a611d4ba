"""Checksums of the c3 meshes after the deposit, and the deposit times of a clustered c3-size set (tools, not product).

    python tools/partition_probe.py OUT TAG    # one JSON line; ASTRILD_PK_LIB=<other build> for the A/B arm

mesh: per-plane sums of the meshes' float32 BIT PATTERNS (as int64, plain and position-weighted), hashed, after each
of two calls: deposits that agree bit for bit print the same digest.  (Bricks of more than 8191 particles -- 26 of the
c3 set's 198144 -- are several chunks whose make-up follows the order of the partition's atomics, so the digest may
change from call to call.)  The per-plane float64 sums of both meshes go to <out>/plane_sums_<tag>.npy.
clustered: the c3 particles with a tenth of them moved into one 32^3-cell corner of the 1024^3 mesh (bricks far beyond
8191 particles); deposit_pair's time (CUDA events around the call, synchronised) on five consecutive calls of one plan,
with the library's split of each (apk_plan_last_deposit_ms).
"""
import hashlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def digest(mesh):
    flat = mesh.view(torch.int32).reshape(mesh.shape[0], -1)
    w = torch.arange(flat.shape[1], device=mesh.device, dtype=torch.int64) % 1000003 + 1
    h = hashlib.sha256()
    for a in range(0, flat.shape[0], 64):
        b = flat[a:a + 64].long()
        h.update(b.sum(1).cpu().numpy().tobytes())
        h.update((b * w).sum(1).cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def timed_pair(eng, pos, m1, m2):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    eng.deposit_pair(pos, None, "tsc", 1.0, "sorted", out=(m1, m2))
    ev[1].record()
    torch.cuda.synchronize()
    return round(ev[0].elapsed_time(ev[1]), 3), {k: round(v, 3) for k, v in eng.last_deposit_ms().items()}


def main():
    import astrild_b200 as ab
    from astrild_b200.engine import PkEngine
    dev = torch.device("cuda", 0)
    wl = bench.WORKLOADS["c3"]
    N, n = wl["mesh"], wl["n"]
    pos, _ = bench.make_particles(wl, dev)
    out = {"lib": os.environ.get("ASTRILD_PK_LIB", "in-tree"), "gpu": torch.cuda.get_device_name(0)}
    eng = ab.get_engine(N, wl["box"], dev)
    eng.enable_timing(True)
    eng.ensure_workspace(n ** 3, False, True)
    m1, m2 = eng.new_mesh(), eng.new_mesh()
    out["uniform_ms"], out["mesh_digest"] = [], []
    for _ in range(2):
        out["uniform_ms"].append(timed_pair(eng, pos, m1, m2))
        out["mesh_digest"].append([digest(m1), digest(m2)])
    sums = torch.stack([m1[:, :, :N].double().sum((1, 2)), m2[:, :, :N].double().sum((1, 2))]).cpu().numpy()
    np.save(os.path.join(sys.argv[1], f"plane_sums_{sys.argv[2]}.npy"), sums)
    eng.close()

    k = pos[0].numel() // 10
    g = torch.Generator(device=dev).manual_seed(12)
    for c in pos:
        c[:k] = torch.rand(k, device=dev, generator=g) * (32.0 / N)
    eng = PkEngine(N, wl["box"], dev)
    eng.enable_timing(True)
    eng.ensure_workspace(n ** 3, False, True)
    out["clustered_ms"] = [timed_pair(eng, pos, m1, m2) for _ in range(5)]
    out["clustered_digest"] = [digest(m1), digest(m2)]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
