"""Seeded stacked (ragged) ball-query cases shared by tests/test_stack_ball_query_cpu.py and tests/test_stack_sa_gpu.py
(TEST INFRASTRUCTURE).  A case is (xyz (N,3), xyz_cnt (B,), new_xyz (M,3), new_cnt (B,), radius, nsample), float32 /
int32 numpy."""
from __future__ import annotations

import numpy as np

import synth


def stack(frames_xyz, frames_new):
    """lists of per-frame (n_b,3) / (m_b,3) arrays -> (xyz, xyz_cnt, new_xyz, new_cnt)"""
    xyz = np.concatenate([np.asarray(f, np.float32).reshape(-1, 3) for f in frames_xyz], 0)
    new = np.concatenate([np.asarray(f, np.float32).reshape(-1, 3) for f in frames_new], 0)
    cnt = np.array([len(f) for f in frames_xyz], np.int32)
    mcnt = np.array([len(f) for f in frames_new], np.int32)
    return np.ascontiguousarray(xyz), cnt, np.ascontiguousarray(new), mcnt


def frames(xyz, cnt, new, mcnt):
    """inverse of stack: [(xyz_b, new_b, centre row offset)]"""
    ns, ms = np.concatenate([[0], np.cumsum(cnt)]), np.concatenate([[0], np.cumsum(mcnt)])
    return [(xyz[ns[k]:ns[k + 1]], new[ms[k]:ms[k + 1]], int(ms[k])) for k in range(len(cnt))]


def centres_from(rng, pts, m, jitter=0.3):
    """m centres: about half of them existing points, the rest points moved by up to `jitter` (misses included)"""
    if len(pts) == 0:
        return rng.uniform(-5, 5, size=(m, 3)).astype(np.float32)
    c = pts[rng.integers(0, len(pts), m)].astype(np.float32)
    move = rng.random(m) < 0.5
    c[move] += rng.uniform(-jitter, jitter, size=(int(move.sum()), 3)).astype(np.float32)
    return c


def ragged(seed=0):
    """four frames: 3000 points / 100 centres, 0 points / 30 centres, 1700 points / 0 centres, 2500 / 200"""
    rng = np.random.default_rng(seed)
    sizes, cents = [3000, 0, 1700, 2500], [100, 30, 0, 200]
    fx = [synth.cloud_ground_objects(1, n, seed=seed + k)[0] if n else np.zeros((0, 3), np.float32)
          for k, n in enumerate(sizes)]
    fn = [centres_from(rng, f, m) for f, m in zip(fx, cents)]
    return stack(fx, fn)


def dup_padded(seed=1):
    rng = np.random.default_rng(seed)
    fx = [synth.cloud_dup_padded(1, n, seed=seed + k)[0] for k, n in enumerate([4096, 2000])]
    return stack(fx, [centres_from(rng, f, 256) for f in fx])


def lattice():
    """points on a 0.5 m lattice, centres on lattice points: with r = 0.5 the six axis neighbours lie exactly at r
    (d2 == r*r, not a hit), with r = 0.75 they are in"""
    g = np.arange(-4, 4, dtype=np.float32) * 0.5
    pts = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    pts2 = pts[::-1] + np.float32(0.25)
    return stack([pts, pts2], [pts[::7], pts2[::5]])


def cases():
    """[(id, xyz, xyz_cnt, new_xyz, new_cnt, radius, nsample)] covering the contract's edges"""
    out = []
    rg = ragged()
    for ns in (1, 7, 32, 100):
        out.append((f"ragged-r0.8-ns{ns}", *rg, 0.8, ns))
    out.append(("ragged-r0", *rg, 0.0, 8))
    out.append(("ragged-rneg", *rg, -0.8, 16))
    out.append(("ragged-saturating", *rg, 1000.0, 32))
    dp = dup_padded()
    out.append(("dup-padded-r0.4-ns16", *dp, 0.4, 16))
    out.append(("dup-padded-r2-ns100", *dp, 2.0, 100))
    lt = lattice()
    out.append(("lattice-r0.5-ns7", *lt, 0.5, 7))
    out.append(("lattice-r0.75-ns32", *lt, 0.75, 32))
    return out
