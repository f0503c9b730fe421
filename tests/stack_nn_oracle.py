"""CPU oracle of the stacked (ragged) three_nn / three_interpolate (TEST INFRASTRUCTURE): the batch oracle
(oracle/pointnet2_oracle.c, pinned by tests/golden/interpolate.npz) applied frame by frame, plus the frame's known start.

The stack contract: unknown row p belongs to the first frame k with p < N0 + ... + Nk; its three nearest known points of
that frame, ties to the smaller index, as GLOBAL rows; slots a frame with fewer than three known points cannot fill are
(+inf, the frame's known start).  The interpolation reads 0 for an index outside [0, M) (the kernel's guard: the batch
oracle indexes without a bound, so a zero feature row is appended and such indices are mapped to it)."""
from __future__ import annotations

import numpy as np

from oracle import oracle as orc


def stack_three_nn(unknown, unknown_cnt, known, known_cnt):
    """unknown (N,3), known (M,3) float32, counts (B,) -> (dist2 (N,3) float32, idx (N,3) int32 global rows)"""
    n = unknown.shape[0]
    us = np.concatenate([[0], np.cumsum(unknown_cnt)])
    ks = np.concatenate([[0], np.cumsum(known_cnt)])
    dist2 = np.empty((n, 3), np.float32)
    idx = np.empty((n, 3), np.int32)
    for f in range(len(unknown_cnt)):
        u0, u1 = int(us[f]), (n if f == len(unknown_cnt) - 1 else int(us[f + 1]))  # the last frame takes the rest
        if u1 <= u0:
            continue
        kn = np.ascontiguousarray(known[ks[f]:ks[f + 1]], np.float32).reshape(1, -1, 3)
        d, i = orc.three_nn(np.ascontiguousarray(unknown[u0:u1], np.float32)[None], kn)
        dist2[u0:u1], idx[u0:u1] = d[0], i[0] + ks[f]
    return dist2, idx


def stack_three_interpolate(features, idx, weight):
    """features (M,C), idx / weight (N,3) -> (N,C) float32"""
    m, c = features.shape
    planes = np.concatenate([features, np.zeros((1, c), np.float32)], 0).T[None]  # (1, C, M + 1)
    safe = np.where((idx >= 0) & (idx < m), idx, m).astype(np.int32)
    return orc.three_interpolate(np.ascontiguousarray(planes), safe[None], np.asarray(weight, np.float32)[None])[0].T.copy()
