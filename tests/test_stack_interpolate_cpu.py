"""CPU suite: the stacked 3-NN / interpolation oracle (tests/stack_nn_oracle.py) reproduces the reference's own batch
kernel outputs pinned in tests/golden/interpolate.npz when the two golden clouds run as a 2-frame stack, and follows the
stack contract on frames with 0 / 1 / 2 / 3 known points and frames without unknown points."""
import os

import numpy as np

import stack_nn_oracle as sno

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_stack_oracle_golden_two_frame_stack():
    g = np.load(os.path.join(GOLDEN, "interpolate.npz"))
    b, n, _ = g["unknown"].shape
    m = g["known"].shape[1]
    ucnt, kcnt = np.full((b,), n, np.int32), np.full((b,), m, np.int32)
    d2, idx = sno.stack_three_nn(g["unknown"].reshape(-1, 3), ucnt, g["known"].reshape(-1, 3), kcnt)
    assert np.array_equal(d2.view(np.uint32), g["dist2"].reshape(-1, 3).view(np.uint32))
    assert np.array_equal(idx, (g["idx"] + (np.arange(b) * m)[:, None, None]).reshape(-1, 3))
    feats = g["feats"].transpose(0, 2, 1).reshape(-1, g["feats"].shape[1])  # (B*M, C) rows
    out = sno.stack_three_interpolate(feats, idx, g["weight"].reshape(-1, 3))
    want = g["out"].transpose(0, 2, 1).reshape(-1, g["out"].shape[1])
    assert np.array_equal(out.view(np.uint32), want.view(np.uint32))


def test_stack_oracle_small_frames():
    """frames with 0 / 1 / 2 / 3 known points and one without unknown points"""
    rng = np.random.default_rng(0)
    kcnt = np.array([3, 0, 1, 2, 5], np.int32)
    ucnt = np.array([4, 3, 2, 0, 5], np.int32)
    known = rng.uniform(-2, 2, (int(kcnt.sum()), 3)).astype(np.float32)
    unknown = rng.uniform(-2, 2, (int(ucnt.sum()), 3)).astype(np.float32)
    d2, idx = sno.stack_three_nn(unknown, ucnt, known, kcnt)
    ks, us = np.concatenate([[0], np.cumsum(kcnt)]), np.concatenate([[0], np.cumsum(ucnt)])
    for f in range(len(kcnt)):
        for p in range(us[f], us[f + 1]):
            kn = known[ks[f]:ks[f + 1]]
            d = (((kn - unknown[p]) ** 2).sum(1)).astype(np.float32)
            order = np.lexsort((np.arange(len(d)), d))[:3]
            k = len(order)
            assert np.allclose(d2[p, :k], d[order], rtol=1e-6) and np.array_equal(idx[p, :k], order + ks[f])
            assert np.isinf(d2[p, k:]).all() and (idx[p, k:] == ks[f]).all()
    # frame 1 has no known points: its rows point at its known start (3, the first point of frame 2), an in-range row
    assert (idx[us[1]:us[2]] == 3).all()
    feats = rng.standard_normal((int(kcnt.sum()), 6)).astype(np.float32)
    w = rng.random((unknown.shape[0], 3)).astype(np.float32)
    out = sno.stack_three_interpolate(feats, idx, w)
    want = (w[:, 2:3] * feats[idx[:, 2]]).astype(np.float64)
    want += w[:, 0:1] * feats[idx[:, 0]] + w[:, 1:2] * feats[idx[:, 1]]
    assert np.allclose(out, want, rtol=1e-5, atol=1e-6)


def test_stack_oracle_interpolation_guard():
    """an index outside [0, M) reads a zero feature row"""
    feats = np.arange(12, dtype=np.float32).reshape(4, 3) + 1
    idx = np.array([[4, 0, -1], [1, 4, 4]], np.int32)
    w = np.ones((2, 3), np.float32)
    out = sno.stack_three_interpolate(feats, idx, w)
    assert np.array_equal(out, np.stack([feats[0], feats[1]]))
