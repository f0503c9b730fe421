"""CPU suite: the stacked ball-query oracle (tests/stack_bq_oracle.c) agrees, frame by frame, with
the batch ball-query oracle that tests/golden/ball_query.npz pins, and with those golden rows themselves (outputs of
the reference's own batch CUDA kernel on a B200) when the two golden clouds run as a 2-frame stack.

The two contracts differ only after the hits: the stack kernel repeats the FIRST hit where the batch kernel pads
cyclically, and marks a centre without hits with idx[p, 0] = -1 (other slots untouched) where the batch kernel zeroes
the row."""
import os

import numpy as np
import pytest

import stack_bq_oracle as sbq
import stack_cases

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def check_against_batch(idx, cnt_b, idx_b, nsample):
    """idx (m, nsample) stack rows of one frame vs the batch oracle's (cnt (m,), idx (m, nsample)) of the same frame"""
    for p in range(idx.shape[0]):
        k = min(int(cnt_b[p]), nsample)
        row = idx[p]
        if k == 0:
            assert row[0] == -1 and not row[1:].any(), (p, row)
        else:
            assert np.array_equal(row[:k], idx_b[p, :k]), (p, row, idx_b[p])
            assert (row[k:] == row[0]).all(), (p, row)


@pytest.mark.parametrize("case", stack_cases.cases(), ids=lambda c: c[0])
def test_stack_oracle_matches_batch_oracle_per_frame(orc, case):
    _, xyz, cnt, new, mcnt, radius, nsample = case
    idx = sbq.stack_ball_query(radius, nsample, xyz, cnt, new, mcnt)
    assert idx.shape == (new.shape[0], nsample)
    for fx, fn, m0 in stack_cases.frames(xyz, cnt, new, mcnt):
        if len(fn) == 0:
            continue
        cnt_b, idx_b = orc.ball_query(radius, nsample, fx[None], fn[None])
        check_against_batch(idx[m0:m0 + len(fn)], cnt_b[0], idx_b[0], nsample)


def test_stack_oracle_edge_semantics():
    """radius 0 and an empty frame hit nothing; a negative radius is its absolute value; a saturating radius fills
    every ball of a non-empty frame with its first nsample points"""
    xyz, cnt, new, mcnt = stack_cases.ragged()
    none = sbq.stack_ball_query(0.0, 8, xyz, cnt, new, mcnt)
    assert (none[:, 0] == -1).all() and not none[:, 1:].any()
    assert np.array_equal(sbq.stack_ball_query(-0.8, 16, xyz, cnt, new, mcnt),
                          sbq.stack_ball_query(0.8, 16, xyz, cnt, new, mcnt))
    full = sbq.stack_ball_query(1000.0, 32, xyz, cnt, new, mcnt)
    ms = np.concatenate([[0], np.cumsum(mcnt)])
    for k in range(len(cnt)):
        rows = full[ms[k]:ms[k + 1]]
        if cnt[k] == 0:
            assert (rows[:, 0] == -1).all()
        else:
            assert (rows == np.arange(32)[None, :]).all()


def test_stack_oracle_golden_two_frame_stack():
    """the two golden clouds as one 2-frame stack: every row's first min(cnt, nsample) entries are the reference's"""
    g = np.load(os.path.join(GOLDEN, "ball_query.npz"))
    b, n, _ = g["xyz"].shape
    m = g["new_xyz"].shape[1]
    cnt = np.full((b,), n, np.int32)
    mcnt = np.full((b,), m, np.int32)
    for key, r, ns in (("r08", 0.8, 32), ("r02", 0.2, 16), ("r30", 3.0, 8)):
        idx = sbq.stack_ball_query(r, ns, g["xyz"].reshape(-1, 3), cnt, g["new_xyz"].reshape(-1, 3), mcnt)
        check_against_batch(idx, g[key + "_cnt"].reshape(-1), g[key + "_idx"].reshape(-1, ns), ns)
