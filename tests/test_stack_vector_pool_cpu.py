"""CPU suite of the vector-pool oracle (tests/vector_pool_oracle.c), the restatement the GPU kernels of
csrc/stack_vector_pool.cu are checked against bit for bit:

  * ball lists (no point at exactly D, capped at nsample) equal the golden-pinned stacked ball query's first hits made
    global (tests/stack_bq_oracle.c), which ties the distance expression and the index order to the reference;
  * with D covering whole frames of fewer than 1000 points, the list 3-NN fills the slots the stacked three_nn fills
    (tests/stack_nn_oracle.py), bit for bit;
  * average-pool sums against a float64 sum within fp32 rounding, counts against a histogram of the sub-voxel index,
    random choice taking the lowest row of each sub-voxel;
  * hand-built cases for the 1000 cap, points at exactly D (ball and cube), the +D face and the single-index clamp,
    channel folding (i % cpg), the -1 slots and the random-choice stop rule."""
import numpy as np
import pytest

import stack_bq_oracle as sbq
import stack_cases
import stack_nn_oracle as sno
import vector_pool_oracle as vpo


def _ragged():
    return stack_cases.ragged()  # frames of 3000 / 0 / 1700 / 2500 points with 100 / 30 / 0 / 200 centres


def _global_first_hits(xyz, cnt, new, mcnt, d, nsample):
    """the stacked ball query's hits per centre as GLOBAL rows: its rows hold the ascending hits, then repeat the first"""
    idx = sbq.stack_ball_query(d, nsample, xyz, cnt, new, mcnt)
    ns = np.concatenate([[0], np.cumsum(cnt)])
    out = []
    for (fx, fn, m0), start in zip(stack_cases.frames(xyz, cnt, new, mcnt), ns):
        for p in range(m0, m0 + len(fn)):
            row = idx[p]
            hits = [] if row[0] == -1 else [int(row[0])]
            for v in row[1:] if hits else []:
                if v <= hits[-1]:
                    break
                hits.append(int(v))
            out.append(np.asarray(hits, np.int32) + start)
    return out


@pytest.mark.parametrize("d,nsample", [(0.8, 7), (0.8, 32), (1.5, 100)])
def test_ball_lists_equal_stacked_ball_query(d, nsample):
    xyz, cnt, new, mcnt = _ragged()
    lists = vpo.local_lists(xyz, cnt, new, mcnt, d, nsample, 1)
    ref = _global_first_hits(xyz, cnt, new, mcnt, d, nsample)
    assert len(lists) == len(ref)
    for p, (a, b) in enumerate(zip(lists, ref)):
        assert np.array_equal(a, b), (p, a, b)
    assert sum(len(x) for x in lists) > 0
    # no point at exactly D, the only place the ball query's strict < and the vector pool's <= differ
    assert sum(len(x) for x in vpo.local_lists(xyz, cnt, new, mcnt, d, nsample, 1)) == \
        sum(len(x) for x in _global_first_hits(xyz, cnt, new, mcnt, np.nextafter(np.float32(d), np.float32(9)), nsample))


def test_three_nn_over_whole_frames_equals_stacked_three_nn():
    rng = np.random.default_rng(3)
    fx = [rng.uniform(-2, 2, (n, 3)).astype(np.float32) for n in (600, 2, 900)]
    fn = [rng.uniform(-2, 2, (m, 3)).astype(np.float32) for m in (20, 5, 30)]
    xyz, cnt, new, mcnt = stack_cases.stack(fx, fn)
    lists = vpo.local_lists(xyz, cnt, new, mcnt, 100.0, -1, 0)  # the cube covers every frame
    ns = np.concatenate([[0], np.cumsum(cnt)])
    ms = np.concatenate([[0], np.cumsum(mcnt)])
    for f in range(3):
        for p in range(ms[f], ms[f + 1]):
            assert np.array_equal(lists[p], np.arange(ns[f], ns[f + 1]))
    G = 4
    centres = (new[:, None, :] + rng.uniform(-1, 1, (new.shape[0], G, 3))).astype(np.float32)
    idx, dist2 = vpo.three_nn_local(xyz, centres, lists)
    ucnt = mcnt * G
    d_ref, i_ref = sno.stack_three_nn(centres.reshape(-1, 3), ucnt.astype(np.int32), xyz, cnt)
    filled = idx.reshape(-1, 3) != -1
    assert np.array_equal(idx.reshape(-1, 3)[filled], i_ref[filled])
    assert np.array_equal(dist2.reshape(-1, 3)[filled].view(np.int32), d_ref[filled].view(np.int32))
    # the frame of two points: slot 2 is (+inf, -1)
    rows = slice(int(ms[1]) * G, int(ms[2]) * G)
    assert (idx.reshape(-1, 3)[rows, 2] == -1).all() and np.isinf(dist2.reshape(-1, 3)[rows, 2]).all()
    assert (idx.reshape(-1, 3)[rows, :2] >= ns[1]).all()


def _sub_voxel(l, d, grids):
    gs = np.float32(d) * np.float32(2) / np.float32(np.array(grids, np.float32))
    i = np.floor(((l + np.float32(d)).astype(np.float32) / gs).astype(np.float32)).astype(np.int64)
    nx, ny, nz = grids
    return np.clip(i[:, 0] * ny * nz + i[:, 1] * nz + i[:, 2], 0, nx * ny * nz - 1)


@pytest.mark.parametrize("ball", [0, 1])
def test_avg_pool_against_float64_and_histogram(ball):
    xyz, cnt, new, mcnt = _ragged()
    rng = np.random.default_rng(4)
    C, d, grids = 6, 0.9, (3, 3, 3)
    feats = rng.normal(size=(xyz.shape[0], C)).astype(np.float32)
    nf, nl, pc, tr, total = vpo.vector_pool(xyz, cnt, feats, new, mcnt, grids, C, d, 1, -1, ball, 0)
    G = 27
    lists = vpo.local_lists(xyz, cnt, new, mcnt, d, -1, ball)
    assert total == sum(len(x) for x in lists) and tr.shape[0] == total
    for p in range(new.shape[0]):
        rows = np.asarray(lists[p], np.int64)
        assert len(rows) < 1000
        l = (xyz[rows] - new[p]).astype(np.float32)
        g = _sub_voxel(l, d, grids)
        assert np.array_equal(pc[p], np.bincount(g, minlength=G))
        ref = np.zeros((G, C))
        np.add.at(ref, g, feats[rows].astype(np.float64))
        bound = 1e-6 * (np.abs(feats[rows]).sum() + 1) * 2
        assert np.abs(nf[p].reshape(G, C) - ref).max() <= bound
        refl = np.zeros((G, 3))
        np.add.at(refl, g, l.astype(np.float64))
        assert np.abs(nl[p].reshape(G, 3) - refl).max() <= 1e-5 * (len(rows) + 1)
        sel = tr[:, 1] == p
        assert np.array_equal(tr[sel, 0], rows) and np.array_equal(tr[sel, 2], g)


def test_random_choice_takes_lowest_row_per_sub_voxel():
    xyz, cnt, new, mcnt = _ragged()
    rng = np.random.default_rng(5)
    C, d, grids = 4, 0.9, (2, 2, 2)
    feats = rng.normal(size=(xyz.shape[0], C)).astype(np.float32)
    nf, nl, pc, tr, total = vpo.vector_pool(xyz, cnt, feats, new, mcnt, grids, C, d, 1, -1, 0, 1)
    lists = vpo.local_lists(xyz, cnt, new, mcnt, d, -1, 0)
    for p in range(new.shape[0]):
        rows = np.asarray(lists[p], np.int64)
        g = _sub_voxel((xyz[rows] - new[p]).astype(np.float32), d, grids)
        firsts = {}
        for r, gg in zip(rows, g):
            firsts.setdefault(int(gg), int(r))
        assert set(np.nonzero(pc[p])[0].tolist()) == set(firsts)
        assert pc[p].max(initial=0) <= 1
        for gg, r in firsts.items():
            assert np.array_equal(nf[p].reshape(8, C)[gg], feats[r])
            assert np.array_equal(nl[p].reshape(8, 3)[gg], (xyz[r] - new[p]).astype(np.float32))
        sel = tr[:, 1] == p
        assert sorted(tr[sel, 0].tolist()) == sorted(firsts.values())


def _one_frame(pts, centre):
    pts = np.asarray(pts, np.float32).reshape(-1, 3)
    return pts, np.array([len(pts)], np.int32), np.asarray(centre, np.float32).reshape(-1, 3), np.array([1], np.int32)


def test_cap_of_1000():
    pts = np.zeros((1500, 3), np.float32)
    pts[:, 0] = np.linspace(-0.5, 0.5, 1500)
    lists = vpo.local_lists(*_one_frame(pts, [0, 0, 0]), 1.0, -1, 0)
    assert np.array_equal(lists[0], np.arange(1000))
    assert np.array_equal(vpo.local_lists(*_one_frame(pts, [0, 0, 0]), 1.0, 1200, 0)[0], np.arange(1000))
    assert np.array_equal(vpo.local_lists(*_one_frame(pts, [0, 0, 0]), 1.0, 5, 0)[0], np.arange(5))


def test_points_at_exactly_d_are_hits():
    pts = [[0.5, 0, 0], [0, -0.5, 0], [0.5, 0.5, 0.5], [0.5000001, 0, 0], [0, 0, -0.75]]
    f = _one_frame(pts, [0, 0, 0])
    assert vpo.local_lists(*f, 0.5, -1, 1)[0].tolist() == [0, 1]       # ball: d2 == D*D is in, the corner is out
    assert vpo.local_lists(*f, 0.5, -1, 0)[0].tolist() == [0, 1, 2]    # cube: |l| == D on every axis is in


def test_plus_d_face_and_single_index_clamp():
    d, grids = 1.0, (2, 2, 2)
    # local (-0.5, +1, -0.5): iy = 2 -> g = 0*4 + 2*2 + 0 = 4, the next x slab; local (+1, +1, +1): g = 14 -> 7
    pts = [[-0.5, 1.0, -0.5], [1.0, 1.0, 1.0], [-1.0, -1.0, -1.0]]
    feats = np.array([[1.0], [2.0], [4.0]], np.float32)
    nf, nl, pc, tr, total = vpo.vector_pool(*_one_frame(pts, [0, 0, 0])[:2], feats, *_one_frame(pts, [0, 0, 0])[2:],
                                            grids, 1, d, 1, -1, 0, 0)
    assert total == 3
    assert pc[0].tolist() == [1, 0, 0, 0, 1, 0, 0, 1]
    assert nf[0].tolist() == [4.0, 0, 0, 0, 1.0, 0, 0, 2.0]


def test_channel_folding():
    pts = [[0.1, 0.1, 0.1], [0.2, 0.2, 0.2]]
    feats = np.array([[1, 2, 3, 4, 5, 6], [10, 20, 30, 40, 50, 60]], np.float32)
    x, c, n, m = _one_frame(pts, [0, 0, 0])
    nf, nl, pc, tr, total = vpo.vector_pool(x, c, feats, n, m, (1, 1, 1), 2, 1.0, 1, -1, 0, 0)
    assert nf[0].tolist() == [1 + 3 + 5 + 10 + 30 + 50, 2 + 4 + 6 + 20 + 40 + 60]
    assert pc[0].tolist() == [2]
    nf, nl, pc, tr, total = vpo.vector_pool(x, c, feats, n, m, (1, 1, 1), 2, 1.0, 1, -1, 0, 1)
    assert nf[0].tolist() == [5, 6] and total == 1  # random choice: the last write of the channel loop, first hit only


def test_minus_one_slots_and_the_last_row():
    pts = np.array([[0.1, 0, 0], [5, 5, 5], [9, 9, 9]], np.float32)
    lists = [np.array([0], np.int32)]
    centres = np.array([[[0, 0, 0], [0.2, 0, 0]]], np.float32)
    idx, dist2 = vpo.three_nn_local(pts, centres, lists)
    assert idx[0].tolist() == [[0, -1, -1], [0, -1, -1]]
    assert np.isinf(dist2[0, :, 1:]).all()
    # the module's offsets: a -1 slot reads the LAST support row (Python's negative index)
    off = centres.reshape(-1, 1, 3) - pts[idx.reshape(-1, 3).astype(np.int64)]
    assert np.array_equal(off[0, 1], centres[0, 0] - pts[-1])


def test_random_choice_stop_rule():
    rng = np.random.default_rng(6)
    pts = rng.uniform(-1, 1, (400, 3)).astype(np.float32)
    feats = rng.normal(size=(400, 2)).astype(np.float32)
    x, c, n, m = _one_frame(pts, [0, 0, 0])
    _, _, pc, tr, total = vpo.vector_pool(x, c, feats, n, m, (2, 2, 2), 2, 1.0, 1, -1, 0, 1)
    assert total == 8 and pc[0].tolist() == [1] * 8  # stops once every sub-voxel is taken
    _, _, pc, tr, total = vpo.vector_pool(x, c, feats, n, m, (2, 2, 2), 2, 1.0, 1, 3, 0, 1)
    assert total == 3 and pc[0].sum() == 3  # ... or after nsample taken
    _, _, pc, tr, total = vpo.vector_pool(x, c, feats, n, m, (2, 2, 2), 2, 1.0, 1, 5, 0, 0)
    assert total == 5 and pc[0].sum() == 5 and tr[:, 0].tolist() == list(range(5))  # average: nsample hits
