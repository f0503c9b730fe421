"""CPU suite of the roiaware_pool3d ops: the oracle (tests/roiaware_oracle.c) by hand cases, each of which fails if its
rule changes; the rounding-aware classifier against the oracle; the library's points_in_boxes_cpu (host code) against
the oracle bit for bit; the new C-ABI symbols."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import roiaware_oracle as rao  # noqa: E402
import synth  # noqa: E402
from roiaware_oracle import boxes_on_points  # noqa: E402

NEW_SYMBOLS = ["tsmdet_points_in_boxes", "tsmdet_points_in_boxes_cpu", "tsmdet_roiaware_pool3d",
               "tsmdet_roiaware_pool3d_grad"]


def _box(cx=0.0, cy=0.0, cz=0.0, dx=2.0, dy=2.0, dz=2.0, h=0.0):
    return np.array([cx, cy, cz, dx, dy, dz, h], np.float32)


def _pib(boxes, pts):
    """oracle points_in_boxes (GPU form) of one frame"""
    return rao.points_in_boxes(np.asarray(boxes, np.float32)[None], np.asarray(pts, np.float32)[None])[0]


def _edges(t):
    """the largest float32 below the float64 threshold t and the smallest float32 at or above it"""
    f = np.float32(t)
    if np.float64(f) >= t:
        return np.nextafter(f, np.float32(-np.inf)), f
    return f, np.nextafter(f, np.float32(np.inf))


# ------------------------------------------------------------------------------------------------ oracle hand cases
def test_heading_zero_boundaries_are_the_double_thresholds():
    """heading 0: cosf = 1 and sinf = -0 exactly, so local_x = x - cx bit for bit and the compare is the double one"""
    for margin, cpu in ((1e-5, False), (1e-2, True)):
        t = 1.0 / 2.0 + np.float64(np.float32(margin))
        below, up = _edges(t)
        pts = np.array([[below, 0, 0], [up, 0, 0], [-below, 0, 0], [-up, 0, 0],
                        [0, below, 0], [0, up, 0]], np.float32)
        box = _box(dx=1.0, dy=1.0)
        got = rao.points_in_boxes_cpu(box[None], pts)[0] if cpu else (_pib(box[None], pts) == 0).astype(np.int32)
        assert got.tolist() == [1, 0, 1, 0, 1, 0], (margin, got)


def test_point_on_the_z_face_is_inside():
    box = _box(cz=1.0, dz=2.0)
    # z - cz = 1 + 2^-22 and -(1 + 2^-23): the nearest floats beyond the faces
    pts = np.array([[0, 0, 2.0], [0, 0, 0.0], [0, 0, np.nextafter(np.float32(2.0), np.float32(3))],
                    [0, 0, -2.0 ** -23]], np.float32)
    assert _pib(box[None], pts).tolist() == [0, 0, -1, -1]


def test_zero_padding_box_holds_points_at_the_origin():
    """all seven values 0: |z| > 0 rejects, |x|, |y| < 0 + MARGIN: points within 1e-5 of the origin in x, y, z == 0"""
    box = np.zeros((1, 7), np.float32)
    pts = np.array([[0, 0, 0], [5e-6, -5e-6, 0], [0, 0, -0.0], [0, 0, 1e-30], [2e-5, 0, 0], [5e-3, 0, 0]], np.float32)
    assert _pib(box, pts).tolist() == [0, 0, 0, -1, -1, -1]
    assert rao.points_in_boxes_cpu(box, pts)[0].tolist() == [1, 1, 1, 0, 1, 1]  # the CPU margin is 1e-2


def test_nan_coordinates_are_never_inside():
    box = _box()
    nan = np.float32(np.nan)
    pts = np.array([[nan, 0, 0], [0, nan, 0], [0, 0, nan], [0, 0, 0]], np.float32)
    assert _pib(box[None], pts).tolist() == [-1, -1, -1, 0]
    assert rao.points_in_boxes_cpu(box[None], pts)[0].tolist() == [0, 0, 0, 1]
    for k in range(7):  # a NaN in the box
        b = _box()
        b[k] = nan
        assert _pib(b[None], pts[3:]).tolist() == [-1], k


def test_first_box_wins():
    boxes = np.stack([_box(cx=5.0), _box(cx=0.5), _box(cx=0.0, dx=4.0)])
    pts = np.array([[0.6, 0, 0], [-1.5, 0, 0], [5, 0, 0], [20, 0, 0]], np.float32)
    assert _pib(boxes, pts).tolist() == [1, 2, 0, -1]


def test_list_cap_and_saturating_counter():
    roi = _box(dx=2, dy=2, dz=2)[None]
    pts = np.random.default_rng(0).uniform(-0.9, 0.9, (200, 3)).astype(np.float32)
    feats = np.zeros((200, 1), np.float32)
    for L, want in ((1, 0), (2, 1), (128, 127)):
        idx, _, _ = rao.forward(roi, pts, feats, 1, L, 0)
        assert idx[0, 0, 0, 0, 0] == want
        assert idx[0, 0, 0, 0, 1:1 + want].tolist() == list(range(want))


def test_max_pool_ties_infinities_nans_and_empty_voxels():
    roi = _box(dx=4, dy=2, dz=2)[None]  # out (2,1,1): x < 0 voxel 0, x > 0 voxel 1
    pts = np.array([[-1, 0, 0]] * 4 + [[1, 0, 0]] * 3, np.float32)
    ninf, nan = -np.inf, np.nan
    feats = np.array([[1, ninf, nan], [3, ninf, 1], [3, ninf, nan], [2, ninf, 2],
                      [ninf, nan, 0], [ninf, nan, 0], [ninf, nan, -0.0]], np.float32)
    idx, am, pooled = rao.forward(roi, pts, feats, (2, 1, 1), 128, 0)
    assert idx[0, :, 0, 0, 0].tolist() == [4, 3]
    assert am[0, 0, 0, 0].tolist() == [1, -1, 3]   # first maximum; -inf never taken; NaN never taken
    assert pooled[0, 0, 0, 0].tolist() == [3, 0, 2]
    assert am[0, 1, 0, 0].tolist() == [-1, -1, 4]  # -inf / NaN only: argmax -1, pooled left 0
    assert pooled[0, 1, 0, 0].tolist() == [0, 0, 0]
    idx, am, pooled = rao.forward(_box(cx=50)[None], pts, feats, (2, 1, 1), 128, 0)  # empty RoI
    assert (am == -1).all() and (pooled == 0).all() and (idx == 0).all()


def test_avg_pool_sums_in_list_order():
    roi = _box()[None]
    pts = np.zeros((4, 3), np.float32)
    feats = np.array([[1e8], [1], [-1e8], [1]], np.float32)
    _, am, pooled = rao.forward(roi, pts, feats, 1, 128, 1)
    seq = np.float32(0)
    for v in feats[:, 0]:
        seq = np.float32(seq + v)
    assert seq == np.float32(1) and np.float64(feats[:, 0].astype(np.float64).sum()) == 2.0
    assert pooled[0, 0, 0, 0, 0] == np.float32(seq / np.float32(4)) == np.float32(0.25)  # not 0.5: sequential float
    assert (am == 0).all()  # avg pooling leaves argmax alone
    _, _, pooled = rao.forward(_box(cx=9)[None], pts, feats, 1, 128, 1)
    assert (pooled == 0).all()


def test_degenerate_boxes_use_the_device_float_to_int_conversion():
    """dx = 0: x_res = 0, (l + 0) / 0 is NaN (-> index 0) at l = 0, +-inf (saturated, then the unsigned clamp: both the
    last voxel) otherwise; a tiny box gives a negative index, which the unsigned clamp puts in the last voxel too"""
    roi = _box(dx=0.0, dy=2.0, dz=2.0)[None]
    pts = np.array([[0, 0, 0], [5e-6, 0, 0], [-5e-6, 0, 0], [2e-5, 0, 0]], np.float32)
    idx, _, _ = rao.forward(roi, pts, np.zeros((4, 1), np.float32), (4, 1, 1), 8, 0)
    assert idx[0, :, 0, 0, 0].tolist() == [1, 0, 0, 2]
    assert idx[0, 0, 0, 0, 1] == 0 and idx[0, 3, 0, 0, 1:3].tolist() == [1, 2]
    roi = _box(dx=1e-5)[None]
    pts = np.array([[-9e-6, 0, 0]], np.float32)  # inside (|x| < 5e-6 + 1e-5); (x + 5e-6) / (1e-5 / 256) ~ -102
    idx, _, _ = rao.forward(roi, pts, np.zeros((1, 1), np.float32), (256, 1, 1), 4, 0)
    assert idx[0, 255, 0, 0, 0] == 1 and idx[0, :255].sum() == 0


@pytest.mark.parametrize("out_size", [(1, 1, 1), (7, 5, 3)])
def test_voxel_coordinates_by_hand(out_size):
    roi = _box(dx=7, dy=5, dz=3)[None]  # resolution 1 per axis at (7, 5, 3)
    pts = np.array([[-3.2, 2.1, 0.4], [3.4, -2.4, -1.4], [0.1, 0.1, 0.1]], np.float32)
    idx, _, _ = rao.forward(roi, pts, np.ones((3, 2), np.float32), out_size, 4, 0)
    if out_size == (1, 1, 1):
        assert idx[0, 0, 0, 0].tolist() == [3, 0, 1, 2]
    else:
        assert idx.shape == (1, 7, 5, 3, 4)
        assert idx[0, 0, 4, 1].tolist() == [1, 0, 0, 0]
        assert idx[0, 6, 0, 0].tolist() == [1, 1, 0, 0]
        assert idx[0, 3, 2, 1].tolist() == [1, 2, 0, 0]
        assert idx[..., 0].sum() == 3


def test_rotated_box_local_frame():
    """heading pi/2: local_x = y - cy, local_y = -(x - cx) up to the float rounding of cosf / sinf"""
    roi = _box(dx=4, dy=2, dz=2, h=np.pi / 2)[None]
    pts = np.array([[0, 1.5, 0], [1.5, 0, 0], [0.5, -1.9, 0]], np.float32)
    assert _pib(roi, pts).tolist() == [0, -1, 0]
    idx, _, _ = rao.forward(roi, pts, np.ones((3, 1), np.float32), (4, 2, 1), 4, 0)
    assert idx[0, 3, 0, 0, :2].tolist() == [1, 0]  # local (1.5, -6.6e-8) -> x voxel 3, y voxel int(0.99999994) = 0
    assert idx[0, 0, 0, 0, :2].tolist() == [1, 2]  # local (-1.9, -0.5)


# ------------------------------------------------------------------------------------------------ classifier
def test_classifier_agrees_with_the_oracle_on_decided_pairs_and_decides_almost_all():
    pts = synth.cloud_ground_objects(1, 20000, seed=3)[0]
    for boxes in (boxes_on_points(pts, 64, 1), synth.boxes_clustered(64, seed=2)):
        inside, decided = rao.classify(boxes, pts)
        got = np.stack([_pib(b[None], pts) == 0 for b in boxes])
        assert np.array_equal(got[decided], inside[decided])
        assert (~decided).mean() < 1e-4
        # the voxel classifier only ever removes pairs
        assert not (rao.classify_voxels(boxes, pts, 14) & ~decided).any()


def test_classifier_marks_the_threshold_neighbourhood_undecided():
    h = np.float32(0.3)
    box = _box(dx=2.0, h=h)
    c, s = np.cos(-np.float64(h)), np.sin(-np.float64(h))
    t = 1.0 + np.float64(np.float32(1e-5))
    # points whose exact local_x is t (on the threshold) and t -+ 1e-3 (decided)
    pts = np.array([[lx * c, -lx * s, 0] for lx in (t, t - 1e-3, t + 1e-3)], np.float32)
    inside, decided = rao.classify(box[None], pts)
    assert decided[0].tolist() == [False, True, True] and inside[0].tolist()[1:] == [True, False]


# ------------------------------------------------------------------------------------------------ the library
def _lib_cpu(boxes, pts):
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_utils as ru

    return ru.points_in_boxes_cpu(pts, boxes)


@pytest.mark.parametrize("kind", ["on_points", "clustered", "random", "heading_zero"])
def test_points_in_boxes_cpu_library_equals_oracle(kind):
    pts = synth.cloud_ground_objects(1, 8000, seed=5)[0]
    boxes = {"on_points": boxes_on_points(pts, 48, 7), "clustered": synth.boxes_clustered(48, seed=8),
             "random": synth.boxes_random(48, seed=9), "heading_zero": boxes_on_points(pts, 48, 10)}[kind]
    if kind == "heading_zero":
        boxes[:, 6] = 0
    got = _lib_cpu(boxes, pts)
    assert isinstance(got, np.ndarray) and got.dtype == np.int32 and got.shape == (48, 8000)
    want = rao.points_in_boxes_cpu(boxes, pts)
    assert np.array_equal(got, want)
    if kind in ("on_points", "heading_zero"):
        assert want.sum() > 200


def test_points_in_boxes_cpu_hand_cases_and_empty_shapes():
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_utils as ru

    nan = np.float32(np.nan)
    t = 0.5 + np.float64(np.float32(1e-2))
    below, up = _edges(t)
    pts = np.array([[below, 0, 0], [up, 0, 0], [0, 0, 1.0], [nan, 0, 0], [0, 0, nan], [5e-3, 0, 0]], np.float32)
    boxes = np.stack([_box(dx=1.0), np.zeros(7, np.float32)])
    got = ru.points_in_boxes_cpu(pts, boxes)
    assert got.tolist() == [[1, 0, 1, 0, 0, 1], [0, 0, 0, 0, 0, 1]]
    assert np.array_equal(got, rao.points_in_boxes_cpu(boxes, pts))
    # tensors in -> tensor out
    tg = ru.points_in_boxes_cpu(torch.from_numpy(pts), torch.from_numpy(boxes))
    assert isinstance(tg, torch.Tensor) and tg.dtype == torch.int32 and np.array_equal(tg.numpy(), got)
    assert ru.points_in_boxes_cpu(pts, np.zeros((0, 7), np.float32)).shape == (0, 6)
    assert ru.points_in_boxes_cpu(np.zeros((0, 3), np.float32), boxes).shape == (2, 0)


def test_shim_rejects_wrong_device_dtype_and_layout():
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_cuda as ext

    b, p = torch.zeros(2, 7), torch.zeros(3, 3)
    with pytest.raises(ValueError):
        ext.points_in_boxes_cpu(b, p, torch.zeros(2, 3))  # float output
    with pytest.raises(ValueError):
        ext.points_in_boxes_cpu(b.double(), p, torch.zeros(2, 3, dtype=torch.int32))
    with pytest.raises(ValueError):
        ext.points_in_boxes_cpu(torch.zeros(7, 2).t(), p, torch.zeros(2, 3, dtype=torch.int32))
    with pytest.raises(ValueError):  # CPU tensors into the GPU functions
        ext.points_in_boxes_gpu(b[None], p[None], torch.zeros(1, 3, dtype=torch.int32))
    with pytest.raises(ValueError):
        ext.forward(b, p, torch.zeros(3, 4), torch.zeros(2, 1, 1, 1, 4, dtype=torch.int32),
                    torch.zeros(2, 1, 1, 1, 8, dtype=torch.int32), torch.zeros(2, 1, 1, 1, 4), 0)


def test_c_abi_rejects_invalid_sizes():
    from tsmdet_b200 import _lib

    f = _lib.lib()
    assert f.tsmdet_points_in_boxes_cpu(-1, 3, None, None, None) == 1000001
    assert f.tsmdet_points_in_boxes(1, -1, 3, None, None, None, None) == 1000001
    for dims in [(257, 1, 1), (1, 257, 1), (1, 1, 257), (0, 1, 1)]:
        assert f.tsmdet_roiaware_pool3d(1, 1, 1, *dims, 4, None, None, None, None, None, None, 0, None) == 1000001
        assert f.tsmdet_roiaware_pool3d_grad(1, 1, 1, *dims, 4, None, None, None, None, 0, None) == 1000001
    assert f.tsmdet_roiaware_pool3d(1, 1, 1, 2, 2, 2, 0, None, None, None, None, None, None, 0, None) == 1000001
    assert f.tsmdet_roiaware_pool3d(-1, 1, 1, 2, 2, 2, 4, None, None, None, None, None, None, 0, None) == 1000001
    assert f.tsmdet_roiaware_pool3d(1, -1, 1, 2, 2, 2, 4, None, None, None, None, None, None, 0, None) == 1000001
    assert f.tsmdet_roiaware_pool3d(1, 1, 1, 2, 2, 2, 4, None, None, None, None, None, None, 2, None) == 1000001
    # nothing to do: no device needed
    assert f.tsmdet_roiaware_pool3d(0, 5, 1, 256, 256, 256, 1, None, None, None, None, None, None, 1, None) == 0


def test_new_symbols_declared_and_exported():
    from tsmdet_b200 import _lib

    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                               "tsmdet_b200.h")).read()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in NEW_SYMBOLS:
        assert f"int {name}(" in header
        assert hasattr(lib, name) and name in _lib.SIGNATURES
