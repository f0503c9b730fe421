"""GPU suite of the roiaware_pool3d ops against the CPU oracle (tests/roiaware_oracle.c): points_in_boxes_gpu on every
pair the rounding-aware classifier calls decided (all pairs for heading-0 boxes); the RoIAwarePool3d forward bit for bit
on inputs without undecided points; the backward against a float64 scatter; the module and its CUDA-graph capture."""
import os
import sys

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import roiaware_oracle as rao  # noqa: E402
import synth  # noqa: E402
from roiaware_oracle import boxes_on_points  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _gpu_labels(boxes, pts):
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_utils as ru

    out = ru.points_in_boxes_gpu(torch.from_numpy(pts).to(DEV), torch.from_numpy(boxes).to(DEV))
    assert out.dtype == torch.int32 and out.shape == pts.shape[:2]
    return out.cpu().numpy()


def _comparable(boxes, pts, want):
    """(B, N) bool: every pair that decides the point's label (boxes 0 .. label, or all of them) is decided"""
    ok = np.ones(want.shape, bool)
    for f in range(boxes.shape[0]):
        _, dec = rao.classify(boxes[f], pts[f])
        if dec.shape[0] == 0:
            continue
        prefix_ok = np.logical_and.accumulate(dec, axis=0)  # decided for boxes 0..k
        last = np.where(want[f] < 0, dec.shape[0] - 1, want[f])
        ok[f] = prefix_ok[last, np.arange(pts.shape[1])]
    return ok


def _frames(b, n, t, seed, heading_zero=False, valid=None):
    r = np.random.default_rng(seed)
    pts = synth.cloud_ground_objects(b, n, seed=seed)
    boxes = np.zeros((b, t, 7), np.float32)  # padding boxes: all zeros
    for f in range(b):
        nv = t if valid is None else valid[f]
        if nv:
            boxes[f, :nv] = boxes_on_points(pts[f], nv, seed + 100 + f)
        pts[f, r.integers(0, n, 8)] = 0.0  # points on the padding boxes' origin
    if heading_zero:
        boxes[..., 6] = 0.0
    return boxes, pts


@pytest.mark.parametrize("case", ["b16_t64_padded", "b16_t64_heading0", "b1_180k_t512", "b1_40k_t1500", "ragged"])
def test_points_in_boxes_gpu_matches_oracle(case):
    if case == "b16_t64_padded":
        boxes, pts = _frames(16, 16384, 64, 1, valid=np.random.default_rng(0).integers(0, 65, 16))
    elif case == "b16_t64_heading0":
        boxes, pts = _frames(16, 16384, 64, 2, heading_zero=True, valid=[64, 40, 0, 7] * 4)
    elif case == "b1_180k_t512":
        boxes, pts = _frames(1, 180000, 512, 3)
    elif case == "b1_40k_t1500":  # more boxes than one staging pass (1024) holds
        boxes, pts = _frames(1, 40000, 1500, 6)
    else:
        boxes, pts = _frames(3, 1000, 5, 4, valid=[5, 1, 3])
    got = _gpu_labels(boxes, pts)
    want = rao.points_in_boxes(boxes, pts)
    assert (want >= 0).sum() > 100 * boxes.shape[0] or case == "ragged"
    if case.endswith("heading0"):
        assert np.array_equal(got, want)
        return
    if case == "b1_40k_t1500":
        assert (want >= 1024).sum() > 100  # labels found in the second pass
    ok = _comparable(boxes, pts, want)
    undecided = 1.0 - ok.mean()
    print(f"[points_in_boxes_gpu {case}] undecided points {undecided:.2e}")
    assert undecided < 1e-4
    assert np.array_equal(got[ok], want[ok])


def _edge_case():
    """a heading-0 box (cosf = 1, sinf = -0 exactly on every implementation) and the floats next to its faces: |x| and
    |y| the largest float below / the smallest at or above dx / 2.0 + 1e-5 (double), z on the faces / the next float
    beyond them"""
    t = 0.5 + np.float64(np.float32(1e-5))
    f = np.float32(t)
    below, up = (np.nextafter(f, np.float32(-1)), f) if np.float64(f) >= t else (f, np.nextafter(f, np.float32(1)))
    over = np.float32(1 + 2.0 ** -23)
    pts = np.array([[below, 0, 0], [up, 0, 0], [-below, 0, 0], [-up, 0, 0],
                    [0, below, 0], [0, up, 0], [0, -below, 0], [0, -up, 0],
                    [0, 0, 1], [0, 0, -1], [0, 0, over], [0, 0, -over]], np.float32)
    box = np.array([[0, 0, 0, 1, 1, 2, 0]], np.float32)
    return box, pts, [0, -1, 0, -1, 0, -1, 0, -1, 0, 0, -1, -1]


def test_threshold_edges_on_the_device():
    """the float thresholds the kernels use (rounded up for x / y, down for z) decide these floats exactly as the double
    compares do"""
    box, pts, labels = _edge_case()
    assert _gpu_labels(box[None], pts[None])[0].tolist() == labels
    assert rao.points_in_boxes(box[None], pts[None])[0].tolist() == labels
    feats = np.arange(len(pts) * 2, dtype=np.float32).reshape(-1, 2)
    for method in (0, 1):
        got = _shim_forward(box, pts, feats, (2, 2, 2), 16, method)
        want = rao.forward(box, pts, feats, (2, 2, 2), 16, method)
        assert want[0][..., 0].sum() == labels.count(0)
        _assert_forward_equal(got, want, method)


def test_points_in_boxes_gpu_empty_shapes_keep_the_prefill():
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_cuda as ext

    pts = torch.zeros((2, 5, 3), device=DEV)
    out = torch.full((2, 5), -7, dtype=torch.int32, device=DEV)
    assert ext.points_in_boxes_gpu(torch.zeros((2, 0, 7), device=DEV), pts, out) == 1
    assert (out == -7).all()
    out0 = torch.zeros((2, 0), dtype=torch.int32, device=DEV)
    ext.points_in_boxes_gpu(torch.zeros((2, 3, 7), device=DEV), torch.zeros((2, 0, 3), device=DEV), out0)
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ forward
def _pool_inputs(out_size, c, seed, n=16384, r=32, clump=0, overlap=False, far=0, ties=False, specials=False):
    """RoIs on the cloud (plus `far` empty ones), points the classifier decides for every RoI, features"""
    rng = np.random.default_rng(seed)
    pts = synth.cloud_ground_objects(1, n, seed=seed)[0]
    rois = boxes_on_points(pts, r, seed + 1)
    if overlap:
        rois[r // 2:] = rois[:r - r // 2] + np.array([0.2, -0.1, 0.05, 0, 0, 0, 0.3], np.float32)
    if clump:  # a dense clump at RoI 0's centre: > 127 points in one voxel
        pts = np.concatenate([pts, rois[0, :3] + rng.uniform(-0.05, 0.05, (clump, 3)).astype(np.float32)])
        pts = pts[rng.permutation(len(pts))]
    if far:
        rois = np.concatenate([rois, synth.boxes_random(far, seed + 2) + np.array([500, 0, 0, 0, 0, 0, 0], np.float32)])
    keep = rao.classify_voxels(rois, pts, out_size).all(axis=0)
    pts = np.ascontiguousarray(pts[keep])
    if ties:
        feats = rng.integers(-2, 3, (len(pts), c)).astype(np.float32)
    else:
        feats = rng.standard_normal((len(pts), c)).astype(np.float32)
    if specials and len(pts) > 10:
        feats[rng.integers(0, len(pts), len(pts) // 10), rng.integers(0, c, len(pts) // 10)] = -np.inf
        feats[rng.integers(0, len(pts), len(pts) // 10), rng.integers(0, c, len(pts) // 10)] = np.nan
    return rois, pts, feats, 1.0 - keep.mean()


def _shim_forward(rois, pts, feats, out_size, L, method):
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_cuda as ext

    X, Y, Z = (out_size,) * 3 if isinstance(out_size, int) else out_size
    r, c = rois.shape[0], feats.shape[1]
    am = torch.zeros((r, X, Y, Z, c), dtype=torch.int32, device=DEV)
    idx = torch.zeros((r, X, Y, Z, L), dtype=torch.int32, device=DEV)
    pooled = torch.zeros((r, X, Y, Z, c), device=DEV)
    t = [torch.from_numpy(a).to(DEV) for a in (rois, pts, feats)]
    assert ext.forward(*t, am, idx, pooled, method) == 1
    return idx.cpu().numpy(), am.cpu().numpy(), pooled.cpu().numpy()


def _assert_forward_equal(got, want, method):
    gi, ga, gp = got
    wi, wa, wp = want
    assert np.array_equal(gi, wi), "pts_idx_of_voxels"
    assert np.array_equal(ga, wa), "argmax"
    # bit for bit; a NaN can reach pooled only through avg (either NaN then)
    same = gp.view(np.int32) == wp.view(np.int32)
    if method == 1:
        same |= np.isnan(gp) & np.isnan(wp)
    assert same.all(), f"pooled: {(~same).sum()} elements differ"


FWD_CASES = [  # (method, C, out_size, L, extra)
    (0, 4, 14, 128, {}), (1, 4, 14, 128, {}),
    (0, 128, 12, 128, {}), (1, 128, 12, 128, {}),
    (0, 33, (7, 5, 3), 4, {"ties": True, "specials": True}), (1, 33, (7, 5, 3), 4, {}),
    (0, 1, 1, 128, {"clump": 400}), (1, 1, 1, 128, {"clump": 400}),
    (0, 4, 14, 1, {}), (1, 4, 12, 4, {"overlap": True, "far": 4}),
    (0, 4, (32, 32, 32), 4, {"far": 2}),  # 32768 voxels: counters in global memory
    (1, 5, (40, 20, 24), 8, {"clump": 300}),
]


@pytest.mark.parametrize("method,c,out_size,L,extra", FWD_CASES)
def test_forward_bit_exact_against_oracle(method, c, out_size, L, extra):
    rois, pts, feats, dropped = _pool_inputs(out_size, c, seed=11 + c, **extra)
    assert dropped < 1e-3
    got = _shim_forward(rois, pts, feats, out_size, L, method)
    want = rao.forward(rois, pts, feats, out_size, L, method)
    assert want[0][..., 0].sum() > 100 or L == 1  # the RoIs hold points (L = 1 lists none)
    if extra.get("clump") and L == 128:
        assert want[0][..., 0].max() == 127  # the cap
    _assert_forward_equal(got, want, method)


def test_forward_counters_do_not_depend_on_the_zero_fill():
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_cuda as ext

    rois, pts, feats, _ = _pool_inputs(6, 4, seed=5)
    want = rao.forward(rois, pts, feats, 6, 16, 0)
    r = rois.shape[0]
    idx = torch.full((r, 6, 6, 6, 16), 12345, dtype=torch.int32, device=DEV)
    am = torch.zeros((r, 6, 6, 6, 4), dtype=torch.int32, device=DEV)
    pooled = torch.zeros((r, 6, 6, 6, 4), device=DEV)
    ext.forward(*[torch.from_numpy(a).to(DEV) for a in (rois, pts, feats)], am, idx, pooled, 0)
    gi = idx.cpu().numpy()
    assert np.array_equal(gi[..., 0], want[0][..., 0])
    n = want[0][..., 0]
    for k in range(1, 16):
        m = n >= k
        assert np.array_equal(gi[..., k][m], want[0][..., k][m])
    assert np.array_equal(am.cpu().numpy(), want[1])


def test_forward_empty_shapes():
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_cuda as ext

    z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device=DEV)  # noqa: E731
    ext.forward(z(0, 7), z(5, 3), z(5, 4), z(0, 2, 2, 2, 4, dt=torch.int32), z(0, 2, 2, 2, 8, dt=torch.int32),
                z(0, 2, 2, 2, 4), 0)
    am, idx, pooled = z(3, 2, 2, 2, 4, dt=torch.int32), z(3, 2, 2, 2, 8, dt=torch.int32) + 9, z(3, 2, 2, 2, 4)
    rois = torch.from_numpy(boxes_on_points(np.zeros((1, 3), np.float32), 3, 0)).to(DEV)
    ext.forward(rois, z(0, 3), z(0, 4), am, idx, pooled, 0)  # P = 0
    torch.cuda.synchronize()
    assert (idx[..., 0] == 0).all() and (am == -1).all() and (pooled == 0).all()


# ------------------------------------------------------------------------------------------------ backward
def _scatter64(idx, am, grad_out, p, method):
    """float64 scatter of the device's float terms, and the bound (k - 1) u sum|terms| per element"""
    c = grad_out.shape[-1]
    g = grad_out.reshape(-1, c)
    ref = np.zeros((p, c), np.float64)
    absum = np.zeros((p, c), np.float64)
    cnt = np.zeros((p, c), np.int64)
    if method == 0:
        a = am.reshape(-1, c)
        e, ch = np.nonzero(a >= 0)
        terms = g[e, ch].astype(np.float64)
        np.add.at(ref, (a[e, ch], ch), terms)
        np.add.at(absum, (a[e, ch], ch), np.abs(terms))
        np.add.at(cnt, (a[e, ch], ch), 1)
    else:
        lists = idx.reshape(-1, idx.shape[-1])
        for v in np.nonzero(lists[:, 0] > 0)[0]:
            n = lists[v, 0]
            w = np.float32(1) / np.float32(max(n, 1))
            terms = (g[v] * w).astype(np.float32).astype(np.float64)  # the device's float product
            for pt in lists[v, 1:1 + n]:
                ref[pt] += terms
                absum[pt] += np.abs(terms)
                cnt[pt] += 1
    bound = np.maximum(cnt - 1, 0) * 2.0 ** -24 * absum
    return ref, bound


@pytest.mark.parametrize("method", [0, 1])
@pytest.mark.parametrize("c,out_size,L", [(4, 14, 128), (33, (7, 5, 3), 4), (1, 1, 128)])
def test_backward_matches_float64_scatter(method, c, out_size, L):
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_cuda as ext

    rois, pts, feats, _ = _pool_inputs(out_size, c, seed=21, overlap=True, clump=200, ties=method == 0)
    idx, am, _ = rao.forward(rois, pts, feats, out_size, L, method)
    if method == 1:
        am = np.zeros_like(am)  # avg leaves argmax at the caller's zeros
    gout = np.random.default_rng(3).standard_normal(am.shape).astype(np.float32)
    gin = torch.zeros((len(pts), c), device=DEV)
    ext.backward(torch.from_numpy(idx).to(DEV), torch.from_numpy(am).to(DEV), torch.from_numpy(gout).to(DEV), gin,
                 method)
    ref, bound = _scatter64(idx, am, gout, len(pts), method)
    err = np.abs(gin.cpu().numpy().astype(np.float64) - ref)
    assert (err <= bound).all(), float((err - bound).max())
    assert np.count_nonzero(ref) >= 10


@pytest.mark.parametrize("pool_method", ["max", "avg"])
def test_module_autograd_and_out_size_forms(pool_method):
    from tsmdet_b200.roiaware_pool3d.roiaware_pool3d_utils import RoIAwarePool3d

    rois, pts, feats, _ = _pool_inputs((6, 5, 4), 16, seed=31, overlap=True)
    method = 0 if pool_method == "max" else 1
    want = rao.forward(rois, pts, feats, (6, 5, 4), 32, method)
    tr, tp = torch.from_numpy(rois).to(DEV), torch.from_numpy(pts).to(DEV)
    tf = torch.from_numpy(feats).to(DEV).requires_grad_(True)
    out = RoIAwarePool3d((6, 5, 4), max_pts_each_voxel=32)(tr, tp, tf, pool_method=pool_method)
    assert out.shape == want[2].shape and np.array_equal(out.detach().cpu().numpy().view(np.int32), want[2].view(np.int32))
    w = torch.from_numpy(np.random.default_rng(4).standard_normal(out.shape).astype(np.float32)).to(DEV)
    (out * w).sum().backward()
    am = want[1] if method == 0 else np.zeros_like(want[1])
    ref, bound = _scatter64(want[0], am, w.cpu().numpy(), len(pts), method)
    assert (np.abs(tf.grad.cpu().numpy().astype(np.float64) - ref) <= bound).all()
    # an int out size is the cube
    cube = RoIAwarePool3d(5, 32)(tr, tp, tf.detach(), pool_method)
    assert np.array_equal(cube.cpu().numpy().view(np.int32), rao.forward(rois, pts, feats, 5, 32, method)[2].view(np.int32))


def test_forward_captures_in_a_cuda_graph():
    from tsmdet_b200.roiaware_pool3d.roiaware_pool3d_utils import RoIAwarePool3d

    rois, pts, feats, _ = _pool_inputs(12, 8, seed=41)
    mod = RoIAwarePool3d(12, 64)
    tr, tp, tf = (torch.from_numpy(a).to(DEV) for a in (rois, pts, feats))
    eager = mod(tr, tp, tf, "avg")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        mod(tr, tp, tf, "avg")  # warm-up on the side stream
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        static = mod(tr, tp, tf, "avg")
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(static.view(torch.int32), eager.view(torch.int32))
    tf.mul_(2.0)  # replays see the new features
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(static, mod(tr, tp, tf, "avg"))


def _reference_extension():
    """The reference's unmodified roiaware_pool3d_cuda: oracle/_ref's build if present, else compiled from the reference
    tree (oracle/build_ref.REF_ROOT) into the temporary directory with build_ref's flags; None without the tree."""
    import tempfile

    from oracle import build_ref

    ref = build_ref.load_ref("roiaware_pool3d_cuda")
    src = os.path.join(build_ref.REF_ROOT, "pcdet/ops/roiaware_pool3d/src")
    if ref is not None or not os.path.isdir(src):
        return ref
    from torch.utils.cpp_extension import load

    bdir = os.path.join(tempfile.gettempdir(), f"tsmdet_ref_roiaware_pool3d_{os.getuid()}")
    os.makedirs(bdir, exist_ok=True)
    srcs = sorted(os.path.join(src, f) for f in os.listdir(src) if f.endswith((".cpp", ".cu")))
    return load(name="roiaware_pool3d_cuda", sources=srcs, extra_include_paths=[src], build_directory=bdir,
                extra_cflags=["-fno-strict-overflow", "-DNDEBUG", "-O2"],
                extra_cuda_cflags=["-gencode=arch=compute_100a,code=sm_100a"])


def _reference_utils():
    """The reference's unmodified roiaware_pool3d_utils.py, read from its tree, over THIS package's shim (the module swap
    of INTEGRATION.md); None without the tree."""
    from oracle import build_ref
    from ref_py import _alias
    from ref_stack_py import _load_source
    from tsmdet_b200 import common_utils
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_cuda

    path = os.path.join(build_ref.REF_ROOT, "pcdet/ops/roiaware_pool3d/roiaware_pool3d_utils.py")
    if not os.path.exists(path):
        return None
    _alias("pcdet.ops.roiaware_pool3d.roiaware_pool3d_cuda", roiaware_pool3d_cuda)
    _alias("pcdet.utils.common_utils", common_utils)
    return _load_source("pcdet.ops.roiaware_pool3d.roiaware_pool3d_utils", path)


def test_head_to_head_against_the_reference_extension():
    """The reference's own kernels on rotated boxes and unfiltered points: labels, lists, argmax and pooled equal bit
    for bit (this is what pins the recalled contract, the contraction of local_x / local_y included)."""
    ref = _reference_extension()
    if ref is None:
        pytest.skip("no reference tree: the reference's roiaware_pool3d_cuda cannot be built")
    boxes, pts = _frames(4, 16384, 64, 61, valid=[64, 30, 0, 64])
    tb, tp = torch.from_numpy(boxes).to(DEV), torch.from_numpy(pts).to(DEV)
    want = torch.full(pts.shape[:2], -1, dtype=torch.int32, device=DEV)
    ref.points_in_boxes_gpu(tb, tp, want)
    assert np.array_equal(_gpu_labels(boxes, pts), want.cpu().numpy())
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_cuda as ext

    cw, cg = (torch.zeros((64, 16384), dtype=torch.int32) for _ in range(2))
    ref.points_in_boxes_cpu(torch.from_numpy(boxes[0]), torch.from_numpy(pts[0]), cw)
    ext.points_in_boxes_cpu(torch.from_numpy(boxes[0]), torch.from_numpy(pts[0]), cg)
    assert torch.equal(cw, cg)
    rng = np.random.default_rng(5)
    pts1 = synth.cloud_ground_objects(1, 16384, seed=62)[0]
    rois = boxes_on_points(pts1, 64, 63)
    for out_size, c, L in ((14, 16, 128), ((7, 5, 3), 33, 4)):
        feats = rng.integers(-3, 4, (len(pts1), c)).astype(np.float32)  # ties
        X, Y, Z = (out_size,) * 3 if isinstance(out_size, int) else out_size
        for method in (0, 1):
            am = torch.zeros((len(rois), X, Y, Z, c), dtype=torch.int32, device=DEV)
            idx = torch.zeros((len(rois), X, Y, Z, L), dtype=torch.int32, device=DEV)
            pooled = torch.zeros((len(rois), X, Y, Z, c), device=DEV)
            ref.forward(*[torch.from_numpy(a).to(DEV) for a in (rois, pts1, feats)], am, idx, pooled, method)
            want = (idx.cpu().numpy(), am.cpu().numpy(), pooled.cpu().numpy())
            assert want[0][..., 0].sum() > 100
            _assert_forward_equal(_shim_forward(rois, pts1, feats, out_size, L, method), want, method)


def test_reference_python_over_the_shim():
    """The reference's unmodified roiaware_pool3d_utils.py over this package's shim equals this package's own file."""
    ru_ref = _reference_utils()
    if ru_ref is None:
        pytest.skip("no reference tree: its roiaware_pool3d_utils.py cannot be loaded")
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_utils as ru

    boxes, pts = _frames(2, 8192, 32, 71)
    tb, tp = torch.from_numpy(boxes).to(DEV), torch.from_numpy(pts).to(DEV)
    assert torch.equal(ru_ref.points_in_boxes_gpu(tp, tb), ru.points_in_boxes_gpu(tp, tb))
    assert np.array_equal(ru_ref.points_in_boxes_cpu(pts[0], boxes[0]), ru.points_in_boxes_cpu(pts[0], boxes[0]))
    rois, pts1, feats, _ = _pool_inputs(6, 8, seed=72)
    tr, tq = torch.from_numpy(rois).to(DEV), torch.from_numpy(pts1).to(DEV)
    for pool_method in ("max", "avg"):
        outs = []
        for mod in (ru_ref.RoIAwarePool3d(6, 32), ru.RoIAwarePool3d(6, 32)):
            tf = torch.from_numpy(feats).to(DEV).requires_grad_(True)
            y = mod(tr, tq, tf, pool_method=pool_method)
            y.sum().backward()
            outs.append((y.detach(), tf.grad))
        assert torch.equal(outs[0][0], outs[1][0])
        assert torch.allclose(outs[0][1], outs[1][1], rtol=1e-6, atol=1e-6)
