"""GPU parity: ball query (+dilated), grouping, gather, QueryAndGroup, three_nn / three_interpolate
and their backward kernels, through the C ABI, vs the CPU oracle (bit-exact), the golden fixtures (reference CUDA
output) and oracle/_ref."""
import os

import numpy as np
import pytest
from conftest import knob_delenv, knob_setenv
import torch

import synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def D():
    return torch.device("cuda:0")


def T(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(D())


BQ = [
    # b, n, m, radius_in, radius, nsample, generator
    (2, 4096, 512, None, 0.8, 32, synth.cloud_ground_objects),
    (2, 4096, 512, None, 0.2, 16, synth.cloud_ground_objects),
    (2, 4096, 512, 0.4, 0.8, 32, synth.cloud_ground_objects),
    (1, 1000, 333, None, 3.0, 8, synth.cloud_uniform),       # dense: early exit, n not a multiple of 4
    (3, 1027, 70, 0.0, 1.5, 64, synth.cloud_dup_padded),      # ragged sizes, duplicates
    (2, 37, 5, None, 100.0, 7, synth.cloud_uniform),          # everything hits; nsample not a power of two
    (2, 2048, 130, None, 1e-3, 16, synth.cloud_uniform),      # nothing but the centre itself
    (1, 16384, 4096, None, 0.8, 32, synth.cloud_ground_objects),  # BASELINE config 1 shape
    (2, 4096, 333, None, 0.8, 24, synth.cloud_ground_objects),    # half-warp kernel: two results per lane, odd centre count
    (2, 4096, 511, 0.2, 0.6, 17, synth.cloud_uniform),            # ... nsample just above 16, dilated
    (1, 2048, 100, None, 3.0, 32, synth.cloud_uniform),           # ... every super-round full of hits
    (2, 300, 300, 0.1, 0.9, 40, synth.cloud_uniform),             # under 512 points: brute force only; dilated, nsample > 32
    (1, 511, 511, None, 0.5, 33, synth.cloud_uniform),            # ... one point short of the grid
    (4, 8192, 8192, None, 0.4, 16, synth.cloud_ground_objects),   # many centres per cloud (b * m = 32768)
    (3, 4099, 2000, 0.3, 0.7, 64, synth.cloud_dup_padded),        # annulus through the merge kernel
    (2, 1024, 1024, None, 2.0, 128, synth.cloud_uniform),         # rows four warps wide
    (1, 4096, 2049, None, 0.8, 1, synth.cloud_ground_objects),    # nsample 1; one centre past a multiple of 128
]


@pytest.mark.parametrize("algo", ["grid", "brute"])
@pytest.mark.parametrize("case", BQ, ids=[f"bq{i}" for i in range(len(BQ))])
def test_ball_query(orc, case, algo, monkeypatch):
    """Both query paths: the uniform-grid kernels (ball_query_grid.cu; clouds of >= 512 points whose grid is
    usable) and the brute-force kernel (ball_query.cu), against the oracle."""
    from tsmdet_b200 import pointnet2_utils as pu

    knob_setenv(monkeypatch, "TSMDET_BQ_ALGO", algo)

    b, n, m, rin, r, ns, gen = case
    xyz = gen(b, n, 7)
    sel = np.random.default_rng(1).permutation(n)[:m]
    new_xyz = np.ascontiguousarray(xyz[:, sel, :])
    if m > 3:
        new_xyz[:, 3] += 500.0  # a centre with an empty ball
    if rin is None:
        cnt, idx = pu.ball_query(r, ns, T(xyz), T(new_xyz))
        wc, wi = orc.ball_query(r, ns, xyz, new_xyz)
    else:
        cnt, idx = pu.ball_query_dilated(rin, r, ns, T(xyz), T(new_xyz))
        wc, wi = orc.ball_query_dilated(rin, r, ns, xyz, new_xyz)
    assert np.array_equal(cnt.cpu().numpy(), wc)
    assert np.array_equal(idx.cpu().numpy(), wi)
    assert idx.dtype == torch.int32 and cnt.dtype == torch.int32


def test_ball_query_grid_edge_cases(orc):
    """Grid construction corner cases (flat / collinear / single-point clouds, centres far outside the cloud or
    between samples, radius larger than the cloud, nsample above 32 -> merge kernel) all match the oracle."""
    from tsmdet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(5)
    flat = synth.cloud_uniform(2, 4000, 61)
    flat[:, :, 2] = 1.5
    line = synth.cloud_uniform(2, 3000, 62)
    line[:, :, 1:] = 0.25
    same = np.ones((2, 2000, 3), np.float32)
    dense = (rng.standard_normal((2, 6000, 3)) * 0.05).astype(np.float32)  # everything in a few cells -> brute force
    obj = synth.cloud_ground_objects(2, 8192, 63)
    for name, xyz, r, ns in [("flat", flat, 0.8, 16), ("line", line, 0.5, 16), ("same", same, 0.3, 8), ("dense", dense, 0.4, 32),
                             ("obj64", obj, 1.0, 64), ("obj48", obj, 0.6, 48), ("huge_r", obj, 500.0, 16), ("tiny_r", obj, 1e-4, 16)]:
        new_xyz = np.ascontiguousarray(xyz[:, ::9, :]).copy()
        new_xyz[:, 1] += 1000.0
        new_xyz[:, 2] += np.float32(0.37 * r)
        new_xyz[:, 3, 2] -= np.float32(2.5 * r)
        cnt, idx = pu.ball_query(r, ns, T(xyz), T(new_xyz))
        wc, wi = orc.ball_query(r, ns, xyz, new_xyz)
        assert np.array_equal(cnt.cpu().numpy(), wc), name
        assert np.array_equal(idx.cpu().numpy(), wi), name
        cnt, idx = pu.ball_query_dilated(0.5 * r, r, ns, T(xyz), T(new_xyz))
        wc, wi = orc.ball_query_dilated(0.5 * r, r, ns, xyz, new_xyz)
        assert np.array_equal(cnt.cpu().numpy(), wc), name
        assert np.array_equal(idx.cpu().numpy(), wi), name


def test_ball_query_waymo_scale(orc):
    """BASELINE config 4 shape (65536 points, 16384 centres, r 0.8, ns 32): grid path vs the oracle on one
    cloud, vs the brute-force kernel on all."""
    import os

    from tsmdet_b200 import pointnet2_utils as pu

    xyz = synth.cloud_uniform(2, 65536, 70, synth.WAYMO_RANGE)
    new_xyz = np.ascontiguousarray(xyz[:, ::4, :])
    cnt, idx = pu.ball_query(0.8, 32, T(xyz), T(new_xyz))
    wc, wi = orc.ball_query(0.8, 32, xyz[:1], new_xyz[:1])
    assert np.array_equal(cnt[:1].cpu().numpy(), wc) and np.array_equal(idx[:1].cpu().numpy(), wi)
    from tsmdet_b200 import _lib

    os.environ["TSMDET_BQ_ALGO"] = "brute"
    _lib.reload_options()
    try:
        c2, i2 = pu.ball_query(0.8, 32, T(xyz), T(new_xyz))
    finally:
        os.environ.pop("TSMDET_BQ_ALGO")
        _lib.reload_options()
    assert torch.equal(cnt, c2) and torch.equal(idx, i2)


def test_ball_query_vs_reference_cuda(ref_pointnet2):
    if ref_pointnet2 is None:
        pytest.skip("oracle/_ref not built")
    from tsmdet_b200 import pointnet2_utils as pu

    xyz = synth.cloud_ground_objects(4, 16384, 3)
    new_xyz = np.ascontiguousarray(xyz[:, ::4, :])
    x, q = T(xyz), T(new_xyz)
    for rin, r, ns in [(None, 0.2, 16), (None, 0.8, 32), (0.2, 0.4, 32), (0.4, 0.8, 32)]:
        idx = torch.zeros((4, 4096, ns), dtype=torch.int32, device=D())
        cnt = torch.zeros((4, 4096), dtype=torch.int32, device=D())
        if rin is None:
            ref_pointnet2.ball_query_wrapper(4, 16384, 4096, r, ns, q, x, cnt, idx)
            c2, i2 = pu.ball_query(r, ns, x, q)
        else:
            ref_pointnet2.ball_query_dilated_wrapper(4, 16384, 4096, rin, r, ns, q, x, cnt, idx)
            c2, i2 = pu.ball_query_dilated(rin, r, ns, x, q)
        torch.cuda.synchronize()
        assert torch.equal(c2, cnt) and torch.equal(i2, idx)


def test_ball_query_golden():
    """Ball query (+dilated) through the pybind-name shims vs the reference kernels' stored outputs on the cases of
    tests/golden/ball_query.npz (2 x 4096 points, 512 centres), bit-exact; runs without the reference extension."""
    from tsmdet_b200 import pointnet2_batch_cuda as ext

    g = np.load(os.path.join(GOLD, "ball_query.npz"))
    (b, n, _), m = g["xyz"].shape, g["new_xyz"].shape[1]
    x, q = T(g["xyz"]), T(g["new_xyz"])
    for tag, rin, r, ns in [("r08", None, 0.8, 32), ("r02", None, 0.2, 16), ("d0408", 0.4, 0.8, 32), ("r30", None, 3.0, 8)]:
        idx = torch.zeros((b, m, ns), dtype=torch.int32, device=D())
        cnt = torch.zeros((b, m), dtype=torch.int32, device=D())
        if rin is None:
            ext.ball_query_wrapper(b, n, m, r, ns, q, x, cnt, idx)
        else:
            ext.ball_query_dilated_wrapper(b, n, m, rin, r, ns, q, x, cnt, idx)
        assert np.array_equal(cnt.cpu().numpy(), g[f"{tag}_cnt"]), tag
        assert np.array_equal(idx.cpu().numpy(), g[f"{tag}_idx"]), tag


@pytest.mark.parametrize("b,c,n,m,s", [(2, 5, 1000, 64, 16), (1, 131, 1024, 512, 32), (3, 1, 333, 7, 3), (2, 35, 4096, 100, 32)])
def test_group_and_gather(orc, b, c, n, m, s):
    from tsmdet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(b * 100 + c)
    feats = rng.normal(size=(b, c, n)).astype(np.float32)
    idx = rng.integers(0, n, size=(b, m, s)).astype(np.int32)
    got = pu.grouping_operation(T(feats), T(idx))
    assert np.array_equal(got.cpu().numpy().view(np.uint32), orc.group_points(feats, idx).view(np.uint32))
    gidx = rng.integers(0, n, size=(b, m)).astype(np.int32)
    got = pu.gather_operation(T(feats), T(gidx))
    assert np.array_equal(got.cpu().numpy().view(np.uint32), orc.gather_points(feats, gidx).view(np.uint32))


def test_group_gather_backward(orc):
    from tsmdet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(5)
    b, c, n, m, s = 2, 6, 500, 40, 8
    feats = torch.from_numpy(rng.normal(size=(b, c, n)).astype(np.float32)).to(D()).requires_grad_(True)
    idx = rng.integers(0, n, size=(b, m, s)).astype(np.int32)
    g = rng.normal(size=(b, c, m, s)).astype(np.float32)
    out = pu.grouping_operation(feats, T(idx))
    out.backward(T(g))
    # atomic float adds: order-dependent rounding, so tolerance not bits
    np.testing.assert_allclose(feats.grad.cpu().numpy(), orc.group_points_grad(g, idx, n), rtol=1e-5, atol=1e-5)
    feats.grad = None
    gidx = rng.integers(0, n, size=(b, m)).astype(np.int32)
    g2 = rng.normal(size=(b, c, m)).astype(np.float32)
    pu.gather_operation(feats, T(gidx)).backward(T(g2))
    np.testing.assert_allclose(feats.grad.cpu().numpy(), orc.gather_points_grad(g2, gidx, n), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("dilated", [False, True])
@pytest.mark.parametrize("with_feats,use_xyz", [(True, True), (True, False), (False, True)])
def test_query_and_group_tuple(orc, dilated, with_feats, use_xyz):
    """QueryAndGroup(.Dilated).forward returns the reference's 3-tuple (SURVEY.md section 0, bug 1)."""
    from tsmdet_b200 import pointnet2_utils as pu

    xyz = synth.cloud_ground_objects(2, 2048, 11)
    new_xyz = np.ascontiguousarray(xyz[:, ::16, :])
    feats = np.random.default_rng(2).normal(size=(2, 5, 2048)).astype(np.float32) if with_feats else None
    mod = pu.QueryAndGroupDilated(0.3, 0.9, 16, use_xyz=use_xyz) if dilated else pu.QueryAndGroup(0.9, 16, use_xyz=use_xyz)
    out = mod(T(xyz), T(new_xyz), T(feats) if with_feats else None)
    assert isinstance(out, tuple) and len(out) == 3
    cnt, nf, gx = out
    wc, wnf, wgx, _ = orc.query_and_group(xyz, new_xyz, feats, 0.9, 16, radius_in=0.3 if dilated else None, use_xyz=use_xyz)
    assert np.array_equal(cnt.cpu().numpy(), wc)
    assert np.array_equal(gx.cpu().numpy().view(np.uint32), wgx.view(np.uint32))
    assert np.array_equal(nf.cpu().numpy().view(np.uint32), wnf.view(np.uint32))


@pytest.mark.parametrize("b,n,m", [(2, 1024, 256), (1, 777, 100), (2, 50, 2), (1, 5000, 3000)])
def test_three_nn(orc, b, n, m):
    from tsmdet_b200 import pointnet2_utils as pu

    unknown = synth.cloud_ground_objects(b, n, 21)
    known = np.ascontiguousarray(synth.cloud_ground_objects(b, max(m, 8), 22)[:, :m, :])
    if m > 6:
        known[:, 5] = known[:, 4]
    dist, idx = pu.three_nn(T(unknown), T(known))
    wd2, wi = orc.three_nn(unknown, known)
    assert np.array_equal(idx.cpu().numpy(), wi)
    assert np.array_equal(dist.cpu().numpy().view(np.uint32), np.sqrt(wd2).view(np.uint32))


def test_three_nn_grid_equals_brute_force(orc, monkeypatch):
    """The grid search (three_nn_grid.cu) returns exactly what the brute-force kernel returns -- (d2, k) ties
    included -- on lattices (many equal distances), duplicated known points, unknown points outside the known
    cloud, flat and collinear clouds, and at the Waymo FP-layer size (65536 unknown, 16384 known)."""
    from tsmdet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(9)
    cases = []
    lat = synth.cloud_lattice(2, 4000, 41)
    cases.append(("lattice", synth.cloud_lattice(2, 6000, 40), lat))
    dup = synth.cloud_dup_padded(2, 4096, 42, unique_frac=0.5)
    cases.append(("dup", synth.cloud_uniform(2, 5000, 43), dup))
    out = synth.cloud_uniform(2, 3000, 44) * 3.0 - 40.0
    cases.append(("outside", out.astype(np.float32), synth.cloud_ground_objects(2, 2048, 45)))
    flat = synth.cloud_uniform(2, 3000, 46)
    flat[:, :, 2] = 0.5
    cases.append(("flat", synth.cloud_uniform(2, 2000, 47), flat))
    line = synth.cloud_uniform(2, 1500, 48)
    line[:, :, 1:] = 1.0
    cases.append(("line", synth.cloud_uniform(2, 2000, 49), line))
    same = np.ones((1, 600, 3), np.float32)
    cases.append(("same", synth.cloud_uniform(1, 500, 50), same))
    w_unknown = synth.cloud_uniform(2, 65536, 51, synth.WAYMO_RANGE)
    cases.append(("waymo", w_unknown, np.ascontiguousarray(w_unknown[:, ::4, :])))
    for name, unknown, known in cases:
        knob_setenv(monkeypatch, "TSMDET_NN_ALGO", "brute")
        d0, i0 = pu.three_nn(T(unknown), T(known))
        knob_delenv(monkeypatch, "TSMDET_NN_ALGO")
        d1, i1 = pu.three_nn(T(unknown), T(known))
        assert torch.equal(i0, i1), name
        assert torch.equal(d0.view(torch.int32), d1.view(torch.int32)), name
    # and against the oracle on the tie-heavy ones
    for name, unknown, known in cases[:2]:
        d1, i1 = pu.three_nn(T(unknown[:1]), T(known[:1]))
        wd2, wi = orc.three_nn(unknown[:1], known[:1])
        assert np.array_equal(i1.cpu().numpy(), wi), name


def test_three_interpolate_and_grad(orc):
    from tsmdet_b200 import pointnet2_utils as pu

    rng = np.random.default_rng(3)
    b, c, m, n = 2, 19, 300, 1111
    feats = rng.normal(size=(b, c, m)).astype(np.float32)
    idx = rng.integers(0, m, size=(b, n, 3)).astype(np.int32)
    w = rng.uniform(0, 1, size=(b, n, 3)).astype(np.float32)
    w /= w.sum(-1, keepdims=True)
    f = T(feats).requires_grad_(True)
    out = pu.three_interpolate(f, T(idx), T(w))
    assert np.array_equal(out.detach().cpu().numpy().view(np.uint32), orc.three_interpolate(feats, idx, w).view(np.uint32))
    g = rng.normal(size=(b, c, n)).astype(np.float32)
    out.backward(T(g))
    np.testing.assert_allclose(f.grad.cpu().numpy(), orc.three_interpolate_grad(g, idx, w, m), rtol=1e-5, atol=1e-5)


def test_interpolate_vs_reference_cuda(ref_pointnet2):
    if ref_pointnet2 is None:
        pytest.skip("oracle/_ref not built")
    from tsmdet_b200 import pointnet2_batch_cuda as ext

    unknown = T(synth.cloud_ground_objects(2, 8192, 31))
    known = T(synth.cloud_ground_objects(2, 2048, 32))
    outs = []
    for mod in (ref_pointnet2, ext):
        d2 = torch.zeros((2, 8192, 3), device=D())
        idx = torch.zeros((2, 8192, 3), dtype=torch.int32, device=D())
        mod.three_nn_wrapper(2, 8192, 2048, unknown, known, d2, idx)
        feats = torch.sin(torch.arange(2 * 32 * 2048, device=D(), dtype=torch.float32)).view(2, 32, 2048).contiguous()
        w = torch.softmax(-d2, dim=2).contiguous()
        o = torch.zeros((2, 32, 8192), device=D())
        mod.three_interpolate_wrapper(2, 32, 2048, 8192, feats, idx, w, o)
        torch.cuda.synchronize()
        outs.append((d2, idx, o))
    for a, bb in zip(outs[0], outs[1]):
        assert torch.equal(a, bb)


def test_interpolate_golden():
    """three_nn / three_interpolate vs the reference kernels' stored outputs on the case of tests/golden/interpolate.npz
    (2 x 1024 unknown, 256 known points), bit-exact; runs without the reference extension."""
    from tsmdet_b200 import pointnet2_batch_cuda as ext

    g = np.load(os.path.join(GOLD, "interpolate.npz"))
    (b, n, _), (_, c, m) = g["unknown"].shape, g["feats"].shape
    d2 = torch.zeros((b, n, 3), device=D())
    idx = torch.zeros((b, n, 3), dtype=torch.int32, device=D())
    ext.three_nn_wrapper(b, n, m, T(g["unknown"]), T(g["known"]), d2, idx)
    out = torch.zeros((b, c, n), device=D())
    ext.three_interpolate_wrapper(b, c, m, n, T(g["feats"]), T(g["idx"]), T(g["weight"]), out)
    assert np.array_equal(idx.cpu().numpy(), g["idx"])
    assert np.array_equal(d2.cpu().numpy().view(np.uint32), g["dist2"].view(np.uint32))
    assert np.array_equal(out.cpu().numpy().view(np.uint32), g["out"].view(np.uint32))
