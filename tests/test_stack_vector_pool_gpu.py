"""GPU suite of the vector-pool ops of pointnet2_stack (csrc/stack_vector_pool.cu) and VectorPoolAggregationModule(MSG):

  * the local neighbour lists, the list 3-NN and vector_pool_wrapper bit for bit against the CPU oracle
    (tests/vector_pool_oracle.c): lists, dist2 bits, idx, sums and counts per centre, the triples as a sorted multiset
    with the exact total; on ragged frames, empty frames, frames without centres, far-away centres, frames the grid
    cannot take (NaN / inf, a pile of > 256 points in one cell), a neighbourhood of > 1000 hits on the grid and a
    150k-point frame; ball and cube, nsample -1 / 1 / 32, G 1 / 8 / 27 / 64 / (2,3,4), C 1 / 2 / 30 / 33 / 128;
  * the per-frame grids against TSMDET_BQ_ALGO=brute on all of them, bit for bit;
  * the fused 3-NN (no list) against the two-step result, bit for bit;
  * the overflow contract: a tiny first buffer forces one retry and gives what a generous one gives;
  * the gradient against a float64 index_add;
  * the modules: eager against a plain restatement fed by the oracle, the eval planes bit-identical to the eager
    tensor for all three aggregation types, outputs within fp32 tolerance, reference-shaped state_dicts,
    build_local_aggregation_module, a CUDA-graph capture of the eval forward (it must not synchronise);
  * head to head against the reference's stack .so and its stack Python over this package's shim, when built."""
import numpy as np
import pytest
import torch
from conftest import knob_setenv

import stack_cases
import synth
import vector_pool_oracle as vpo

pytestmark = pytest.mark.gpu


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


# ---------------------------------------------------------------------------------------------- cases
def _edge():
    """frames: 0 points / 20 centres, 800 points / 0 centres, 900 points / 40 centres of which half far away, 1 point"""
    rng = np.random.default_rng(11)
    f2 = synth.cloud_ground_objects(1, 900, seed=11)[0]
    far = rng.uniform(50, 60, (20, 3)).astype(np.float32)
    fx = [np.zeros((0, 3), np.float32), rng.uniform(-3, 3, (800, 3)), f2, rng.uniform(-1, 1, (1, 3))]
    fn = [rng.uniform(-2, 2, (20, 3)), np.zeros((0, 3), np.float32),
          np.concatenate([stack_cases.centres_from(rng, f2, 20), far]), rng.uniform(-1, 1, (5, 3))]
    return stack_cases.stack(fx, fn)


def _unusable():
    """a frame with a NaN and an inf coordinate, a frame with 300 copies of one point (> 256 in a cell), a normal one"""
    rng = np.random.default_rng(12)
    a = rng.uniform(-2, 2, (600, 3)).astype(np.float32)
    a[7, 1] = np.nan
    a[100, 0] = np.inf
    pile = np.concatenate([np.full((300, 3), 0.25, np.float32), rng.uniform(-2, 2, (300, 3)).astype(np.float32)])
    c = synth.cloud_ground_objects(1, 1500, seed=12)[0]
    fn = [stack_cases.centres_from(rng, x[np.isfinite(x).all(1)], 40) for x in (a, pile, c)]
    return stack_cases.stack([a, pile, c], fn)


def _dense():
    """a 0.05 lattice (216 points per grid cell at D = 0.25): > 1000 hits per cube on the grid path"""
    g = (np.arange(40, dtype=np.float32) * np.float32(0.05) - np.float32(1)).astype(np.float32)
    pts = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    rng = np.random.default_rng(13)
    return stack_cases.stack([pts], [rng.uniform(-0.6, 0.6, (64, 3))])


def _big():
    pts = synth.cloud_ground_objects(1, 150000, seed=14)[0]
    rng = np.random.default_rng(14)
    return stack_cases.stack([pts], [stack_cases.centres_from(rng, pts, 512)])


CASES = {"ragged": stack_cases.ragged, "edge": _edge, "unusable": _unusable, "dense": _dense, "150k": _big}
_cache = {}


def case(name):
    if name not in _cache:
        _cache[name] = CASES[name]()
    return _cache[name]


# ---------------------------------------------------------------------------------------------- function 1 / 2
def _lists_gpu(c, d, nsample, ntype, avg=1000):
    from tsmdet_b200.pointnet2_stack import pointnet2_stack_cuda as ps

    xyz, cnt, new, mcnt = c
    m = new.shape[0]
    buf = torch.full((avg * m,), -5, dtype=torch.int32, device="cuda")
    start_len = torch.zeros((m, 2), dtype=torch.int32, device="cuda")
    cumsum = torch.zeros((1,), dtype=torch.int32, device="cuda")
    assert ps.query_stacked_local_neighbor_idxs_wrapper_stack(T(xyz), T(cnt), T(new), T(mcnt), buf, start_len, cumsum,
                                                              avg, d, nsample, ntype) == 1
    return buf, start_len, int(cumsum.item())


def _split(buf, start_len):
    b, sl = buf.cpu().numpy(), start_len.cpu().numpy()
    return [b[o:o + n] for o, n in sl]


def _centres(new, grids, d):
    from tsmdet_b200.pointnet2_stack.pointnet2_modules import VectorPoolAggregationModule as V

    return V.get_dense_voxels_by_center(T(new), d, grids).contiguous()


def _nn_gpu(c, buf, start_len, total, centres):
    from tsmdet_b200.pointnet2_stack import pointnet2_stack_cuda as ps

    xyz, cnt, new, mcnt = c
    m, G = centres.shape[0], centres.shape[1]
    idx = torch.full((m, G, 3), -9, dtype=torch.int32, device="cuda")
    d2 = torch.full((m, G, 3), -1.0, device="cuda")
    assert ps.query_three_nn_by_stacked_local_idxs_wrapper_stack(T(xyz), T(new), centres, idx, d2, buf[:total],
                                                                 start_len, m, G) == 1
    return idx, d2


def _fused_nn(c, centres, d, nsample, ntype):
    from tsmdet_b200._lib import call, ptr, stream_ptr

    xyz, cnt, new, mcnt = c
    m, G = centres.shape[0], centres.shape[1]
    idx = torch.full((m, G, 3), -9, dtype=torch.int32, device="cuda")
    d2 = torch.full((m, G, 3), -1.0, device="cuda")
    x, xc, n, nc = T(xyz), T(cnt), T(new), T(mcnt)
    call("tsmdet_stack_vector_three_nn", len(cnt), m, xyz.shape[0], G, ptr(x), ptr(xc), ptr(n), ptr(nc), ptr(centres),
         float(d), nsample, ntype, ptr(idx), ptr(d2), stream_ptr())
    return idx, d2


NN_CFGS = [(1, -1, (3, 3, 3)), (0, 32, (2, 2, 2)), (0, 1, (1, 1, 1)), (1, 32, (4, 4, 4)), (0, -1, (2, 3, 4))]
D_OF = {"ragged": 0.8, "edge": 0.9, "unusable": 0.7, "dense": 0.25, "150k": 0.6}


def _run_lists_nn(name, cfg):
    c = case(name)
    ntype, nsample, grids = cfg
    d = D_OF[name]
    buf, sl, total = _lists_gpu(c, d, nsample, ntype)
    centres = _centres(c[2], grids, d)
    idx, d2 = _nn_gpu(c, buf, sl, total, centres)
    fidx, fd2 = _fused_nn(c, centres, d, nsample, ntype)
    return _split(buf, sl), total, idx.cpu().numpy(), d2.cpu().numpy(), fidx.cpu().numpy(), fd2.cpu().numpy(), centres


@pytest.mark.parametrize("cfg", NN_CFGS, ids=lambda c: f"t{c[0]}-ns{c[1]}-g{c[2][0]}{c[2][1]}{c[2][2]}")
@pytest.mark.parametrize("name", list(CASES))
def test_lists_and_three_nn_match_oracle_grid_and_brute(monkeypatch, name, cfg):
    if name == "150k" and cfg[2] != (3, 3, 3):
        pytest.skip("the 150k-point frame runs one configuration")
    xyz, cnt, new, mcnt = case(name)
    ntype, nsample, grids = cfg
    d = D_OF[name]
    lists, total, idx, d2, fidx, fd2, centres = _run_lists_nn(name, cfg)
    want = vpo.local_lists(xyz, cnt, new, mcnt, d, nsample, ntype)
    assert total == sum(len(x) for x in want)
    for p, (a, b) in enumerate(zip(lists, want)):
        assert np.array_equal(a, b), (name, p, a[:8], b[:8])
    if name == "dense" and ntype == 0:  # the cube holds > 1000 lattice points, the ball fewer
        assert max(len(x) for x in want) == (1000 if nsample < 0 else min(nsample, 1000))
    oi, od = vpo.three_nn_local(xyz, centres.cpu().numpy(), want)
    assert np.array_equal(idx, oi) and np.array_equal(_bits(d2), _bits(od))
    assert np.array_equal(fidx, oi) and np.array_equal(_bits(fd2), _bits(od))
    knob_setenv(monkeypatch, "TSMDET_BQ_ALGO", "brute")
    lists_b, total_b, idx_b, d2_b, fidx_b, fd2_b, _ = _run_lists_nn(name, cfg)
    assert total_b == total and all(np.array_equal(a, b) for a, b in zip(lists_b, want))
    assert np.array_equal(idx_b, oi) and np.array_equal(_bits(d2_b), _bits(od))
    assert np.array_equal(fidx_b, oi) and np.array_equal(_bits(fd2_b), _bits(od))


def test_list_buffer_truncation_and_exact_total():
    c = case("ragged")
    full, sl_full, total = _lists_gpu(c, 0.8, -1, 1)
    small, sl, total_small = _lists_gpu(c, 0.8, -1, 1, avg=2)
    assert total_small == total > 2 * c[2].shape[0]
    assert torch.equal(sl[:, 1], sl_full[:, 1])
    buf = small.cpu().numpy()
    for (o, n), lst in zip(sl.cpu().numpy(), _split(full, sl_full)):
        k = max(0, min(n, buf.shape[0] - o))
        assert np.array_equal(buf[o:o + k], lst[:k])


# ---------------------------------------------------------------------------------------------- function 3
POOL_CFGS = [  # (pooling, neighbor_type, nsample, grids, c_in, cpg, use_xyz)
    (0, 0, -1, (3, 3, 3), 30, 30, 1), (0, 1, 32, (2, 2, 2), 64, 32, 0), (1, 0, 32, (3, 3, 3), 128, 128, 1),
    (1, 1, -1, (4, 4, 4), 33, 33, 1), (0, 0, 1, (1, 1, 1), 1, 1, 1), (0, 0, -1, (2, 3, 4), 2, 1, 1),
    (1, 0, -1, (2, 3, 4), 30, 15, 0),
]


def _pool_gpu(c, feats, cfg, d, max_sum):
    from tsmdet_b200.pointnet2_stack import pointnet2_stack_cuda as ps

    pooling, ntype, nsample, (nx, ny, nz), cin, cpg, use_xyz = cfg
    xyz, cnt, new, mcnt = c
    m, G = new.shape[0], nx * ny * nz
    nf = torch.zeros((m, G * cpg), device="cuda")
    nl = torch.zeros((m, 3 * G), device="cuda")
    pc = torch.zeros((m, G), dtype=torch.int32, device="cuda")
    tr = torch.zeros((max_sum, 3), dtype=torch.int32, device="cuda")
    total = ps.vector_pool_wrapper(T(xyz), T(cnt), T(feats), T(new), T(mcnt), nf, nl, pc, tr, nx, ny, nz, d, use_xyz,
                                   max_sum, nsample, ntype, pooling)
    assert isinstance(total, int)
    return nf.cpu().numpy(), nl.cpu().numpy(), pc.cpu().numpy(), tr.cpu().numpy(), total


def _sorted_rows(a):
    a = np.asarray(a).reshape(-1, 3)
    return a[np.lexsort(a.T[::-1])] if len(a) else a


@pytest.mark.parametrize("cfg", POOL_CFGS, ids=lambda c: f"p{c[0]}-t{c[1]}-ns{c[2]}-g{c[3][0]}{c[3][1]}{c[3][2]}-c{c[4]}")
@pytest.mark.parametrize("name", list(CASES))
def test_vector_pool_matches_oracle_grid_and_brute(monkeypatch, name, cfg):
    if name == "150k" and cfg not in POOL_CFGS[:3]:
        pytest.skip("the 150k-point frame runs three configurations")
    c = case(name)
    d = D_OF[name]
    feats = np.random.default_rng(20).normal(size=(c[0].shape[0], cfg[4])).astype(np.float32)
    pooling, ntype, nsample, grids, cin, cpg, use_xyz = cfg
    want = vpo.vector_pool(c[0], c[1], feats, c[2], c[3], grids, cpg, d, use_xyz, nsample, ntype, pooling)
    runs = [_pool_gpu(c, feats, cfg, d, max(want[4], 1))]
    knob_setenv(monkeypatch, "TSMDET_BQ_ALGO", "brute")
    runs.append(_pool_gpu(c, feats, cfg, d, max(want[4], 1)))
    for nf, nl, pc, tr, total in runs:
        assert total == want[4]
        assert np.array_equal(_bits(nf), _bits(want[0])) and np.array_equal(pc, want[2])
        assert np.array_equal(_bits(nl), _bits(want[1]))
        assert np.array_equal(_sorted_rows(tr[:total]), _sorted_rows(want[3]))


def test_vector_pool_overflow_returns_the_exact_total():
    c = case("ragged")
    cfg = POOL_CFGS[0]
    feats = np.random.default_rng(21).normal(size=(c[0].shape[0], 30)).astype(np.float32)
    big = _pool_gpu(c, feats, cfg, 0.8, 200000)
    small = _pool_gpu(c, feats, cfg, 0.8, 5)
    assert small[4] == big[4] > 5
    assert np.array_equal(_bits(small[0]), _bits(big[0])) and np.array_equal(small[2], big[2])


def test_retry_loops_give_the_generous_result():
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu

    xyz, cnt, new, mcnt = case("ragged")
    centres = _centres(new, (3, 3, 3), 0.8)
    args = (T(xyz), T(cnt), T(new), centres, T(mcnt), 0.8, -1, 0)
    d_a, i_a, avg_a = pu.three_nn_for_vector_pool_by_two_step(*args, 1, 27, 2.0)
    d_b, i_b, avg_b = pu.three_nn_for_vector_pool_by_two_step(*args, 100000, 27, 2.0)
    assert torch.equal(i_a, i_b) and torch.equal(d_a, d_b) and int(avg_a) == int(avg_b) > 1
    feats = T(np.random.default_rng(22).normal(size=(xyz.shape[0], 16)).astype(np.float32))
    outs = [pu.vector_pool_with_voxel_query_op(T(xyz), T(cnt), feats, T(new), T(mcnt), 3, 3, 3, 0.8, 16, 1, nm, -1, 0, 0)
            for nm in (1, 100000)]
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a.cpu(), b.cpu())
    assert int(outs[0][2]) == int(outs[1][2]) > 1


# ---------------------------------------------------------------------------------------------- function 4
@pytest.mark.parametrize("pooling", [0, 1])
def test_gradient_against_float64_index_add(pooling):
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu

    xyz, cnt, new, mcnt = case("ragged")
    rng = np.random.default_rng(23)
    feats = T(rng.normal(size=(xyz.shape[0], 8)).astype(np.float32)).requires_grad_(True)
    nf, nl, nm, pc = pu.vector_pool_with_voxel_query_op(T(xyz), T(cnt), feats, T(new), T(mcnt), 2, 2, 2, 0.8, 4, 1, 20,
                                                        -1, 0, pooling)
    go = torch.randn_like(nf)
    nf.backward(go)
    want = vpo.vector_pool(xyz, cnt, feats.detach().cpu().numpy(), new, mcnt, (2, 2, 2), 4, 0.8, 1, -1, 0, pooling)
    tr, pcn = want[3].astype(np.int64), want[2]
    assert np.array_equal(pc.cpu().numpy(), pcn)
    g = go.double().cpu().numpy().reshape(len(new), 8, 4)
    ref = np.zeros((xyz.shape[0], 8))
    w = 1.0 / np.maximum(pcn[tr[:, 1], tr[:, 2]], 1)
    for i in range(8):
        np.add.at(ref[:, i], tr[:, 0], g[tr[:, 1], tr[:, 2], i % 4] * w)
    assert np.allclose(feats.grad.double().cpu().numpy(), ref, rtol=1e-5, atol=1e-6)


# ---------------------------------------------------------------------------------------------- modules
class Cfg(dict):
    __getattr__ = dict.__getitem__


def _module(kind, c_in=64, reduced=32, grids=(3, 3, 3), d=1.2, nsample=-1, ntype=0, seed=0):
    from tsmdet_b200.pointnet2_stack.pointnet2_modules import VectorPoolAggregationModule

    torch.manual_seed(seed)
    mod = VectorPoolAggregationModule(c_in, num_local_voxel=grids, local_aggregation_type=kind,
                                      num_reduced_channels=reduced, num_channels_of_local_aggregation=16,
                                      post_mlps=(64,), max_neighbor_distance=d, neighbor_nsample=nsample,
                                      neighbor_type=ntype).cuda()
    for m in mod.modules():  # non-trivial batch-norm statistics
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.uniform_(-0.1, 0.1)
            m.running_var.uniform_(0.5, 1.5)
    return mod.eval()


def _module_inputs(c_in=64, name="ragged"):
    xyz, cnt, new, mcnt = case(name)
    feats = np.random.default_rng(30).normal(size=(xyz.shape[0], c_in)).astype(np.float32)
    return dict(xyz=T(xyz), xyz_batch_cnt=T(cnt), new_xyz=T(new), new_xyz_batch_cnt=T(mcnt), features=T(feats))


KINDS = ["local_interpolation", "voxel_avg_pool", "voxel_random_choice"]


def _eager_planes(mod, inp):
    feats = inp["features"].view(inp["features"].shape[0], -1, mod.num_reduced_channels).sum(dim=1)
    args = dict(xyz=inp["xyz"], xyz_batch_cnt=inp["xyz_batch_cnt"], features=feats, new_xyz=inp["new_xyz"],
                new_xyz_batch_cnt=inp["new_xyz_batch_cnt"])
    if mod.local_aggregation_type == "local_interpolation":
        vf = mod.vector_pool_with_local_interpolate(**args)
    else:
        vf = mod.vector_pool_with_voxel_query(**args)[0]
    return feats, vf.permute(1, 0)[None, :, :]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("ntype,nsample", [(0, -1), (1, 32)])
def test_eval_planes_bit_identical_to_eager(kind, ntype, nsample):
    mod = _module(kind, ntype=ntype, nsample=nsample)
    for name in ("ragged", "edge"):
        inp = _module_inputs(name=name)
        feats, eager = _eager_planes(mod, inp)
        fused = mod.input_planes(inp["xyz"], inp["xyz_batch_cnt"], feats, inp["new_xyz"], inp["new_xyz_batch_cnt"])
        assert fused.shape == eager.shape
        assert torch.equal(fused.view(torch.int32), eager.contiguous().view(torch.int32)), (kind, name)


@pytest.mark.parametrize("kind", KINDS)
def test_eager_matches_restatement_fed_by_the_oracle(kind):
    mod = _module(kind, ntype=1)
    inp = _module_inputs()
    feats, eager = _eager_planes(mod, inp)
    xyz, cnt, new, mcnt = case("ragged")
    f = feats.cpu().numpy()
    G, C, d = 27, 32, 1.2
    if kind == "local_interpolation":
        import stack_nn_oracle as sno

        lists = vpo.local_lists(xyz, cnt, new, mcnt, np.float32(d * 2.0), -1, 1)
        centres = _centres(new, (3, 3, 3), d)
        idx, d2 = vpo.three_nn_local(xyz, centres.cpu().numpy(), lists)
        dist = torch.sqrt(T(d2))
        dist_recip = 1.0 / (dist + 1e-8)
        w = (dist_recip / torch.clamp_min(torch.sum(dist_recip, dim=-1, keepdim=True), min=1e-8)).cpu().numpy()
        idx = idx.reshape(-1, 3)
        empty = idx[:, 0] == -1
        idx[empty] = 0
        interp = sno.stack_three_interpolate(f, idx, w.reshape(-1, 3))
        local = (centres.cpu().numpy().reshape(-1, 1, 3) - xyz[idx]).reshape(-1, 9)
        rows = np.concatenate([interp, local], 1)
        rows[empty] = 0
        want = rows.reshape(len(new), -1).T[None]
    else:
        pooling = 0 if kind == "voxel_avg_pool" else 1
        nf, nl, pc, _, _ = vpo.vector_pool(xyz, cnt, f, new, mcnt, (3, 3, 3), C, d, 1, -1, 1, pooling)
        norm = np.maximum(pc.astype(np.float32), np.float32(1e-6))[:, :, None]
        rows = np.concatenate([(nl.reshape(-1, G, 3) / norm).astype(np.float32),
                               (nf.reshape(-1, G, C) / norm).astype(np.float32)], -1)
        want = rows.reshape(len(new), -1).T[None]
    assert np.array_equal(_bits(eager.cpu().numpy()), _bits(want))


@pytest.mark.parametrize("kind", KINDS)
def test_fused_module_output_within_fp32_tolerance(kind):
    mod = _module(kind)
    inp = _module_inputs()
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            fused = mod(**inp)[1]
            mod.fused = False
            eager = mod(**inp)[1]
    finally:
        torch.backends.cudnn.allow_tf32 = old
        mod.fused = True
    assert torch.allclose(fused, eager, rtol=1e-5, atol=1e-5)


def _msg_config(kind):
    return Cfg(NAME="VectorPoolAggregationModuleMSG", NUM_GROUPS=2, LOCAL_AGGREGATION_TYPE=kind, NUM_REDUCED_CHANNELS=2,
               NUM_CHANNELS_OF_LOCAL_AGGREGATION=32, MSG_POST_MLPS=[128],
               GROUP_CFG_0=Cfg(NUM_LOCAL_VOXEL=[2, 2, 2], MAX_NEIGHBOR_DISTANCE=0.2, NEIGHBOR_NSAMPLE=-1, POST_MLPS=[32, 32]),
               GROUP_CFG_1=Cfg(NUM_LOCAL_VOXEL=[3, 3, 3], MAX_NEIGHBOR_DISTANCE=0.4, NEIGHBOR_NSAMPLE=-1, POST_MLPS=[32, 32]))


def test_state_dict_keys_and_loading_and_builder():
    from tsmdet_b200.pointnet2_stack import pointnet2_modules as pm

    mod, c_out = pm.build_local_aggregation_module(4, _msg_config("local_interpolation"))
    assert isinstance(mod, pm.VectorPoolAggregationModuleMSG) and c_out == 128
    keys = set(mod.state_dict())
    for k in (0, 1):
        for s in ("separate_local_aggregation_layer.0.weight", "separate_local_aggregation_layer.1.running_var",
                  "post_mlps.0.weight", "post_mlps.1.weight", "post_mlps.3.weight", "post_mlps.4.num_batches_tracked"):
            assert f"layer_{k}.{s}" in keys
    assert "msg_post_mlps.0.weight" in keys and "msg_post_mlps.1.bias" in keys
    assert mod.layer_1.separate_local_aggregation_layer[0].weight.shape == (27 * 32, 11, 1)
    assert mod.layer_0.separate_local_aggregation_layer[0].groups == 8
    assert mod.msg_post_mlps[0].weight.shape == (128, 32 + 32 + 3, 1)
    # a checkpoint of the reference module: same keys and shapes, loads strictly
    sd = {k: torch.randn_like(v.float()).to(v.dtype) if v.dtype.is_floating_point else v for k, v in mod.state_dict().items()}
    mod2, _ = pm.build_local_aggregation_module(4, _msg_config("local_interpolation"))
    mod2.load_state_dict(sd, strict=True)
    sa, c_sa = pm.build_local_aggregation_module(16, Cfg(NAME="StackSAModuleMSG", MLPS=[[16, 16], [16, 32]],
                                                         POOL_RADIUS=[0.4, 0.8], NSAMPLE=[16, 16]))
    assert isinstance(sa, pm.StackSAModuleMSG) and c_sa == 48
    assert pm.VectorPoolAggregationModule(32, max_neighbor_distance=1.0).num_mean_points_per_grid == 20
    assert pm.VectorPoolAggregationModule(
        32, max_neighbor_distance=1.0).local_interpolate_module.num_avg_length_of_neighbor_idxs == 1000


@pytest.mark.parametrize("kind", KINDS)
def test_msg_module_eval_forward_in_a_cuda_graph(kind):
    from tsmdet_b200.pointnet2_stack import pointnet2_modules as pm

    torch.manual_seed(1)
    mod = pm.VectorPoolAggregationModuleMSG(4, _msg_config(kind)).cuda().eval()
    xyz, cnt, new, mcnt = case("ragged")
    inp = dict(xyz=T(xyz * 0.2), xyz_batch_cnt=T(cnt), new_xyz=T(new * 0.2), new_xyz_batch_cnt=T(mcnt),
               features=T(np.random.default_rng(31).normal(size=(xyz.shape[0], 4)).astype(np.float32)))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s), torch.no_grad():
        want = mod(**inp)[1].clone()  # warm-up on the capture stream: the scratch buffers are keyed by stream
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s), torch.no_grad():
        out = mod(**inp)[1]
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, want)


# ---------------------------------------------------------------------------------------------- head to head
@pytest.fixture(scope="module")
def ref_stack():
    from oracle import build_ref

    return build_ref.load_ref("pointnet2_stack_cuda")


@pytest.mark.parametrize("name", ["ragged", "edge", "dense"])
def test_wrappers_vs_reference_cuda(ref_stack, name):
    if ref_stack is None:
        pytest.skip("oracle/_ref/pointnet2_stack_cuda.so not built (needs the reference tree)")
    xyz, cnt, new, mcnt = c = case(name)
    d, m = D_OF[name], new.shape[0]
    for ntype, nsample in ((0, -1), (1, 32)):
        buf = torch.zeros((1000 * m,), dtype=torch.int32, device="cuda")
        sl = torch.zeros((m, 2), dtype=torch.int32, device="cuda")
        cs = torch.zeros((1,), dtype=torch.int32, device="cuda")
        ref_stack.query_stacked_local_neighbor_idxs_wrapper_stack(T(xyz), T(cnt), T(new), T(mcnt), buf, sl, cs, 1000, d,
                                                                  nsample, ntype)
        mine_buf, mine_sl, total = _lists_gpu(c, d, nsample, ntype)
        assert int(cs.item()) == total
        assert all(np.array_equal(a, b) for a, b in zip(_split(buf, sl), _split(mine_buf, mine_sl)))
        centres = _centres(new, (3, 3, 3), d)
        idx = torch.zeros((m, 27, 3), dtype=torch.int32, device="cuda")
        d2 = torch.zeros((m, 27, 3), device="cuda")
        ref_stack.query_three_nn_by_stacked_local_idxs_wrapper_stack(T(xyz), T(new), centres, idx, d2, buf[:total], sl,
                                                                     m, 27)
        mi, md = _nn_gpu(c, mine_buf, mine_sl, total, centres)
        assert torch.equal(idx, mi) and torch.equal(d2.view(torch.int32), md.view(torch.int32))
        for pooling in (0, 1):
            feats = np.random.default_rng(40).normal(size=(xyz.shape[0], 16)).astype(np.float32)
            cfg = (pooling, ntype, nsample, (3, 3, 3), 16, 16, 1)
            nf, nl, pc, tr, tot = _pool_gpu(c, feats, cfg, d, 200000)
            rf, rl = torch.zeros((m, 27 * 16), device="cuda"), torch.zeros((m, 81), device="cuda")
            rp, rt = torch.zeros((m, 27), dtype=torch.int32, device="cuda"), torch.zeros((200000, 3), dtype=torch.int32,
                                                                                          device="cuda")
            rtot = ref_stack.vector_pool_wrapper(T(xyz), T(cnt), T(feats), T(new), T(mcnt), rf, rl, rp, rt, 3, 3, 3, d, 1,
                                                 200000, nsample, ntype, pooling)
            assert rtot == tot and np.array_equal(pc, rp.cpu().numpy())
            assert np.array_equal(_bits(nf), _bits(rf.cpu().numpy())) and np.array_equal(_bits(nl), _bits(rl.cpu().numpy()))
            assert np.array_equal(_sorted_rows(tr[:tot]), _sorted_rows(rt.cpu().numpy()[:rtot]))


def test_reference_stack_vector_pool_python_over_shims():
    from ref_stack_py import load_reference_stack_python

    ref = load_reference_stack_python()
    if ref is None:
        pytest.skip("the reference tree (its stack pointnet2_utils.py / pointnet2_modules.py) is not present")
    _, ref_modules = ref
    if not hasattr(ref_modules, "VectorPoolAggregationModuleMSG"):
        pytest.skip("the reference's stack modules have no VectorPoolAggregationModuleMSG")
    from tsmdet_b200.pointnet2_stack import pointnet2_modules as pm

    xyz, cnt, new, mcnt = case("ragged")
    inp = dict(xyz=T(xyz * 0.2), xyz_batch_cnt=T(cnt), new_xyz=T(new * 0.2), new_xyz_batch_cnt=T(mcnt),
               features=T(np.random.default_rng(41).normal(size=(xyz.shape[0], 4)).astype(np.float32)))
    for kind in KINDS:
        mine = pm.VectorPoolAggregationModuleMSG(4, _msg_config(kind)).cuda().eval()
        theirs = ref_modules.VectorPoolAggregationModuleMSG(4, _msg_config(kind)).cuda().eval()
        theirs.load_state_dict(mine.state_dict())
        with torch.no_grad():
            want = theirs(**inp)[1]
            got = mine(**inp)[1]
        assert torch.allclose(got, want, rtol=1e-5, atol=1e-5), kind
