"""GPU suite of the stacked (ragged) ball query, QueryAndGroup and StackSAModuleMSG (pointnet2_stack):

  * ball_query_wrapper bit-exact against the CPU oracle (tests/stack_bq_oracle.c), on the cases of tests/stack_cases.py
    plus frames the grid cannot take (a pile of > 256 points in one cell, a non-finite coordinate), a 150k-point frame,
    the grid against TSMDET_BQ_ALGO=brute, and the golden rows of the reference's batch kernel as a 2-frame stack;
  * QueryAndGroup bit-exact against numpy assembled from the oracle's idx, its autograd against an index_add
    restatement;
  * StackSAModuleMSG: eager against a plain-torch restatement, fused fp32 / bf16 / tf32 against eager (tests/parity.py
    bars) and element by element against the float64 reference of tests/mlp_ref.py; the empty-ball ReLU(bias) chain,
    the fold cache and the eager fallbacks of train mode / fused=False;
  * head to head against the reference's own stack ball query (oracle/_ref/pointnet2_stack_cuda.so) and its stack
    Python over this package's shim, when those are built."""
import os

import numpy as np
import pytest
import torch
from conftest import knob_setenv

import mlp_ref
import parity
import stack_bq_oracle as sbq
import stack_cases
import synth

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _query(xyz, cnt, new, mcnt, radius, nsample):
    from tsmdet_b200.pointnet2_stack import pointnet2_stack_cuda as ps

    m = new.shape[0]
    idx = torch.zeros((m, nsample), dtype=torch.int32, device="cuda")
    assert ps.ball_query_wrapper(len(cnt), m, radius, nsample, T(new), T(mcnt), T(xyz), T(cnt), idx) == 1
    return idx.cpu().numpy()


def _native(xyz, cnt, new, mcnt, radius, nsample, global_rows):
    """tsmdet_stack_ball_query with idx_cnt: (idx, idx_cnt); idx pre-filled with a sentinel"""
    from tsmdet_b200._lib import call, ptr, stream_ptr

    m = new.shape[0]
    idx = torch.full((m, nsample), -7, dtype=torch.int32, device="cuda")
    ic = torch.full((m,), -5, dtype=torch.int32, device="cuda")
    args = [T(a) for a in (new, mcnt, xyz, cnt)]
    call("tsmdet_stack_ball_query", len(cnt), m, xyz.shape[0], float(radius), nsample, ptr(args[0]), ptr(args[1]),
         ptr(args[2]), ptr(args[3]), ptr(idx), ptr(ic), global_rows, stream_ptr())
    return idx.cpu().numpy(), ic.cpu().numpy()


def _global_rows(idx, cnt_frames, mcnt):
    """oracle rows (frame-local, -1 marks empty) -> (global rows with zero rows for empty balls, empty mask)"""
    ns = np.concatenate([[0], np.cumsum(cnt_frames)])[:-1]
    owner = np.repeat(np.arange(len(mcnt)), mcnt)
    empty = idx[:, 0] == -1
    g = idx + ns[owner][:, None]
    g[empty] = 0
    return g.astype(np.int32), empty


def _extra_cases():
    rng = np.random.default_rng(11)
    base = synth.cloud_ground_objects(1, 3000, seed=21)[0]
    pile = base.copy()
    pile[100:700] = pile[50] + rng.uniform(-1e-3, 1e-3, size=(600, 3)).astype(np.float32)  # > 256 in one cell
    bad = base.copy()
    bad[17, 1] = np.nan
    bad[29, 2] = np.inf
    fx = [base, pile, bad, base[::-1].copy()]
    fn = [stack_cases.centres_from(rng, f[np.isfinite(f).all(1)], 300) for f in fx]
    fn[1][:50] = pile[50]  # centres inside the pile
    big = synth.cloud_ground_objects(1, 150000, seed=22)[0]
    out = [("grid-unusable-frames", *stack_cases.stack(fx, fn), 0.8, 32),
           ("grid-unusable-frames-ns100", *stack_cases.stack(fx, fn), 0.8, 100)]
    out.append(("150k-frame", *stack_cases.stack([big, base], [stack_cases.centres_from(rng, big, 4096),
                                                              stack_cases.centres_from(rng, base, 500)]), 0.4, 16))
    return out


ALL_CASES = stack_cases.cases() + _extra_cases()


@pytest.mark.parametrize("case", ALL_CASES, ids=lambda c: c[0])
def test_stack_ball_query_matches_oracle(case):
    _, xyz, cnt, new, mcnt, radius, nsample = case
    want = sbq.stack_ball_query(radius, nsample, xyz, cnt, new, mcnt)
    got = _query(xyz, cnt, new, mcnt, radius, nsample)
    assert np.array_equal(got, want), f"{int((got != want).any(1).sum())} rows differ"
    # the fused path's form: global rows, zero rows for empty balls, counts
    g, empty = _global_rows(want, cnt, mcnt)
    idx, ic = _native(xyz, cnt, new, mcnt, radius, nsample, 1)
    assert np.array_equal(idx, g)
    hits = np.array([len(set(r)) for r in want])  # distinct frame-local hits = min(hits, nsample)
    assert np.array_equal(ic, np.where(empty, 0, hits))
    idx0, ic0 = _native(xyz, cnt, new, mcnt, radius, nsample, 0)
    assert np.array_equal(ic0, ic)
    assert np.array_equal(np.where(idx0 == -7, 0, idx0), want)  # slots 1.. of an empty ball are left alone
    assert (idx0[empty, 1:] == -7).all() and not (idx0[~empty] == -7).any()


@pytest.mark.parametrize("case", [c for c in ALL_CASES if c[0] in ("ragged-r0.8-ns32", "ragged-r0.8-ns100",
                                                                   "grid-unusable-frames", "dup-padded-r0.4-ns16")],
                         ids=lambda c: c[0])
def test_stack_ball_query_grid_equals_brute(monkeypatch, case):
    _, xyz, cnt, new, mcnt, radius, nsample = case
    grid = _query(xyz, cnt, new, mcnt, radius, nsample)
    knob_setenv(monkeypatch, "TSMDET_BQ_ALGO", "brute")
    brute = _query(xyz, cnt, new, mcnt, radius, nsample)
    assert np.array_equal(grid, brute)


def test_stack_ball_query_golden_two_frame_stack():
    """the reference's batch kernel's rows (tests/golden/ball_query.npz), first min(cnt, nsample) entries"""
    g = np.load(os.path.join(GOLDEN, "ball_query.npz"))
    b, n, _ = g["xyz"].shape
    m = g["new_xyz"].shape[1]
    cnt, mcnt = np.full((b,), n, np.int32), np.full((b,), m, np.int32)
    for key, r, ns in (("r08", 0.8, 32), ("r02", 0.2, 16), ("r30", 3.0, 8)):
        idx = _query(g["xyz"].reshape(-1, 3), cnt, g["new_xyz"].reshape(-1, 3), mcnt, r, ns)
        gc, gi = g[key + "_cnt"].reshape(-1), g[key + "_idx"].reshape(-1, ns)
        for p in range(b * m):
            k = min(int(gc[p]), ns)
            if k == 0:
                assert idx[p, 0] == -1 and not idx[p, 1:].any()
            else:
                assert np.array_equal(idx[p, :k], gi[p, :k]) and (idx[p, k:] == idx[p, 0]).all(), (key, p)


# ---------------------------------------------------------------------------------------------- QueryAndGroup
@pytest.mark.parametrize("use_xyz,c", [(True, 0), (True, 5), (False, 5)])
def test_query_and_group_matches_oracle(use_xyz, c):
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu

    xyz, cnt, new, mcnt = stack_cases.ragged(seed=3)
    radius, ns = 0.8, 16
    feats = np.random.default_rng(4).standard_normal((xyz.shape[0], c)).astype(np.float32) if c else None
    raw = sbq.stack_ball_query(radius, ns, xyz, cnt, new, mcnt)
    g, empty = _global_rows(raw, cnt, mcnt)
    want_xyz = (xyz[g] - new[:, None, :]).transpose(0, 2, 1)  # (M, 3, ns), fp32 subtraction as the torch op
    want_xyz[empty] = 0
    parts = [want_xyz] if use_xyz else []
    if c:
        wf = feats[g].transpose(0, 2, 1)
        wf[empty] = 0
        parts.append(wf)
    want = np.concatenate(parts, 1)
    qg = pu.QueryAndGroup(radius, ns, use_xyz=use_xyz)
    got, idx = qg(T(xyz), T(cnt), T(new), T(mcnt), None if feats is None else T(feats))
    assert np.array_equal(idx.cpu().numpy(), np.where(raw == -1, 0, raw))
    assert got.shape == want.shape and np.array_equal(got.cpu().numpy(), want)
    idx2, mask = pu.ball_query(radius, ns, T(xyz), T(cnt), T(new), T(mcnt))
    assert np.array_equal(mask.cpu().numpy(), empty) and torch.equal(idx2, idx)


def test_query_and_group_backward():
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu

    xyz, cnt, new, mcnt = stack_cases.ragged(seed=5)
    c, ns = 6, 8
    tx = T(xyz).requires_grad_(True)
    tf = torch.randn((xyz.shape[0], c), device="cuda", requires_grad=True)
    out, idx = pu.QueryAndGroup(0.8, ns)(tx, T(cnt), T(new), T(mcnt), tf)
    go = torch.randn_like(out)
    out.backward(go)
    starts = torch.from_numpy(np.concatenate([[0], np.cumsum(cnt)])[:-1]).cuda()
    owner = torch.repeat_interleave(torch.arange(len(mcnt), device="cuda"), T(mcnt).long())
    gidx = (idx.long() + starts[owner][:, None]).reshape(-1)
    _, empty = pu.ball_query(0.8, ns, T(xyz), T(cnt), T(new), T(mcnt))
    live = (~empty).float()[:, None, None]
    gx = (go[:, :3] * live).permute(0, 2, 1).reshape(-1, 3)
    gf = (go[:, 3:] * live).permute(0, 2, 1).reshape(-1, c)
    want_x = torch.zeros_like(tx).index_add_(0, gidx, gx)
    want_f = torch.zeros_like(tf).index_add_(0, gidx, gf)
    assert torch.allclose(tx.grad, want_x, atol=1e-5, rtol=1e-5)
    assert torch.allclose(tf.grad, want_f, atol=1e-5, rtol=1e-5)


# ---------------------------------------------------------------------------------------------- StackSAModuleMSG
def _randomise_bn(mod, seed):
    g = torch.Generator().manual_seed(seed)
    for m in mod.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.1)


# PV-RCNN's keypoint SA shapes: C = 1 (planes) and C = 64 (feature rows); nsample 16 / 32
CFGS = {
    "c1": dict(radii=[0.4, 0.8], nsamples=[16, 16], mlps=[[1, 16, 16], [1, 16, 16]], c=1),
    "c64": dict(radii=[1.2, 2.4], nsamples=[16, 32], mlps=[[64, 64, 64], [64, 64, 64]], c=64),
    "c5_noxyz": dict(radii=[0.8], nsamples=[16], mlps=[[5, 32, 48]], c=5, use_xyz=False),
}


def _sa_inputs(c, seed=7):
    rng = np.random.default_rng(seed)
    sizes = [9000, 0, 14000, 11000]
    fx = [synth.cloud_ground_objects(1, n, seed=seed + k)[0] if n else np.zeros((0, 3), np.float32)
          for k, n in enumerate(sizes)]
    fn = [stack_cases.centres_from(rng, f, m, jitter=1.0) for f, m in zip(fx, [512, 40, 512, 0])]
    xyz, cnt, new, mcnt = stack_cases.stack(fx, fn)
    new[3] += 1000.0  # an empty ball in a populated frame
    feats = rng.standard_normal((xyz.shape[0], c)).astype(np.float32)
    return xyz, cnt, new, mcnt, feats


def _module(cfg, precision="fp32", seed=0):
    from tsmdet_b200.pointnet2_stack import StackSAModuleMSG

    torch.manual_seed(seed)
    mod = StackSAModuleMSG(radii=cfg["radii"], nsamples=cfg["nsamples"], mlps=cfg["mlps"],
                           use_xyz=cfg.get("use_xyz", True), precision=precision).cuda().eval()
    _randomise_bn(mod, seed + 1)
    return mod


def _run(mod, xyz, cnt, new, mcnt, feats, fused):
    mod.fused = fused
    with torch.no_grad():
        return mod(T(xyz), T(cnt), T(new), T(mcnt), T(feats))


@pytest.mark.parametrize("name", list(CFGS))
def test_stack_sa_eager_matches_torch_restatement(name):
    cfg = CFGS[name]
    mlps_arg = [list(s) for s in cfg["mlps"]]
    mod = _module(dict(cfg, mlps=mlps_arg))
    assert mlps_arg == cfg["mlps"], "the caller's list was mutated"
    assert all(k.startswith(("groupers.", "mlps.")) for k in mod.state_dict())
    xyz, cnt, new, mcnt, feats = _sa_inputs(cfg["c"])
    use_xyz = cfg.get("use_xyz", True)
    outs = []
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        new_xyz, got = _run(mod, xyz, cnt, new, mcnt, feats, fused=False)
        assert np.array_equal(new_xyz.cpu().numpy(), new)
        for r, ns, seq in zip(cfg["radii"], cfg["nsamples"], mod.mlps):
            g, empty = _global_rows(sbq.stack_ball_query(r, ns, xyz, cnt, new, mcnt), cnt, mcnt)
            parts = [(xyz[g] - new[:, None, :])] if use_xyz else []
            parts.append(feats[g])
            x = np.concatenate(parts, 2)
            x[empty] = 0
            h = T(x).permute(2, 0, 1).unsqueeze(0)  # (1, C, M, ns)
            with torch.no_grad():
                for layer in seq:
                    h = layer(h)
            outs.append(h.max(dim=3)[0][0].t())
    finally:
        torch.backends.cudnn.allow_tf32 = old
    want = torch.cat(outs, 1)
    assert got.shape == want.shape
    assert torch.allclose(got, want, atol=1e-5, rtol=1e-5)


@pytest.mark.parametrize("name,precision", [(k, p) for k in CFGS for p in ("fp32", "bf16", "tf32")])
def test_stack_sa_fused_matches_eager_and_reference(name, precision):
    from tsmdet_b200.pointnet2_modules import _effective_precision

    cfg = CFGS[name]
    mod = _module(cfg, precision)
    xyz, cnt, new, mcnt, feats = _sa_inputs(cfg["c"])
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        _, want = _run(mod, xyz, cnt, new, mcnt, feats, fused=False)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    _, got = _run(mod, xyz, cnt, new, mcnt, feats, fused=True)
    _, again = _run(mod, xyz, cnt, new, mcnt, feats, fused=True)
    torch.cuda.synchronize()
    assert torch.equal(got, again)
    assert got.shape == want.shape and got.is_contiguous()
    m = parity.err_metrics(got, want)
    print(f"STACKSA {name} {precision}: {m}")
    parity.check_metrics(m, precision, f"{name} fused {precision} vs eager")

    # element by element: the stack as ONE cloud (B = 1), global rows from the oracle
    use_xyz = cfg.get("use_xyz", True)
    c0 = 0
    for (r, ns), layers, img in zip(zip(cfg["radii"], cfg["nsamples"]), mod._folded, mod._packed[1]):
        prec = _effective_precision(precision, img)
        kernel = {"fp32": "fp32"}.get(prec, "tc2" if img is not None else "v1")
        g, empty = _global_rows(sbq.stack_ball_query(r, ns, xyz, cnt, new, mcnt), cnt, mcnt)
        ic = (~empty).astype(np.int32)
        rows = mlp_ref.sa_rows(xyz[None], new[None], feats.T[None], g[None], ic[None], use_xyz, mlp_ref.QUANT[prec])
        lnp = [(w.cpu().numpy(), b.cpu().numpy()) for w, b in layers]
        want_k, bound = mlp_ref.mlp_reference(rows, lnp, ns, prec, kernel)
        cout = lnp[-1][0].shape[0]
        ratio, rel, n_out = mlp_ref.compare(got[:, c0:c0 + cout].double().cpu().numpy(), want_k, bound)
        print(f"MLPREF stack {name} {precision}->{prec} {kernel}: max err/B {ratio:.3f} rel_l2 {rel:.2e}")
        assert n_out == 0 and ratio <= 1.0, (ratio, n_out)
        assert rel <= mlp_ref.REL_L2_BAR[prec], rel
        c0 += cout


def test_stack_sa_empty_ball_relu_bias_chain():
    """an empty ball sees an all-zero INPUT and outputs the ReLU(bias) chain, in both modes"""
    cfg = CFGS["c64"]
    mod = _module(cfg)
    xyz, cnt, new, mcnt, feats = _sa_inputs(cfg["c"])
    _, fused = _run(mod, xyz, cnt, new, mcnt, feats, fused=True)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False  # the eager convolutions and the chain below in fp32
    try:
        _, eager = _run(mod, xyz, cnt, new, mcnt, feats, fused=False)
        chain = []
        for seq in mod.mlps:
            h = torch.zeros((1, seq[0].in_channels, 1, 1), device="cuda")
            with torch.no_grad():
                for layer in seq:
                    h = layer(h)
            chain.append(h.reshape(-1))
    finally:
        torch.backends.cudnn.allow_tf32 = old
    chain = torch.cat(chain)
    assert float(chain.abs().max()) > 0
    assert torch.allclose(eager[3], chain, atol=1e-5) and torch.allclose(fused[3], chain, atol=1e-5)
    # the 40 centres of the frame without points are empty balls too
    assert torch.allclose(fused[512:552], chain.expand(40, -1), atol=1e-5)


def test_stack_sa_fold_cache_and_eager_paths(monkeypatch):
    from tsmdet_b200.pointnet2_stack import pointnet2_modules as pm

    cfg = CFGS["c1"]
    mod = _module(cfg, seed=3)
    xyz, cnt, new, mcnt, feats = _sa_inputs(cfg["c"])
    _, a = _run(mod, xyz, cnt, new, mcnt, feats, fused=True)
    other = _module(cfg, seed=9)
    mod.load_state_dict(other.state_dict())
    assert mod._folded is None
    _, b = _run(mod, xyz, cnt, new, mcnt, feats, fused=True)
    _, want = _run(other, xyz, cnt, new, mcnt, feats, fused=True)
    assert torch.equal(b, want) and not torch.equal(a, b)
    mod.train()
    assert mod._folded is None
    mod.eval()

    # fused=False and train mode never reach the fused path
    calls = []
    real = pm.StackSAModuleMSG._forward_fused
    monkeypatch.setattr(pm.StackSAModuleMSG, "_forward_fused", lambda self, *a: calls.append(1) or real(self, *a))
    _run(mod, xyz, cnt, new, mcnt, feats, fused=False)
    mod.train()
    with torch.no_grad():
        mod(T(xyz), T(cnt), T(new), T(mcnt), T(feats))
    assert calls == []
    mod.eval()
    _run(mod, xyz, cnt, new, mcnt, feats, fused=True)
    assert calls == [1]


# ---------------------------------------------------------------------------------------------- head to head
@pytest.fixture(scope="module")
def ref_stack():
    from oracle import build_ref

    return build_ref.load_ref("pointnet2_stack_cuda")


@pytest.mark.parametrize("case", [c for c in ALL_CASES if c[0] != "150k-frame"], ids=lambda c: c[0])
def test_stack_ball_query_vs_reference_cuda(ref_stack, case):
    if ref_stack is None:
        pytest.skip("oracle/_ref/pointnet2_stack_cuda.so not built (needs the reference tree)")
    _, xyz, cnt, new, mcnt, radius, nsample = case
    m = new.shape[0]
    idx = torch.zeros((m, nsample), dtype=torch.int32, device="cuda")
    ref_stack.ball_query_wrapper(len(cnt), m, radius, nsample, T(new), T(mcnt), T(xyz), T(cnt), idx)
    assert np.array_equal(_query(xyz, cnt, new, mcnt, radius, nsample), idx.cpu().numpy())


def test_reference_stack_python_over_shims():
    from ref_stack_py import load_reference_stack_python

    ref = load_reference_stack_python()
    if ref is None:
        pytest.skip("the reference tree (its stack pointnet2_utils.py / pointnet2_modules.py) is not present")
    ref_utils, ref_modules = ref
    cfg = CFGS["c64"]
    xyz, cnt, new, mcnt, feats = _sa_inputs(cfg["c"])
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu

    want = pu.QueryAndGroup(1.2, 16)(T(xyz), T(cnt), T(new), T(mcnt), T(feats))
    got = ref_utils.QueryAndGroup(1.2, 16)(T(xyz), T(cnt), T(new), T(mcnt), T(feats))
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    mod = _module(cfg)
    ref_mod = ref_modules.StackSAModuleMSG(radii=cfg["radii"], nsamples=cfg["nsamples"],
                                           mlps=[list(s) for s in cfg["mlps"]]).cuda().eval()
    ref_mod.load_state_dict(mod.state_dict())
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            _, ref_out = ref_mod(T(xyz), T(cnt), T(new), T(mcnt), T(feats))
        _, eager = _run(mod, xyz, cnt, new, mcnt, feats, fused=False)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert torch.allclose(ref_out, eager, atol=1e-6, rtol=0)
    _, fused = _run(mod, xyz, cnt, new, mcnt, feats, fused=True)
    parity.check_metrics(parity.err_metrics(fused, ref_out), "fp32", "fused vs the reference module")
