"""GPU suite of the stacked (ragged) three_nn / three_interpolate and StackPointnetFPModule (pointnet2_stack):

  * three_nn_wrapper bit-exact (idx and the dist2 bits) against the CPU oracle (tests/stack_nn_oracle.py) on the frames of
    tests/stack_cases.py, ragged frames with 0 / 1 / 2 known points and without unknown points, frames the grid cannot
    take (a non-finite coordinate, a pile of > 256 points in one cell), lattice and duplicate ties, unknown points far
    outside their frame and a 150k-point frame; the grid against TSMDET_NN_ALGO=brute on all of them;
  * three_interpolate bit-exact against the oracle, the (C,N) planes output against the rows, the gradient against a
    float64 index_add, and an empty last known frame (no read out of bounds, NaN rows as the reference's module gives);
  * StackPointnetFPModule: eager against a plain-torch restatement, fused fp32 / bf16 / tf32 against eager
    (tests/parity.py bars) and element by element against the float64 reference of tests/mlp_ref.py, the NaN rows of an
    empty known frame, the fold cache and the eager paths of train mode / fused=False;
  * head to head against the reference's own stack wrappers (oracle/_ref/pointnet2_stack_cuda.so) and its stack Python
    over this package's shim, when those are built."""
import numpy as np
import pytest
import torch
from conftest import knob_setenv

import mlp_ref
import parity
import stack_cases
import stack_nn_oracle as sno
import synth

pytestmark = pytest.mark.gpu


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _three_nn(unknown, ucnt, known, kcnt):
    from tsmdet_b200.pointnet2_stack import pointnet2_stack_cuda as ps

    n = unknown.shape[0]
    d2 = torch.full((n, 3), -3.0, device="cuda")
    idx = torch.full((n, 3), -7, dtype=torch.int32, device="cuda")
    assert ps.three_nn_wrapper(T(unknown), T(ucnt), T(known), T(kcnt), d2, idx) is None
    return d2.cpu().numpy(), idx.cpu().numpy()


def _small_frames(seed=0):
    """frames with 3000 / 0 / 1 / 2 / 2500 known points; the frame with 2 known points has no unknown points"""
    rng = np.random.default_rng(seed)
    big = synth.cloud_ground_objects(1, 3000, seed=seed)[0]
    big2 = synth.cloud_ground_objects(1, 2500, seed=seed + 1)[0]
    fk = [big, np.zeros((0, 3), np.float32), rng.uniform(-3, 3, (1, 3)), rng.uniform(-3, 3, (2, 3)), big2]
    fu = [stack_cases.centres_from(rng, big, 700, jitter=2.0), rng.uniform(-5, 5, (40, 3)), rng.uniform(-3, 3, (30, 3)),
          np.zeros((0, 3), np.float32), stack_cases.centres_from(rng, big2, 500, jitter=2.0)]
    known, kcnt, unknown, ucnt = stack_cases.stack(fk, fu)
    return unknown, ucnt, known, kcnt


def _nn_cases():
    rng = np.random.default_rng(5)
    out = []
    for cid, xyz, cnt, new, mcnt, *_ in stack_cases.cases():
        if cid in ("ragged-r0.8-ns1", "dup-padded-r0.4-ns16", "lattice-r0.5-ns7"):
            out.append((cid.split("-r")[0], new, mcnt, xyz, cnt))  # known = xyz, unknown = new_xyz
    out.append(("small-frames", *_small_frames()))
    base = synth.cloud_ground_objects(1, 3000, seed=21)[0]
    pile = base.copy()
    pile[100:700] = pile[50] + rng.uniform(-1e-3, 1e-3, size=(600, 3)).astype(np.float32)  # > 256 in one cell
    bad = base.copy()
    bad[17, 1] = np.nan
    bad[29, 2] = np.inf
    fk = [base, pile, bad]
    fu = [stack_cases.centres_from(rng, f[np.isfinite(f).all(1)], 300) for f in fk]
    fu[1][:50] = pile[50]
    known, kcnt, unknown, ucnt = stack_cases.stack(fk, fu)
    out.append(("grid-unusable-frames", unknown, ucnt, known, kcnt))
    far = [stack_cases.centres_from(rng, base, 200) + np.float32(500.0), rng.uniform(-1e4, 1e4, (200, 3))]
    known, kcnt, unknown, ucnt = stack_cases.stack([base, base[::-1].copy()], far)
    out.append(("far-outside", unknown, ucnt, known, kcnt))
    g = np.arange(-4, 4, dtype=np.float32) * 0.5  # lattice unknown points midway between lattice known points: 3-way ties
    lat = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    dup = np.repeat(lat[::3], 3, 0)  # every point three times
    known, kcnt, unknown, ucnt = stack_cases.stack([lat, dup], [lat + np.float32(0.25), dup[::2] + np.float32(0.1)])
    out.append(("lattice-duplicate-ties", unknown, ucnt, known, kcnt))
    big = synth.cloud_ground_objects(1, 150000, seed=22)[0]
    known, kcnt, unknown, ucnt = stack_cases.stack([big, base], [stack_cases.centres_from(rng, big, 20000),
                                                                 stack_cases.centres_from(rng, base, 500)])
    out.append(("150k-frame", unknown, ucnt, known, kcnt))
    return out


NN_CASES = _nn_cases()


def _bits_equal(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


@pytest.mark.parametrize("case", NN_CASES, ids=lambda c: c[0])
def test_stack_three_nn_matches_oracle(case):
    _, unknown, ucnt, known, kcnt = case
    wd, wi = sno.stack_three_nn(unknown, ucnt, known, kcnt)
    d2, idx = _three_nn(unknown, ucnt, known, kcnt)
    bad = (idx != wi).any(1) | ~(d2.view(np.uint32) == wd.view(np.uint32)).all(1)
    assert not bad.any(), f"{int(bad.sum())} rows differ, first {np.flatnonzero(bad)[:5]}"


@pytest.mark.parametrize("case", NN_CASES, ids=lambda c: c[0])
def test_stack_three_nn_grid_equals_brute(monkeypatch, case):
    _, unknown, ucnt, known, kcnt = case
    grid = _three_nn(unknown, ucnt, known, kcnt)
    knob_setenv(monkeypatch, "TSMDET_NN_ALGO", "brute")
    brute = _three_nn(unknown, ucnt, known, kcnt)
    assert np.array_equal(grid[1], brute[1]) and _bits_equal(grid[0], brute[0])


def test_three_nn_python_returns_sqrt():
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu

    _, unknown, ucnt, known, kcnt = NN_CASES[0]
    dist, idx = pu.three_nn(T(unknown), T(ucnt), T(known), T(kcnt))
    wd, wi = sno.stack_three_nn(unknown, ucnt, known, kcnt)
    assert idx.dtype == torch.int32 and np.array_equal(idx.cpu().numpy(), wi)
    assert torch.equal(dist, torch.sqrt(T(wd)))


# ---------------------------------------------------------------------------------------------- three_interpolate
def _interp_inputs(c, seed=1):
    _, unknown, ucnt, known, kcnt = NN_CASES[3]  # small-frames: 0 / 1 / 2 known points included
    rng = np.random.default_rng(seed)
    _, idx = sno.stack_three_nn(unknown, ucnt, known, kcnt)
    w = rng.random(idx.shape).astype(np.float32)
    feats = rng.standard_normal((known.shape[0], c)).astype(np.float32)
    return feats, idx, w


def _interp(feats, idx, w, planes):
    from tsmdet_b200._lib import call, ptr, stream_ptr

    n, c = idx.shape[0], feats.shape[1]
    out = torch.full((c, n) if planes else (n, c), -9.0, device="cuda")
    tf, ti, tw = T(feats), T(idx), T(w)
    call("tsmdet_stack_three_interpolate", n, c, feats.shape[0], ptr(tf), ptr(ti), ptr(tw), ptr(out), int(planes),
         stream_ptr())
    return out.cpu().numpy()


@pytest.mark.parametrize("c", [1, 3, 32, 45, 128, 300])
def test_stack_three_interpolate_matches_oracle(c):
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu

    feats, idx, w = _interp_inputs(c)
    want = sno.stack_three_interpolate(feats, idx, w)
    got = pu.three_interpolate(T(feats), T(idx), T(w))
    assert got.shape == want.shape and _bits_equal(got.cpu().numpy(), want)
    assert _bits_equal(_interp(feats, idx, w, planes=True), want.T)


def test_stack_three_interpolate_backward():
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu

    feats, idx, w = _interp_inputs(40)
    tf = T(feats).requires_grad_(True)
    out = pu.three_interpolate(tf, T(idx), T(w))
    go = torch.randn_like(out)
    out.backward(go)
    want = torch.zeros(feats.shape, dtype=torch.float64, device="cuda")
    for s in range(3):
        want.index_add_(0, T(idx[:, s]).long(), go.double() * T(w[:, s:s + 1]).double())
    assert torch.allclose(tf.grad.double(), want, rtol=1e-5, atol=1e-6)


def _empty_last_known_frame():
    """the last frame with known points is frame 1; frames 2 and 3 have unknown points but no known points, so their
    idx is the known start M: one past the last row"""
    rng = np.random.default_rng(9)
    a, b = synth.cloud_ground_objects(1, 900, seed=3)[0], synth.cloud_ground_objects(1, 700, seed=4)[0]
    fk = [a, b, np.zeros((0, 3), np.float32), np.zeros((0, 3), np.float32)]
    fu = [stack_cases.centres_from(rng, a, 300), stack_cases.centres_from(rng, b, 200), rng.uniform(-5, 5, (64, 3)),
          rng.uniform(-5, 5, (33, 3))]
    known, kcnt, unknown, ucnt = stack_cases.stack(fk, fu)
    return unknown, ucnt, known, kcnt


def test_stack_three_interpolate_empty_last_known_frame():
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu

    unknown, ucnt, known, kcnt = _empty_last_known_frame()
    m = known.shape[0]
    dist, idx = pu.three_nn(T(unknown), T(ucnt), T(known), T(kcnt))
    empty = slice(500, None)
    assert (idx[empty] == m).all() and torch.isinf(dist[empty]).all()
    # the module's weights: 0/0 = NaN rows; the out-of-range index reads 0, so no read past the features
    w = 1.0 / (dist + 1e-8)
    w = w / w.sum(-1, keepdim=True)
    feats = torch.randn((m, 24), device="cuda")
    out = pu.three_interpolate(feats, idx, w)
    torch.cuda.synchronize()
    assert torch.isnan(out[empty]).all() and not torch.isnan(out[:500]).any()
    want = sno.stack_three_interpolate(feats.cpu().numpy(), idx.cpu().numpy(), w.cpu().numpy())
    np.testing.assert_array_equal(out.cpu().numpy(), want)  # (NaN payloads may differ between CPU and GPU)
    # finite weights on the same indices: the guard reads zeros
    ones = torch.ones_like(w)
    assert (pu.three_interpolate(feats, idx, ones)[empty] == 0).all()
    g = torch.zeros_like(feats)
    from tsmdet_b200.pointnet2_stack import pointnet2_stack_cuda as ps

    ps.three_interpolate_grad_wrapper(torch.ones((idx.shape[0], 24), device="cuda"), idx, ones, g)
    want_g = torch.zeros_like(g).index_add_(0, idx[:500].reshape(-1).long(), torch.ones((1500, 24), device="cuda"))
    assert torch.equal(g, want_g)


# ---------------------------------------------------------------------------------------------- StackPointnetFPModule
def _randomise_bn(mod, seed):
    g = torch.Generator().manual_seed(seed)
    for m in mod.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.1)


# (C2 known feature channels, C1 skip channels | 0 for unknown_feats=None, mlp after the input width)
FP_CFGS = {
    "c128_c64": (128, 64, [128, 128]),
    "c4_none": (4, 0, [32, 16]),
    "c3_c5": (3, 5, [24]),
    "c256_c32": (256, 32, [256, 64]),
}


def _fp_inputs(c2, c1, seed=7):
    rng = np.random.default_rng(seed)
    ksz, usz = [2000, 0, 1500, 2600], [8000, 0, 6000, 9000]
    fk = [synth.cloud_ground_objects(1, k, seed=seed + i)[0] if k else np.zeros((0, 3), np.float32)
          for i, k in enumerate(ksz)]
    fu = [stack_cases.centres_from(rng, f, u, jitter=1.0) if u else np.zeros((0, 3), np.float32)
          for f, u in zip(fk, usz)]
    known, kcnt, unknown, ucnt = stack_cases.stack(fk, fu)
    kf = rng.standard_normal((known.shape[0], c2)).astype(np.float32)
    uf = rng.standard_normal((unknown.shape[0], c1)).astype(np.float32) if c1 else None
    return unknown, ucnt, known, kcnt, uf, kf


def _fp_module(c2, c1, spec, precision="fp32", seed=0):
    from tsmdet_b200.pointnet2_stack import StackPointnetFPModule

    torch.manual_seed(seed)
    mod = StackPointnetFPModule(mlp=[c2 + c1] + spec, precision=precision).cuda().eval()
    _randomise_bn(mod, seed + 1)
    return mod


def _fp_run(mod, inputs, fused):
    unknown, ucnt, known, kcnt, uf, kf = inputs
    mod.fused = fused
    with torch.no_grad():
        return mod(T(unknown), T(ucnt), T(known), T(kcnt), None if uf is None else T(uf), T(kf))


def _eager_fp32(mod, inputs):
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        return _fp_run(mod, inputs, fused=False)
    finally:
        torch.backends.cudnn.allow_tf32 = old


@pytest.mark.parametrize("name", list(FP_CFGS))
def test_stack_fp_eager_matches_torch_restatement(name):
    c2, c1, spec = FP_CFGS[name]
    mod = _fp_module(c2, c1, spec)
    assert list(mod.state_dict())[:2] == ["mlp.0.weight", "mlp.1.weight"]
    inputs = _fp_inputs(c2, c1)
    unknown, ucnt, known, kcnt, uf, kf = inputs
    got = _eager_fp32(mod, inputs)
    d2, idx = sno.stack_three_nn(unknown, ucnt, known, kcnt)
    dist = torch.sqrt(T(d2))
    w = 1.0 / (dist + 1e-8)
    w = w / torch.sum(w, dim=-1, keepdim=True)
    ti = T(idx).long()
    x = sum(w[:, s:s + 1] * T(kf)[ti[:, s]] for s in (1, 0, 2))
    if uf is not None:
        x = torch.cat([x, T(uf)], 1)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            want = mod.mlp(x.t()[None, :, :, None])[0, :, :, 0].t()
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert got.shape == (unknown.shape[0], spec[-1])
    assert torch.allclose(got, want, atol=1e-4, rtol=1e-4)
    assert not torch.isnan(got).any()  # no frame here has unknown points without known points


@pytest.mark.parametrize("name,precision", [(k, p) for k in FP_CFGS for p in ("fp32", "bf16", "tf32")])
def test_stack_fp_fused_matches_eager_and_reference(name, precision):
    from tsmdet_b200.pointnet2_stack.pointnet2_modules import _dense_precision

    c2, c1, spec = FP_CFGS[name]
    mod = _fp_module(c2, c1, spec, precision)
    inputs = _fp_inputs(c2, c1)
    unknown, ucnt, known, kcnt, uf, kf = inputs
    want = _eager_fp32(mod, inputs)
    got = _fp_run(mod, inputs, fused=True)
    again = _fp_run(mod, inputs, fused=True)
    torch.cuda.synchronize()
    assert torch.equal(got, again)
    assert got.shape == want.shape and got.is_contiguous()
    m = parity.err_metrics(got, want)
    print(f"STACKFP {name} {precision}: {m}")
    parity.check_metrics(m, precision, f"{name} fused {precision} vs eager")

    # element by element: the MLP input the fused kernel sees (interpolated planes from the oracle, skip planes)
    img = mod._packed[1]
    prec = _dense_precision(precision, img)
    kernel = "fp32" if prec == "fp32" else "tc2"
    d2, idx = sno.stack_three_nn(unknown, ucnt, known, kcnt)
    dist = torch.sqrt(T(d2))
    w = 1.0 / (dist + 1e-8)
    w = (w / torch.sum(w, dim=-1, keepdim=True)).cpu().numpy()
    src0 = sno.stack_three_interpolate(kf, idx, w).T[None]
    rows = mlp_ref.dense_rows(src0, None if uf is None else uf.T[None], mlp_ref.QUANT[prec])
    lnp = [(wt.cpu().numpy(), b.cpu().numpy()) for wt, b in mod._folded]
    want_k, bound = mlp_ref.mlp_reference(rows, lnp, 1, prec, kernel)
    ratio, rel, n_out = mlp_ref.compare(got.double().cpu().numpy(), want_k, bound)
    print(f"MLPREF stackfp {name} {precision}->{prec} {kernel}: max err/B {ratio:.3f} rel_l2 {rel:.2e}")
    assert n_out == 0 and ratio <= 1.0, (ratio, n_out)
    assert rel <= mlp_ref.REL_L2_BAR[prec], rel


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_stack_fp_nan_rows_of_empty_known_frame(precision):
    unknown, ucnt, known, kcnt = _empty_last_known_frame()
    rng = np.random.default_rng(2)
    inputs = (unknown, ucnt, known, kcnt, rng.standard_normal((unknown.shape[0], 8)).astype(np.float32),
              rng.standard_normal((known.shape[0], 16)).astype(np.float32))
    mod = _fp_module(16, 8, [32, 32], precision)
    eager = _eager_fp32(mod, inputs)
    fused = _fp_run(mod, inputs, fused=True)
    for out in (eager, fused):
        assert torch.isnan(out[500:]).all() and not torch.isnan(out[:500]).any()
    parity.check_metrics(parity.err_metrics(fused[:500], eager[:500]), precision, "fused vs eager, populated frames")


def test_stack_fp_fold_cache_and_eager_paths(monkeypatch):
    from tsmdet_b200.pointnet2_stack import pointnet2_modules as pm

    c2, c1, spec = FP_CFGS["c128_c64"]
    mod = _fp_module(c2, c1, spec, seed=3)
    inputs = _fp_inputs(c2, c1)
    a = _fp_run(mod, inputs, fused=True)
    other = _fp_module(c2, c1, spec, seed=9)
    mod.load_state_dict(other.state_dict())
    assert mod._folded is None
    b = _fp_run(mod, inputs, fused=True)
    want = _fp_run(other, inputs, fused=True)
    assert torch.equal(b, want) and not torch.equal(a, b)
    mod.train()
    assert mod._folded is None
    mod.eval()

    calls = []
    real = pm.StackPointnetFPModule._forward_fused
    monkeypatch.setattr(pm.StackPointnetFPModule, "_forward_fused", lambda self, *a: calls.append(1) or real(self, *a))
    _fp_run(mod, inputs, fused=False)
    mod.train()
    unknown, ucnt, known, kcnt, uf, kf = inputs
    tk = T(kf).requires_grad_(True)
    out = mod(T(unknown), T(ucnt), T(known), T(kcnt), T(uf), tk)
    out.sum().backward()  # train mode runs the autograd path, three_interpolate's backward included
    assert tk.grad is not None and torch.isfinite(tk.grad).all()
    assert calls == []
    mod.eval()
    _fp_run(mod, inputs, fused=True)
    assert calls == [1]


# ---------------------------------------------------------------------------------------------- head to head
@pytest.fixture(scope="module")
def ref_stack():
    from oracle import build_ref

    return build_ref.load_ref("pointnet2_stack_cuda")


def _every_unknown_frame_has_known(case):
    _, _, ucnt, _, kcnt = case
    return bool(((ucnt == 0) | (kcnt > 0)).all())


# the reference's interpolation reads out of bounds for unknown points of a frame without known points: never feed it one
@pytest.mark.parametrize("case", [c for c in NN_CASES if c[0] != "150k-frame" and _every_unknown_frame_has_known(c)],
                         ids=lambda c: c[0])
def test_stack_three_nn_interpolate_vs_reference_cuda(ref_stack, case):
    if ref_stack is None:
        pytest.skip("oracle/_ref/pointnet2_stack_cuda.so not built (needs the reference tree)")
    _, unknown, ucnt, known, kcnt = case
    n = unknown.shape[0]
    d2 = torch.zeros((n, 3), device="cuda")
    idx = torch.zeros((n, 3), dtype=torch.int32, device="cuda")
    ref_stack.three_nn_wrapper(T(unknown), T(ucnt), T(known), T(kcnt), d2, idx)
    got_d2, got_idx = _three_nn(unknown, ucnt, known, kcnt)
    assert np.array_equal(got_idx, idx.cpu().numpy()) and _bits_equal(got_d2, d2.cpu().numpy())
    feats = torch.randn((known.shape[0], 33), device="cuda")
    w = torch.rand((n, 3), device="cuda")
    out = torch.zeros((n, 33), device="cuda")
    ref_stack.three_interpolate_wrapper(feats, idx, w, out)
    assert _bits_equal(_interp(feats.cpu().numpy(), idx.cpu().numpy(), w.cpu().numpy(), planes=False),
                       out.cpu().numpy())
    go = torch.randn((n, 33), device="cuda")
    g_ref, g = torch.zeros_like(feats), torch.zeros_like(feats)
    ref_stack.three_interpolate_grad_wrapper(go, idx, w, g_ref)
    from tsmdet_b200.pointnet2_stack import pointnet2_stack_cuda as ps

    ps.three_interpolate_grad_wrapper(go, idx, w, g)
    assert torch.allclose(g, g_ref, rtol=1e-5, atol=1e-6)


def test_reference_stack_fp_python_over_shims():
    from ref_stack_py import load_reference_stack_python

    ref = load_reference_stack_python()
    if ref is None:
        pytest.skip("the reference tree (its stack pointnet2_utils.py / pointnet2_modules.py) is not present")
    ref_utils, ref_modules = ref
    c2, c1, spec = FP_CFGS["c128_c64"]
    inputs = _fp_inputs(c2, c1)
    unknown, ucnt, known, kcnt, uf, kf = inputs
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu

    want = pu.three_nn(T(unknown), T(ucnt), T(known), T(kcnt))
    got = ref_utils.three_nn(T(unknown), T(ucnt), T(known), T(kcnt))
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    mod = _fp_module(c2, c1, spec)
    ref_mod = ref_modules.StackPointnetFPModule(mlp=[c2 + c1] + spec).cuda().eval()
    ref_mod.load_state_dict(mod.state_dict())
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            ref_out = ref_mod(T(unknown), T(ucnt), T(known), T(kcnt), T(uf), T(kf))
        eager = _fp_run(mod, inputs, fused=False)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert torch.allclose(ref_out, eager, atol=1e-6, rtol=0)
    fused = _fp_run(mod, inputs, fused=True)
    parity.check_metrics(parity.err_metrics(fused, ref_out), "fp32", "fused vs the reference module")
