"""Width-class tiles of the fused SA MLP (csrc/mlp_tc2.cu): a centre whose idx slots from w = 2^k on repeat slots
0 .. w-1 -- next_pow2(cnt) under the batch ball query's cyclic padding row[j] = row[j mod cnt], next_pow2(t) when slots
t.. repeat slot 0 -- is computed on w rows instead of nsample.  Dropped rows are byte copies of kept rows, so the result
must be BIT-IDENTICAL to the fixed-width tiles that TSMDET_MLP_WIDTH=fixed selects -- for every class mix, both operand types,
one and two threads per tile row, the tf32 cluster pair and the nsample-128 exchange -- and stay within the rounding-
aware float64 reference of tests/mlp_ref.py.  The classes are sorted on the device, so a captured CUDA graph replayed on
new neighbour lists must follow them."""
import numpy as np
import pytest
import torch

import mlp_ref
from conftest import knob_delenv, knob_setenv

pytestmark = pytest.mark.gpu

ROW_DT = {"bf16": (torch.bfloat16, 8), "tf32": (torch.float32, 4)}


def D():
    return torch.device("cuda:0")


def T(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(D())


def _inputs(kind, seed, b, n, m, s, c_feat):
    """xyz, new_xyz, features, idx, idx_cnt (numpy) with the neighbour lists of `kind`."""
    xyz, new_xyz, feats, idx, cnt = mlp_ref.synth_sa_case(seed, b, n, m, s, c_feat)
    rng = np.random.default_rng(seed + 5)
    if kind == "width1":  # every ball holds one point: all slots repeat slot 0
        idx = np.repeat(idx[:, :, :1], s, axis=2)
        cnt = np.ones((b, m), np.int32)
    elif kind == "full":  # every ball full: nsample distinct neighbours
        idx = np.stack([rng.permutation(n)[:m * s].reshape(m, s) for _ in range(b)]).astype(np.int32)
        cnt = np.full((b, m), s, np.int32)
    elif kind == "cyclic":  # the batch ball query's padding: row[j] = row[j mod cnt]
        idx = idx[:, :, :1] + np.zeros_like(idx)
        for p in range(m):
            for bi in range(b):
                c = int(cnt[bi, p])
                if c > 0:
                    idx[bi, p] = np.resize(rng.permutation(n)[:c], s)
    elif kind == "empty":  # many empty balls (rows zeroed), the rest of one hit
        idx = np.repeat(idx[:, :, :1], s, axis=2)
        cnt = (rng.random((b, m)) < 0.5).astype(np.int32)
    # "mixed": synth_sa_case as is -- random hit counts, some empty balls, and every eighth centre's LAST slot is the
    # frame's last point (full width whatever its count says)
    return xyz, new_xyz, feats, np.ascontiguousarray(idx, dtype=np.int32), np.ascontiguousarray(cnt, dtype=np.int32)


def _run(args, tl, s, c_feat, prec, packed, cout, m, b):
    row_dt, row_q = ROW_DT[prec]
    out = torch.full((b, cout, m), float("nan"), device=D())
    out_t = torch.full((b, m, -(-cout // row_q) * row_q), float("nan"), dtype=row_dt, device=D())
    from tsmdet_b200.pointnet2_modules import sa_mlp_maxpool

    sa_mlp_maxpool(*args, tl, out, 0, precision=prec, packed=packed, out_t=out_t)
    torch.cuda.synchronize()
    return out, out_t


def _both(monkeypatch, args, tl, s, c_feat, prec, cout, m, b):
    from tsmdet_b200.pointnet2_modules import pack_mlp

    packed = pack_mlp(tl, dense=False, nsample=s, c_feat=c_feat, precision=prec)
    assert packed is not None, "the second-generation kernel should take this shape"
    knob_setenv(monkeypatch, "TSMDET_MLP_WIDTH", "classes")  # the call fails rather than run fixed-width tiles
    classed = _run(args, tl, s, c_feat, prec, packed, cout, m, b)
    knob_setenv(monkeypatch, "TSMDET_MLP_WIDTH", "fixed")
    fixed = _run(args, tl, s, c_feat, prec, packed, cout, m, b)
    knob_delenv(monkeypatch, "TSMDET_MLP_WIDTH")
    return classed, fixed


def _assert_same(classed, fixed):
    for got, want in zip(classed, fixed):
        assert not bool(got.float().isnan().any()), "output element not written"
        assert torch.equal(got.view(torch.int16) if got.dtype == torch.bfloat16 else got.view(torch.int32),
                           want.view(torch.int16) if want.dtype == torch.bfloat16 else want.view(torch.int32)), \
            f"width classes differ from fixed-width tiles in {int((got != want).sum())} elements"


# name: (kind, nsample, c_feat, widths, b, m, precisions, knobs)
CASES = {
    "width1_ns16": ("width1", 16, 1, [16, 16, 32], 3, 300, ("bf16", "tf32"), {}),
    "full_ns16": ("full", 16, 1, [16, 16, 32], 2, 64, ("bf16", "tf32"), {}),
    "mixed_ns8": ("mixed", 8, 13, [16, 32, 36], 3, 100, ("bf16", "tf32"), {}),
    "mixed_ns16": ("mixed", 16, 32, [64, 64, 128], 3, 70, ("bf16", "tf32"), {}),
    "mixed_ns32": ("mixed", 32, 32, [64, 64, 128], 4, 257, ("bf16", "tf32"), {}),
    "empty_ns32": ("empty", 32, 4, [32, 64], 3, 90, ("bf16", "tf32"), {}),
    "cyclic_ns16": ("cyclic", 16, 32, [64, 64, 128], 3, 70, ("bf16", "tf32"), {}),
    "cyclic_ns32": ("cyclic", 32, 128, [128, 128, 256], 3, 130, ("bf16", "tf32"), {}),
    "full_ns32": ("full", 32, 32, [64, 64, 128], 2, 50, ("bf16",), {}),
    "mixed_ns64": ("mixed", 64, 8, [32, 128], 3, 15, ("bf16", "tf32"), {}),
    "mixed_ns128": ("mixed", 128, 8, [32, 128], 3, 9, ("bf16", "tf32"), {}),
    # two threads per tile row, incl. the halves of a 128-row centre meeting in shared memory
    "nh2_mixed_ns16": ("mixed", 16, 64, [64, 128], 3, 60, ("bf16",), {"TSMDET_MLP_NH": "2"}),
    "nh2_mixed_ns32": ("mixed", 32, 136, [128, 256], 3, 30, ("bf16",), {"TSMDET_MLP_NH": "2"}),
    "nh2_mixed_ns128": ("mixed", 128, 32, [64, 256], 3, 9, ("bf16",), {"TSMDET_MLP_NH": "2"}),
    # SA layer 3 of the KITTI stack: two tile groups (bf16), the cluster pair (tf32)
    "l3_mixed_ns32": ("mixed", 32, 128, [128, 128, 256], 3, 130, ("bf16", "tf32"), {}),
    "l3_width1_ns32": ("width1", 32, 128, [128, 128, 256], 2, 512, ("bf16", "tf32"), {}),
    "l3_full_ns32": ("full", 32, 128, [128, 128, 256], 1, 40, ("bf16", "tf32"), {}),
    # many tiles per CTA (one resident CTA per SM): the loop over the device-side tile count
    "occ1_width1": ("width1", 16, 4, [16, 32], 4, 4096, ("bf16",), {"TSMDET_MLP_OCC": "1"}),
}


@pytest.mark.parametrize("name,prec", [(k, p) for k, v in CASES.items() for p in v[6]])
def test_width_classes_bitwise_equal_fixed(name, prec, monkeypatch):
    kind, s, c_feat, widths, b, m, _, knobs = CASES[name]
    for k, v in knobs.items():
        knob_setenv(monkeypatch, k, v)
    seed = sum(map(ord, name))
    n = max(1000, m * s + 17)
    xyz, new_xyz, feats, idx, cnt = _inputs(kind, seed, b, n, m, s, c_feat)
    layers = mlp_ref.synth_layers(seed + 1, [3 + c_feat] + widths)
    tl = [(T(w), T(bb)) for w, bb in layers]
    args = (T(xyz), T(new_xyz), T(feats) if feats is not None else None, T(idx), T(cnt))
    classed, fixed = _both(monkeypatch, args, tl, s, c_feat, prec, widths[-1], m, b)
    _assert_same(classed, fixed)
    if kind in ("mixed", "cyclic"):  # and element by element against the float64 reference
        rows = mlp_ref.sa_rows(xyz, new_xyz, feats, idx, cnt, True, mlp_ref.QUANT[prec])
        want, bound = mlp_ref.mlp_reference(rows, layers, s, prec, "tc2")
        got = classed[0].permute(0, 2, 1).reshape(b * m, widths[-1]).double().cpu().numpy()
        ratio, rel, n_out = mlp_ref.compare(got, want, bound)
        print(f"MLPREF {prec:4s} tc2w {name:24s} max err/B {ratio:.3f} rel_l2 {rel:.2e}")
        assert n_out == 0 and rel <= mlp_ref.REL_L2_BAR[prec], (ratio, rel)


@pytest.mark.parametrize("prec", ["bf16", "tf32"])
def test_width_classes_ball_query_duplicate_points(prec, monkeypatch):
    """Neighbour lists from the ball query on clouds padded by repeating their points (duplicate coordinates under
    different indices): the classes follow the hit counts, frames of 2 000 centres make tiles straddle frames."""
    from tsmdet_b200 import pointnet2_utils

    rng = np.random.default_rng(11)
    b, n0, rep, m, s = 3, 3000, 3, 2000, 16
    base = rng.uniform(-20, 20, size=(b, n0, 3)).astype(np.float32)
    xyz = T(np.concatenate([base] * rep, axis=1))
    new_xyz = xyz[:, :m].contiguous()
    feats = T(rng.standard_normal((b, 8, n0 * rep)).astype(np.float32))
    cnt, idx = pointnet2_utils.ball_query(0.8, s, xyz, new_xyz)
    layers = mlp_ref.synth_layers(5, [3 + 8, 32, 64])
    tl = [(T(w), T(bb)) for w, bb in layers]
    classed, fixed = _both(monkeypatch, (xyz, new_xyz, feats, idx, cnt), tl, s, 8, prec, 64, m, b)
    _assert_same(classed, fixed)


def test_width_classes_follow_new_inputs_in_a_captured_graph(monkeypatch):
    """One captured call replayed on neighbour lists of other class mixes equals eager fixed-width calls bit for bit:
    the tile table is built on the device each replay."""
    from tsmdet_b200.pointnet2_modules import pack_mlp, sa_mlp_maxpool

    b, m, s, c_feat, n = 2, 600, 32, 32, 20000
    layers = mlp_ref.synth_layers(3, [3 + c_feat, 64, 64, 128])
    tl = [(T(w), T(bb)) for w, bb in layers]
    packed = pack_mlp(tl, dense=False, nsample=s, c_feat=c_feat, precision="bf16")
    sets = [_inputs(kind, 20 + i, b, n, m, s, c_feat) for i, kind in enumerate(("mixed", "width1", "full", "empty", "cyclic"))]
    static = [T(a) for a in sets[0]]
    knob_setenv(monkeypatch, "TSMDET_MLP_WIDTH", "classes")
    out = torch.empty((b, 128, m), device=D())
    call = lambda: sa_mlp_maxpool(*static, tl, out, 0, precision="bf16", packed=packed)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        call()  # warm-up on the capture stream: its scratch buffers are allocated outside the capture
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        call()
    for arrs in sets[1:] + sets[:1]:
        for dst, src in zip(static, arrs):
            dst.copy_(T(src))
        g.replay()
        torch.cuda.synchronize()
        got = out.clone()
        knob_setenv(monkeypatch, "TSMDET_MLP_WIDTH", "fixed")
        want, _ = _run(tuple(static), tl, s, c_feat, "bf16", packed, 128, m, b)
        knob_setenv(monkeypatch, "TSMDET_MLP_WIDTH", "classes")
        assert torch.equal(got.view(torch.int32), want.view(torch.int32))
