"""The shared-MLP kernels through their C ABI (``sa_mlp_maxpool``, ``pointwise_mlp``, ``pack_mlp``) against the
rounding-aware float64 reference of tests/mlp_ref.py, element by element.

Inputs are synthetic: folded random weights, hand-placed ``idx`` / ``idx_cnt`` (no ball query, no BatchNorm), so every
edge a launch path has -- padded channels, tiles straddling frames, empty balls, the last point -- is there on purpose.
Every case checks (a) |kernel - reference| <= the elementwise bound B, (b) rel_l2 <= mlp_ref.REL_L2_BAR, and exactly:
the output written into a NaN-filled wider tensor at out_c0 > 0 leaves the other channels and a guard region after it
untouched; two calls are bit-identical; the pre-packed call is bit-identical to the per-call one (same kernel); the
row copy ``out_t`` is q(out) with zero padding columns, and a next layer fed ``feat_t = out_t`` is bit-identical to one
fed ``features = out``.  Every case prints max(err/B) and rel_l2 (lines starting with MLPREF).

The path each row reaches is read off ``tc2_plan_cl`` / ``tsm_mlp_tc2`` (csrc/mlp_tc2.cu) and ``tsmdet_sa_mlp_maxpool``
(csrc/sa_mlp.cu): tc2 = second-generation kernel (bf16 or tf32 operands), v1 = first-generation bf16 kernel
(sa_mlp_tc.cu: nsample < 8, or TSMDET_MLP_V1=1), fp32 = FMA kernel.  PF = feature chunks prefetched into registers
(4: <= 32 bf16 / 16 tf32 channels, 16: <= 128 bf16 / 64 tf32), planar = <= 4 channels read from the fp32 planes,
cp.async = wider rows; SC = min(nsample, 32); a tile is 128 rows, nsample-128 tiles pool across the two halves of a
row through shared memory (the exchange path)."""
import numpy as np
import pytest
import torch

import mlp_ref
from conftest import knob_setenv

pytestmark = pytest.mark.gpu

B_DEF, N_DEF = 3, 1000  # n % 64 != 0: the feature transpose has a partial tile
ROW_DT = {"bf16": (torch.bfloat16, 8), "tf32": (torch.float32, 4)}


def C(s, c, w, m=None, precs=("bf16", "tf32", "fp32"), b=B_DEF, n=N_DEF, use_xyz=True, knobs=None, cnt=True,
      empty_frame=None, chain=False):
    # m: centres per frame, default so that m % (128 / s) != 0 (tiles straddle frames)
    if m is None:
        m = {1: 90, 2: 70, 4: 50, 8: 100, 12: 50, 16: 60, 24: 30, 32: 30, 64: 15, 128: 9}[s]
    return dict(s=s, c=c, w=w, m=m, precs=precs, b=b, n=max(n, m + 17), use_xyz=use_xyz, knobs=knobs or {}, cnt=cnt,
                empty_frame=empty_frame, chain=chain)


SA = {
    # ---- nsample sweep (SC 8 / 16 / 32, nsample-128 exchange), B = 3, partial tiles straddling frames
    "ns8_c13": C(8, 13, [16, 32, 36], empty_frame=1),   # tc2 SC8, whole_tiles = 0, PF4; last cout 36 padded to 128
    "ns16_c32": C(16, 32, [64, 64, 128], chain=True),    # tc2 SC16, bf16 PF4 / tf32 PF16
    "ns32_c64": C(32, 64, [128, 128, 256], chain=True),  # tc2 SC32, two 128-channel blocks; bf16 PF16, two groups;
                                                         # tf32: 242 KB of operands -> cluster pair, PF16 split over it
    "ns64_c128": C(64, 128, [64, 200]),                  # tc2 SC32, S=64; bf16 PF16; tf32 > 64 channels: cp.async rows
    "ns128_c8": C(128, 8, [32, 128], chain=True),        # tc2 SC32, S=128 one centre per tile, NH 1
    # ---- input channels at nsample 16 (planar gather <= 4, register prefetch PF 4 / 16, cp.async > 128)
    "c0_xyz_only": C(16, 0, [16, 32]),                   # tc2, xyz chunk only, no feature rows
    "c1_planar": C(16, 1, [16, 16, 32]),                 # tc2 planar gather (fp32 planes, 1 channel)
    "c3_planar_w24": C(16, 3, [24, 40]),                 # tc2 planar, mid width 24 outside the epilogue switch
    "c4_planar_w48": C(16, 4, [48, 80, 96]),             # tc2 planar (4 channels), mid widths 48 / 80, last 96
    "c5_w8": C(16, 5, [8, 16]),                          # tc2 PF4 (transpose), mid width 8
    "c8_w256": C(16, 8, [256, 128], precs=("bf16", "fp32")),  # tc2 PF4, mid width 256, two groups (tf32: no fit)
    "c136_cpasync": C(16, 136, [64, 128], chain=True),   # tc2 > 128 (bf16) / 64 (tf32, two groups) channels: cp.async
    "c200_cpasync": C(16, 200, [96, 128], precs=("bf16", "fp32")),  # tc2 cp.async, mid width 96
    "c256_cpasync": C(8, 256, [64, 64], precs=("bf16", "fp32")),    # tc2 cp.async, K0 = 264 -> 272
    "no_xyz_c32": C(16, 32, [64, 128], use_xyz=False),   # tc2 use_xyz=False: no coordinate chunk
    "no_cnt": C(32, 13, [32, 64], cnt=False),            # idx_cnt = None: every row live
    # ---- two tile groups per CTA ([131,128,128,256] bf16: one CTA per SM, two operand buffers)
    "two_group": C(32, 128, [128, 128, 256], precs=("bf16", "fp32")),
    "two_group_one_tile": C(32, 128, [128, 128, 256], b=1, m=3, precs=("bf16",)),  # 96 rows: one tile, group 1 idle
    "two_group_knob_one": C(32, 128, [128, 128, 256], precs=("bf16",), knobs={"TSMDET_MLP_ONE_GROUP": "1"}),
    # ---- TSMDET_MLP_NH=2 on bf16 SA scales (two threads per tile row)
    "nh2_ns8": C(8, 13, [32, 64], precs=("bf16",), knobs={"TSMDET_MLP_NH": "2"}),
    "nh2_ns16": C(16, 64, [64, 128], precs=("bf16",), knobs={"TSMDET_MLP_NH": "2"}),
    "nh2_ns32": C(32, 136, [128, 256], precs=("bf16",), knobs={"TSMDET_MLP_NH": "2"}),  # NH 2 + cp.async
    "nh2_ns128": C(128, 32, [64, 256], precs=("bf16",), knobs={"TSMDET_MLP_NH": "2"}),  # halves meet in shared memory
    # ---- TSMDET_MLP_OCC=1: 4096 tiles on one CTA per SM, > 20 tiles per CTA (the mbarrier phase flips many times)
    "occ1_many_tiles": C(32, 4, [16, 32], b=4, m=4096, precs=("bf16", "tf32"), knobs={"TSMDET_MLP_OCC": "1"}),
    # ---- tf32 cluster pair: last layer 256, mid widths multiples of 32 (run-time epilogue widths 48 / 80 per CTA)
    "pair_odd_tiles": C(16, 64, [96, 160, 256], m=40, precs=("tf32",)),    # 15 tiles
    "pair_one_tile": C(16, 64, [96, 160, 256], b=1, m=8, precs=("tf32",)),  # 1 tile
    # ---- first-generation kernel: nsample < 8, and TSMDET_MLP_V1=1
    "v1_ns1": C(1, 5, [16, 32], precs=("bf16",)),
    "v1_ns2": C(2, 13, [32, 64], precs=("bf16",)),
    "v1_ns4": C(4, 3, [32, 48, 128], precs=("bf16",), empty_frame=2),
    "v1_knob_ns16": C(16, 32, [64, 64, 128], precs=("bf16",), knobs={"TSMDET_MLP_V1": "1"}),
    "v1_knob_ns32": C(32, 64, [128, 128, 256], precs=("bf16",), knobs={"TSMDET_MLP_V1": "1"}),
    "v1_knob_ns128": C(128, 8, [32, 128], precs=("bf16",), knobs={"TSMDET_MLP_V1": "1"}),
    # ---- fp32 kernel: non-power-of-two nsample (centres straddle its 64-row tiles: atomicMax pooling)
    "fp32_ns12": C(12, 5, [24, 40], precs=("fp32",)),
    "fp32_ns24": C(24, 32, [64, 128], precs=("fp32",)),
}


def _kernel(prec, case):
    if prec == "fp32":
        return "fp32"
    if prec == "bf16" and (case["s"] < 8 or case["knobs"].get("TSMDET_MLP_V1") == "1"):
        return "v1"
    return "tc2"


def D():
    return torch.device("cuda:0")


def T(x):
    return None if x is None else torch.from_numpy(np.ascontiguousarray(x)).to(D())


def _wide_out(b, cout, m, c0=3, extra=5, guard=1024):
    """(b, c0 + cout + extra, m) view of a NaN-filled buffer with a guard region after it; the layer writes out_c0 = c0."""
    ctot = c0 + cout + extra
    buf = torch.full((b * ctot * m + guard,), float("nan"), device=D())
    return buf, buf[:b * ctot * m].view(b, ctot, m), c0


def _check_untouched(buf, out, c0, cout):
    n = out.numel()
    assert bool(buf[n:].isnan().all()), "write past the end of the output"
    assert bool(out[:, :c0].isnan().all()) and bool(out[:, c0 + cout:].isnan().all()), "write outside the channel range"
    assert not bool(out[:, c0:c0 + cout].isnan().any()), "output element not written"


def _q_torch(x, prec):
    q = mlp_ref.QUANT[prec]
    return torch.from_numpy(q(x.cpu().numpy()))


def _judge(name, prec, kernel, got, want, bound):
    ratio, rel, n_out = mlp_ref.compare(got, want, bound)
    print(f"MLPREF {prec:4s} {kernel:4s} {name:24s} max err/B {ratio:.3f} rel_l2 {rel:.2e}")
    assert n_out == 0, f"{n_out} outputs outside the bound, max err/B {ratio:.3g}"
    assert rel <= mlp_ref.REL_L2_BAR[prec], rel


@pytest.mark.parametrize("name,prec", [(k, p) for k, v in SA.items() for p in v["precs"]])
def test_sa_mlp_maxpool_matches_reference(name, prec, monkeypatch):
    from tsmdet_b200.pointnet2_modules import pack_mlp, sa_mlp_maxpool

    cs = SA[name]
    for k, v in cs["knobs"].items():
        knob_setenv(monkeypatch, k, v)
    b, n, m, s, c_feat, use_xyz = cs["b"], cs["n"], cs["m"], cs["s"], cs["c"], cs["use_xyz"]
    kernel = _kernel(prec, cs)
    seed = sum(map(ord, name))
    xyz, new_xyz, feats, idx, cnt = mlp_ref.synth_sa_case(seed, b, n, m, s, c_feat, empty_frame=cs["empty_frame"])
    if not cs["cnt"]:
        cnt = None
    cin = (3 if use_xyz else 0) + c_feat
    layers = mlp_ref.synth_layers(seed + 1, [cin] + cs["w"])
    tl = [(T(w), T(bb)) for w, bb in layers]
    cout = cs["w"][-1]
    args = (T(xyz), T(new_xyz), T(feats), T(idx), T(cnt))

    packed = pack_mlp(tl, dense=False, nsample=s, c_feat=c_feat, use_xyz=use_xyz, precision=prec) if prec != "fp32" else None
    if kernel == "tc2":
        assert packed is not None, "expected the second-generation kernel to take this shape"
    if kernel == "v1" and s < 8:
        assert packed is None
    outs = []
    for _ in range(2):  # determinism
        buf, out, c0 = _wide_out(b, cout, m)
        sa_mlp_maxpool(*args, tl, out, c0, use_xyz=use_xyz, precision=prec)
        torch.cuda.synchronize()
        _check_untouched(buf, out, c0, cout)
        outs.append(out[:, c0:c0 + cout].clone())
    assert torch.equal(outs[0], outs[1]), "two calls differ"
    got = outs[0]

    rows = mlp_ref.sa_rows(xyz, new_xyz, feats, idx, cnt, use_xyz, mlp_ref.QUANT[prec])
    want, bound = mlp_ref.mlp_reference(rows, layers, s, prec, kernel)
    g = got.permute(0, 2, 1).reshape(b * m, cout).double().cpu().numpy()
    _judge(name, prec, kernel, g, want, bound)

    if packed is None or kernel != "tc2":
        return
    # the pre-packed call, with the operand-type row copy out_t
    row_dt, row_q = ROW_DT[prec]
    cpo = -(-cout // row_q) * row_q
    out_t = torch.full((b, m, cpo), float("nan"), dtype=row_dt, device=D())
    buf, out, c0 = _wide_out(b, cout, m)
    sa_mlp_maxpool(*args, tl, out, c0, use_xyz=use_xyz, precision=prec, packed=packed, out_t=out_t)
    torch.cuda.synchronize()
    _check_untouched(buf, out, c0, cout)
    assert torch.equal(out[:, c0:c0 + cout], got), "pre-packed call differs from the per-call packing"
    rows_t = out_t.float().cpu()
    assert torch.equal(rows_t[:, :, :cout], _q_torch(got.permute(0, 2, 1), prec)), "out_t != q(out)"
    assert bool((rows_t[:, :, cout:] == 0).all()), "out_t padding columns not zero"
    if not cs["chain"]:
        return
    # chaining: a next layer fed feat_t = out_t equals the same layer fed features = out, bit for bit
    m2, s2 = max(m // 2, 1), 16
    rng = np.random.default_rng(seed + 2)
    idx2 = T(rng.integers(0, m, size=(b, m2, s2)).astype(np.int32))
    cnt2 = T(rng.integers(0, 3, size=(b, m2)).astype(np.int32))
    xyz2 = args[1]
    new2 = xyz2[:, :m2].contiguous()
    l2 = [(T(w), T(bb)) for w, bb in mlp_ref.synth_layers(seed + 3, [3 + cout, 64, 256])]
    p2 = pack_mlp(l2, dense=False, nsample=s2, c_feat=cout, precision=prec)
    assert p2 is not None
    r = []
    for kw in (dict(features=got.contiguous()), dict(features=None, feat_t=out_t)):
        o = torch.empty((b, 256, m2), device=D())
        f = kw.pop("features")
        sa_mlp_maxpool(xyz2, new2, f, idx2, cnt2, l2, o, 0, precision=prec, packed=p2, **kw)
        r.append(o)
    torch.cuda.synchronize()
    assert torch.equal(r[0], r[1]), "feat_t = out_t differs from features = out"


DENSE = {
    # name: (c0, c1, n, widths, precisions, knobs); dense tc2 = two threads per tile row unless TSMDET_MLP_NH=1 (bf16)
    "c1_n1": (1, 0, 1, [16, 32], ("bf16", "tf32", "fp32"), {}),          # 3 rows: one tile across three frames
    "c5_c2_n127": (5, 2, 127, [24, 40], ("bf16", "tf32", "fp32"), {}),   # run-time epilogue width 24 / 12 per thread
    "c21_c5_n129": (21, 5, 129, [64, 36], ("bf16", "tf32", "fp32"), {}),
    "c128_c2_n2999": (128, 2, 2999, [128, 128], ("bf16", "tf32", "fp32"), {}),  # FP-module shape, partial last tile
    "c21_n2999_nh1": (21, 0, 2999, [32, 64, 200], ("bf16",), {"TSMDET_MLP_NH": "1"}),
    "c5_c5_n129_nh2": (5, 5, 129, [48, 96], ("bf16",), {"TSMDET_MLP_NH": "2"}),
    "two_group": (128, 3, 2999, [128, 128, 256], ("bf16", "fp32"), {}),  # [131,128,128,256]: two tile groups
}


@pytest.mark.parametrize("name,prec", [(k, p) for k, v in DENSE.items() for p in v[4]])
def test_pointwise_mlp_matches_reference(name, prec, monkeypatch):
    from tsmdet_b200.pointnet2_modules import pack_mlp, pointwise_mlp

    c0, c1, n, widths, _, knobs = DENSE[name]
    for k, v in knobs.items():
        knob_setenv(monkeypatch, k, v)
    b = B_DEF
    seed = sum(map(ord, name)) + 7
    rng = np.random.default_rng(seed)
    src0 = rng.standard_normal((b, c0, n)).astype(np.float32)
    src1 = rng.standard_normal((b, c1, n)).astype(np.float32) if c1 else None
    layers = mlp_ref.synth_layers(seed + 1, [c0 + c1] + widths)
    tl = [(T(w), T(bb)) for w, bb in layers]
    cout = widths[-1]
    packed = pack_mlp(tl, dense=True, c_feat=c0, c1=c1, precision=prec) if prec != "fp32" else None
    if prec != "fp32":
        assert packed is not None
    outs = []
    for pk in (None, None, packed):
        if pk is None and len(outs) == 2:
            break
        buf, out, oc0 = _wide_out(b, cout, n)
        pointwise_mlp(T(src0), T(src1), tl, out=out, out_c0=oc0, precision=prec, packed=pk)
        torch.cuda.synchronize()
        _check_untouched(buf, out, oc0, cout)
        outs.append(out[:, oc0:oc0 + cout].clone())
    assert torch.equal(outs[0], outs[1]), "two calls differ"
    if len(outs) == 3:
        assert torch.equal(outs[0], outs[2]), "pre-packed call differs from the per-call packing"
    kernel = "fp32" if prec == "fp32" else "tc2"
    want, bound = mlp_ref.mlp_reference(mlp_ref.dense_rows(src0, src1, mlp_ref.QUANT[prec]), layers, 1, prec, kernel)
    g = outs[0].permute(0, 2, 1).reshape(b * n, cout).double().cpu().numpy()
    _judge("dense_" + name, prec, kernel, g, want, bound)
