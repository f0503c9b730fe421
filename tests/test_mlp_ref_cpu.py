"""The float64 shared-MLP reference and its elementwise bound (tests/mlp_ref.py), tested on their own, without a GPU.

A numpy model of the kernels -- exact operand products, fp32 accumulation in a random order, the bias as the hi + lo
K step (second-generation kernel) or an fp32 add (first-generation and fp32 kernels) -- must satisfy the two checks a
kernel is held to against the reference: (a) every output within the bound, (b) rel_l2 under the precision's bar.  Numeric mutants of the model
(the bugs those checks exist for) must fail one of them."""
import numpy as np
import pytest
import torch

import mlp_ref
from mlp_ref import QUANT, REL_L2_BAR, q_bf16, q_tf32


def q_rz(precision):
    keep = {"bf16": 0xFFFF0000, "tf32": 0xFFFFE000}[precision]
    return lambda x: (np.asarray(x, np.float32).view(np.uint32) & np.uint32(keep)).view(np.float32)


def model_kernel(a0, layers, s, precision, kernel, seed, *, q_act=None, drop_lo=False, drop_sample=False):
    """Surrogate kernel: exact products of operand-rounded values, accumulated in fp32 in a random order per layer;
    mid-layer bias as two extra K terms q(b), q(b - q(b)) (kernel 'tc2') or an fp32 add after the sum ('v1', 'fp32');
    last layer: tc2 pools then adds the bias, the others add bias + ReLU per row and pool."""
    rng = np.random.default_rng(seed)
    q = QUANT[precision]
    q_act = q_act or q
    a = a0.astype(np.float32)
    nl = len(layers)
    for l, (w, b) in enumerate(layers):
        last = l + 1 == nl
        wq = q(w).astype(np.float64)
        terms = [(a[:, k:k + 1].astype(np.float64) * wq[None, :, k]).astype(np.float32) for k in range(w.shape[1])]
        if kernel == "tc2" and not last:
            hi = q(b)
            lo = np.zeros_like(hi) if drop_lo else q(b - hi)
            terms += [np.broadcast_to(hi, terms[0].shape), np.broadcast_to(lo, terms[0].shape)]
        acc = np.zeros(terms[0].shape, np.float32)
        for k in rng.permutation(len(terms)):
            acc = acc + terms[k]  # float32 + float32: one IEEE round-to-nearest add
        if kernel != "tc2":
            acc = acc + b
        if not last:
            a = acc if precision == "fp32" else q_act(np.maximum(acc, 0))
            a = np.maximum(a, 0).astype(np.float32)
            continue
        z = acc.reshape(-1, s, acc.shape[1])
        if drop_sample:
            z = z[:, :-1]
        if kernel == "tc2":
            return np.maximum(z.max(axis=1) + b, 0).astype(np.float32)
        return np.maximum(z, 0).max(axis=1).astype(np.float32)


SHAPES = {  # name: (b, n, m, s, c_feat, mlp widths behind the input)
    "kitti_l2": (2, 600, 96, 16, 32, [64, 64, 128]),
    "narrow": (1, 300, 128, 8, 1, [16, 16, 32]),
    "wide_odd": (1, 200, 40, 32, 13, [40, 96, 200]),
    "one_layer": (2, 256, 64, 8, 5, [36]),
}


def _case(shape, seed, precision, kernel="tc2", coord_round_first=False):
    b, n, m, s, c_feat, widths = SHAPES[shape]
    xyz, new_xyz, feats, idx, cnt = mlp_ref.synth_sa_case(seed, b, n, m, s, c_feat)
    layers = mlp_ref.synth_layers(seed + 1, [3 + c_feat] + widths)
    q = QUANT[precision]
    want, bound = mlp_ref.mlp_reference(mlp_ref.sa_rows(xyz, new_xyz, feats, idx, cnt, True, q), layers, s, precision, kernel)
    if coord_round_first:  # mutant rows: the coordinates rounded before the subtraction
        rows = mlp_ref.sa_rows(q(xyz), q(new_xyz), feats, idx, cnt, True, q)
    else:
        rows = mlp_ref.sa_rows(xyz, new_xyz, feats, idx, cnt, True, q)
    return rows, layers, s, want, bound


CONFIGS = [("bf16", "tc2"), ("bf16", "v1"), ("tf32", "tc2"), ("fp32", "fp32")]


@pytest.mark.parametrize("precision,kernel", CONFIGS)
@pytest.mark.parametrize("shape", list(SHAPES))
def test_model_kernel_within_bound(shape, precision, kernel):
    worst_ratio = worst_rel = 0.0
    for seed in (0, 1, 2):
        rows, layers, s, want, bound = _case(shape, 10 * seed, precision, kernel)
        got = model_kernel(rows, layers, s, precision, kernel, seed)
        ratio, rel, n_out = mlp_ref.compare(got, want, bound)
        worst_ratio, worst_rel = max(worst_ratio, ratio), max(worst_rel, rel)
        assert n_out == 0, (seed, ratio)
        assert rel <= REL_L2_BAR[precision], (seed, rel)
    print(f"{shape} {precision}/{kernel}: max err/B {worst_ratio:.3f}, rel_l2 {worst_rel:.2e} "
          f"(bar {REL_L2_BAR[precision]:.0e}, margin {REL_L2_BAR[precision] / max(worst_rel, 1e-30):.1f}x)")


MUTANTS = {
    "rz_activations": dict(q_act="rz"),
    "bias_lo_dropped": dict(drop_lo=True),
    "pooled_sample_dropped": dict(drop_sample=True),
    "output_channels_swapped": dict(swap=True),
    "coords_rounded_first": dict(coord_round_first=True),
}


@pytest.mark.parametrize("precision,kernel", CONFIGS)
@pytest.mark.parametrize("mutant", list(MUTANTS))
@pytest.mark.parametrize("shape,seed", [("kitti_l2", 0), ("wide_odd", 10)])
def test_mutant_rejected(shape, seed, mutant, precision, kernel):
    kw = dict(MUTANTS[mutant])
    if precision == "fp32" and mutant in ("rz_activations", "coords_rounded_first"):
        pytest.skip("the fp32 kernel rounds no operand")
    if kernel != "tc2" and mutant == "bias_lo_dropped":
        pytest.skip("only the second-generation kernel splits the bias")
    rows, layers, s, want, bound = _case(shape, seed, precision, kernel, coord_round_first=kw.pop("coord_round_first", False))
    swap = kw.pop("swap", False)
    if kw.pop("q_act", None):
        kw["q_act"] = q_rz(precision)
    got = model_kernel(rows, layers, s, precision, kernel, seed, **kw)
    if swap:
        got = got[:, [1, 0] + list(range(2, got.shape[1]))]
    ratio, rel, n_out = mlp_ref.compare(got, want, bound)
    print(f"{mutant} {shape} {precision}/{kernel}: max err/B {ratio:.3g}, {n_out} outputs outside the bound, rel_l2 {rel:.2e} "
          f"(bar {REL_L2_BAR[precision]:.0e})")
    assert n_out > 0 or rel > REL_L2_BAR[precision]


DENSE_SHAPES = {  # name: (b, n, c0, c1, mlp widths): the point-wise MLP, no pooling (last layer relu(z + b) per row)
    "fp_module": (2, 300, 32, 5, [64, 64]),
    "one_layer_c1": (3, 129, 1, 0, [36]),
    "wide": (1, 200, 130, 2, [128, 200]),
}


@pytest.mark.parametrize("precision,kernel", [("bf16", "tc2"), ("tf32", "tc2"), ("fp32", "fp32")])
@pytest.mark.parametrize("shape", list(DENSE_SHAPES))
def test_model_kernel_dense_within_bound(shape, precision, kernel):
    """Dense mode of the reference (dense_rows, nsample 1) against the model kernel; RZ activations and a dropped
    bias-lo term are rejected here too."""
    b, n, c0, c1, widths = DENSE_SHAPES[shape]
    rng = np.random.default_rng(len(shape))
    src0 = rng.standard_normal((b, c0, n)).astype(np.float32)
    src1 = rng.standard_normal((b, c1, n)).astype(np.float32) if c1 else None
    layers = mlp_ref.synth_layers(5, [c0 + c1] + widths)
    rows = mlp_ref.dense_rows(src0, src1, QUANT[precision])
    assert rows.shape == (b * n, c0 + c1)
    np.testing.assert_array_equal(rows[(b - 1) * n + 7, :c0], QUANT[precision](src0[b - 1, :, 7]))  # row f * n + i: point i of frame f
    want, bound = mlp_ref.mlp_reference(rows, layers, 1, precision, kernel)
    ratio, rel, n_out = mlp_ref.compare(model_kernel(rows, layers, 1, precision, kernel, 0), want, bound)
    print(f"dense {shape} {precision}/{kernel}: max err/B {ratio:.3f}, rel_l2 {rel:.2e}")
    assert n_out == 0 and rel <= REL_L2_BAR[precision], (ratio, rel)
    if precision == "fp32" or len(layers) < 2:
        return
    for kw in (dict(q_act=q_rz(precision)), dict(drop_lo=True)):
        _, rel, n_out = mlp_ref.compare(model_kernel(rows, layers, 1, precision, kernel, 0, **kw), want, bound)
        assert n_out > 0 or rel > REL_L2_BAR[precision], kw


def test_bf16_rounding_matches_torch():
    rng = np.random.default_rng(0)
    x = np.concatenate([
        rng.standard_normal(500_000).astype(np.float32) * np.float32(10.0) ** rng.integers(-30, 30, 500_000).astype(np.float32),
        rng.integers(0, 2 ** 32, 500_000, dtype=np.uint64).astype(np.uint32).view(np.float32),  # every bit pattern
    ])
    x = x[np.isfinite(x)]
    x = x[np.abs(x) < 3.3e38]  # rounding up to infinity is not a case the kernels meet
    want = torch.from_numpy(x).to(torch.bfloat16).float().numpy()
    got = q_bf16(x)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    # ties: exactly halfway between two bf16 values goes to the even one
    ties = np.array([1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, -(1.0 + 2.0 ** -8)], np.float32)
    assert q_bf16(ties).tolist() == [1.0, 1.0 + 2.0 ** -6, -1.0]


def test_tf32_rounding_ties_away_from_zero():
    u = 2.0 ** -10  # tf32 spacing at 1
    x = np.array([1.0 + u / 2, 1.0 + 3 * u / 2, -(1.0 + u / 2), 1.0 + u / 2 - 2.0 ** -23, 1.0 + u / 2 + 2.0 ** -23,
                  3.0, 0.0, 1.5 * 2.0 ** -136], np.float32)
    want = np.array([1.0 + u, 1.0 + 2 * u, -(1.0 + u), 1.0, 1.0 + u, 3.0, 0.0, 2.0 ** -135], np.float32)
    assert np.array_equal(q_tf32(x), want)
    # every tf32 result keeps 10 mantissa bits and is within half a tf32 ulp
    x = np.random.default_rng(1).standard_normal(100_000).astype(np.float32)
    r = q_tf32(x)
    assert not (r.view(np.uint32) & 0x1FFF).any()
    assert (np.abs(r.astype(np.float64) - x) <= np.abs(x).astype(np.float64) * 2.0 ** -11).all()


def test_reference_empty_ball_is_relu_bias_chain():
    """An empty ball sees all-zero input rows: its output is the ReLU(bias) chain of the rounded layers."""
    xyz, new_xyz, feats, idx, cnt = mlp_ref.synth_sa_case(3, 1, 100, 16, 8, 4)
    layers = mlp_ref.synth_layers(4, [7, 16, 32])
    rows = mlp_ref.sa_rows(xyz, new_xyz, feats, idx, cnt, True, q_bf16)
    want, _ = mlp_ref.mlp_reference(rows, layers, 8, "bf16")
    a = q_bf16(np.maximum(layers[0][1], 0)).astype(np.float64)
    chain = np.maximum(q_bf16(layers[1][0]).astype(np.float64) @ a + layers[1][1], 0)
    assert (cnt.reshape(-1) == 0).any()
    for c in np.flatnonzero(cnt.reshape(-1) == 0):
        np.testing.assert_array_equal(want[c], chain)
