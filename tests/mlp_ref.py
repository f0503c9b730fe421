"""Float64 reference of the shared-MLP kernels with an elementwise error bound (TEST INFRASTRUCTURE, numpy, CPU).

The kernels (``csrc/mlp_tc2.cu``, ``csrc/sa_mlp_tc.cu``, ``csrc/sa_mlp_fp32.cu``) take folded layers
``[(W (cout, cin) fp32, b (cout,) fp32)]`` and compute, per row, ``[1x1 conv + bias + ReLU]*`` followed by a max over
the ``nsample`` rows of a centre (SA mode) or nothing (dense mode).  This module restates that in float64 and models
exactly what the kernels round:

  * operand rounding ``q``: bf16 round-to-nearest-even, tf32 ``cvt.rna`` (round half away from zero), identity for
    the fp32 kernel.  Weights are ``q(W)``; layer-0 feature rows are ``q(f)``; coordinate rows are
    ``q(fp32(p - centre))`` (``__fsub_rn``, then rounded); rows of an empty ball (``idx_cnt <= 0``) are zero;
  * mid layers: ``z = q(W) a + b`` exactly, then ``a' = q(fp32(relu(z)))``;
  * last layer: SA ``relu(max_s z_s + b)``, dense ``relu(z + b)``.

Alongside it, ``B`` bounds ``|kernel - reference|`` elementwise by forward propagation:

  * pre-activation: ``E_z = |q(W)| E_a + gamma (|q(W)| |a| + |b|)`` with ``gamma = (K + 2) 2^-23``, ``K`` the layer's
    padded input width -- twice the fp32 unit roundoff per addition, because the tensor core's fp32 accumulation is
    not an IEEE sequential sum.  The second-generation kernel adds a mid layer's bias inside the accumulator as
    ``q(b) + q(b - q(b))``; the error of that split, ``|b - (q(b) + q(b - q(b)))|``, is added to ``E_z``;
  * after rounding: ``E_a' = max |q(fp32(relu(z +- E_z))) - a'|``.  ``q o fp32 o relu`` is monotone, so this is zero
    unless a rounding boundary lies within ``+-E_z``: most activations are pinned exactly, and the kernel may differ
    only where it could legitimately have rounded the other way;
  * output: ``B = max_s E_z + 2^-23 (|max_s z| + |b|)`` (the fp32 add of the last bias, with a factor 2 to spare).
    The fp32 kernel has no operand rounding, so its ``E_a`` simply propagates.

The per-element margin is thin by construction.  Where a kernel legitimately rounds one activation the other way, the
output moves by |w| times that activation's rounding step, and ``B`` holds exactly that term plus the gamma allowances:
max(err/B) close to 1 (0.998 in the model kernel of tests/test_mlp_ref_cpu.py, 0.999 bf16 / 0.995 tf32 measured on a
B200) is the expected worst case, not a near miss.  What is left of ``B`` beyond such a flip is the gamma term, i.e.
the assumption that the tensor core's fp32 accumulation strays from an IEEE sum by at most twice the unit roundoff
per term.  A kernel that accumulates worse than that, rounds an operand differently or drops a term lands outside.
"""
from __future__ import annotations

import numpy as np

U = 2.0 ** -23  # twice the fp32 unit roundoff

# rel_l2 bars of check (b).  Derivation: the unmutated model (tests/test_mlp_ref_cpu.py), over the shapes and seeds of
# test_model_kernel_within_bound, gives a worst rel_l2 against the float64 reference of 5.1e-5 (bf16), 7.9e-6 (tf32)
# and 2.0e-7 (fp32; it rounds every product, the FMA kernel does not), printed by that test.  Each bar is 10x the
# model's worst value: 5e-4 for bf16 still rejects the model with the bias-lo row dropped (1.2e-3) or RZ activations
# (7e-3), 8e-5 for tf32 (its operands carry 3 more mantissa bits) the bias-lo mutant (1.25e-4).  The printed margins
# show how much room each shape has.  Measured on one B200 (1000 W power limit) over tests/test_mlp_kernels_gpu.py, the
# worst rel_l2 is 2.2e-4 for bf16 (the one-tile case, 3 centres), 1.2e-5 for the first-generation bf16 kernel, 2.0e-5
# for tf32 and 3.8e-7 for fp32.
REL_L2_BAR = {"bf16": 5e-4, "tf32": 8e-5, "fp32": 2e-6}


def q_bf16(x):
    """fp32 -> bf16 -> fp32, round to nearest even (``__float2bfloat16_rn``, ``cvt.rn.bf16x2.f32``)."""
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000).astype(np.uint32).view(np.float32)


def q_tf32(x):
    """fp32 -> tf32 bit pattern, round half away from zero (``cvt.rna.tf32.f32``)."""
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x1000) & 0xFFFFE000).astype(np.uint32).view(np.float32)


def q_fp32(x):
    return np.asarray(x, np.float32)


QUANT = {"bf16": q_bf16, "tf32": q_tf32, "fp32": q_fp32}


def sa_rows(xyz, new_xyz, features, idx, idx_cnt, use_xyz, q):
    """Layer-0 operand rows of a fused SA scale, reference channel order [dx, dy, dz, features...].
    xyz (B,N,3), new_xyz (B,M,3), features (B,C,N) | None, idx (B,M,S), idx_cnt (B,M) | None -> (B*M*S, cin) fp32."""
    b, m, s = idx.shape
    bi = np.arange(b)[:, None, None]
    parts = []
    if use_xyz:
        d = xyz[bi, idx] - new_xyz[:, :, None, :]  # float32 - float32: the kernel's __fsub_rn
        parts.append(q(d))
    if features is not None:
        f = np.transpose(features, (0, 2, 1))[bi, idx]  # (B,M,S,C)
        parts.append(q(f))
    rows = np.concatenate(parts, axis=3)
    if idx_cnt is not None:
        rows = rows * (idx_cnt > 0)[:, :, None, None]
    return np.ascontiguousarray(rows.reshape(b * m * s, -1), dtype=np.float32)


def dense_rows(src0, src1, q):
    """Layer-0 rows of the point-wise MLP: cat([src0, src1], 1) (B,C,n) -> (B*n, C)."""
    x = src0 if src1 is None else np.concatenate([src0, src1], axis=1)
    return np.ascontiguousarray(q(np.transpose(x, (0, 2, 1)).reshape(-1, x.shape[1])))


def padded_k(cin, layer):
    """An upper bound of the padded input width a kernel contracts over: 16-channel K steps (8 for tf32), and on layer
    0 the features padded to a 16-byte chunk plus one chunk for the coordinates."""
    return -(-cin // 16) * 16 + (16 if layer == 0 else 0)


def mlp_reference(a0, layers, nsample, precision, kernel="tc2"):
    """a0 (R, cin) operand-rounded layer-0 rows (sa_rows / dense_rows), R = centres * nsample, rows of a centre
    consecutive; layers [(W, b)] fp32 numpy; precision 'bf16' | 'tf32' | 'fp32'; kernel 'tc2' (mlp_tc2.cu: mid biases
    as a hi + lo K step), 'v1' (sa_mlp_tc.cu) or 'fp32' (sa_mlp_fp32.cu: fp32 adds of the biases).
    Returns (want, bound), both (R / nsample, cout) float64."""
    q = QUANT[precision]

    def qa(x):
        return q(np.maximum(x, 0.0).astype(np.float32)).astype(np.float64)

    a = a0.astype(np.float64)
    ea = np.zeros_like(a)
    nl = len(layers)
    for l, (w, b) in enumerate(layers):
        wq = np.abs(q(w).astype(np.float64)).T
        wqs = q(w).astype(np.float64).T
        b64 = b.astype(np.float64)
        gamma = (padded_k(w.shape[1], l) + 2) * U
        z = a @ wqs
        ez = ea @ wq + gamma * (np.abs(a) @ wq + np.abs(b64))
        if l + 1 < nl:
            z += b64
            if kernel == "tc2":
                hi = q(b)
                lo = q(b - hi)
                ez += np.abs(b64 - (hi.astype(np.float64) + lo.astype(np.float64)))
            if precision == "fp32":
                a, ea = np.maximum(z, 0.0), ez
            else:
                an = qa(z)
                ea = np.maximum(np.abs(qa(z + ez) - an), np.abs(qa(z - ez) - an))
                a = an
        else:
            zc = z.reshape(-1, nsample, z.shape[1])
            ec = ez.reshape(-1, nsample, z.shape[1])
            mz = zc.max(axis=1)
            want = np.maximum(mz + b64, 0.0)
            bound = ec.max(axis=1) + U * (np.abs(mz) + np.abs(b64))
            return want, bound


def synth_sa_case(seed, b, n, m, s, c_feat, empty_frac=0.1, empty_frame=None, extent=40.0):
    """Seeded inputs of one fused SA scale with every edge placed on purpose: M centres per frame spread over a
    +-extent metre box, point i of a frame lies within ~1 m of centre i % M (so coordinate offsets are small against
    the coordinates, as after a ball query); a centre's neighbours are drawn from its own points, the samples behind
    a random hit count repeat the first one (ball-query padding), one neighbour of every eighth centre is the frame's
    last point (idx = n - 1).  idx_cnt is 0 (empty ball) for about ``empty_frac`` of the centres, for the first
    centres of the first two 128-row tiles and the last of the first, and for every centre of frame ``empty_frame``.
    Returns float32 / int32 numpy arrays xyz (b,n,3), new_xyz (b,m,3), features (b,c_feat,n) | None, idx (b,m,s),
    idx_cnt (b,m)."""
    rng = np.random.default_rng(seed)
    new_xyz = rng.uniform(-extent, extent, size=(b, m, 3)).astype(np.float32)
    owner = np.arange(n) % m
    xyz = (new_xyz[:, owner] + rng.normal(0, 0.6, size=(b, n, 3))).astype(np.float32)
    p = np.arange(m)[None, :, None]
    per = (n - 1 - p) // m + 1  # points owned by centre p (n >= m: at least one)
    idx = p + m * np.floor(rng.random((b, m, s)) * per).astype(np.int64)
    hits = rng.integers(1, s + 1, size=(b, m))
    idx = np.where(np.arange(s)[None, None, :] < hits[:, :, None], idx, idx[:, :, :1])
    idx[:, ::8, -1] = n - 1
    cnt = hits.astype(np.int32)
    cnt[rng.random((b, m)) < empty_frac] = 0
    cpt = max(128 // s, 1)
    flat = cnt.reshape(-1)
    for c in (0, cpt - 1, cpt):
        if c < flat.size:
            flat[c] = 0
    if empty_frame is not None:
        cnt[empty_frame] = 0
    feats = rng.standard_normal((b, c_feat, n)).astype(np.float32) if c_feat else None
    return xyz, new_xyz, feats, np.ascontiguousarray(idx, dtype=np.int32), cnt


def synth_layers(seed, chans, bias_scale=0.2):
    """Random folded layers [(W (cout, cin), b)] for channel list chans = [cin, c1, ..., cout], fp32 numpy:
    W ~ N(0, 1/cin) keeps activations O(1) through the stack, as BatchNorm folding does."""
    rng = np.random.default_rng(seed)
    out = []
    for ci, co in zip(chans[:-1], chans[1:]):
        w = (rng.standard_normal((co, ci)) / np.sqrt(ci)).astype(np.float32)
        out.append((w, (rng.standard_normal(co) * bias_scale).astype(np.float32)))
    return out


def compare(got, want, bound):
    """(max err / bound, rel_l2, number of elements outside the bound) of float arrays of the same shape; a NaN in
    ``got`` counts as outside."""
    got = np.asarray(got, np.float64)
    err = np.abs(got - want)
    ratio = float(np.nan_to_num(err / np.maximum(bound, 1e-300), nan=np.inf).max()) if err.size else 0.0
    rel = float(np.linalg.norm(got - want) / max(np.linalg.norm(want), 1e-300))
    return ratio, rel, int((~(err <= bound)).sum())
