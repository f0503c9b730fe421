"""Width classes of the fused SA MLP on the benchmark's inputs: per SA layer of config 2 (bench.SA_LAYERS, 16 frames of
bench.make_inputs), the histogram of the row width each centre is computed at (next_pow2(cnt) for the ball query's
cyclic padding, 1 for an empty ball; see sa_width_classify_kernel), the 128-row tiles that makes against nsample-wide tiles, and the MLP time
with width-class tiles and with TSMDET_MLP_WIDTH=fixed (one call replayed from a CUDA graph, CUDA events, bf16, chained
bf16 rows as in the pipeline; the classed time includes the classification kernel).  Needs a GPU.

    python scripts/bench_sa_width.py [--frames 16] [--iters 200]
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import bench  # noqa: E402
import mlp_ref  # noqa: E402
from tsmdet_b200 import _lib, pointnet2_utils  # noqa: E402
from tsmdet_b200.pointnet2_modules import gather_xyz, pack_mlp, sa_mlp_maxpool  # noqa: E402


def widths(idx, cnt):
    """The row width sa_width_classify_kernel gives each centre (csrc/mlp_tc2.cu)."""
    s = idx.shape[-1]
    idx = idx.reshape(-1, s)
    c = np.minimum(cnt.reshape(-1), s)
    diff = idx != idx[:, :1]
    t = np.where(diff.any(1), s - np.argmax(diff[:, ::-1], axis=1), 1)
    j = np.arange(s)
    cyc = np.array([ci > 0 and bool((row[ci:] == row[j[ci:] % ci]).all()) for row, ci in zip(idx, c)])
    t = np.where(cyc, np.minimum(t, c), t)
    t[c <= 0] = 1
    return 1 << np.ceil(np.log2(t)).astype(int)


def time_ms(fn, iters):
    """Device time of one call, replayed from a CUDA graph (the mode is fixed at capture; inputs stay L2-resident)."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        fn()
    for _ in range(5):
        g.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--iters", type=int, default=200)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    print(f"# {torch.cuda.get_device_name(dev)}")
    xyz_np, feats_np, _, _ = bench.make_inputs(args.frames, 0)
    xyz, feat = torch.from_numpy(xyz_np).to(dev), torch.from_numpy(feats_np).to(dev)
    feat_t, c_feat = None, feat.shape[1]
    for li, (npoint, radius, ns, chans) in enumerate(bench.SA_LAYERS):
        new_xyz = gather_xyz(xyz, pointnet2_utils.farthest_point_sample(xyz, npoint))
        cnt, idx = pointnet2_utils.ball_query(radius, ns, xyz, new_xyz)
        w = widths(idx.cpu().numpy(), cnt.cpu().numpy())
        hist = {int(k): int(v) for k, v in zip(*np.unique(w, return_counts=True))}
        tiles = sum(-(-v // (128 // k)) for k, v in hist.items())
        layers = [(torch.from_numpy(a).to(dev), torch.from_numpy(bb).to(dev))
                  for a, bb in mlp_ref.synth_layers(li, list(chans))]
        packed = pack_mlp(layers, dense=False, nsample=ns, c_feat=c_feat, precision="bf16")
        cout = chans[-1]
        out_t = torch.empty((args.frames, npoint, -(-cout // 8) * 8), dtype=torch.bfloat16, device=dev)
        run = lambda: sa_mlp_maxpool(xyz, new_xyz, feat if feat_t is None else None, idx, cnt, layers, None, 0,
                                     precision="bf16", packed=packed, feat_t=feat_t, out_t=out_t)
        t = {}
        for mode in ("fixed", "classes"):
            if mode == "fixed":
                os.environ["TSMDET_MLP_WIDTH"] = "fixed"
            else:
                os.environ.pop("TSMDET_MLP_WIDTH", None)
            _lib.reload_options()
            t[mode] = time_ms(run, args.iters)
        fixed_tiles = args.frames * npoint * ns // 128
        print(f"L{li + 1} {xyz.shape[1]}->{npoint} r {radius} ns {ns}: widths {hist}, mean {w.mean():.2f}; "
              f"tiles {tiles} (fixed {fixed_tiles}); MLP ms fixed {t['fixed']:.4f} classes {t['classes']:.4f}")
        xyz, feat, feat_t, c_feat = new_xyz, None, out_t, cout


if __name__ == "__main__":
    main()
