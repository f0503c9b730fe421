"""Benchmark of the roiaware_pool3d ops on one GPU; prints ONE JSON line.

    python scripts/bench_roiaware_pool3d.py [--iters 20] [--warmup 5] [--seed 0]

Shapes (chosen here, not read from configuration files):
  points_in_boxes_gpu: B = 16 frames x N = 16384 points x T = 64 boxes, a random number of them padding (all zeros);
                       B = 2 x N = 180000 x T = 128;
  RoIAwarePool3d:      16384 points, R = 128 RoIs on the cloud, out sizes 12 and 14, max_pts_each_voxel 128,
                       C = 4 and 128, max and avg, forward and backward.
Reported per call: the median of CUDA-event timings in ms, with a 256 MB buffer overwritten before every timed call (the
inputs would otherwise sit in L2), and the compulsory HBM bytes against that time:
  points_in_boxes_gpu: boxes and points read, labels written (the kernel alone: the -1 pre-fill is done once, outside
                       the timed call -- a label the kernel writes is the same on every call);
  forward:  RoIs and points read (once), every voxel counter and the listed indices written, the listed feature rows
            read, pooled written for the non-empty voxels and (max) argmax for every voxel -- the rest of the caller's
            zero-filled tensors is never touched;
  backward: max: argmax read, grad_out read where argmax >= 0; avg: the counters, the lists and the non-empty voxels'
            grad_out read; grad_in written once.
The GPU's name and power limit are read in the same run.  The reference's kernels are not timed: "not measured".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def timed(fn, iters, warmup, flush):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(iters):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


def rate(nbytes, ms):
    return {"ms": round(ms, 4), "MB": round(nbytes / 1e6, 2), "GBps": round(nbytes / ms / 1e6, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_roiaware_pool3d.py measures on a CUDA device; none is visible")

    import synth
    from roiaware_oracle import boxes_on_points
    from tsmdet_b200.roiaware_pool3d import roiaware_pool3d_cuda as ext

    dev = torch.device("cuda:0")
    name, power = gpu_identity()
    rng = np.random.default_rng(args.seed)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"metric": "roiaware_pool3d", "gpu": name, "power_limit": power, "iters": args.iters,
           "reference_kernels": "not measured", "points_in_boxes_gpu": {}, "roiaware_pool3d": {}}

    for b, n, t, padded in ((16, 16384, 64, True), (2, 180000, 128, False)):
        pts = synth.cloud_ground_objects(b, n, seed=args.seed)
        boxes = np.zeros((b, t, 7), np.float32)
        valid = rng.integers(t // 4, t + 1, b) if padded else np.full(b, t)
        for f in range(b):
            boxes[f, :valid[f]] = boxes_on_points(pts[f], int(valid[f]), args.seed + f)
        tb, tp = torch.from_numpy(boxes).to(dev), torch.from_numpy(pts).to(dev)
        lab = torch.empty((b, n), dtype=torch.int32, device=dev)

        lab.fill_(-1)
        ms = timed(lambda: ext.points_in_boxes_gpu(tb, tp, lab), args.iters, args.warmup, flush)
        rec = rate(28 * b * t + 12 * b * n + 4 * b * n, ms)
        rec["inside_share"] = round(float((lab >= 0).float().mean()), 4)
        rec["valid_boxes"] = int(valid.sum())
        out["points_in_boxes_gpu"][f"B{b}_N{n}_T{t}" + ("_padded" if padded else "")] = rec

    n, r, L = 16384, 128, 128
    pts = synth.cloud_ground_objects(1, n, seed=args.seed + 1)[0]
    rois = boxes_on_points(pts, r, args.seed + 2)
    tr, tp = torch.from_numpy(rois).to(dev), torch.from_numpy(pts).to(dev)
    for c in (4, 128):
        feats = torch.from_numpy(rng.standard_normal((n, c)).astype(np.float32)).to(dev)
        for size in (12, 14):
            V = size ** 3
            for method, mname in ((0, "max"), (1, "avg")):
                am = torch.zeros((r, size, size, size, c), dtype=torch.int32, device=dev)
                idx = torch.zeros((r, size, size, size, L), dtype=torch.int32, device=dev)
                pooled = torch.zeros((r, size, size, size, c), device=dev)

                def fwd():
                    ext.forward(tr, tp, feats, am, idx, pooled, method)
                fms = timed(fwd, args.iters, args.warmup, flush)
                fwd()
                listed = int(idx[..., 0].sum())
                full = int((idx[..., 0] > 0).sum())
                fbytes = (28 * r + 12 * n + 4 * r * V + 4 * listed + 4 * listed * c + 4 * full * c +
                          (4 * r * V * c if method == 0 else 0))
                gout = torch.randn((r, size, size, size, c), device=dev)
                gin = torch.zeros((n, c), device=dev)

                def bwd():
                    gin.zero_()
                    ext.backward(idx, am, gout, gin, method)
                bms = timed(bwd, args.iters, args.warmup, flush)
                taken = int((am >= 0).sum()) if method == 0 else 0
                bbytes = 4 * n * c + (4 * r * V * c + 4 * taken if method == 0 else 4 * r * V + 4 * listed + 4 * full * c)
                out["roiaware_pool3d"][f"C{c}_out{size}_{mname}"] = {
                    "forward": rate(fbytes, fms), "backward": rate(bbytes, bms), "listed_points": listed,
                    "non_empty_voxels": full}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
