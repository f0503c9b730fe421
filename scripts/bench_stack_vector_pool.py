"""Benchmark of the vector-pool ops of pointnet2_stack and VectorPoolAggregationModuleMSG on one GPU; prints ONE JSON line.

    python scripts/bench_stack_vector_pool.py [--iters 20] [--warmup 5] [--seed 0]

Shapes in the spirit of PV-RCNN++ (chosen here, not read from its configuration files), B = 2 frames:
  vsa_raw:   ~16k raw points per frame, 4096 centres per frame, C = 2 reduced to NUM_REDUCED_CHANNELS 2,
             groups (2,2,2) at 0.2 and (3,3,3) at 0.4, local_interpolation;
  vsa_voxel: ~6k voxel-feature points per frame, 4096 centres per frame, C 64 -> 32, (3,3,3) at 1.2 and 2.4,
             local_interpolation;
  roi_grid:  128 RoIs x 216 grid points per frame over 4096 keypoints per frame, C 120 -> 30 (the module needs a
             multiple of the reduced width), voxel_random_choice,
             nsample 32, (3,3,3) at 0.8 and 1.6.
Reported per shape:
  * the wrappers of the first group (neighbour lists, the list 3-NN, vector_pool_wrapper) on the per-frame grids and under
    TSMDET_BQ_ALGO=brute, in ms (vector_pool_wrapper includes its one device-to-host read of the total);
  * how many frames the grid cannot take (a host restatement of the grid's cell sizing: no points, a non-finite
    coordinate, > 256 points in one cell), i.e. fall back to brute force;
  * the module eager against fused (eval), in ms, their largest absolute difference and whether the fused input planes
    equal the eager ones bit for bit;
  * each planes writer's compulsory HBM bytes against its time;
  * the GPU's name and power limit, read in the same run.
A 256 MB buffer is overwritten before every timed call (the inputs would otherwise sit in L2), and the median of CUDA-event
timings is reported.  The reference's kernels are not timed: "not measured".
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


class Cfg(dict):
    __getattr__ = dict.__getitem__


SHAPES = {
    "vsa_raw": dict(support=16384, centres=4096, c=2, reduced=2, kind="local_interpolation", nsample=-1,
                    groups=[((2, 2, 2), 0.2), ((3, 3, 3), 0.4)]),
    "vsa_voxel": dict(support=6000, centres=4096, c=64, reduced=32, kind="local_interpolation", nsample=-1,
                      groups=[((3, 3, 3), 1.2), ((3, 3, 3), 2.4)]),
    "roi_grid": dict(support=4096, centres=128 * 216, c=120, reduced=30, kind="voxel_random_choice", nsample=32,
                     groups=[((3, 3, 3), 0.8), ((3, 3, 3), 1.6)]),
}


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


def grid_unusable(pts, d):
    """the grid build's verdict (ball_query_grid.cu): cells >= 1.01 d per axis, <= 2048 per axis and 32768 in all
    (the smallest-extent axis halved first), usable iff the points are finite, there are some and no cell holds > 256"""
    if len(pts) == 0 or not np.isfinite(pts).all():
        return True
    lo, hi = pts.min(0), pts.max(0)
    ext = (hi - lo).astype(np.float32)
    s0 = np.float32(d) * np.float32(1.01)
    nc = np.clip(np.floor(ext / s0), 1, 2048).astype(np.int64)
    while nc.prod() > 32768:
        a = min((c for c in range(3) if nc[c] > 1), key=lambda c: ext[c])
        nc[a] = (nc[a] + 1) // 2
    inv = np.where(ext > 0, nc / np.maximum(ext, 1e-30), 0).astype(np.float32)
    inv = np.where(inv * s0 > 1, 1 / s0, inv).astype(np.float32)
    q = np.clip(np.floor((pts - lo) * inv).astype(np.int64), 0, nc - 1)
    cell = (q[:, 2] * nc[1] + q[:, 1]) * nc[0] + q[:, 0]
    return bool(np.bincount(cell).max() > 256)


def frames(shape, rng, seed):
    import synth

    sup = [synth.cloud_ground_objects(1, int(shape["support"] * rng.uniform(0.9, 1.1)), seed=seed + k)[0] for k in range(2)]
    cen = [f[rng.choice(len(f), min(shape["centres"], len(f)), replace=len(f) < shape["centres"])] +
           rng.uniform(-0.3, 0.3, (min(shape["centres"], len(f)), 3)).astype(np.float32) for f in sup]
    if shape["centres"] > shape["support"]:  # RoI grid points: 216 points on a 6^3 lattice in each of 128 boxes
        cen = []
        for f in sup:
            boxes = f[rng.choice(len(f), 128, replace=False)]
            g = (np.arange(6, dtype=np.float32) - 2.5) * np.float32(0.6)
            lat = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
            cen.append((boxes[:, None, :] + lat[None]).reshape(-1, 3).astype(np.float32))
    return sup, cen


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stack_vector_pool.py measures on a CUDA device; none is visible")

    from tsmdet_b200 import _lib
    from tsmdet_b200._lib import call, ptr, stream_ptr
    from tsmdet_b200.pointnet2_stack import pointnet2_stack_cuda as ps
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu
    from tsmdet_b200.pointnet2_stack.pointnet2_modules import VectorPoolAggregationModuleMSG

    dev = torch.device("cuda:0")
    name, power = gpu_identity()
    rng = np.random.default_rng(args.seed)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.backends.cudnn.allow_tf32 = False
    out = {"metric": "stack_vector_pool", "gpu": name, "power_limit": power, "iters": args.iters,
           "reference_kernels": "not measured", "shapes": {}}

    for key, sh in SHAPES.items():
        sup, cen = frames(sh, rng, args.seed)
        xyz = torch.from_numpy(np.concatenate(sup)).to(dev)
        new = torch.from_numpy(np.concatenate(cen)).to(dev)
        cnt = torch.tensor([len(f) for f in sup], dtype=torch.int32, device=dev)
        mcnt = torch.tensor([len(f) for f in cen], dtype=torch.int32, device=dev)
        feats = torch.from_numpy(rng.standard_normal((xyz.shape[0], sh["c"])).astype(np.float32)).to(dev)
        n, m = xyz.shape[0], new.shape[0]
        rec = {"frames_support": cnt.tolist(), "frames_centres": mcnt.tolist(), "c": sh["c"], "reduced": sh["reduced"],
               "kind": sh["kind"], "groups": sh["groups"], "wrappers": {}}
        grids, d = sh["groups"][0]
        G = grids[0] * grids[1] * grids[2]
        dq = d * 2.0 if sh["kind"] == "local_interpolation" else d
        rec["brute_force_frames"] = {f"D={dd}": sum(grid_unusable(f, dd * (2.0 if sh["kind"] == "local_interpolation"
                                                                           else 1.0)) for f in sup)
                                     for _, dd in sh["groups"]}
        red = feats.view(n, -1, sh["reduced"]).sum(1).contiguous()
        centres = (new[:, None, :] + torch.zeros((1, G, 3), device=dev)).contiguous()
        for impl in ("grid", "brute"):
            os.environ.pop("TSMDET_BQ_ALGO", None)
            if impl == "brute":
                os.environ["TSMDET_BQ_ALGO"] = "brute"
            _lib.reload_options()
            buf = torch.zeros((1000 * m,), dtype=torch.int32, device=dev)
            sl = torch.zeros((m, 2), dtype=torch.int32, device=dev)
            cs = torch.zeros((1,), dtype=torch.int32, device=dev)

            def lists():
                cs.zero_()
                ps.query_stacked_local_neighbor_idxs_wrapper_stack(xyz, cnt, new, mcnt, buf, sl, cs, 1000, dq,
                                                                   sh["nsample"], 0)
            r = {"local_neighbor_idxs_ms": round(timed(lists, args.iters, args.warmup, flush), 4)}
            lists()
            total = int(cs.item())
            idx = torch.empty((m, G, 3), dtype=torch.int32, device=dev)
            d2 = torch.empty((m, G, 3), device=dev)
            r["three_nn_local_ms"] = round(timed(lambda: ps.query_three_nn_by_stacked_local_idxs_wrapper_stack(
                xyz, new, centres, idx, d2, buf[:total], sl, m, G), args.iters, args.warmup, flush), 4)
            nf = torch.zeros((m, G * sh["reduced"]), device=dev)
            nl = torch.zeros((m, 3 * G), device=dev)
            pc = torch.zeros((m, G), dtype=torch.int32, device=dev)
            tr = torch.zeros((m * G, 3), dtype=torch.int32, device=dev)

            def pool():
                nf.zero_(), nl.zero_(), pc.zero_()
                ps.vector_pool_wrapper(xyz, cnt, red, new, mcnt, nf, nl, pc, tr, *grids, d, 1, m * G, sh["nsample"], 0,
                                       0 if sh["kind"] == "voxel_avg_pool" else 1)
            r["vector_pool_ms"] = round(timed(pool, args.iters, args.warmup, flush), 4)
            r["mean_list_length"] = round(total / max(m, 1), 1)
            rec["wrappers"][impl] = r
        os.environ.pop("TSMDET_BQ_ALGO", None)
        _lib.reload_options()

        cfg = Cfg(NAME="VectorPoolAggregationModuleMSG", NUM_GROUPS=2, LOCAL_AGGREGATION_TYPE=sh["kind"],
                  NUM_REDUCED_CHANNELS=sh["reduced"], NUM_CHANNELS_OF_LOCAL_AGGREGATION=32, MSG_POST_MLPS=[128])
        for k, (gr, dd) in enumerate(sh["groups"]):
            cfg[f"GROUP_CFG_{k}"] = Cfg(NUM_LOCAL_VOXEL=list(gr), MAX_NEIGHBOR_DISTANCE=dd, NEIGHBOR_NSAMPLE=sh["nsample"],
                                        POST_MLPS=[64, 64])
        torch.manual_seed(args.seed)
        mod = VectorPoolAggregationModuleMSG(sh["c"], cfg).to(dev).eval()
        kw = dict(xyz=xyz, xyz_batch_cnt=cnt, new_xyz=new, new_xyz_batch_cnt=mcnt, features=feats)
        layers = [getattr(mod, f"layer_{k}") for k in range(2)]
        with torch.no_grad():
            for lay in layers:
                lay.fused = False
            want = mod(**kw)[1]
            rec["module_eager_ms"] = round(timed(lambda: mod(**kw), args.iters, args.warmup, flush), 4)
            for lay in layers:
                lay.fused = True
            got = mod(**kw)[1]
            rec["module_fused_ms"] = round(timed(lambda: mod(**kw), args.iters, args.warmup, flush), 4)
            rec["module_max_abs_diff"] = float(f"{(got - want).abs().max().item():.3e}")
            planes_equal, writers = True, {}
            for k, lay in enumerate(layers):
                lay.fused = False
                args_e = dict(xyz=xyz, xyz_batch_cnt=cnt, features=red, new_xyz=new, new_xyz_batch_cnt=mcnt)
                if sh["kind"] == "local_interpolation":
                    eager_pl = lay.vector_pool_with_local_interpolate(**args_e).permute(1, 0)[None]
                else:
                    eager_pl = lay.vector_pool_with_voxel_query(**args_e)[0].permute(1, 0)[None]
                lay.fused = True
                fused_pl = lay.input_planes(xyz, cnt, red, new, mcnt)
                planes_equal &= bool(torch.equal(fused_pl.view(torch.int32), eager_pl.contiguous().view(torch.int32)))
                Gk = lay.total_voxels
                if sh["kind"] == "local_interpolation":
                    li = lay.local_interpolate_module
                    cen_k = lay.get_dense_voxels_by_center(new, lay.max_neighbour_distance, lay.num_local_voxel).contiguous()
                    idx = torch.empty((m, Gk, 3), dtype=torch.int32, device=dev)
                    d2 = torch.empty((m, Gk, 3), device=dev)
                    call("tsmdet_stack_vector_three_nn", 2, m, n, Gk, ptr(xyz), ptr(cnt), ptr(new), ptr(mcnt), ptr(cen_k),
                         float(li.max_neighbour_distance * li.neighbor_distance_multiplier), int(li.nsample),
                         int(li.neighbor_type), ptr(idx), ptr(d2), stream_ptr(dev))
                    w = pu.local_interp_weights(torch.sqrt(d2)).contiguous()
                    pl = torch.empty_like(fused_pl)
                    c = red.shape[1]
                    t = timed(lambda: call("tsmdet_stack_vector_interp_planes", m, Gk, n, c, ptr(red), ptr(xyz),
                                           ptr(cen_k), ptr(idx), ptr(w), ptr(pl), stream_ptr(dev)),
                              args.iters, args.warmup, flush)
                    # planes written + idx / weight / centres read + (at most) every support row and point read once
                    nbytes = 4 * pl.numel() + 36 * m * Gk + n * (4 * c + 12)
                    writers[f"group{k}_interp_planes"] = {"ms": round(t, 4), "MB": round(nbytes / 1e6, 1),
                                                          "GBps": round(nbytes / t / 1e6, 1)}
                    t = timed(lambda: call("tsmdet_stack_vector_three_nn", 2, m, n, Gk, ptr(xyz), ptr(cnt), ptr(new),
                                           ptr(mcnt), ptr(cen_k), float(li.max_neighbour_distance *
                                                                        li.neighbor_distance_multiplier),
                                           int(li.nsample), int(li.neighbor_type), ptr(idx), ptr(d2), stream_ptr(dev)),
                              args.iters, args.warmup, flush)
                    writers[f"group{k}_fused_three_nn_ms"] = round(t, 4)
                else:
                    t = timed(lambda: lay.input_planes(xyz, cnt, red, new, mcnt), args.iters, args.warmup, flush)
                    # planes written + centres and counts read + (at most) every support row and point read once
                    nbytes = 4 * fused_pl.numel() + 12 * m + n * (4 * red.shape[1] + 12)
                    writers[f"group{k}_pool_planes"] = {"ms": round(t, 4), "MB": round(nbytes / 1e6, 1),
                                                        "GBps": round(nbytes / t / 1e6, 1),
                                                        "note": "includes the neighbour search"}
            rec["planes_bit_identical"] = planes_equal
            rec["planes_writers"] = writers
        out["shapes"][key] = rec
    print(json.dumps(out))


if __name__ == "__main__":
    main()
