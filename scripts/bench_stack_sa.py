"""Benchmark of the stacked (ragged) ball query and StackSAModuleMSG on one GPU; prints ONE JSON line.

    python scripts/bench_stack_sa.py [--iters 20] [--warmup 5] [--seed 0]

Shapes are PV-RCNN's keypoint set abstraction: B = 4 ragged frames of 9k-20k points (seeded sizes), 2048 centres each;
scale A: C = 1, radii 0.4 / 0.8, nsample 16 / 16, MLPs [1,16,16] x 2; scale B: C = 64, radii 1.2 / 2.4, nsample 16 / 32,
MLPs [64,64,64] x 2.  Reported:
  * query: grid (default), brute force (TSMDET_BQ_ALGO=brute) and the reference's ball_query_wrapper
    (oracle/_ref/pointnet2_stack_cuda.so; "not measured" without it), in ms and in GB/s of the compulsory bytes
    12 N + 12 M + 4 M nsample;
  * StackSAModuleMSG: eager and fused fp32 / bf16 / tf32, in ms, with the fused MLP's TFLOP/s from
    2 M S sum(C_i C_i+1) (C_0 including the 3 coordinates) over the whole module call (ball queries and feature rows
    included, so a lower bound of the MLP kernel's own rate);
  * eager vs fused parity metrics (tests/parity.py) at the timed size;
  * the GPU's name and power limit, read in the same run.
The inputs are a few MB, so they would sit in L2 after the first pass: a 256 MB buffer is overwritten before every
timed call, and CUDA events time the call alone.
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

SCALES = {
    "A": dict(c=1, radii=[0.4, 0.8], nsamples=[16, 16], mlps=[[1, 16, 16], [1, 16, 16]]),
    "B": dict(c=64, radii=[1.2, 2.4], nsamples=[16, 32], mlps=[[64, 64, 64], [64, 64, 64]]),
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


def inputs(seed, frames=4, centres=2048):
    import synth

    rng = np.random.default_rng(seed)
    sizes = rng.integers(9000, 20001, frames)
    fx = [synth.cloud_ground_objects(1, int(n), seed=seed + 1 + k)[0] for k, n in enumerate(sizes)]
    fn = [f[rng.choice(len(f), centres, replace=False)] for f in fx]
    xyz = np.concatenate(fx, 0)
    new = np.concatenate(fn, 0)
    return xyz, sizes.astype(np.int32), new, np.full((frames,), centres, np.int32), rng


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stack_sa.py measures on a CUDA device; none is visible")

    import parity
    from oracle import build_ref
    from tsmdet_b200 import _lib
    from tsmdet_b200.pointnet2_stack import StackSAModuleMSG
    from tsmdet_b200.pointnet2_stack import pointnet2_stack_cuda as ps

    dev = torch.device("cuda:0")
    name, power = gpu_identity()
    xyz_np, cnt_np, new_np, mcnt_np, rng = inputs(args.seed)
    xyz, cnt, new, mcnt = (torch.from_numpy(a).to(dev) for a in (xyz_np, cnt_np, new_np, mcnt_np))
    n, m, b = xyz.shape[0], new.shape[0], len(cnt_np)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ref = build_ref.load_ref("pointnet2_stack_cuda")
    out = {"metric": "stack_sa", "gpu": name, "power_limit": power, "frames": b, "points": int(n), "centres": int(m),
           "frame_sizes": cnt_np.tolist(), "iters": args.iters, "query": {}, "module": {}}

    def query_fn(impl, r, ns):
        idx = torch.zeros((m, ns), dtype=torch.int32, device=dev)
        wrapper = ref.ball_query_wrapper if impl == "reference" else ps.ball_query_wrapper
        return lambda: wrapper(b, m, r, ns, new, mcnt, xyz, cnt, idx)

    seen = set()
    for cfg in SCALES.values():
        for r, ns in zip(cfg["radii"], cfg["nsamples"]):
            if (r, ns) in seen:
                continue
            seen.add((r, ns))
            rec = {}
            nbytes = 12 * n + 12 * m + 4 * m * ns
            for impl in ("grid", "brute", "reference"):
                if impl == "reference" and ref is None:
                    rec[impl] = "not measured"
                    continue
                os.environ.pop("TSMDET_BQ_ALGO", None)
                if impl == "brute":
                    os.environ["TSMDET_BQ_ALGO"] = "brute"
                _lib.reload_options()
                t = timed(query_fn(impl, r, ns), args.iters, args.warmup, flush)
                rec[impl] = {"ms": round(t, 4), "GBps": round(nbytes / t / 1e6, 1)}
            os.environ.pop("TSMDET_BQ_ALGO", None)
            _lib.reload_options()
            out["query"][f"r{r}_ns{ns}"] = rec

    for key, cfg in SCALES.items():
        feats = torch.from_numpy(rng.standard_normal((n, cfg["c"])).astype(np.float32)).to(dev)
        torch.manual_seed(args.seed)
        mod = StackSAModuleMSG(radii=cfg["radii"], nsamples=cfg["nsamples"], mlps=cfg["mlps"]).to(dev).eval()
        flop = sum(2 * m * ns * sum(a * c for a, c in zip([s[0] + 3] + s[1:-1], s[1:]))
                   for ns, s in zip(cfg["nsamples"], cfg["mlps"]))
        rec = {"mlp_gflop": round(flop / 1e9, 3)}
        torch.backends.cudnn.allow_tf32 = False
        mod.fused = False
        with torch.no_grad():
            want = mod(xyz, cnt, new, mcnt, feats)[1]
            rec["eager_fp32"] = {"ms": round(timed(lambda: mod(xyz, cnt, new, mcnt, feats), args.iters, args.warmup,
                                                   flush), 4)}
            mod.fused = True
            for prec in ("fp32", "bf16", "tf32"):
                mod.precision = prec
                mod._folded = None
                got = mod(xyz, cnt, new, mcnt, feats)[1]
                t = timed(lambda: mod(xyz, cnt, new, mcnt, feats), args.iters, args.warmup, flush)
                met = parity.err_metrics(got, want)
                rec[f"fused_{prec}"] = {"ms": round(t, 4), "TFLOPs": round(flop / t / 1e9, 2),
                                        "parity": {k: float(f"{v:.3e}") for k, v in met.items()},
                                        "within_bars": all(met[k] <= bar for k, bar in parity.BARS[prec].items())}
        out["module"][f"scale_{key}"] = rec
    print(json.dumps(out))


if __name__ == "__main__":
    main()
