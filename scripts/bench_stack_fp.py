"""Benchmark of the stacked (ragged) three_nn / three_interpolate and StackPointnetFPModule on one GPU; prints ONE JSON line.

    python scripts/bench_stack_fp.py [--iters 20] [--warmup 5] [--seed 0]

Shapes: B = 4 ragged frames.
  layer a: 12k-18k unknown points per frame (seeded sizes) <- a quarter of them known, C2 = 128, C1 = 64,
           mlp [192, 128, 128];
  layer b: 1024 unknown <- 256 known points per frame, C2 = 512, C1 = 256, mlp [768, 512, 512].
Reported per layer:
  * three_nn: the per-frame grids (default) and brute force (TSMDET_NN_ALGO=brute), in ms;
  * three_interpolate (rows), in ms and in GB/s of the compulsory bytes 4 M C2 + 24 N + 4 N C2;
  * the module: eager and fused fp32 / bf16 / tf32, in ms, with the kernel the layer's MLP ran in (an MLP the tensor
    path does not pack runs in the fp32 FMA kernel);
  * eager vs fused parity metrics (tests/parity.py) at the timed size;
  * the GPU's name and power limit, read in the same run.
The inputs are a few MB to a few tens of MB, so they would sit in L2 after the first pass: a 256 MB buffer is overwritten
before every timed call, and CUDA events time the call alone.
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

LAYERS = {
    "a": dict(c2=128, c1=64, mlp=[192, 128, 128]),
    "b": dict(c2=512, c1=256, mlp=[768, 512, 512]),
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


def inputs(layer, rng, seed, frames=4):
    import synth

    if layer == "a":
        usz = rng.integers(12000, 18001, frames)
        ksz = usz // 4
    else:
        usz, ksz = np.full(frames, 1024), np.full(frames, 256)
    fu = [synth.cloud_ground_objects(1, int(n), seed=seed + 1 + k)[0] for k, n in enumerate(usz)]
    fk = [f[rng.choice(len(f), int(m), replace=False)] for f, m in zip(fu, ksz)]
    return (np.concatenate(fu, 0), usz.astype(np.int32), np.concatenate(fk, 0), ksz.astype(np.int32))


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
        raise SystemExit("bench_stack_fp.py measures on a CUDA device; none is visible")

    import parity
    from tsmdet_b200 import _lib
    from tsmdet_b200.pointnet2_stack import StackPointnetFPModule
    from tsmdet_b200.pointnet2_stack import pointnet2_utils as pu
    from tsmdet_b200.pointnet2_stack.pointnet2_modules import _dense_precision

    dev = torch.device("cuda:0")
    name, power = gpu_identity()
    rng = np.random.default_rng(args.seed)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"metric": "stack_fp", "gpu": name, "power_limit": power, "iters": args.iters, "layers": {}}

    for key, cfg in LAYERS.items():
        un_np, ucnt_np, kn_np, kcnt_np = inputs(key, rng, args.seed)
        un, ucnt, kn, kcnt = (torch.from_numpy(a).to(dev) for a in (un_np, ucnt_np, kn_np, kcnt_np))
        n, m = un.shape[0], kn.shape[0]
        kf = torch.from_numpy(rng.standard_normal((m, cfg["c2"])).astype(np.float32)).to(dev)
        uf = torch.from_numpy(rng.standard_normal((n, cfg["c1"])).astype(np.float32)).to(dev)
        rec = {"frames_unknown": ucnt_np.tolist(), "frames_known": kcnt_np.tolist(), "c2": cfg["c2"], "c1": cfg["c1"],
               "mlp": cfg["mlp"], "three_nn": {}}
        for impl in ("grid", "brute"):
            os.environ.pop("TSMDET_NN_ALGO", None)
            if impl == "brute":
                os.environ["TSMDET_NN_ALGO"] = "brute"
            _lib.reload_options()
            rec["three_nn"][impl] = {"ms": round(timed(lambda: pu.three_nn(un, ucnt, kn, kcnt), args.iters, args.warmup,
                                                       flush), 4)}
        os.environ.pop("TSMDET_NN_ALGO", None)
        _lib.reload_options()

        dist, idx = pu.three_nn(un, ucnt, kn, kcnt)
        w = 1.0 / (dist + 1e-8)
        w = w / w.sum(-1, keepdim=True)
        t = timed(lambda: pu.three_interpolate(kf, idx, w), args.iters, args.warmup, flush)
        nbytes = 4 * m * cfg["c2"] + 24 * n + 4 * n * cfg["c2"]
        rec["three_interpolate"] = {"ms": round(t, 4), "GBps": round(nbytes / t / 1e6, 1)}

        torch.manual_seed(args.seed)
        mod = StackPointnetFPModule(mlp=cfg["mlp"]).to(dev).eval()
        torch.backends.cudnn.allow_tf32 = False
        mod.fused = False
        with torch.no_grad():
            want = mod(un, ucnt, kn, kcnt, uf, kf)
            rec["eager_fp32"] = {"ms": round(timed(lambda: mod(un, ucnt, kn, kcnt, uf, kf), args.iters, args.warmup,
                                                   flush), 4)}
            mod.fused = True
            for prec in ("fp32", "bf16", "tf32"):
                mod.precision = prec
                mod._folded = None
                got = mod(un, ucnt, kn, kcnt, uf, kf)
                t = timed(lambda: mod(un, ucnt, kn, kcnt, uf, kf), args.iters, args.warmup, flush)
                met = parity.err_metrics(got, want)
                kernel = {"fp32": "fp32 FMA"}.get(_dense_precision(prec, mod._packed[1]), f"tcgen05 {prec}")
                rec[f"fused_{prec}"] = {"ms": round(t, 4), "kernel": kernel,
                                        "parity": {k: float(f"{v:.3e}") for k, v in met.items()},
                                        "within_bars": all(met[k] <= bar for k, bar in parity.BARS[prec].items())}
        out["layers"][key] = rec
    print(json.dumps(out))


if __name__ == "__main__":
    main()
