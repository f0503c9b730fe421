#!/usr/bin/env python
"""bench.py -- frames/s of the SA backbone + rotated NMS hot path (BASELINE.json metric).

    python bench.py --gpus 1 --steps 50 --warmup 8                  # this repo's sm_100a path
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...                             # reference CPU arm (oracle port)

A "step" = one pass of the hot path over one batch of synthetic frames per GPU:
  config 2  KITTI SA stack 16384 -> 4096 -> 1024 -> 512 (radii 0.2/0.8/1.6, nsample 16/32/32,
            MLPs [4,16,16,32] [35,64,64,128] [131,128,128,256]), batch 16 frames per GPU, plus
  config 3  rotated NMS on 4096 proposals per frame, IoU 0.01 then 0.1 on the survivors; at N > 1 the
            padded detections are gathered on every rank (frames are sharded, weak scaling): one kernel of
            peer-memory stores per step by default, the NCCL all_gather with TSMDET_GATHER=nccl.
Prints ONE JSON line (rank 0).  `value` = frames/s with inputs resident in HBM; `e2e` = the same through the
host-buffer API (one pinned collated input buffer H2D + one packed result buffer D2H per step, inside the timed
region).  Each is measured over exactly K = `--steps` timed steps (split into `--repeats` regions, one by default).
After the timed regions the last step's results are verified against the oracle (`verified`), the unmodified reference
CUDA extension is timed on the same inputs (`ref_cuda_baseline`) and the other BASELINE configs are measured
(`secondary`).  `--dump-outputs DIR` writes the arrays the last timed device-resident step returned as DIR/<name>.npy; the
inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")  # before any CUDA call: see tsmdet_b200/__init__.py (both arms)
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FRAMES_PER_GPU = 16
N_POINTS = 16384
N_PROPOSALS = 4096
METRIC = "frames/sec (SA backbone+NMS, 16384 pts/frame)"
WORKLOAD = ("KITTI SA stack 16384->4096->1024->512 (r 0.2/0.8/1.6, ns 16/32/32) batch 16/GPU + rotated NMS "
            "4096 proposals/frame IoU 0.01 then 0.1")
# (npoint, radius, nsample, MLP incl. the +3 xyz channels) per SA layer of config 2
SA_LAYERS = ((4096, 0.2, 16, (4, 16, 16, 32)), (1024, 0.8, 32, (35, 64, 64, 128)), (512, 1.6, 32, (131, 128, 128, 256)))


def common_config(world: int) -> dict:
    """The `config` object, identical in both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "frames_per_gpu": FRAMES_PER_GPU, "points_per_frame": N_POINTS,
            "proposals_per_frame": N_PROPOSALS, "parallelism": f"frames sharded x{world}",
            "l2": "GPU arm: a 256 MB buffer is written before every step, inside the timed region"}


# ------------------------------------------------------------------------------------ inputs
def make_inputs(frames: int, seed: int):
    import numpy as np
    import synth

    xyz = np.concatenate([synth.cloud_ground_objects(frames // 2, N_POINTS, seed),
                          synth.cloud_dup_padded(frames - frames // 2, N_POINTS, seed + 1)], 0)
    feats = np.random.default_rng(seed + 2).uniform(0, 1, size=(frames, 1, N_POINTS)).astype(np.float32)
    boxes = np.stack([synth.boxes_clustered(N_PROPOSALS, seed + 10 + i, centres=200) for i in range(frames)])
    scores = np.stack([synth.scores_random(N_PROPOSALS, seed + 100 + i) for i in range(frames)])
    return xyz, feats, boxes, scores


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: an in-process NVML thread (about 250 Hz;
    only the samples whose timestamps fall inside [start(), stop()] are kept), nvidia-smi -lms as the fallback."""

    REASONS = (("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40), ("sw_power_cap", 0x4))

    def __init__(self, device):
        self.device, self.rows, self.proc, self.nvml, self.handle = device, [], None, None, None
        self._stop = threading.Event()
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            props = torch.cuda.get_device_properties(device)
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(props.uuid)).encode())
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(device.index or 0)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _loop(self):
        nv, h = self.nvml, self.handle
        while not self._stop.is_set():
            try:
                self.rows.append((time.perf_counter(), float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                                  int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))))
            except Exception:
                break
            time.sleep(0.004)  # ~250 Hz: NVML calls hold the GIL, the timed loop needs it

    def start(self):
        self.t0 = time.perf_counter()
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
            return
        try:
            q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                 "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20", "-i", str(self.device.index or 0)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        t1 = time.perf_counter()
        if self.nvml is not None:
            self._stop.set()
            self.thread.join(timeout=1.0)
            nv = self.nvml
            inside = [r for r in self.rows if self.t0 <= r[0] <= t1]
            sm = sorted(r[1] for r in inside)
            bits = 0
            for r in inside:
                bits |= r[2]
            try:
                mx = float(nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM))
            except Exception:
                mx = None
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx,
                    "reasons": sorted(n for n, b in self.REASONS if bits & b), "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------ reference-shaped MLPs
def build_eager_mlps(device=None):
    """The shared MLPs of config 2 as the reference builds them (Conv2d 1x1 without bias -> BatchNorm2d -> ReLU,
    pointnet2_modules.py:1549-1555), plain torch.nn -- nothing from this repo's package."""
    import torch
    from torch import nn

    torch.manual_seed(0)
    mlps = []
    for _, _, _, spec in SA_LAYERS:
        mods = []
        for k in range(len(spec) - 1):
            mods += [nn.Conv2d(spec[k], spec[k + 1], kernel_size=1, bias=False), nn.BatchNorm2d(spec[k + 1]), nn.ReLU()]
        mlps.append(nn.Sequential(*mods))
    g = torch.Generator().manual_seed(1)
    for seq in mlps:
        for m in seq:
            if isinstance(m, nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
        seq.eval()
        if device is not None:
            seq.to(device)
    return mlps


# ------------------------------------------------------------------------------------ CPU arm
def cpu_frames_per_second(frames: int, threads: int, seed: int = 0, mlps=None):
    """The oracle port (this repo's C restatement of the reference kernels + torch-CPU fp32 MLP) on the
    host cores, over `frames` frames of the same workload.  Returns (frames/s, seconds)."""
    import numpy as np
    import torch

    from oracle import oracle as orc

    orc.build()
    orc.set_threads(threads)
    torch.set_num_threads(threads)
    xyz, feats, boxes, scores = make_inputs(max(frames, 2), seed)
    xyz, feats, boxes, scores = xyz[:frames], feats[:frames], boxes[:frames], scores[:frames]
    mlps = mlps if mlps is not None else build_eager_mlps()
    t0 = time.perf_counter()
    cur_xyz, cur_f = xyz, feats
    with torch.no_grad():
        for (npoint, radius, nsample, _), mlp in zip(SA_LAYERS, mlps):
            idx = orc.fps(cur_xyz, npoint)
            new_xyz = np.take_along_axis(cur_xyz, idx.astype(np.int64)[..., None], axis=1)
            cnt, nf, _, _ = orc.query_and_group(cur_xyz, new_xyz, cur_f, radius, nsample)
            x = torch.from_numpy(nf) * torch.from_numpy((cnt > 0).astype(np.float32))[:, None, :, None]
            y = mlp(x).max(dim=3)[0]
            cur_xyz, cur_f = new_xyz, y.numpy()
    for i in range(frames):
        order = np.argsort(-scores[i], kind="stable")
        k1 = orc.nms_sorted(boxes[i][order], 0.01)
        orc.nms_sorted(boxes[i][order][k1], 0.1)
    dt = time.perf_counter() - t0
    return frames / dt, dt


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path (the pointnet2 ops are CUDA-only in
    the reference, so this is the oracle port of those kernels + its rotated-IoU CPU code), all host threads.
    Nothing of this repo's product package is imported."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    mlps = build_eager_mlps()
    t_w = time.perf_counter()
    for _ in range(args.warmup):  # W warm-up steps on a 2-frame sample (page-in, thread pools, oracle build)
        cpu_frames_per_second(2, cores, mlps=mlps)
    per_frame = (time.perf_counter() - t_w) / max(1, 2 * args.warmup)
    # every step is a bounded sample of the per-GPU batch, sized so that K steps end within ~4 minutes
    frames_per_step = FRAMES_PER_GPU
    while frames_per_step > 2 and frames_per_step * per_frame * args.steps > 200.0:
        frames_per_step //= 2
    secs = []
    for _ in range(args.steps):
        _, dt = cpu_frames_per_second(frames_per_step, cores, mlps=mlps)
        secs.append(dt)
    value = len(secs) * frames_per_step / sum(secs)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * sum(secs) / len(secs),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": common_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{frames_per_step} frame(s) of the same workload per step, {len(secs)} steps, "
                                   f"OpenMP C oracle of the reference kernels + torch-CPU fp32 MLP + oracle rotated "
                                   f"NMS on {cores} threads"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ host affinity
def pin_to_gpu_numa_node(dev_index: int):
    """Run this rank's host thread (and so first-touch its pinned buffers) on the NUMA node its GPU hangs off:
    eight ranks' pinned copies through one socket's memory controllers were the e2e wall of round 1."""
    try:
        import torch

        bus = torch.cuda.get_device_properties(dev_index).pci_bus_id
        dom = torch.cuda.get_device_properties(dev_index).pci_domain_id
        devid = torch.cuda.get_device_properties(dev_index).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{devid:02x}.0/numa_node"
        with open(path) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        cpus &= allowed
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": node, "cpus": len(cpus)}
    except Exception:  # noqa: BLE001 -- affinity is an optimisation, never a requirement
        return None
    return None


# ------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--repeats", type=int, default=1, help="timed regions the K steps are split into")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("TSMDET_BENCH_PRECISION", "bf16"), choices=["fp32", "bf16", "tf32"])
    ap.add_argument("--depth", type=int, default=int(os.environ.get("TSMDET_BENCH_DEPTH", "8")),
                    help="steps kept in flight (each on its own stream / CUDA graph / buffers)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip verify / ref_cuda_baseline / secondary configs")
    ap.add_argument("--profile-kernels", action="store_true", help="per-kernel CUDA-event breakdown to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step as DIR/<name>.npy (float32, integers as float64)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        return run_reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    affinity = pin_to_gpu_numa_node(local_rank) if os.environ.get("TSMDET_BENCH_NO_AFFINITY", "0") == "0" else None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from tsmdet_b200 import _lib
    from tsmdet_b200.pipeline import PipelinedRunner

    depth = max(1, args.depth)
    xyz_np, feats_np, boxes_np, scores_np = make_inputs(FRAMES_PER_GPU, seed=1000 * rank)
    d0 = [torch.from_numpy(a).to(dev) for a in (xyz_np, feats_np, boxes_np, scores_np)]
    runner = PipelinedRunner(depth=depth, device=dev, precision=args.precision)
    lane_inputs = runner.prepare(*d0)  # captures one CUDA graph per lane; inputs stay resident in HBM
    # the host front door: every lane gets a pinned, collated copy of the batch (filled once, outside the timed region,
    # as a data loader's collate would) and captures its staged graph
    ios = runner.prepare_host(*[torch.from_numpy(a) for a in (xyz_np, feats_np, boxes_np, scores_np)])
    engine = runner.engines[0]
    gather = world > 1 and os.environ.get("TSMDET_BENCH_NO_GATHER", "0") == "0"  # (experiments only)
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def flush():
        flush_buf.zero_()  # L2 flush before every step, inside the timed region (on the step's own stream)

    def timed(submit, steps):
        """K steps, `depth` in flight; device time between one start and one end event on the main stream."""
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        runner.fork()
        t_host = time.perf_counter()
        for _ in range(steps):
            submit()
        host_ms.append((time.perf_counter() - t_host) * 1e3 / max(1, steps))  # host time to ENQUEUE one step
        runner.join()
        e.record()
        torch.cuda.synchronize(dev)
        return s.elapsed_time(e)

    host_ms = []

    def timed_repeats(submit):
        """Exactly K steps in `--repeats` regions, each bracketed by barrier + synchronize; per region the MAX over
        ranks; returns (list of region ms, total ms)."""
        regions = max(1, min(args.repeats, args.steps))
        out = []
        for i in range(regions):
            barrier()
            steps = args.steps // regions + (i < args.steps % regions)
            t = torch.tensor([timed(submit, steps)], dtype=torch.float64, device=dev)
            barrier()
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            out.append(float(t))
        return out, sum(out)

    last = {}

    def dev_step():
        last["res"] = runner.submit_device(lane_inputs, gather=gather, pre=flush)[1]

    host_step = lambda: runner.submit_host(gather=gather, pre=flush)  # noqa: E731

    for _ in range(depth):  # prime every lane once (graph upload, first collective) whatever --warmup is
        dev_step()
    runner.sync()
    for _ in range(args.warmup):
        dev_step()
    runner.sync()
    barrier()
    gather_transport = None
    if gather:
        # outside the timed region: whatever transport the gather uses, every rank must now hold exactly what an NCCL
        # all_gather of the last step's packed records returns
        from tsmdet_b200.sharding import gather_packed

        for eng in runner.engines[:2]:
            res = eng.forward_device(*lane_inputs[0], gather=True)
            all_det, all_num = res["all_det"].clone(), res["all_num"].clone()
            torch.cuda.synchronize(dev)
            gather_transport = ("peer-memory stores (tsmdet_peer_put: ring of 4 slots + credits), one kernel per step"
                                if eng._pg is not None else "nccl all_gather")
            f, k = res["det"].shape[0], res["det"].shape[1]
            ref_det, ref_num, _ = gather_packed(res["det_packed"], f, k)
            torch.cuda.synchronize(dev)
            if not (torch.equal(all_det, ref_det) and torch.equal(all_num, ref_num)):
                raise RuntimeError("detection gather differs from the NCCL all_gather of the same records")
        barrier()
    sampler = ClockSampler(dev)
    sampler.start()
    l0 = _lib.launch_count
    t_wall = time.perf_counter()
    dev_regions, ms_total = timed_repeats(dev_step)
    wall = time.perf_counter() - t_wall
    launches = _lib.launch_count - l0
    clocks = sampler.stop()
    # copied before any later step can replay the last timed step's graph and overwrite its results
    # (`packed` / `det_packed` are left out: they are the same bytes as features | xyz | det | det_num)
    dumped = ({k: v.cpu().numpy().astype(np.float32 if v.is_floating_point() else np.float64)
               for k, v in last["res"].items() if k not in ("packed", "det_packed")}
              if args.dump_outputs and rank == 0 else None)
    for _ in range(depth + args.warmup):
        host_step()
    runner.sync()
    barrier()
    e2e_regions, ms_e2e_total = timed_repeats(host_step)
    runner.sync()
    runner.check()
    status = _lib.read_status()
    if status != 0:
        raise RuntimeError(f"watchdog status {status} after the timed regions")

    # the ceiling of the host side: the same pinned copies (same bytes, same lanes / streams), no compute
    def copy_step():
        lane_id = copy_step.i % depth
        copy_step.i += 1
        io, lane = ios[lane_id], runner.lanes[lane_id]
        ent = runner.engines[lane_id]._graph_for_host(io, dev)
        with torch.cuda.stream(lane):
            ent["in"][0].copy_(io.inp, non_blocking=True)
            io.out.copy_(ent["out"]["packed"], non_blocking=True)
            if gather and rank == 0 and io.all is not None:
                io.all.copy_(ent["out"]["packed"][: io.all.numel()].view_as(io.all), non_blocking=True)
    copy_step.i = 0
    for _ in range(depth):
        copy_step()
    runner.sync()
    _, ms_copy_total = timed_repeats(copy_step)

    # single-step latency (one step in flight, no flush inside the events)
    lat = []
    for _ in range(5):
        flush()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        engine.forward_device(*lane_inputs[0])
        e.record()
        torch.cuda.synchronize(dev)
        lat.append(s.elapsed_time(e))
    lat.sort()

    t_dev, t_e2e, t_copy = ms_total / 1000.0, ms_e2e_total / 1000.0, ms_copy_total / 1000.0
    frames_total = FRAMES_PER_GPU * world * args.steps
    value = frames_total / t_dev
    e2e = frames_total / t_e2e
    d = lane_inputs[0]

    # ---- per-kernel breakdown + roofline (CUDA events on the launching stream)
    roof, kernels = kernel_breakdown(engine, d, dev, args, ms_total / args.steps)

    cfg = common_config(world)
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * t_dev / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": {"bf16": "bf16", "tf32": "tf32", "fp32": "f32"}[args.precision],
        "data": "synthetic", "config": cfg,
        "e2e": {"value": e2e, "unit": "frames/s", "h2d_bytes_per_step": int(ios[0].h2d_bytes),
                "d2h_bytes_per_step": int(ios[0].d2h_bytes(rank == 0 and gather)),
                "copies_per_step": "1 H2D (collated points | boxes | scores, one pinned buffer) + 1 D2H (features | xyz | "
                                   "records, one packed buffer)" + (" + 1 D2H of the gathered records on rank 0" if gather else ""),
                "copy_ceiling": {"value": frames_total / t_copy, "unit": "frames/s",
                                 "what": "the same pinned copies on the same streams with no compute"},
                "host_affinity": affinity},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roof,
        "fps_ms_per_cloud": next((k["ms"] for k in kernels if k["name"] == "fps_L1"), None),
        "repeats": {"n": len(dev_regions), "statistic": "sum", "ms_per_region_device": dev_regions,
                    "ms_per_region_e2e": e2e_regions},
        "execution": {"mlp_precision": args.precision, "pipeline_depth": depth,
                      "graph": "one CUDA graph per step (FPS chain, query+MLP, NMS on 3 concurrent streams); "
                               f"{depth} step(s) in flight on separate streams/buffers",
                      "fps": "one CTA per cloud, exact spatial pruning, rounds of up to 8 picks (fps_bucket_kernel); levels "
                             "2/3 CHAINED (look-ups proven exact by level 1's record; the un-chained stand-alone times are "
                             "fps_L2 / fps_L3 in roofline.per_kernel)",
                      "ms_per_step_single_in_flight": lat[len(lat) // 2], "gather": gather_transport,
                      "cuda_device_max_connections": os.environ.get("CUDA_DEVICE_MAX_CONNECTIONS"),
                      # host time to ENQUEUE one step (python + graph launch [+ gather kernels]), median over the regions:
                      # when it approaches ms_per_step the host, not the GPU, sets the pace
                      "host_enqueue_ms_per_step": {"device": sorted(host_ms[:len(dev_regions)])[len(dev_regions) // 2],
                                                   "e2e": sorted(host_ms[len(dev_regions):2 * len(dev_regions)])[len(dev_regions) // 2]}},
        "kernels": kernels, "wall_s_timed_region": wall,
    }
    extras = rank == 0 and world == 1 and not args.no_extras
    if extras:
        from oracle import oracle as orc  # the checker, outside every timed region

        import parity

        orc.build()
        _, res = runner.submit_device(lane_inputs)
        runner.sync()
        m = parity.verify_step(engine, orc, xyz_np, feats_np, boxes_np, scores_np, res, args.precision)
        io = ios[(runner._i - 1) % depth]
        host = {"xyz": io.xyz, "features": io.features, "det": io.det, "det_num": io.det_num}
        parity.verify_step(engine, orc, xyz_np, feats_np, boxes_np, scores_np, host, args.precision, frames=[0, 15])
        line["verified"] = True
        line["verification"] = {"against": "CPU oracle (FPS chain, greedy NMS sweep) + eager fp32 stack, all 16 frames of the "
                                           "last device-resident step; frames 0 and 15 of the last host-API step",
                                "indices_and_keep_lists": "bit-exact", **{k: m[k] for k in
                                ("max_abs_over_scale", "rel_l2", "max_rel_big", "max_rel_all", "detections_checked")}}
        try:
            line["ref_cuda_baseline"] = ref_cuda_baseline(d, dev)
        except Exception as ex:  # noqa: BLE001 -- a baseline leg must not void the measured line
            line["ref_cuda_baseline"] = {"unavailable": f"{type(ex).__name__}: {ex}"}
        try:
            line["secondary"] = secondary_configs(dev)
        except Exception as ex:  # noqa: BLE001
            line["secondary"] = {"unavailable": f"{type(ex).__name__}: {ex}"}
        try:
            line["secondary"]["tf32_stack"] = tf32_stack(d, dev, args, (xyz_np, feats_np, boxes_np, scores_np), orc)
        except Exception as ex:  # noqa: BLE001
            line["secondary"]["tf32_stack"] = {"unavailable": f"{type(ex).__name__}: {ex}"}
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        n_cpu = 32  # two per-GPU batches: about 10 s of host work, every core busy in the OpenMP loops over clouds
        v, dt = cpu_frames_per_second(n_cpu, cores)
        line["cpu_baseline"] = {"value": v, "unit": "frames/s", "cores": cores, "kind": "port",
                                "sample": f"{n_cpu} frames of the same workload ({dt:.1f} s): OpenMP C oracle of the reference "
                                          f"kernels + torch-CPU fp32 MLP + oracle rotated NMS"}
    elif rank == 0:
        line["cpu_baseline"] = None
    if dumped is not None:  # 8.8 MB for the 16-frame step
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        # Leave at once.  Tearing the process down piece by piece (NCCL communicator, the IPC mappings of
        # every peer's receive rings, 8 captured graphs per rank) took more than a minute after the line was printed in
        # one 8-GPU run of round 2; nothing below this point is needed, and the driver reclaims a dead process's resources.
        # (No collective here either: the last one -- the all_reduce of the copy-ceiling regions -- lies seconds back on
        # every rank, behind the per-kernel timing.)
        torch.cuda.synchronize(dev)
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def _graph_timer(dev, flush_mb: int = 256):
    """Returns t(fn, reps): device time of one stage, captured into a CUDA graph (as the timed step runs it -- no
    per-launch host cost between its kernels) and replayed between two events on the launching stream, cold L2."""
    import torch

    flush_buf = torch.empty(flush_mb * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def t(fn, reps=5):
        fn()
        torch.cuda.synchronize(dev)
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            fn()  # warm on the capture stream: grows that stream's scratch buffers
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                fn()
            graph.replay()
            times = []
            for _ in range(reps):
                flush_buf.zero_()  # cold L2 for every replay, as in the timed step
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record(side)
                graph.replay()
                e.record(side)
                e.synchronize()
                times.append(s.elapsed_time(e))
        torch.cuda.synchronize(dev)
        times.sort()
        return times[len(times) // 2]

    return t


def _peaks():
    peaks = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = dict(peaks, **json.load(f), src="measured")
    except OSError:
        pass
    return peaks


def _ncu_facts():
    """Per-launch facts taken from the committed `ncu --set full` captures (profiles/*_ncu_traffic.jsonl, newest
    round last): DRAM traffic, tensor-pipe activity, shared-memory wavefronts."""
    facts = {}
    pdir = os.path.join(ROOT, "profiles")
    for name in sorted(f for f in os.listdir(pdir) if f.endswith("_ncu_traffic.jsonl")) if os.path.isdir(pdir) else []:
        with open(os.path.join(pdir, name)) as f:
            for ln in f:
                try:
                    rec = json.loads(ln)
                except ValueError:
                    continue
                for fam in ("fps_bucket_kernel", "sa_mlp_tc", "mlp_tc2_kernel", "bq_grid_query", "bq_grid_build", "nms_lazy", "group_points",
                            "pointwise_mlp_tc", "voxel_centroid"):
                    if fam in rec.get("kernel", ""):
                        facts[fam] = dict(rec, source=name)
    return facts


def kernel_breakdown(engine, d, dev, args, ms_step):
    """Times each stage of one step on its own (CUDA events, graph replay, cold L2, median of 5) and builds the
    `roofline` object: `per_kernel` = one entry per kernel family with the bound that really limits it
    (SURVEY.md 8d: tensor for the MLP, HBM for query / group, a latency chain for FPS, pairs/s for NMS) and its
    share of the pipelined step's SM-time; the top-level entry = the family with the largest share."""
    import torch

    from tsmdet_b200 import iou3d_nms_utils, pointnet2_utils
    from tsmdet_b200.pointnet2_modules import gather_xyz, sa_mlp_maxpool

    peaks = _peaks()
    facts = _ncu_facts()
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    xyz, feats, boxes, scores = d
    b = xyz.shape[0]
    t = _graph_timer(dev)
    kernels = []
    ctx = {}
    cur_xyz, cur_f, cur_t = xyz, feats, None
    tot = {"fps": [0.0, 0.0], "mlp": [0.0, 0.0, 0.0], "bq": [0.0, 0.0, 0.0]}  # ms, sm_ms, (flops | bytes)
    with torch.no_grad():
        for li, layer in enumerate(engine.backbone.layers):
            n = cur_xyz.shape[1]
            m = layer.npoint_list[0]
            g = layer.groupers[0]
            ns = g.nsample
            c = cur_f.shape[1]
            idx = pointnet2_utils.farthest_point_sample(cur_xyz, m)
            ms_fps = t(lambda: pointnet2_utils.farthest_point_sample(cur_xyz, m))
            new_xyz = gather_xyz(cur_xyz, idx)
            cnt, bidx = pointnet2_utils.ball_query(g.radius, ns, cur_xyz, new_xyz)
            ms_bq = t(lambda: pointnet2_utils.ball_query(g.radius, ns, cur_xyz, new_xyz))
            layers = layer._folded_layers()[0]
            img = layer._packed_layers(c, True)[0]
            cout = layers[-1][0].shape[0]
            out = torch.empty((b, cout, m), device=dev)
            # as in the pipelined step: layers hand their features on as bf16 rows (no fp32 tensor / transpose between)
            chain_out = img is not None and li + 1 < len(engine.backbone.layers)
            row_dt, row_q = (torch.bfloat16, 8) if layer.precision == "bf16" else (torch.float32, 4)
            out_t = torch.empty((b, m, (cout + row_q - 1) // row_q * row_q), dtype=row_dt, device=dev) if chain_out else None
            f_in, t_in = (None, cur_t) if cur_t is not None else (cur_f, None)
            ms_mlp = t(lambda: sa_mlp_maxpool(cur_xyz, new_xyz, f_in, bidx, cnt, layers, out, 0, precision=layer.precision,
                                              packed=img, feat_t=t_in, out_t=out_t))
            next_t = out_t
            fps_bytes = b * (12 * n + 4 * m)
            bq_bytes = b * (12 * n + 12 * m + 4 * m * ns + 4 * m)
            chans = [3 + c] + [w.shape[0] for w, _ in layers]
            flops = b * 2 * m * ns * sum(chans[i] * chans[i + 1] for i in range(len(chans) - 1))
            sa_bytes = b * (12 * n + 4 * c * n + 12 * m + 4 * chans[-1] * m + 4 * m * ns)
            kernels += [
                {"name": f"fps_L{li + 1}", "ms": ms_fps, "alg_bytes": fps_bytes, "gbs": fps_bytes / ms_fps / 1e6,
                 "us_per_iter": 1000.0 * ms_fps / max(m - 1, 1), "point_updates_per_s": b * n * (m - 1) / ms_fps * 1e3},
                {"name": f"ball_query_L{li + 1}", "ms": ms_bq, "alg_bytes": bq_bytes, "gbs": bq_bytes / ms_bq / 1e6,
                 "tests_per_s": b * n * m / ms_bq * 1e3},
                {"name": f"sa_mlp_maxpool_L{li + 1}", "ms": ms_mlp, "alg_bytes": sa_bytes, "gbs": sa_bytes / ms_mlp / 1e6,
                 "tflops": flops / ms_mlp / 1e9, "flops": flops},
            ]
            if li == 0:  # in the pipelined step levels 2/3 are chained look-ups: only level 1 costs sampler SM-time
                tot["fps"][0] += ms_fps
                tot["fps"][1] += ms_fps * min(b, sms)  # one CTA (one SM) per cloud
            tot["mlp"][0] += ms_mlp
            tot["mlp"][1] += ms_mlp * sms                # persistent: every SM
            tot["mlp"][2] += flops
            tot["bq"][0] += ms_bq
            tot["bq"][1] += ms_bq * sms * 0.6            # build: one CTA per cloud; query: every SM (ncu: 0.049 / 0.034 ms)
            tot["bq"][2] += bq_bytes
            ctx = {"xyz": cur_xyz, "f": cur_f, "idx": bidx}
            cur_xyz, cur_f, cur_t = new_xyz, out, next_t
        # the API-level (materialising) grouping op on the last layer's shape: the HBM-bound kernel of the path
        lay = engine.backbone.layers[-1]
        g3 = lay.groupers[0]
        src_xyz, src_f = ctx["xyz"], ctx["f"]
        c3, n3, m3, s3 = src_f.shape[1], src_xyz.shape[1], lay.npoint_list[0], g3.nsample
        ms_grp = t(lambda: pointnet2_utils.grouping_operation(src_f, ctx["idx"]))
        grp_bytes = b * (4 * c3 * n3 + 4 * m3 * s3 + 4 * c3 * m3 * s3)
        kernels.append({"name": f"grouping_operation_L{len(engine.backbone.layers)} (API op, not on the fused path)",
                        "ms": ms_grp, "alg_bytes": grp_bytes, "gbs": grp_bytes / ms_grp / 1e6,
                        "hbm_frac": grp_bytes / ms_grp / 1e6 / float(peaks["hbm_gbs"])})
        ms_nms = t(lambda: iou3d_nms_utils.nms_gpu_batch(boxes, scores, 0.01))
        p = boxes.shape[1]
        pairs = b * p * (p - 1) / 2
        kernels.append({"name": "nms_batch(0.01)", "ms": ms_nms, "alg_bytes": b * 36 * p, "gbs": b * 36 * p / ms_nms / 1e6,
                        "pairs_per_s": pairs / ms_nms * 1e3})

    hbm, tens = float(peaks["hbm_gbs"]), float(peaks["bf16_tflops"])
    k1 = next(k for k in kernels if k["name"] == "fps_L1")
    # latency floor of one pick: a pick cannot take less than one dependent pass argmax -> broadcast -> update of a
    # single SM: LDS 29 + REDUX ~30 + BAR ~30 + 4 dependent FMA/MNMX ~20 + winner's coordinate LDS 29 ~= 140 cycles
    floor_us = 140.0 / (float(peaks.get("sm_max_mhz", 1965.0)))
    step_sm_ms = ms_step * sms
    fam = [
        {"kernel": "fps_bucket_kernel<1024,16,8> (FPS 16384->4096; levels 2/3 chained)", "bound": "latency",
         "achieved": k1["us_per_iter"], "peak": floor_us, "unit": "us/pick (lower is better; peak = dependent-chain floor)",
         "frac": floor_us / k1["us_per_iter"], "ms": tot["fps"][0], "sm_ms": tot["fps"][1],
         "hbm_gbs": k1["gbs"], "hbm_frac": k1["gbs"] / hbm,
         "smem_wavefronts_per_launch": facts.get("fps_bucket_kernel", {}).get("smem_wavefronts"),
         "traffic": facts.get("fps_bucket_kernel", {}).get("dram_bytes")},
        {"kernel": "mlp_tc2_kernel (3 launches: SA L1+L2+L3, tcgen05 bf16)", "bound": "tensor",
         "achieved": tot["mlp"][2] / tot["mlp"][0] / 1e9, "peak": tens, "unit": "TFLOP/s",
         "frac": tot["mlp"][2] / tot["mlp"][0] / 1e9 / tens, "ms": tot["mlp"][0], "sm_ms": tot["mlp"][1],
         "per_layer": [{"layer": i + 1, "ms": k["ms"], "tflops": k["tflops"], "frac": k["tflops"] / tens}
                       for i, k in enumerate(k for k in kernels if k["name"].startswith("sa_mlp"))],
         "tensor_pipe_pct": facts.get("mlp_tc2_kernel", {}).get("tensor_pct"),  # layer 3, ncu --set full (profiles/)
         "traffic": facts.get("mlp_tc2_kernel", {}).get("dram_bytes")},
        {"kernel": "bq_grid_build + bq_grid_query (3 layers)", "bound": "hbm", "achieved": tot["bq"][2] / tot["bq"][0] / 1e6,
         "peak": hbm, "unit": "GB/s", "frac": tot["bq"][2] / tot["bq"][0] / 1e6 / hbm, "ms": tot["bq"][0],
         "sm_ms": tot["bq"][1], "traffic": facts.get("bq_grid_query", {}).get("dram_bytes")},
        {"kernel": "nms_lazy_kernel (IoU 0.01 pass, 4096 boxes/frame)", "bound": "alu", "achieved": pairs / ms_nms * 1e3 / 1e9,
         "peak": None, "unit": "G nominal pairs/s", "frac": None, "ms": ms_nms, "sm_ms": ms_nms * min(b, sms)},
        {"kernel": "group_points (API op, K-L3 shape; not on the fused path)", "bound": "hbm",
         "achieved": grp_bytes / ms_grp / 1e6, "peak": hbm, "unit": "GB/s", "frac": grp_bytes / ms_grp / 1e6 / hbm,
         "ms": ms_grp, "sm_ms": 0.0, "traffic": facts.get("group_points", {}).get("dram_bytes")},
    ]
    for f in fam:
        f["sm_time_share_of_step"] = f["sm_ms"] / step_sm_ms if step_sm_ms > 0 else None
    top = max(fam, key=lambda f: f["sm_ms"])
    roof = {"kernel": top["kernel"], "bound": top["bound"], "achieved": top["achieved"], "peak": top["peak"],
            "unit": top["unit"], "frac": top["frac"], "traffic": top.get("traffic"), "peak_source": peaks["src"],
            "chosen_by": "largest share of the pipelined step's SM-time (ms x SMs occupied)",
            "timing": "each stage replayed from its own CUDA graph, cold L2, CUDA events on the launching stream, median of 5; "
                      "tensor fractions are against the BURST bf16 peak (isolated timing), HBM against the measured copy",
            "per_kernel": fam}
    if args.profile_kernels:
        for k in kernels:
            print(json.dumps(k), file=sys.stderr)
    return roof, kernels


def ref_cuda_baseline(d, dev):
    """The bar to beat (SURVEY.md 8d 'three things side by side'): the UNMODIFIED reference CUDA extension
    (oracle/_ref, rebuilt for sm_100a) + the reference's eager sequence (transpose / group / cat / mask / Conv2d /
    BatchNorm2d / ReLU / max_pool2d in fp32, pointnet2_utils.py:544-568, pointnet2_modules.py:1259-1300) + its
    nms_gpu (blocking mask copy + CPU sweep), on the SAME inputs and box, outside the timed region."""
    import torch

    from oracle import build_ref

    pn = build_ref.load_ref("pointnet2_batch_cuda")
    iou = build_ref.load_ref("iou3d_nms_cuda")
    if pn is None or iou is None:
        return {"unavailable": "oracle/_ref not built (needs /root/reference at build time)"}
    xyz, feats, boxes, scores = d
    b = xyz.shape[0]
    mlps = build_eager_mlps(dev)
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    per_op = {"fps": 0.0, "ball_query": 0.0, "group": 0.0, "mlp_maxpool": 0.0, "nms": 0.0}

    def step(record):
        cur_xyz, cur_f = xyz, feats
        marks = []

        def mark(name):
            if record:
                e = ev()
                e.record()
                marks.append((name, e))
        mark("start")
        with torch.no_grad():
            for (npoint, radius, nsample, _), mlp in zip(SA_LAYERS, mlps):
                n = cur_xyz.shape[1]
                idx = torch.empty((b, npoint), dtype=torch.int32, device=dev)
                temp = torch.full((b, n), 1e10, dtype=torch.float32, device=dev)
                pn.farthest_point_sampling_wrapper(b, n, npoint, cur_xyz, temp, idx)
                xyz_t = cur_xyz.transpose(1, 2).contiguous()
                new_t = torch.empty((b, 3, npoint), dtype=torch.float32, device=dev)
                pn.gather_points_wrapper(b, 3, n, npoint, xyz_t, idx, new_t)
                new_xyz = new_t.transpose(1, 2).contiguous()
                mark("fps")
                cnt = torch.zeros((b, npoint), dtype=torch.int32, device=dev)
                bidx = torch.zeros((b, npoint, nsample), dtype=torch.int32, device=dev)
                pn.ball_query_wrapper(b, n, npoint, radius, nsample, new_xyz, cur_xyz, cnt, bidx)
                mark("ball_query")
                gx = torch.empty((b, 3, npoint, nsample), dtype=torch.float32, device=dev)
                pn.group_points_wrapper(b, 3, n, npoint, nsample, xyz_t, bidx, gx)
                gx = gx - new_xyz.transpose(1, 2).unsqueeze(-1)
                c = cur_f.shape[1]
                gf = torch.empty((b, c, npoint, nsample), dtype=torch.float32, device=dev)
                pn.group_points_wrapper(b, c, n, npoint, nsample, cur_f.contiguous(), bidx, gf)
                nf = torch.cat([gx, gf], dim=1) * (cnt > 0).float().unsqueeze(1).unsqueeze(-1)
                mark("group")
                y = torch.nn.functional.max_pool2d(mlp(nf), kernel_size=[1, nsample]).squeeze(-1)
                mark("mlp_maxpool")
                cur_xyz, cur_f = new_xyz, y.contiguous()
            for f in range(b):
                order = scores[f].sort(0, descending=True)[1]
                sb = boxes[f][order].contiguous()
                keep = torch.empty((sb.shape[0],), dtype=torch.int64)
                k1 = iou.nms_gpu(sb, keep, 0.01)
                sb2 = sb[keep[:k1].to(dev)].contiguous()
                keep2 = torch.empty((sb2.shape[0],), dtype=torch.int64)
                iou.nms_gpu(sb2, keep2, 0.1)
            mark("nms")
        return marks

    try:
        step(False)
        torch.cuda.synchronize(dev)
        reps = 3
        total = 0.0
        for _ in range(reps):
            t0 = time.perf_counter()
            marks = step(True)
            torch.cuda.synchronize(dev)
            total += time.perf_counter() - t0
            for (_, e0), (name, e1) in zip(marks[:-1], marks[1:]):
                per_op[name] += e0.elapsed_time(e1) / reps
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    sec = total / reps
    return {"value": b / sec, "unit": "frames/s", "ms_per_step": 1000.0 * sec, "per_op_ms": per_op,
            "what": "unmodified reference CUDA kernels (oracle/_ref, sm_100a build) + reference eager fp32 MLP (cuDNN, TF32 off) "
                    "+ reference nms_gpu, one 16-frame step at a time on the legacy default stream, wall clock with a "
                    "synchronize (its NMS blocks the host anyway), mean of 3"}


def tf32_stack(d, dev, args, d_np, orc):
    """The same SA stack with tf32 tensor-core operands (tcgen05 kind::tf32; layer 3 on a cluster pair): per-layer times
    measured like roofline.per_kernel, one whole step verified like the headline configuration with the tf32 bars."""
    import parity
    import torch

    from tsmdet_b200.pipeline import SABackboneNMS

    torch.manual_seed(0)
    eng = SABackboneNMS(precision="tf32").to(dev)
    res = eng.forward_device(*d)
    torch.cuda.synchronize(dev)
    m = parity.verify_step(eng, orc, *d_np, res, "tf32", frames=[0, 15])
    roof, _ = kernel_breakdown(eng, d, dev, args, 1.0)
    mlp = next(f for f in roof["per_kernel"] if f["bound"] == "tensor")
    tf32_peak = float(_peaks()["bf16_tflops"]) / 2  # kind::tf32 runs at half the bf16 rate
    return {"what": "SA L1+L2+L3 with tf32 operands (precision='tf32'), fp32 accumulate; L3 [131,128,128,256] on cluster pairs",
            "stack_ms": mlp["ms"], "per_layer": [{"layer": k["layer"], "ms": k["ms"], "tflops": k["tflops"],
                                                   "frac_of_tf32_peak": k["tflops"] / tf32_peak} for k in mlp["per_layer"]],
            "vs_eager_fp32": {k: m[k] for k in ("max_abs_over_scale", "rel_l2", "max_rel_big")},
            "indices_and_keep_lists": "bit-exact"}


def secondary_configs(dev):
    """The other BASELINE configs as bounded measurements (parity for these shapes lives in tests/): config 2b
    reference-true KITTI layer 0, config 4 Waymo frame FPS + query/group + FP layer, config 5 sweep-stack FPS."""
    import numpy as np
    import synth
    import torch

    from tsmdet_b200 import pointnet2_utils as pu
    from tsmdet_b200.pointnet2_modules import PointnetFPModule, PointnetSAModuleFSMSG

    t = _graph_timer(dev)
    peaks = _peaks()
    hbm = float(peaks["hbm_gbs"])
    out = {}
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
    with torch.no_grad():
        # ---- config 2b: N = 20000 -> 4096 (fast_cpc.yaml:52-56, 78-122), B = 16
        x = T(synth.cloud_ground_objects(16, 20000, 5))
        ms = t(lambda: pu.farthest_point_sample(x, 4096), reps=3)
        torch.manual_seed(0)
        layer0 = PointnetSAModuleFSMSG(npoint_list=[4096], sample_range_list=[[0, None]], sample_method_list=['d-fps'],
                                       radii=[0.2, 0.4, 0.8], nsamples=[32, 32, 32],
                                       mlps=[[1, 16, 16, 32], [1, 16, 16, 32], [1, 32, 32, 64]], dilated_radius_group=True,
                                       aggregation_mlp=[64], fused=True, precision="bf16").to(dev).eval()
        f1 = torch.rand((16, 1, 20000), device=dev)
        ms_layer = t(lambda: layer0(x, f1), reps=3)
        w = torch.rand((16, 4096), device=dev)
        x4 = x[:, :4096].contiguous()
        ms_sfps = t(lambda: pu.furthest_point_sample_weights(x4, w, 512), reps=3)
        out["config_2b"] = {"shape": "B=16, 20000->4096 d-FPS, dilated (0-0.2/0.2-0.4/0.4-0.8) ns 32, MLPs [4,16,16,32]x2 "
                                     "[4,32,32,64], agg 128->64, then s-FPS 4096->512",
                            "fps_ms": ms, "fps_ms_per_cloud": ms / 16, "fps_us_per_pick": 1000 * ms / 4095,
                            "layer0_ms": ms_layer, "frames_per_s_unpipelined": 16 / ((ms_layer + ms_sfps) / 1000),
                            "s_fps_ms": ms_sfps}
        del x, f1, layer0
        # ---- config 4: Waymo frame B = 8, N = 65536, 2 extra features
        x = T(synth.cloud_uniform(8, 65536, 7, synth.WAYMO_RANGE))
        ms_fps = t(lambda: pu.farthest_point_sample(x, 16384), reps=3)
        idx = pu.farthest_point_sample(x, 16384)
        from tsmdet_b200.pointnet2_modules import gather_xyz
        nx = gather_xyz(x, idx)
        ms_bq = t(lambda: pu.ball_query(0.8, 32, x, nx), reps=3)
        cnt, bidx = pu.ball_query(0.8, 32, x, nx)
        f2 = torch.rand((8, 2, 65536), device=dev)
        qg = pu.QueryAndGroup(0.8, 32, use_xyz=True)
        ms_qg = t(lambda: qg(x, nx, f2), reps=3)
        n, m, ns, c = 65536, 16384, 32, 2
        qg_bytes = 8 * ((12 * n + 12 * m + 4 * m * ns + 4 * m) + (4 * 3 * n + 4 * m * ns + 4 * 3 * m * ns)
                        + (4 * c * n + 4 * m * ns + 4 * c * m * ns) + 4 * (3 + c) * m * ns)
        kf = torch.rand((8, 128, 16384), device=dev)
        ms_nn = t(lambda: pu.three_nn(x, nx), reps=3)
        dist, nidx = pu.three_nn(x, nx)
        wgt = torch.rand((8, 65536, 3), device=dev)
        ms_int = t(lambda: pu.three_interpolate(kf, nidx, wgt), reps=3)
        int_bytes = 8 * (4 * 128 * m + 24 * n + 4 * 128 * n)
        torch.manual_seed(0)
        fp = PointnetFPModule(mlp=[128 + 2, 128, 128], precision="bf16").to(dev).eval()
        ms_fp = t(lambda: fp(x, nx, f2, kf), reps=3)
        fp_flops = 8 * 2 * n * (130 * 128 + 128 * 128)
        out["config_4"] = {"shape": "B=8, N=65536 (+2 features): FPS ->16384, ball query + group r=0.8 ns=32, FP layer "
                                    "three_nn(65536,16384) + three_interpolate C=128 + MLP [130,128,128]",
                           "fps_ms": ms_fps, "fps_ms_per_cloud": ms_fps / 8, "fps_us_per_pick": 1000 * ms_fps / 16383,
                           "ball_query_ms": ms_bq, "query_and_group_ms": ms_qg,
                           "query_and_group_gbs": qg_bytes / ms_qg / 1e6, "query_and_group_hbm_frac": qg_bytes / ms_qg / 1e6 / hbm,
                           "three_nn_ms": ms_nn, "three_interpolate_ms": ms_int,
                           "three_interpolate_gbs": int_bytes / ms_int / 1e6,
                           "three_interpolate_hbm_frac": int_bytes / ms_int / 1e6 / hbm,
                           "fp_module_ms": ms_fp, "fp_module_mlp_tflops_incl_nn_and_interp": fp_flops / ms_fp / 1e9}
        del x, nx, kf, f2, wgt, dist, nidx, cnt, bidx, fp
        # ---- config 5: sweep stack, ~180k points per sample, 2 clouds per GPU
        for npts in (163840, 180000):
            x = T(synth.cloud_uniform(2, npts, 9, synth.WAYMO_RANGE))
            ms5 = t(lambda: pu.farthest_point_sample(x, 16384), reps=2)
            idx = pu.farthest_point_sample(x, 16384)
            nx = gather_xyz(x, idx)
            ms5q = t(lambda: pu.ball_query(0.8, 32, x, nx), reps=2)
            out[f"config_5_n{npts}"] = {"shape": f"B=2 per GPU, N={npts}: FPS ->16384, ball query r=0.8 ns=32",
                                        "fps_ms": ms5, "fps_ms_per_cloud": ms5 / 2, "fps_us_per_pick": 1000 * ms5 / 16383,
                                        "ball_query_ms": ms5q}
            del x, nx
    return out


if __name__ == "__main__":
    main()
