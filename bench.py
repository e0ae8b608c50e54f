#!/usr/bin/env python
"""Benchmark of the DA-MVSNet cost-volume hot path (BASELINE.json metric: views/sec).

A "step" is one reference view's three-stage hot path (fused warp+aggregate ->
CostRegNet -> softmax/regression head, models/cas_mvsnet.py:18-134 of the
reference, three times) on synthetic DTU-test-shaped inputs: 1152x1600, N=5,
D=48/32/8, batch 1 (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W]        # this implementation
    python bench.py --impl reference ...                         # the reference's own DepthNet on the host cores
    python bench.py ... --dump-outputs DIR                       # also write the last timed step's outputs as DIR/*.npy

One process per GPU (torchrun for N>1); reference views are independent, so ranks
share nothing on the data path and the scaling is weak (K views per rank).
Prints ONE JSON line on rank 0.

Legs of the main line (all on the same box, same run):
  value          exactly K steps of the hot path, inputs resident in HBM, timed as one batch (max over ranks)
  e2e            the same through HotPathRunner.submit_host/collect from pinned host buffers
  roofline(s)    per-kernel-class device time (CUDA events around every C-ABI call) against SURVEY.md 8d's algorithmic
                 bytes / flops
  cpu_baseline   one full-size pass of the reference's own DepthNet x3 on the host cores (rank 0, N=1)
  incumbent_gpu  the reference's own PyTorch DepthNet x3 (nn.Conv3d / F.grid_sample, cudnn.benchmark as test_uni.py:29)
                 on this B200, fp32 with TF32 off and with PyTorch's defaults: the same-box number to beat
  extras         fp32-mode throughput, Tanks-and-Temples shape (configs[2]), training step with the NCCL gradient
                 all-reduce (configs[3]), full CascadeMVSNet forward images-in -> dict-out through the drop-in
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import math
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "views/sec at 1152x1600 N=5 D=48/32/8 (hot path: warp+aggregate, CostRegNet, regression head)"
UNIT = "views/s"


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400,
                    help="timed steps, run as one batch (the default covers about 1 s of device time on a B200)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16", "fp32"],
                    help="fp16 (default): fp16 features / cost volume / activations, tcgen05 convolutions, fp32 accumulate; "
                         "bf16: the same in bf16 (round 1's mode); fp32: the <= 1e-4 parity mode")
    ap.add_argument("--conv-impl", default="auto", choices=["auto", "direct", "tcgen05"])
    ap.add_argument("--mode", default="adaptive", choices=["adaptive", "variance"])
    ap.add_argument("--height", type=int, default=1152)
    ap.add_argument("--width", type=int, default=1600)
    ap.add_argument("--nviews", type=int, default=5)
    ap.add_argument("--ndepths", default="48,32,8")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-incumbent", action="store_true", help="skip the reference-on-this-GPU legs")
    ap.add_argument("--no-extras", action="store_true", help="skip the fp32 / T&T / training / full-forward legs")
    ap.add_argument("--min-seconds", type=float, default=1.0,
                    help="device time the e2e and Tanks-and-Temples legs must cover (their batches are repeated)")
    ap.add_argument("--budget-s", type=float, default=150.0, help="--impl reference: wall-clock budget of the timed passes")
    ap.add_argument("--detail", action="store_true", help="print a per-layer device-time table to stderr")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying a CUDA graph")
    ap.add_argument("--fuse-prob-head", action="store_true", help="run CostRegNet's last layer fused with the head (one launch)")
    ap.add_argument("--inflight", type=int, default=4, help="independent views in flight on separate streams (graph mode)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the per-stage outputs of the last one (rank 0) as DIR/stage<s>_<key>.npy "
                         "in float32; see dump_outputs()")
    args = ap.parse_args(argv)
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this implementation's timed path; it does not apply to --impl reference")
    return args


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"hbm": p["hbm_gbs"], "tensor": p["bf16_tflops"], "tensor_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "src": "measured"}
    return {"hbm": 6650.0, "tensor": 1590.0, "tensor_sustained": 1400.0, "src": "fallback"}


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# SURVEY.md 8d: algorithmic bytes / flops per view of each kernel class (what roofline.achieved is computed from)
# ---------------------------------------------------------------------------------------------
def stage_dims(height, width, ndepths, channels=(32, 16, 8), scales=(4, 2, 1)):
    return [(height // s, width // s, c, d) for s, c, d in zip(scales, channels, ndepths)]


def algorithmic_per_view(height, width, nviews, ndepths, precision, base=8):
    """{class: {"bytes": per view, "flops": per view}} for the layer-by-layer pipeline.
    warp+aggregate: N*C*h*w*f + D*h*w*4 read, C*D*h*w*v written (f = 2 for the fp16 features the bf16 pipeline gathers,
    4 in fp32; v = 2 for a bf16 cost volume, 4 for fp32).  CostRegNet: sum over the 11 layers of input + output activation
    bytes at v bytes per element (skip-tensor re-reads and the fp32 width of the logits are NOT counted: they are waste the
    roofline fraction should show).  Head: 2*V*4 read, V*4 + 3*h*w*4 written.  FLOPs: 2*27*Cin*Cout*V_out (V_in for the
    transposed layers)."""
    f = 4 if precision == "fp32" else 2
    v = 4 if precision == "fp32" else 2
    out = {"warp_agg": {"bytes": 0.0, "flops": 0.0}, "conv": {"bytes": 0.0, "flops": 0.0}, "head": {"bytes": 0.0, "flops": 0.0},
           "repack": {"bytes": 0.0, "flops": 0.0}}
    b = base
    for (h, w, c, d) in stage_dims(height, width, ndepths):
        V = d * h * w
        out["warp_agg"]["bytes"] += nviews * c * h * w * f + V * 4 + c * V * v
        out["head"]["bytes"] += 2 * V * 4 + V * 4 + 3 * h * w * 4
        out["repack"]["bytes"] += nviews * c * h * w * (4 + f) if precision != "fp32" else 0.0
        # (cin, cout, input-volume divisor, output-volume divisor, transposed)
        layers = [(c, b, 1, 1, 0), (b, 2 * b, 1, 8, 0), (2 * b, 2 * b, 8, 8, 0), (2 * b, 4 * b, 8, 64, 0), (4 * b, 4 * b, 64, 64, 0),
                  (4 * b, 8 * b, 64, 512, 0), (8 * b, 8 * b, 512, 512, 0), (8 * b, 4 * b, 512, 64, 1), (4 * b, 2 * b, 64, 8, 1),
                  (2 * b, b, 8, 1, 1), (b, 1, 1, 1, 0)]
        for cin, cout, di, do, tr in layers:
            out["conv"]["bytes"] += (cin * V / di + cout * V / do) * v
            out["conv"]["flops"] += 2.0 * 27 * cin * cout * (V / di if tr else V / do)
    return out


# ---------------------------------------------------------------------------------------------
# CPU legs: the reference's own DepthNet on the host cores (oracle/_ref), else the oracle port.
# The only place bench.py touches oracle/.
# ---------------------------------------------------------------------------------------------
def cpu_step_fn(args, height, width):
    """-> (step(), kind): one three-stage pass of the hot path on the CPU at the given image size."""
    from damvsnet_b200 import synthetic
    from damvsnet_b200.runner import make_workload
    nd = [int(x) for x in args.ndepths.split(",")]
    sd = synthetic.hot_path_state_dict(seed=0, mode=args.mode)
    stages = make_workload(height, width, args.nviews, nd, seed=0)
    # hypotheses as the cascade produces them (the GPU arm's workload): stage 1 = the plane-sweep range, stages 2/3 =
    # uncertainty-aware samples of smooth previous-stage maps -- here through the oracle's CPU samplers
    from oracle import damvs_oracle as O
    rng = synthetic.make_depth_range(1, 192)
    for s in range(len(stages)):
        fs, p, _ = stages[s]
        b, _, h, w = fs[0].shape
        if s == 0:
            dv = O.first_stage_samples(rng, nd[s]).view(b, nd[s], 1, 1).expand(b, nd[s], h, w).contiguous()
        else:
            pd, pv = synthetic.make_prev_maps(s, b, height, width, seed=0)
            dv = O.stage_hypotheses(pd, pv, nd[s], height, width, synthetic.STAGE_SCALES[s])
        stages[s] = (fs, p, dv)
    from oracle import ref_loader
    if ref_loader.available():
        import warnings
        depthnet, crs = ref_loader.build_hot_path(sd, args.mode)

        def step():
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                ref_loader.hot_path_forward(depthnet, crs, stages)
        return step, "reference"
    def step():
        with torch.no_grad():
            for s, (f, p, d) in enumerate(stages):
                O.depthnet_forward(s, f, p, d, sd, args.mode)
    return step, "port"


def cpu_leg(args, max_steps, budget_s):
    """Time full-size passes (no crop, no extrapolation) with all host threads: one untimed small-shape pass to spin up
    the thread pool, then timed passes at the workload's own size until `max_steps` or until the next pass would not
    fit in `budget_s` (at least one)."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    small, _ = cpu_step_fn(args, 128, 160)
    small()
    step, kind = cpu_step_fn(args, args.height, args.width)
    times = []
    t_start = time.perf_counter()
    while len(times) < max(1, max_steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if (time.perf_counter() - t_start) + 1.05 * max(times) > budget_s:
            break
    sec = statistics.median(times)
    what = "the reference's own DepthNet + CostRegNet (oracle/_ref, staged unmodified by oracle/make_ref.py)" if kind == "reference" \
        else "torch-CPU fp32 oracle port (oracle/_ref not staged)"
    return {"value": 1.0 / sec, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": f"{len(times)} full-size pass(es) of the {args.height}x{args.width} view (all 3 stages, N={args.nviews}, "
                      f"D={args.ndepths}; no crop, no extrapolation), median; {what}, fp32, {cores} threads",
            "sec_per_sample": sec, "passes": len(times), "timed_s": sum(times)}


def config_of(args, extra=None):
    c = {"workload": f"DTU-test {args.height}x{args.width}, N={args.nviews}, D={args.ndepths.replace(',', '/')}, batch 1, "
                     f"agg={args.mode} (BASELINE.json configs[1])",
         "hypotheses": "as the cascade produces them: stage 1 = plane-sweep range [425, 931] mm, stages 2/3 = uncertainty-aware "
                       "samples (+-12 / +-3 mm) of smooth synthetic previous-stage depth / variance maps (teacher forcing)",
         "precision": args.precision,
         "l2": "no flush needed: per-step inputs (0.4 GB) and intermediates (>2 GB) exceed the 126 MB L2"}
    if extra:
        c.update(extra)
    return c


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_leg(args, max_steps=max(args.steps, 1), budget_s=args.budget_s)
    note = ("the reference's own models/cas_mvsnet.py DepthNet + models/module.py CostRegNet, unmodified, eval(), no_grad, fp32, "
            "on the host cores at the full workload size") if r["kind"] == "reference" else \
        "CPU oracle port of the reference path (oracle/_ref was not staged on this box)"
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": r["passes"], "steps_requested": args.steps, "warmup": 1, "ms_per_step": 1e3 * r["sec_per_sample"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args, {"precision": "fp32", "note": note,
                                       "bounded": f"timed passes stop when the next one would exceed --budget-s {args.budget_s:.0f}; "
                                                  "the untimed warm-up is one 128x160 pass"}),
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "timed_region_s": r["timed_s"], "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# helpers of the GPU legs
# ---------------------------------------------------------------------------------------------
def device_workload(height, width, nviews, ndepths, dev, seed=0, batch=1):
    """Synthetic three-stage inputs built ON the device (same construction as damvsnet_b200.synthetic.make_stage_inputs,
    GPU generator): for legs that are timed only, where a minute of host-side synthesis buys nothing."""
    from damvsnet_b200 import synthetic
    import torch.nn.functional as F
    g = torch.Generator(device=dev).manual_seed(seed)
    projs, _ = synthetic.make_cameras(batch, nviews, height, width, seed=seed)
    stages = []
    for s, d in enumerate(ndepths):
        sc, c = synthetic.STAGE_SCALES[s], synthetic.STAGE_CHANNELS[s]
        h, w = height // sc, width // sc

        def smooth(shared=None):
            coarse = torch.randn(batch, c, max(h // 4, 1), max(w // 4, 1), generator=g, device=dev)
            x = 0.6 * F.interpolate(coarse, size=(h, w), mode="bilinear", align_corners=False) + \
                0.4 * torch.randn(batch, c, h, w, generator=g, device=dev)
            return (0.7 * shared + 0.3 * x if shared is not None else x).contiguous()
        base = smooth()
        feats = [base] + [smooth(base) for _ in range(1, nviews)]
        if s == 0:
            lo, hi = synthetic.DTU_DEPTH_MIN, synthetic.DTU_DEPTH_MIN + synthetic.DTU_DEPTH_INTERVAL * 191
            dv = torch.linspace(lo, hi, d, device=dev).view(1, d, 1, 1).expand(batch, d, h, w).clone()
        else:
            half = 12.0 if s == 1 else 3.0
            lo, hi = -half, half
            yy, xx = torch.meshgrid(torch.linspace(0, 1, h, device=dev), torch.linspace(0, 1, w, device=dev), indexing="ij")
            surf = 600.0 + 120.0 * torch.sin(3.0 * xx + 0.5) * torch.cos(2.0 * yy)
            dv = (surf.view(1, 1, h, w) + torch.linspace(lo, hi, d, device=dev).view(1, d, 1, 1)).expand(batch, d, h, w).clone()
        dv += (torch.rand(batch, 1, h, w, generator=g, device=dev) - 0.5) * 0.5 * (hi - lo) / max(d - 1, 1)
        stages.append((feats, projs[f"stage{s + 1}"].to(dev), dv.contiguous()))
    return stages


def shifted_sets(dev_stages, inflight):
    """K input sets with distinct data for K views in flight: set k is set 0 shifted by a few pixels plus a small offset."""
    sets = [dev_stages]
    for k in range(1, inflight):
        sets.append([([torch.roll(f, shifts=(3 * k, 5 * k), dims=(2, 3)).add_(0.01 * k).contiguous() for f in fs], p.clone(),
                      (d + 0.05 * k).contiguous()) for fs, p, d in dev_stages])
    return sets


def timed_batches(run_views, steps, min_seconds, barrier, dev, max_reps=40):
    """Time batches of exactly `steps` views, each bracketed by barrier + synchronize and CUDA events, until the batches
    cover >= min_seconds of device time.  -> (median batch ms [max over ranks per batch], all batch ms, reps)."""
    import torch.distributed as dist
    world = dist.get_world_size() if dist.is_initialized() else 1
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def one():
        barrier()
        e0.record()
        run_views(steps)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()
    first = one()
    reps = int(min(max_reps, max(1, math.ceil(min_seconds * 1e3 / max(first, 1e-3)))))
    times = [first] + [one() for _ in range(reps - 1)]
    return statistics.median(times), times, len(times)


DUMP_BYTES = 60_000_000


def dump_outputs(out_dir, outs, seed=0):
    """Write one step's per-stage output dicts (what HotPathRunner.run_device returns) as out_dir/stage<s>_<key>.npy in
    float32, so that two builds run with the same arguments can be compared array for array.  The arrays share
    DUMP_BYTES equally: one larger than its share is stored as a 1-D sample of its flattened values at fixed indices (a
    seeded random subset, sorted, that depends only on the array's size); the others keep their shape."""
    import numpy as np
    arrays = {f"stage{s + 1}_{k}": v for s, out in enumerate(outs) for k, v in out.items()}
    cap = DUMP_BYTES // 4 // len(arrays)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().float()
        if a.numel() > cap:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(seed))[:cap].sort().values
            a = a.flatten()[idx.to(a.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def numa_pin(local_rank: int) -> str:
    """Bind this process to the CPUs of the NUMA node its GPU hangs off, BEFORE the pinned host buffers are allocated
    (first touch places them on that node), so that 8 ranks do not all stream their uploads out of node 0."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(int(os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",")[local_rank])
                                              if os.environ.get("CUDA_VISIBLE_DEVICES") else local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return "numa node unknown"
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        ids &= os.sched_getaffinity(0)
        if ids:
            os.sched_setaffinity(0, ids)
            return f"node {node} ({len(ids)} cpus)"
        return f"node {node} (no allowed cpus)"
    except Exception as exc:  # noqa: BLE001
        return f"unavailable: {type(exc).__name__}"


# ---------------------------------------------------------------------------------------------
# incumbent: the reference's own PyTorch path on this GPU
# ---------------------------------------------------------------------------------------------
def incumbent_gpu_leg(args, dev, dev_stages, sd, iters=3):
    """The reference's DepthNet x3 (unmodified, oracle/_ref) on the B200 on the SAME device-resident inputs:
    (a) strict fp32 (cudnn / matmul TF32 off), (b) PyTorch defaults (cudnn TF32 allowed); cudnn.benchmark on as
    test_uni.py:29 sets it.  Also returns the max relative depth difference of our result from (a)."""
    from oracle import ref_loader
    if not ref_loader.available():
        return {"unavailable": "oracle/_ref not staged (run oracle/make_ref.py where /root/reference exists)"}
    import warnings
    depthnet, crs = ref_loader.build_hot_path(sd, args.mode, device=dev)
    out = {"what": "reference models/cas_mvsnet.py DepthNet + models/module.py CostRegNet (nn.Conv3d, nn.ConvTranspose3d, "
                   "F.grid_sample), eval, no_grad, cudnn.benchmark=True, same device-resident inputs, batch 1"}
    old = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.benchmark = True
    try:
        for tag, tf32 in (("fp32_strict", False), ("torch_defaults_tf32_convs", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = False
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                for _ in range(2):
                    res = ref_loader.hot_path_forward(depthnet, crs, dev_stages)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(iters):
                    res = ref_loader.hot_path_forward(depthnet, crs, dev_stages)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / iters
            out[tag] = {"views_s": 1e3 / ms, "ms_per_view": ms}
            if not tf32:
                out["_depths"] = [r["depth"].clone() for r in res]
            del res
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    del depthnet, crs
    torch.cuda.empty_cache()
    return out


def full_forward_leg(args, dev, sd, iters=3, with_reference=True, seed=0):
    """Full CascadeMVSNet.forward (models/cas_mvsnet.py:190-319), images in pinned host memory -> output dict, final
    depth + confidence read back to the host (test_uni.py:229-237): the reference as is on this GPU, then the SAME class
    with the hot path re-bound to this package by dropin.install() (FPN / GeoFeatureFusion stay the reference's PyTorch)."""
    from oracle import ref_loader
    if not ref_loader.available():
        return {"unavailable": "oracle/_ref not staged"}
    import warnings
    import damvsnet_b200.dropin as dropin
    from damvsnet_b200 import synthetic
    nd = [int(x) for x in args.ndepths.split(",")]
    H, W, N = args.height, args.width, args.nviews
    imgs = synthetic.make_images(1, N, H, W, seed=seed).pin_memory()
    projs, intr = synthetic.make_cameras(1, N, H, W, seed=seed)
    dvals = synthetic.make_depth_range(1, 192)
    out = {"what": f"CascadeMVSNet.forward {H}x{W} N={N} D={args.ndepths}: imgs [1,{N},3,{H},{W}] fp32 from pinned host memory "
                   "(H2D inside the timed region), stage-3 depth + confidence read back; random-init FPN / GeoFeatureFusion "
                   "(reference PyTorch code in both arms), hot-path weights = the benchmark's", "h2d_bytes": imgs.numel() * 4}

    def timed(model):
        def once():
            x = imgs.to(dev, non_blocking=True)
            p = {k: v.to(dev, non_blocking=True) for k, v in projs.items()}
            k = {k2: v.to(dev, non_blocking=True) for k2, v in intr.items()}
            with contextlib.redirect_stdout(io.StringIO()):
                o = model(x, p, dvals.to(dev), k)
            return o["depth"].cpu(), o["photometric_confidence"].cpu()
        with torch.no_grad(), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            for _ in range(2):
                once()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(iters):
                d, c = once()
            torch.cuda.synchronize()
            sec = (time.perf_counter() - t0) / iters
        return sec, d
    old_b = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    try:
        ref_model = ref_loader.build_cascade(nd, args.mode, hot_state_dict=sd).to(dev)
        state = ref_model.state_dict()
        d_ref = None
        if with_reference:
            sec, d_ref = timed(ref_model)
            out["reference_torch_defaults"] = {"views_s": 1.0 / sec, "ms_per_view": sec * 1e3}
        del ref_model
        torch.cuda.empty_cache()
        dropin.install(precision=args.precision)
        try:
            cas, _ = ref_loader.load()
            with contextlib.redirect_stdout(io.StringIO()):
                ours = cas.CascadeMVSNet(refine=False, ndepths=nd, depth_interals_ratio=[4, 2, 1], share_cr=False,
                                         cr_base_chs=[8, 8, 8], grad_method="detach", agg_mode=args.mode)
            ours.load_state_dict(state, strict=True)
            ours = ours.eval().to(dev)
            sec, d_ours = timed(ours)
            out["dropin_" + args.precision] = {"views_s": 1.0 / sec, "ms_per_view": sec * 1e3}
            out["_sec"] = sec
            if d_ref is not None:
                out["final_depth_median_rel_diff"] = ((d_ours - d_ref).abs() / d_ref.abs().clamp_min(1.0)).median().item()
            del ours
        finally:
            dropin.uninstall()
    finally:
        torch.backends.cudnn.benchmark = old_b
        torch.cuda.empty_cache()
    return out


def train_leg(dev, rank, world, barrier, steps=6, warmup=3, batch=4, height=512, width=640, nviews=5, ndepths=(48, 32, 8)):
    """BASELINE.json configs[3]: DTU training step 512x640, N=5, batch 4 per GPU, forward + backward through warp / cost
    volume / CostRegNet / head with batch-statistics BatchNorm, per-stage bucketed NCCL gradient all-reduce started from
    gradient hooks (damvsnet_b200/training.py), Adam step.  -> samples/s over all ranks (max device time over ranks)."""
    import torch.distributed as dist
    import damvsnet_b200 as dm
    from damvsnet_b200 import _lib, synthetic
    from damvsnet_b200.training import HotPathTrainer
    with dm.precision("bf16"):
        trainer = HotPathTrainer(synthetic.hot_path_state_dict(seed=0), device=dev)
        stages = device_workload(height, width, nviews, list(ndepths), dev, seed=rank, batch=batch)
        stages = [([f.requires_grad_(True) for f in fs], p, d) for fs, p, d in stages]
        g = torch.Generator(device=dev).manual_seed(100 + rank)
        gts, masks = [], []
        for _, _, d in stages:
            b, _, h, w = d.shape
            gts.append((d[:, d.shape[1] // 2] + torch.randn(b, h, w, generator=g, device=dev)).contiguous())
            masks.append((torch.rand(b, h, w, generator=g, device=dev) > 0.2).float())

        def step():
            for fs, _, _ in stages:
                for f in fs:
                    f.grad = None
            return trainer.train_step(stages, gts, masks)
        for _ in range(warmup):
            step()
        barrier()
        n0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            loss = step()
        e1.record()
        barrier()
        launches = (_lib.launch_count() - n0) // steps
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms_step = ms.item() / steps
        res = {"samples_s": world * batch / (ms_step / 1e3), "ms_per_step": ms_step, "steps": steps, "batch_per_gpu": batch,
               "workload": f"DTU-train {height}x{width}, N={nviews}, D={'/'.join(map(str, ndepths))} (BASELINE.json configs[3]), bf16",
               "collective": f"{len(trainer.overlap.buckets)} per-stage fp32 gradient buckets ({trainer.bucket.numel * 4} bytes in total), "
                             f"NCCL all-reduce (SUM, then / world) over {world} rank(s), started from gradient hooks inside backward",
               "loss": float(loss), "gpu_launches_per_step": int(launches)}
        trainer.overlap.close()
    del trainer, stages, gts, masks
    torch.cuda.empty_cache()
    return res


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    numa = numa_pin(local)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import damvsnet_b200 as dm
    from damvsnet_b200 import _lib, synthetic
    from damvsnet_b200.runner import HotPathRunner, ViewPipeline, make_workload
    _lib.check(_lib.load().damvs_check_device(local))
    dm.set_precision(args.precision, args.conv_impl)
    dm.ops.set_fusion(prob_head=args.fuse_prob_head)
    nd = [int(x) for x in args.ndepths.split(",")]
    sd = synthetic.hot_path_state_dict(seed=0, mode=args.mode)
    runner = HotPathRunner(sd, mode=args.mode, device=dev)
    host_stages = make_workload(args.height, args.width, args.nviews, nd, seed=rank)
    # Hypotheses as the cascade produces them (reference models/cas_mvsnet.py:236-296): stage 1 sweeps the plane-sweep
    # range, stages 2/3 are uncertainty-aware samples of the previous stage's depth / variance -- here smooth synthetic
    # maps (teacher forcing), sampled on the device by the fused sampler.  The device-resident leg (`value`) and the
    # host-buffer leg (`e2e`) run on exactly these hypotheses; the latter uploads the maps, not the hypotheses.
    depth_range = synthetic.make_depth_range(1, 192)
    prev_maps = [None] + [synthetic.make_prev_maps(s, 1, args.height, args.width, seed=rank) for s in range(1, len(nd))]
    dev_stages = []
    for s, (fs, p, _) in enumerate(host_stages):
        b, _, h, w = fs[0].shape
        if s == 0:
            dv = runner.range_hypotheses(depth_range, nd[s], b, h, w)
        else:
            dv = dm.ops.stage_hypotheses(prev_maps[s][0].to(dev), prev_maps[s][1].to(dev), nd[s], args.height, args.width, args.height // h)
        dev_stages.append(([f.to(dev) for f in fs], p.to(dev), dv))
    host_inputs = [(fs, p, prev_maps[s]) for s, (fs, p, _) in enumerate(host_stages)]
    cascade = (depth_range.pin_memory(), nd, args.height, args.width)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    steps, warmup = max(args.steps, 1), max(args.warmup, 3)
    inflight = 1 if args.no_graph else max(1, args.inflight)

    def make_run_views(rn, stages):
        pipe = None if args.no_graph else ViewPipeline(rn, shifted_sets(stages, inflight))
        last = [None]

        def run_views(n):
            if pipe is None:
                for _ in range(n):
                    last[0] = rn.run_device(stages)
            else:
                pipe.fork()
                pipe.submit(n)
                pipe.join()
                last[0] = pipe.last_outputs()
        run_views.last_outputs = lambda: last[0]
        return run_views

    run_views = make_run_views(runner, dev_stages)
    run_views(max(warmup, inflight))
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    batch_ms, all_ms, _ = timed_batches(run_views, steps, 0.0, barrier, dev, max_reps=1)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, run_views.last_outputs())
    # kernels per step = C-ABI launches of one eager pass (graph replays do not pass through the C ABI)
    n0 = _lib.launch_count()
    runner.run_device(dev_stages)
    torch.cuda.synchronize()
    launches = _lib.launch_count() - n0
    value = world * steps / (batch_ms / 1e3)

    # ---- end to end: host buffers in, host results out, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        fmt = "nhwc_f16" if args.precision != "fp32" else "nchw_f32"
        pinned = runner.pin_stages(host_inputs, feature_format=fmt)
        warm = [runner.submit_host(pinned, cascade=cascade) for _ in range(3)]      # also allocates the pinned result buffers
        for t in warm:
            runner.collect(t)
            runner.release(t)

        def run_host(n):
            # two views in flight: the upload of view i+1 overlaps the kernels of view i; every view's results are
            # read back to pinned host memory and waited for inside the timed region
            pending = None
            for _ in range(n):
                t = runner.submit_host(pinned, cascade=cascade)
                if pending is not None:
                    runner.collect(pending)
                    runner.release(pending)
                pending = t
            runner.collect(pending)
            runner.release(pending)
        e_steps = max(3, min(steps, 20))
        e_ms, _, e_reps = timed_batches(run_host, e_steps, args.min_seconds, barrier, dev, max_reps=20)
        e2e = {"value": world * e_steps / (e_ms / 1e3), "unit": UNIT,
               "h2d_bytes_per_step": runner.h2d_bytes(pinned) + depth_range.numel() * 4, "d2h_bytes_per_step": runner.d2h_bytes(host_stages),
               "steps": e_steps, "repetitions": e_reps, "numa": numa,
               "api": "HotPathRunner.submit_host/collect, 2 views in flight; pinned host inputs: features "
                      + ("fp16 channels_last [B,C,h,w] (the layout and width the gather kernel consumes; zero-copy on the device)"
                         if fmt == "nhwc_f16" else "fp32 NCHW")
                      + ", projection matrices, the plane-sweep range (stage 1) and the previous stage's depth / variance maps (stages 2, 3: "
                        "hypotheses are sampled on the device by the fused sampler, as in the cascade); depth, confidence, variance of 3 "
                        "stages out to pinned host memory"}
        del pinned

    # ---- roofline: per-call device times of the hot kernels, measured live with CUDA events (eager pass, one view)
    roof, kernels, rooflines = None, None, None
    if rank == 0:
        pk = peaks()
        alg = algorithmic_per_view(args.height, args.width, args.nviews, nd, args.precision)
        # A spin kernel (~12 ms) is queued ahead of every eager pass so that the CPU -- which needs ~0.1 ms of Python per
        # launch -- is always ahead of the GPU: the event pairs then bracket back-to-back kernel executions, not the gaps in
        # which the GPU waits for the next launch to arrive (those gaps inflated round 1's per-kernel times of short
        # kernels: 69 us per head launch here against 35 us under ncu).
        runner.run_device(dev_stages)
        torch.cuda.synchronize()
        with dm.ops.CallTimer() as timer:
            for _ in range(3):
                torch.cuda._sleep(int(12e-3 * 1.9e9))
                runner.run_device(dev_stages)
        summ = timer.summary()
        if args.detail:
            for tag, d in timer.summary(detail=True).items():
                ms = d["ms"] / d["calls"]
                print(f"  {tag:48s} {ms * 1e3:9.1f} us  {d['bytes'] / d['calls'] / ms / 1e6:8.0f} GB/s  {d['flops'] / d['calls'] / ms / 1e9:8.1f} TF/s",
                      file=sys.stderr)
        cls = {"conv3d_tc": "conv", "conv3d_direct": "conv", "conv_head": "conv"}
        kernels = {}
        for tag, d in summ.items():
            per_step_ms = d["ms"] / 3
            kernels[tag] = {"ms_per_step": per_step_ms, "launches_per_step": d["calls"] // 3}
        # class totals (conv3d_tc + fused conv+head launches are one class: CostRegNet)
        klass = {}
        for tag, k in kernels.items():
            c = cls.get(tag, tag)
            a = klass.setdefault(c, {"ms_per_step": 0.0, "launches_per_step": 0})
            a["ms_per_step"] += k["ms_per_step"]
            a["launches_per_step"] += k["launches_per_step"]
        traffic = {}
        tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            traffic = {k2: v for k2, v in tj.get("kernels", {}).items()}

        def roof_of(c):
            k = klass[c]
            a = alg.get(c, {"bytes": 0.0, "flops": 0.0})
            avg_ms = k["ms_per_step"] / max(k["launches_per_step"], 1)
            gbs = a["bytes"] / k["ms_per_step"] / 1e6
            # measured DRAM bytes (ncu launch list of this same step, profiles/r02_traffic.json), per C-ABI call like `achieved`;
            # only trusted when the list holds exactly the kernels this step launches (conv6 is two kernels in one call)
            tr = traffic.get(c)
            tr_per_launch = None
            if tr and sum(v.get("launches_per_step", 0) for v in traffic.values()) == int(launches):
                tr_per_launch = (tr["dram_read_per_step"] + tr["dram_write_per_step"]) / max(k["launches_per_step"], 1)
            r = {"kernel": c, "bound": "hbm", "achieved": gbs, "peak": pk["hbm"], "unit": "GB/s", "frac": gbs / pk["hbm"],
                 "traffic": tr_per_launch, "peak_source": pk["src"], "avg_launch_ms": avg_ms,
                 "algorithmic_bytes_per_step": a["bytes"], "algorithmic_bytes_per_launch": a["bytes"] / max(k["launches_per_step"], 1),
                 "launches_per_step": k["launches_per_step"], "ms_per_step": k["ms_per_step"]}
            if c == "conv":
                tf = a["flops"] / k["ms_per_step"] / 1e9
                r.update({"arithmetic_intensity_flop_per_byte": a["flops"] / a["bytes"],
                          "ridge_flop_per_byte": pk["tensor_sustained"] * 1e3 / pk["hbm"],
                          "also_tensor": {"achieved": tf, "peak": pk["tensor_sustained"], "unit": "TFLOP/s",
                                          "frac": tf / pk["tensor_sustained"], "frac_of_burst": tf / pk["tensor"],
                                          "peak_source": pk["src"] + " (sustained bf16)"}})
            return r
        if "head" not in klass and "conv_head" in kernels:
            # the head ran fused into CostRegNet's last layer: its bytes belong to the conv class, minus the logits that no
            # longer travel (written as 2-byte elements in 8d's conv figure, read as fp32 in its head figure)
            V = sum(d * h * w for (h, w, _, d) in stage_dims(args.height, args.width, nd))
            alg["conv"]["bytes"] += alg["head"]["bytes"] - V * 4 - V * (4 if args.precision == "fp32" else 2)
        rooflines = [roof_of(c) for c in klass]
        roof = max(rooflines, key=lambda r: r["ms_per_step"])

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_leg(args, max_steps=1, budget_s=30.0)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}

    # ---- incumbent: the reference's own PyTorch hot path on this GPU (rank 0, N = 1)
    incumbent = None
    if rank == 0 and world == 1 and not args.no_incumbent:
        try:
            ours = runner.run_device(dev_stages)
            incumbent = incumbent_gpu_leg(args, dev, dev_stages, sd)
            ref_depths = incumbent.pop("_depths", None)
            if ref_depths is not None:
                incumbent["our_depth_vs_reference_gpu_fp32"] = [
                    {"median_rel": ((o["depth"] - r).abs() / r.abs()).median().item(),
                     "p99_rel": ((o["depth"] - r).abs() / r.abs()).flatten().float().quantile(0.99).item() if r.numel() < 2 ** 24
                     else ((o["depth"] - r).abs() / r.abs()).flatten()[::4].float().quantile(0.99).item()}
                    for o, r in zip(ours, ref_depths)]
            if incumbent.get("fp32_strict"):
                incumbent["speedup_vs_fp32_strict"] = value / incumbent["fp32_strict"]["views_s"]
                incumbent["speedup_vs_torch_defaults"] = value / incumbent["torch_defaults_tf32_convs"]["views_s"]
            del ours, ref_depths
        except Exception as exc:  # noqa: BLE001
            incumbent = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        torch.cuda.empty_cache()

    # ---- extras: the other configurations of BASELINE.json, so the driver's line carries them too
    extras = None
    if not args.no_extras:
        extras = {}
        del run_views
        # (1) the other precision modes on the same workload, rank 0 at N = 1: fp32 (the <= 1e-4 parity mode) and the
        #     other 2-byte pipeline (bf16 when the headline is fp16)
        if rank == 0 and world == 1:
            others = [("fp32", "fp32 features / cost volume, direct fp32 convolutions: the <= 1e-4 parity mode")]
            if args.precision != "fp32":
                o = "bf16" if args.precision == "fp16" else "fp16"
                others.append((o, f"fp16 features, {o} cost volume / weights / activations, tcgen05 convolutions"))
            if args.precision == "fp16":
                others.append(("fp16+fp32feat", "fp32 features (fp32 gather kernel), fp16 cost volume / weights / activations, tcgen05 "
                                                "convolutions: meets SURVEY H7's bound, depth rel p99 <= 1e-3 / max <= 5e-3"))
            for prec, note in others:
                try:
                    with dm.precision(prec.split("+")[0], features="fp32" if "+" in prec else "auto"):
                        r2 = HotPathRunner(sd, mode=args.mode, device=dev)
                        rv = make_run_views(r2, dev_stages)
                        rv(inflight)
                        n2 = max(3, min(steps, 5)) if prec == "fp32" else steps
                        ms2, _, _ = timed_batches(rv, n2, 0.0, barrier, dev, max_reps=1)
                        extras[f"{prec}_views_s"] = {"value": n2 / (ms2 / 1e3), "note": "same workload, precision " + prec + " (" + note + ")"}
                        del rv, r2
                except Exception as exc:  # noqa: BLE001
                    extras[f"{prec}_views_s"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
                torch.cuda.empty_cache()
        del dev_stages, host_stages
        torch.cuda.empty_cache()
        # (2) Tanks-and-Temples shape, views sharded over the ranks (configs[2])
        try:
            tnt = device_workload(1056, 1920, 7, nd, dev, seed=rank)
            rv = make_run_views(runner, tnt)
            rv(max(3, inflight))
            t_steps = max(4, min(steps, 20))
            t_ms, _, t_reps = timed_batches(rv, t_steps, min(args.min_seconds, 0.5), barrier, dev, max_reps=10)
            extras["tnt_views_s"] = {"value": world * t_steps / (t_ms / 1e3), "ms_per_view": t_ms / t_steps, "steps": t_steps,
                                     "repetitions": t_reps,
                                     "workload": f"Tanks-and-Temples 1056x1920, N=7, D={args.ndepths.replace(',', '/')}, batch 1, "
                                                 f"{args.precision}; views sharded x{world} (BASELINE.json configs[2])"}
            del rv, tnt
        except Exception as exc:  # noqa: BLE001
            extras["tnt_views_s"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        torch.cuda.empty_cache()
        # (3) training step with the gradient all-reduce (configs[3])
        try:
            extras["train_samples_s"] = train_leg(dev, rank, world, barrier)
        except Exception as exc:  # noqa: BLE001
            extras["train_samples_s"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        dm.set_precision(args.precision, args.conv_impl)
        # (4) full forward, images in -> dict out: the drop-in on every rank (one view stream per GPU, sharded like the hot
        #     path; throughput = ranks / slowest rank's seconds per view), the unmodified reference beside it on rank 0 at N = 1
        try:
            ff = full_forward_leg(args, dev, sd, with_reference=(rank == 0 and world == 1), seed=rank)
        except Exception as exc:  # noqa: BLE001
            ff = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        dm.set_precision(args.precision, args.conv_impl)
        sec_t = torch.tensor([ff.pop("_sec", -1.0) if isinstance(ff, dict) else -1.0], dtype=torch.float64, device=dev)
        bad_t = (sec_t < 0).to(torch.float64)
        if world > 1:
            dist.all_reduce(sec_t, op=dist.ReduceOp.MAX)
            dist.all_reduce(bad_t, op=dist.ReduceOp.MAX)
        if rank == 0:
            if bad_t.item() == 0 and sec_t.item() > 0:
                ff["dropin_" + args.precision] = {"views_s": world / sec_t.item(), "ms_per_view_slowest_rank": sec_t.item() * 1e3, "ranks": world}
            extras["full_forward"] = ff

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
                "ms_per_step": batch_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": args.precision, "data": "synthetic",
                "config": config_of(args, {"parallelism": f"views sharded x{world}, no data-path collective",
                                           "launch": "eager" if args.no_graph else f"cuda-graph replay of the 3-stage step, {inflight} independent views in flight on {inflight} streams",
                                           "timing": f"one batch of {steps} steps (bracketed by barrier + synchronize, CUDA events, max over ranks); "
                                                     f"{sum(all_ms) / 1e3:.2f} s of device time"}),
                "batches_ms": all_ms, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof,
                "rooflines": rooflines, "kernels": kernels, "cpu_baseline": cpu, "incumbent_gpu": incumbent, "extras": extras}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
