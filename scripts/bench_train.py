#!/usr/bin/env python
"""Training-step benchmark of the hot path (BASELINE.json configs[3]): DTU training shape 512x640, N=5, batch 4
per GPU, D=48/32/8, forward + backward through warp / cost volume / CostRegNet / head with batch-statistics
BatchNorm, bucketed NCCL gradient all-reduce, Adam step.  Not the headline metric (bench.py is); one JSON line.

    python scripts/bench_train.py [--steps K] [--warmup W] [--batch 4] [--mode adaptive|variance|groupwise --groups 8,8,4]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        scripts/bench_train.py --gpus N
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--height", type=int, default=512)
    ap.add_argument("--width", type=int, default=640)
    ap.add_argument("--nviews", type=int, default=5)
    ap.add_argument("--ndepths", default="48,32,8")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--detail", action="store_true")
    ap.add_argument("--mode", default="adaptive", choices=["adaptive", "variance", "groupwise"],
                    help="cost-volume aggregation; groupwise (not in the reference) needs --groups")
    ap.add_argument("--groups", default=None, help="group-wise correlation groups per stage, e.g. 8,8,4")
    args = ap.parse_args()

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import damvsnet_b200 as dm
    from damvsnet_b200 import _lib, synthetic
    from damvsnet_b200.runner import make_workload
    from damvsnet_b200.cas_mvsnet import stage_volume_channels
    from damvsnet_b200.training import HotPathTrainer
    dm.set_precision(args.precision)
    nd = [int(x) for x in args.ndepths.split(",")]
    groups = [int(x) for x in args.groups.split(",")] if args.groups else None
    if args.mode == "groupwise":
        if groups is None:
            ap.error("--mode groupwise needs --groups")
        vol_channels = stage_volume_channels(args.mode, synthetic.STAGE_CHANNELS, groups)
        sd = synthetic.hot_path_state_dict(in_channels=vol_channels, seed=0, mode=args.mode)
    else:
        sd = synthetic.hot_path_state_dict(seed=0, mode=args.mode)
    trainer = HotPathTrainer(sd, mode=args.mode, device=dev, groups=groups)
    stages = make_workload(args.height, args.width, args.nviews, nd, batch=args.batch, seed=rank, device=dev)
    # features come out of the (PyTorch) FPN in real training and need gradients: keep that work in the step
    stages = [([f.requires_grad_(True) for f in fs], p, d) for fs, p, d in stages]
    g = torch.Generator().manual_seed(100 + rank)
    gts, masks = [], []
    for _, _, d in stages:
        b, _, h, w = d.shape
        gts.append((d[:, d.shape[1] // 2] + torch.randn(b, h, w, generator=g).to(dev)).contiguous())
        masks.append((torch.rand(b, h, w, generator=g) > 0.2).float().to(dev))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        for fs, _, _ in stages:
            for f in fs:
                f.grad = None
        return trainer.train_step(stages, gts, masks)

    for _ in range(max(args.warmup, 3)):
        loss = step()
    barrier()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step()
    e1.record()
    barrier()
    launches = (_lib.launch_count() - n0) // args.steps
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = ms.item() / args.steps
    detail = None
    if args.detail and rank == 0:
        # forward-only and forward+backward without the collective / optimizer, for the breakdown
        def timed(fn, n=3):
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n

        def fwd():
            with torch.no_grad():
                trainer.forward(stages)

        def fwd_bwd():
            from damvsnet_b200.training import depth_loss
            depth_loss(trainer.forward(stages), gts, masks).backward()
        detail = {"forward_ms": timed(fwd), "forward_backward_ms": timed(fwd_bwd)}
    if rank == 0:
        metric = "training samples/sec, hot path fwd+bwd+allreduce+Adam at 512x640 N=5 D=48/32/8"
        if args.mode != "adaptive":     # the default keeps its metric name (and output) unchanged
            metric += f", {args.mode} aggregation" + (f" groups {args.groups}" if args.mode == "groupwise" else "")
        print(json.dumps({"metric": metric, "value": world * args.batch / (ms_step / 1e3),
                          "unit": "samples/s", "n_gpus": world, "steps": args.steps, "ms_per_step": ms_step, "scaling": "weak",
                          "dtype": args.precision, "data": "synthetic", "loss": float(loss), "gpu_launches": int(launches),
                          "config": {"workload": f"DTU-train {args.height}x{args.width}, N={args.nviews}, D={args.ndepths}, batch {args.batch}/GPU (BASELINE.json configs[3])",
                                     "allreduce_bytes": trainer.bucket.numel * 4, "bn": "batch statistics, per GPU"},
                          "detail": detail}), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
