#!/usr/bin/env python
"""Per-stage device time of the group-wise correlation training kernels against the variance-mode backward at the
training shape of BASELINE.json configs[3] (512x640 image, N = 5, batch 4, D = 48/32/8, feature widths 32/16/8, bf16
volume gradient).  Each kernel is called through the C ABI on preallocated buffers (no allocation or zeroing in the
timed window), the variants alternate round by round, and every timing is CUDA events around `--iters` launches; the
median over `--rounds` is printed as one JSON line, with the card's name and power limit.

    python scripts/time_gwc_train.py [--groups 8,8,4] [--iters 20] [--rounds 5]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--groups", default="8,8,4")
    ap.add_argument("--batch", type=int, default=4)
    ap.add_argument("--nviews", type=int, default=5)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()

    from damvsnet_b200 import _lib, ops, synthetic
    from damvsnet_b200.cas_mvsnet import DepthNet
    dev = torch.device("cuda:0")
    lib = _lib.load()
    groups = [int(x) for x in args.groups.split(",")]
    st = ops._stream
    res = {}
    for s, (D, G) in enumerate(zip((48, 32, 8), groups)):
        feats, proj, dv = synthetic.make_stage_inputs(s, args.batch, args.nviews, 512, 640, D, seed=s)
        feats = [f.to(dev) for f in feats]
        rt = DepthNet.stage_rot_trans(proj.to(dev))
        dv = dv.to(dev).contiguous()
        nhwc = [ops.features_to_nhwc(f).contiguous() for f in feats]
        ref, srcs = nhwc[0], nhwc[1:]
        B, H, W, C = ref.shape
        n = len(srcs)
        sp = (ctypes.c_void_p * n)(*[t.data_ptr() for t in srcs])
        g_ref = torch.empty_like(ref)
        g_src = [torch.zeros_like(t) for t in srcs]
        gp = (ctypes.c_void_p * n)(*[t.data_ptr() for t in g_src])
        vol_g = torch.empty((B, max(G, 8) // 8, D, H, W, 8), dtype=torch.bfloat16, device=dev)
        gv_g = torch.randn(vol_g.shape, device=dev).bfloat16()
        gv_v = torch.randn((B, C // 8, D, H, W, 8), device=dev).bfloat16()
        p = ops._p
        calls = {
            "warp_gwc_train_fwd": lambda: lib.damvs_warp_gwc_train_fwd(p(ref), sp, n, p(rt), p(dv), p(vol_g), B, C, G, D, H, W, 1,
                                                                       _lib.BF16, st()),
            "warp_gwc_bwd": lambda: lib.damvs_warp_gwc_bwd(p(ref), sp, n, p(rt), p(dv), p(gv_g), _lib.BF16, p(g_ref), gp, B, C, G, D,
                                                           H, W, 1, st()),
            "warp_agg_bwd_variance": lambda: lib.damvs_warp_agg_bwd(p(ref), sp, n, p(rt), p(dv), None, p(gv_v), _lib.BF16, p(g_ref), gp,
                                                                    None, B, C, D, H, W, _lib.AGG_VARIANCE, 1, st()),
        }
        for fn in calls.values():              # warm-up, and the launch must succeed
            _lib.check(fn())
        torch.cuda.synchronize()
        times = {k: [] for k in calls}
        for _ in range(args.rounds):
            for k, fn in calls.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.iters):
                    fn()
                b.record()
                b.synchronize()
                times[k].append(a.elapsed_time(b) / args.iters * 1e3)
        res[f"stage{s + 1}"] = {"shape": f"B={B} C={C} G={G} D={D} {H}x{W} n_src={n}",
                                **{k: round(sorted(v)[len(v) // 2], 1) for k, v in times.items()}}
    print(json.dumps({"unit": "us per launch (median of rounds)", "card": card(), "stages": res}), flush=True)


if __name__ == "__main__":
    main()
