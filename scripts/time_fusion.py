#!/usr/bin/env python
"""Scan-level fusion (reference filter/dypcd.py:filter_depth) at the DTU-test size, old composition against the native
point emission.  The scan is 11 seeded views of tests/golden/make_golden_filter.make_scene at 1152x1600; every view is
a reference view with the next 4 views (cyclically) as its sources.

- old: per view filter_reference_view, backproject_valid, the colours at the final mask, then torch.cat -- what
  fusion.fuse_views did before its points came from damvs_geo_consistency_points (two host synchronisations, pageable
  copies and ~15 torch launches per view);
- new: fusion.fuse_views (one library launch per view, one synchronisation per scan).

The arms alternate round by round in one process.  Per arm and round: wall time per scan (host clock around `reps`
back-to-back scans ending in a device synchronise; `reps` is sized so that a round lasts about `--seconds`), the CUDA
event span per scan over the same window, library launches per scan and the point count.  The medians over `--rounds`
are printed as one JSON line with the card's name and power limit.  Both arms' points are compared before timing.
`new_enqueue_event_ms_per_scan` is the event span of the new arm's device work alone (the zeroing of the count and the
workspace, and the 11 launches, without the count's read-back and the copy out of the scan-wide buffer).

    python scripts/time_fusion.py [--rounds 5] [--seconds 1.0]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def old_fuse(depths, confidences, images, Ks, Es, pairs):
    from damvsnet_b200 import fusion
    xyz, rgb = [], []
    for ref, srcs in pairs:
        out = fusion.filter_reference_view(depths[ref], confidences[ref], Ks[ref], Es[ref], [depths[s] for s in srcs],
                                           [Ks[s] for s in srcs], [Es[s] for s in srcs])
        m = out["final_mask"]
        xyz.append(fusion.backproject_valid(out["depth_est_averaged"], m, Ks[ref], Es[ref]))
        rgb.append((images[ref][m] * 255).to(torch.uint8))
    return torch.cat(xyz, 0), torch.cat(rgb, 0)


def run(fn, reps):
    from damvsnet_b200 import _lib
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    t0 = time.perf_counter()
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / reps
    return {"wall_ms": wall * 1e3, "event_ms": a.elapsed_time(b) / reps, "launches": (_lib.launch_count() - n0) / reps,
            "points": len(out[0])}, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--seconds", type=float, default=1.0)
    args = ap.parse_args()

    from damvsnet_b200 import fusion
    from make_golden_filter import make_scene
    assert torch.cuda.is_available(), "time_fusion.py needs a GPU"
    H, W, V, n_src = 1152, 1600, 11, 4
    Ks, Es, d = make_scene(3, H, W, V - 1)
    rs = np.random.RandomState(0)
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    depths = [t(x) for x in d]
    confidences = [[t(rs.rand(H, W).astype(np.float32)) for _ in range(3)] for _ in range(V)]
    images = [t(rs.rand(H, W, 3).astype(np.float32)) for _ in range(V)]
    pairs = [(v, [(v + k) % V for k in range(1, n_src + 1)]) for v in range(V)]
    scan = (depths, confidences, images, Ks, Es, pairs)
    arms = {"old": lambda: old_fuse(*scan), "new": lambda: fusion.fuse_views(*scan)}

    reps, outs = {}, {}
    for k, fn in arms.items():                  # warm-up, and size each round to about --seconds
        run(fn, 2)
        r, outs[k] = run(fn, 3)
        reps[k] = max(3, int(args.seconds / (r["wall_ms"] / 1e3)))
    (ox, orgb), (nx, nrgb) = outs["old"], outs["new"]
    assert len(ox) == len(nx) and torch.equal(orgb, nrgb), "the arms disagree on the points"
    a, b = ox.cpu().numpy(), nx.cpu().numpy()
    ulps = (np.abs(a.astype(np.float64) - b) / np.spacing(np.maximum(np.abs(a), np.abs(b)))).max() if len(a) else 0.0
    rounds = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            rounds[k].append(run(fn, reps[k])[0])
    enqueue = run(lambda: fusion._enqueue_points(*scan, (0.1, 0.15, 0.9), 1 / 4, 1 / 1300)[1:], reps["new"])[0]["event_ms"]
    med = lambda k, f: sorted(r[f] for r in rounds[k])[len(rounds[k]) // 2]
    res = {k: {"wall_ms_per_scan": round(med(k, "wall_ms"), 3), "event_ms_per_scan": round(med(k, "event_ms"), 3),
               "wall_ms_rounds": [round(r["wall_ms"], 3) for r in rounds[k]], "library_launches_per_scan": rounds[k][0]["launches"],
               "points": rounds[k][0]["points"], "scans_per_round": reps[k]} for k in arms}
    print(json.dumps({"scan": f"{V} views x {n_src} sources, {H}x{W}", "card": card(), "rounds": args.rounds,
                      "max_xyz_diff_ulp": float(ulps), **res, "new_enqueue_event_ms_per_scan": round(enqueue, 3)}), flush=True)


if __name__ == "__main__":
    main()
