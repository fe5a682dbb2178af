#!/usr/bin/env python
"""corners_bench.py -- cost of the Shi-Tomasi corner detector (ofb_detect_corners_device) on one GPU.

    python scripts/corners_bench.py [--reps 20] [--warmup 3] [--out FILE]

Workload: 1920x1080 frames of bench.py's synthetic pairs (value noise), 1 and 64 images per call, windows 3 and 9,
max_corners 1000 and 16384, min_distance 0, 5 and 10 px, quality_level 0.01.  Per configuration, CUDA events around
whole calls (median of --reps, every configuration warmed up first) give the call time; a separate profiled pass reads
the OFB_PROFILE_CORNERS record (all of the call's kernels).  Per (images, window) the score kernel alone is timed
through ofb_min_eig_map_device (events around --reps calls), with the bytes it must move (every image byte read once,
the float map written once) and their share of the copy peak, measured in the same run as fb_bench.py does (a
device-to-device copy of 4 GiB).  One torch.profiler pass per one-image configuration splits the call into its kernels
(score, candidates, sort, selection).  The card's name, power limit and clocks are read in the same run.  Prints one
JSON line (and writes it to --out).
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

W, H = 1920, 1080
IMAGES = [1, 64]
WINS = [3, 9]
MAX_CORNERS = [1000, 16384]
MIN_DIST = [0.0, 5.0, 10.0]
QUALITY = 0.01


def timed(torch, fn, reps):
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


def kernel_split(torch, call, reps):
    """Device time per kernel group over `reps` calls (torch.profiler), in ms per call."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            call()
        torch.cuda.synchronize()
    groups = {"score": 0.0, "candidates": 0.0, "sort": 0.0, "select": 0.0, "other": 0.0}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        name = ev.key
        g = ("score" if "corner_score" in name else "candidates" if "corner_cand" in name else
             "select" if "corner_select" in name else "sort" if ("cub" in name or "Segmented" in name) else "other")
        groups[g] += t / 1e3 / reps
    return {k: round(v, 4) for k, v in groups.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch

    from bench import synth_pairs_torch
    from cuda_optical_flow_2_b200 import PROFILE_CORNERS, Context
    from fb_bench import card_info, copy_peak_gbs

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device"}), flush=True)
        return 1
    card = card_info(torch)
    dev = torch.device("cuda", 0)
    peak = copy_peak_gbs(torch, args.reps)
    ctx = Context(0)
    rows, score_rows = [], []
    for n in IMAGES:
        imgs, _, _ = synth_pairs_torch(n, W, H, dev, seed=1)
        imgs = imgs.contiguous()
        for win in WINS:
            ctx.reserve_corners(W, H, n, win, max(MAX_CORNERS))
            smap = lambda: ctx.min_eig_map_device(imgs, W, win)
            for _ in range(args.warmup):
                smap()
            torch.cuda.synchronize()
            ms = float(np.median(timed(torch, smap, args.reps)))
            nbytes = n * (H * W + H * W * 4)  # each image byte read once, the map written once
            gbs = nbytes / (ms * 1e-3) / 1e9
            score_rows.append({"images": n, "win": win, "score_kernel_ms": round(ms, 4), "bytes": nbytes,
                               "gb_per_s": round(gbs, 1), "copy_peak_share": round(gbs / peak, 3)})
            print(json.dumps(score_rows[-1]), file=sys.stderr, flush=True)
            for mc in MAX_CORNERS:
                for md in MIN_DIST:
                    call = lambda: ctx.detect_corners_device(imgs, W, win, mc, QUALITY, md)
                    for _ in range(args.warmup):
                        out = call()
                    torch.cuda.synchronize()
                    ms = timed(torch, call, args.reps)
                    ctx.profile_enable(True)
                    for _ in range(args.reps):
                        call()
                    kern_ms, nk = ctx.profile_read(PROFILE_CORNERS)
                    ctx.profile_enable(False)
                    counts = out[2].cpu().numpy()
                    row = {"images": n, "win": win, "max_corners": mc, "min_distance": md, "call_ms": round(float(np.median(ms)), 4),
                           "call_ms_min": round(float(np.min(ms)), 4), "corners_kernels_ms": round(kern_ms / nk, 4),
                           "mean_count": round(float(counts.mean()), 1)}
                    if n == 1:
                        row["kernels_ms"] = kernel_split(torch, call, args.reps)
                    rows.append(row)
                    print(json.dumps(row), file=sys.stderr, flush=True)
        del imgs
        torch.cuda.empty_cache()
    ctx.close()
    out = {"workload": {"w": W, "h": H, "quality_level": QUALITY, "content": "bench.py synth_pairs_torch prev frames"},
           "card": card, "reps": args.reps, "copy_peak_gb_per_s": round(peak, 1), "score_kernel": score_rows, "rows": rows}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
