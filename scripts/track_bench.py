#!/usr/bin/env python
"""track_bench.py -- cost of the sparse point tracker (ofb_track_points_device) on one GPU.

    python scripts/track_bench.py [--reps 10] [--warmup 2] [--out FILE]

Workload: 1920x1080, 3 levels, 9x9 window, flow_scale 8/15, bench.py's synthetic pairs (value noise shifted by up to
+-4 px), 1 k, 16 k and 256 k uniformly random sub-pixel points per pair, 1 and 64 pairs, 30 iterations per level with
eps = 0 (fixed work: every point runs every iteration) and with eps = 0.01 px (OpenCV's default stop).  Per configuration,
CUDA events around whole calls (median of --reps, every configuration warmed up first) give the call time, which includes
the pyramid build of both frames; a separate profiled pass reads the OFB_PROFILE_TRACK (kernel) and OFB_PROFILE_PYRAMID
records.  Also reported: points per second (points / call time), the share of points TRACKED and their median position
error against the known shift.  The card's name and power limit are read in the same run.  Prints one JSON line (and
writes it to --out).
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

W, H, LEVELS, WIN, S = 1920, 1080, 3, 9, 8 / 15
POINTS = [1 << 10, 1 << 14, 1 << 18]
PAIRS = [1, 64]
EPS = [0.0, 0.01]
ITERS = 30


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch

    from bench import synth_pairs_torch
    from cuda_optical_flow_2_b200 import PROFILE_PYRAMID, PROFILE_TRACK, PT_TRACKED, Context
    from fb_bench import card_info

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device"}), flush=True)
        return 1
    card = card_info(torch)
    dev = torch.device("cuda", 0)
    ctx = Context(0)
    ctx.reserve_pairs(W, H, LEVELS, WIN, max(PAIRS))
    rng = np.random.default_rng(5)
    rows = []
    for n in PAIRS:
        prev, nxt, _, shifts = synth_pairs_torch(n, W, H, dev, seed=1, return_shifts=True)
        prev, nxt = prev.contiguous(), nxt.contiguous()
        shifts = np.asarray(shifts, np.float32)
        for m in POINTS:
            pts_np = np.stack([rng.uniform(0, W - 1, (n, m)), rng.uniform(0, H - 1, (n, m))], -1).astype(np.float32)
            pts = torch.from_numpy(pts_np).to(dev)
            for eps in EPS:
                call = lambda: ctx.track_points_device(prev, nxt, W, LEVELS, WIN, pts, S, ITERS, eps)
                for _ in range(args.warmup):
                    call()
                torch.cuda.synchronize()
                ms = []
                for _ in range(args.reps):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    flow, st = call()
                    e1.record()
                    torch.cuda.synchronize()
                    ms.append(e0.elapsed_time(e1))
                ctx.profile_enable(True)
                for _ in range(args.reps):
                    call()
                kern_ms, nk = ctx.profile_read(PROFILE_TRACK)
                pyr_ms, npy = ctx.profile_read(PROFILE_PYRAMID)
                ctx.profile_enable(False)
                flow, st = flow.cpu().numpy(), st.cpu().numpy()
                ok = st == PT_TRACKED
                err = np.hypot(S * flow[..., 0] - shifts[:, None, 0], S * flow[..., 1] - shifts[:, None, 1])[ok]
                call_ms = float(np.median(ms))
                rows.append({"pairs": n, "points_per_pair": m, "iters": ITERS, "eps": eps, "call_ms": round(call_ms, 4),
                             "call_ms_min": round(float(np.min(ms)), 4), "track_kernel_ms": round(kern_ms / nk, 4),
                             "pyramid_ms": round(pyr_ms / npy, 4), "points_per_s": float(f"{n * m / (call_ms * 1e-3):.4g}"),
                             "tracked_share": round(float(ok.mean()), 4),
                             "median_err_px": round(float(np.median(err)), 4) if err.size else None})
                print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
        del prev, nxt
        torch.cuda.empty_cache()
    ctx.close()
    out = {"workload": {"w": W, "h": H, "levels": LEVELS, "win": WIN, "flow_scale": "8/15", "iters": ITERS},
           "card": card, "reps": args.reps, "rows": rows}
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
