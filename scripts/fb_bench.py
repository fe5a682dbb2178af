#!/usr/bin/env python
"""fb_bench.py -- cost of the forward-backward consistency check on one GPU.

    python scripts/fb_bench.py [--pairs 512] [--reps 20] [--warmup 3] [--out FILE]

Workload: bench.py's headline settings (1920x1080, 3 levels, 9x9 window, bilinear warp, tolerance-mode solve) on `--pairs`
of bench.py's synthetic pairs, all resident in HBM.  Timed with CUDA events, every shape warmed up first, the three calls
interleaved round by round so that drift hits them alike:
  fwd     ofb_flow_pairs_device with the total flow (one direction, what bench.py's headline does plus the total)
  fb      ofb_flow_pairs_fb_device without err2 (both directions from one pyramid build + the check)
  fb_err2 the same with err2
The check kernel alone is read from its OFB_PROFILE_FB_CHECK records in the fb calls.  Its algorithmic bytes are
17 B/px (8 B fwd + 8 B bwd + 1 B status) or 21 B/px with err2; the copy peak beside it is a device-to-device copy of
a 4 GB buffer measured in the same run (read + write bytes over time).  Prints one JSON line (and writes it to --out).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

W, H, LEVELS, WIN = 1920, 1080, 3, 9


def card_info(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        pl, clk = [x.strip() for x in r.stdout.strip().split(",")]
        info.update({"power_limit": pl, "clocks_max_sm": clk})
    except Exception as e:  # (reported, not guessed)
        info.update({"power_limit": None, "nvidia_smi_error": repr(e)})
    return info


def copy_peak_gbs(torch, reps=10):
    n = 4 << 30
    src = torch.empty(n, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    src.fill_(1)
    for _ in range(3):
        dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        dst.copy_(src)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del src, dst
    torch.cuda.empty_cache()
    return 2 * n / (ms * 1e-3) / 1e9


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=512)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch

    from bench import synth_pairs_torch
    from cuda_optical_flow_2_b200 import PROFILE_FB_CHECK, SOLVE_FAST, WARP_BILINEAR, Context, OfbParams, _lib

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device"}), flush=True)
        return 1
    card = card_info(torch)
    n = args.pairs
    dev = torch.device("cuda", 0)
    prev, nxt, pitch = synth_pairs_torch(n, W, H, dev, seed=1)
    ctx = Context(0)
    ctx.solve = SOLVE_FAST
    lib, h = ctx._lib, ctx._h
    st = torch.cuda.current_stream().cuda_stream
    p = OfbParams(W, H, LEVELS, WIN, WARP_BILINEAR, 1.0, n)
    flows = [torch.empty((n, H >> k, W >> k, 2), dtype=torch.float32, device=dev) for k in range(LEVELS)]
    fptrs = (C.c_void_p * LEVELS)(*[f.data_ptr() for f in flows])
    fwd = torch.empty((n, H, W, 2), dtype=torch.float32, device=dev)
    bwd = torch.empty_like(fwd)
    status = torch.empty((n, H, W), dtype=torch.uint8, device=dev)
    err2 = torch.empty((n, H, W), dtype=torch.float32, device=dev)
    _lib.check(lib.ofb_ctx_reserve_pairs_fb(h, C.byref(p)))

    def call_fwd():
        _lib.check(lib.ofb_flow_pairs_device(h, C.byref(p), prev.data_ptr(), nxt.data_ptr(), pitch, pitch * H, fptrs,
                                             fwd.data_ptr(), C.c_void_p(st)))

    def call_fb(e2):
        _lib.check(lib.ofb_flow_pairs_fb_device(h, C.byref(p), prev.data_ptr(), nxt.data_ptr(), pitch, pitch * H,
                                                C.c_float(0.01), C.c_float(0.5), fwd.data_ptr(), bwd.data_ptr(),
                                                status.data_ptr(), e2, C.c_void_p(st)))

    calls = {"fwd": call_fwd, "fb": lambda: call_fb(None), "fb_err2": lambda: call_fb(err2.data_ptr())}
    for fn in calls.values():
        for _ in range(args.warmup):
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in calls}
    check_ms = {"fb": [], "fb_err2": []}
    for _ in range(args.reps):
        for k, fn in calls.items():
            if k != "fwd":
                ctx.profile_enable(True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1))
            if k != "fwd":
                cms, cn = ctx.profile_read(PROFILE_FB_CHECK)
                assert cn == 1
                check_ms[k].append(cms)
                ctx.profile_enable(False)
    counts = np.bincount(status.flatten().cpu().numpy(), minlength=5).tolist()
    del flows, fwd, bwd, status, err2, prev, nxt
    torch.cuda.empty_cache()
    peak = copy_peak_gbs(torch)
    mpx = W * H / 1e6 * n
    px = W * H * n
    rec = {"what": "forward-backward consistency check", "card": card, "pairs": n, "size": f"{W}x{H}", "levels": LEVELS,
           "win": WIN, "warp": "bilinear", "solve": "fast", "reps": args.reps, "copy_peak_gbs": peak,
           "status_counts_last_call": dict(zip(["consistent", "inconsistent", "outside", "fwd_nonfinite", "bwd_nonfinite"],
                                               counts))}
    for k in calls:
        med = float(np.median(ms[k]))
        rec[k] = {"ms_median": med, "ms_min": float(np.min(ms[k])), "ms_max": float(np.max(ms[k])),
                  "mpx_pairs_per_s": mpx / (med * 1e-3)}
    for k, bpp in (("fb", 17), ("fb_err2", 21)):
        med = float(np.median(check_ms[k]))
        gbs = bpp * px / (med * 1e-3) / 1e9
        rec[k]["check_kernel"] = {"ms_median": med, "ms_min": float(np.min(check_ms[k])), "bytes_per_px": bpp,
                                  "algorithmic_gbs": gbs, "frac_of_copy_peak": gbs / peak}
    rec["fb_over_fwd"] = rec["fb"]["ms_median"] / rec["fwd"]["ms_median"]
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    ctx.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
