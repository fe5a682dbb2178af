#!/usr/bin/env python
"""fb_e2e_bench.py -- the forward-backward check with host buffers: batched (ofb_flow_pairs_fb_host) and on the frame
stream (ofb_stream_push_bgr_host_fb), on one GPU.

    python scripts/fb_e2e_bench.py [--pairs 32] [--rounds 7] [--pushes 60] [--out FILE]

Workload: bench.py's headline settings (1920x1080, 3 levels, 9x9 window, bilinear warp, tolerance-mode solve) on bench.py's
synthetic frames, every host buffer pinned (ofb_host_alloc).  Every call is synchronous, so a host clock around it is the
call's time.  Everything is warmed up first, and the compared calls alternate round by round so that drift hits them alike;
medians over the rounds are reported.
  host  `lean`: ofb_flow_pairs_host_ex, planar gray in, total flow out (8 B/px: bench.py's `e2e.lean`);
        `fb`:   ofb_flow_pairs_fb_host on the same pairs, planar gray in, forward total + status out (9 B/px).
  stream (ms per push of a 1080p BGR frame): `push` (ofb_stream_push_bgr_host with the total flow: the residual flow of
        every level and the total come back, 18.5 B/px at 3 levels), `push_no_total` (the same without the total, 10.5 B/px:
        level 0 composes the cumulative flow on the fly, level 1 does not write its own), `push_fb` (forward total + status back, 9 B/px) with the
        backward level loop on the stream's second CUDA stream (the default) and with OFB_FB_SERIAL=1 (after the forward
        loop on the context stream).  The override is read once per process, so each mode runs in child processes of its
        own, which alternate; `push` and `push_no_total` are timed in both, alternating with `push_fb`.  The children also hash their last
        outputs: the two modes must give the same bytes.  `push` downloads twice the bytes of `push_fb`, so the
        difference of the two is no cost of the check; the fork is judged by `push_fb` forked against serial.
The card's name, power limit and maximum SM clock are read with nvidia-smi, the SM clock under load (and any throttle
reason) sampled through NVML while the host rounds and each stream child's timed rounds run.  Prints one JSON line (and writes it to --out).
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

W, H, LEVELS, WIN = 1920, 1080, 3, 9
ALPHA, BETA = 0.01, 0.5


def card_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30)
        return dict(zip(["name", "power_limit", "clocks_max_sm", "clocks_sm_idle"], [x.strip() for x in r.stdout.split(",")]))
    except Exception as e:  # (reported, not guessed)
        return {"nvidia_smi_error": repr(e)}


def stream_child(mode, rounds, pushes):
    """One process, one mode of the check's fork: rounds of `pushes` plain pushes and `pushes` pushes with the check."""
    from bench import ClockSampler, Pinned, synth_pairs_numpy
    from cuda_optical_flow_2_b200 import SOLVE_FAST, WARP_BILINEAR, Context, _lib

    a, b = synth_pairs_numpy(4, W, H, 31)
    pin = Pinned()
    frames = [pin.array((H, W, 3), np.uint8) for _ in range(8)]
    for i, f in enumerate(frames):
        f[...] = (a if i % 2 == 0 else b)[i // 2]
    flows = [pin.array((H >> k, W >> k, 2), np.float32) for k in range(LEVELS)]
    total, fwd = pin.array((H, W, 2), np.float32), pin.array((H, W, 2), np.float32)
    status = pin.array((H, W), np.uint8)
    lib = _lib.load()
    f32, u8 = lambda x: x.ctypes.data_as(_lib.f32p), lambda x: x.ctypes.data_as(_lib.u8p)
    fptrs = (_lib.f32p * LEVELS)(*[f32(x) for x in flows])
    ctx = Context(0)
    ctx.solve = SOLVE_FAST
    st = ctx.open_stream(W, H, LEVELS, WIN, warp_mode=WARP_BILINEAR)
    has = C.c_int()
    t = [0]

    def push():
        _lib.check(lib.ofb_stream_push_bgr_host(st._h, u8(frames[t[0] % 8]), fptrs, f32(total), C.byref(has)))
        t[0] += 1

    def push_no_total():
        _lib.check(lib.ofb_stream_push_bgr_host(st._h, u8(frames[t[0] % 8]), fptrs, None, C.byref(has)))
        t[0] += 1

    def push_fb():
        _lib.check(lib.ofb_stream_push_bgr_host_fb(st._h, u8(frames[t[0] % 8]), ALPHA, BETA, None, f32(fwd), None, u8(status), None,
                                                   C.byref(has)))
        t[0] += 1

    def block(fn):
        t0 = time.perf_counter()
        for _ in range(pushes):
            fn()
        return (time.perf_counter() - t0) / pushes * 1e3

    arms = {"push": push, "push_no_total": push_no_total, "push_fb": push_fb}
    for _ in range(2):  # warm-up: kernels loaded, buffers and the second stream created
        for fn in arms.values():
            block(fn)
    ms = {k: [] for k in arms}
    clocks = ClockSampler(0)
    clocks.start()
    for _ in range(rounds):
        for k, fn in arms.items():
            ms[k].append(block(fn))
    clk = clocks.stop()
    # the last push_fb's frames are fixed by the counter: identical inputs in every child
    digest = hashlib.sha256(fwd.tobytes() + status.tobytes()).hexdigest()
    st.close()
    ctx.close()
    pin.free()
    print(json.dumps({"mode": mode, "ms": ms, "last_push_fb_sha256": digest, "pushes_total": t[0], "clocks_under_load": clk}),
          flush=True)
    return 0


def run_children(rounds, pushes, children):
    res = {"fork": [], "serial": []}
    for _ in range(children):
        for mode in ("fork", "serial"):
            env = {k: v for k, v in os.environ.items() if k != "OFB_FB_SERIAL"}
            if mode == "serial":
                env["OFB_FB_SERIAL"] = "1"
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--stream-child", mode, "--rounds", str(rounds),
                                "--pushes", str(pushes)], env=env, capture_output=True, text=True, timeout=1200)
            if r.returncode != 0:
                raise RuntimeError(f"stream child ({mode}) failed: {r.stderr[-2000:]}")
            res[mode].append(json.loads(r.stdout.strip().splitlines()[-1]))
    return res


def host_block(rounds, pairs, warmup):
    from bench import ClockSampler, Pinned, synth_pairs_numpy
    from cuda_optical_flow_2_b200 import SOLVE_FAST, WARP_BILINEAR, Context, OfbParams, _lib

    a, b = synth_pairs_numpy(min(pairs, 4), W, H, 2000)
    pin = Pinned()
    gprev, gnext = pin.array((pairs, H, W), np.uint8), pin.array((pairs, H, W), np.uint8)
    for i in range(pairs):
        gprev[i], gnext[i] = a[i % len(a)][:, :, 0], b[i % len(b)][:, :, 0]
    total = pin.array((pairs, H, W, 2), np.float32)
    fwd = pin.array((pairs, H, W, 2), np.float32)
    status = pin.array((pairs, H, W), np.uint8)
    lib = _lib.load()
    f32, u8 = lambda x: x.ctypes.data_as(_lib.f32p), lambda x: x.ctypes.data_as(_lib.u8p)
    ctx = Context(0)
    ctx.solve = SOLVE_FAST
    p = OfbParams(W, H, LEVELS, WIN, WARP_BILINEAR, 1.0, pairs)

    def lean():
        _lib.check(lib.ofb_flow_pairs_host_ex(ctx._h, C.byref(p), u8(gprev), u8(gnext), 1, None, f32(total)))

    def fb():
        _lib.check(lib.ofb_flow_pairs_fb_host(ctx._h, C.byref(p), u8(gprev), u8(gnext), 1, ALPHA, BETA, f32(fwd), None, u8(status),
                                              None))

    calls = {"lean": lean, "fb": fb}
    for fn in calls.values():
        for _ in range(warmup):
            fn()
    clocks = ClockSampler(0)
    clocks.start()
    sec = {k: [] for k in calls}
    for _ in range(rounds):
        for k, fn in calls.items():
            t0 = time.perf_counter()
            fn()
            sec[k].append(time.perf_counter() - t0)
    clk = clocks.stop()
    same = bool(np.array_equal(fwd.view(np.uint32), total.view(np.uint32)))
    counts = np.bincount(status.reshape(-1), minlength=5).tolist()
    ctx.close()
    pin.free()
    mpx = W * H / 1e6 * pairs
    rec = {"pairs_per_call": pairs, "clocks_under_load": clk, "fb_forward_total_equals_lean_total": same,
           "status_counts": dict(zip(["consistent", "inconsistent", "outside", "fwd_nonfinite", "bwd_nonfinite"], counts))}
    for k, bpp in (("lean", 2 + 8), ("fb", 2 + 9)):
        med = float(np.median(sec[k]))
        rec[k] = {"ms_median": med * 1e3, "ms_min": float(np.min(sec[k])) * 1e3, "ms_max": float(np.max(sec[k])) * 1e3,
                  "mpx_pairs_per_s": mpx / med, "pcie_bytes_per_px": bpp}
    rec["fb_over_lean_time"] = rec["fb"]["ms_median"] / rec["lean"]["ms_median"]
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=32, help="pairs per host-batch call (bench.py's e2e uses 32)")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--pushes", type=int, default=60, help="pushes per timed stream block")
    ap.add_argument("--children", type=int, default=3, help="child processes per stream mode (they alternate)")
    ap.add_argument("--stream-child", choices=["fork", "serial"], help=argparse.SUPPRESS)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.stream_child:
        return stream_child(args.stream_child, args.rounds, args.pushes)

    card = card_info()
    host = host_block(args.rounds, args.pairs, args.warmup)
    kids = run_children(args.rounds, args.pushes, args.children)
    level_bytes = sum(8 / 4 ** k for k in range(LEVELS))  # residual flow of every level, per level-0 pixel
    stream = {"pushes_per_block": args.pushes, "rounds_per_child": args.rounds, "children_per_mode": args.children,
              "d2h_bytes_per_px": {"push": level_bytes + 8, "push_no_total": level_bytes, "push_fb": 9}, "h2d_bytes_per_px": 3}
    for mode in ("fork", "serial"):
        stream[mode] = {"clocks_under_load_per_child": [c["clocks_under_load"] for c in kids[mode]]}
        for arm in ("push", "push_no_total", "push_fb"):
            v = [x for c in kids[mode] for x in c["ms"][arm]]
            stream[mode].update({f"{arm}_ms_median": float(np.median(v)), f"{arm}_ms_min": float(np.min(v)),
                                 f"{arm}_ms_max": float(np.max(v))})
    digests = {c["last_push_fb_sha256"] for m in ("fork", "serial") for c in kids[m]}
    stream["fork_and_serial_same_bytes"] = len(digests) == 1
    stream["fork_saves_ms"] = stream["serial"]["push_fb_ms_median"] - stream["fork"]["push_fb_ms_median"]
    rec = {"what": "forward-backward check with host buffers: batched host call and frame stream", "card": card,
           "size": f"{W}x{H}", "levels": LEVELS, "win": WIN, "warp": "bilinear", "solve": "fast", "alpha": ALPHA, "beta": BETA,
           "host_memory": "pinned (ofb_host_alloc)", "host": host, "stream": stream}
    line = json.dumps(rec)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
