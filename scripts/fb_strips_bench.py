#!/usr/bin/env python
"""fb_strips_bench.py -- the forward-backward check on row strips of one large pair: plain against checked pairs.

    python scripts/fb_strips_bench.py [--size 7680x4320x4] [--win 9] [--reps 40] [--rounds 5] [--out FILE]
    torchrun --nproc-per-node N scripts/fb_strips_bench.py ...    (one rank per GPU, peer-memory transport over CUDA IPC)

Workload: one WxH pair of bench.py's synthetic frames (the same on every rank), L levels, the given window, bilinear warp,
the context's default (bit-exact) solve, fb_reach 16, alpha 0.01, beta 0.5, no err2.  Four check-capable handles per rank
(dist.NativeStrips with fb_reach), each pair replayed as a CUDA graph captured per handle and kind (eager if capture fails).
Timed as ms per pair between CUDA events, the maximum over the ranks, medians over rounds in which the configurations
alternate:
  plain_1 / checked_1      one pair at a time on one stream: the latency of a pair's whole dependency chain
  plain_4 / checked_4      four handles on four streams, pairs in flight (the throughput of a frame sequence)
  alternated_4             plain and checked pairs alternating on each of the four handles
plus check_kernel_ms: the check kernel alone on a rank's own rows (ofb_fb_check_device on a field of that size), to split
a checked pair's extra time into the check and the backward level loop with its exchanges.  bit_identical_to_whole_frame:
every rank's forward total, backward total, status and err2 after a checked pair equal its rows of ofb_flow_pairs_fb_device
on the whole frame (computed on each rank's GPU).  The card's name, power limit and SM clocks (nvidia-smi, and the SM clock
sampled through NVML while the timed rounds run) are recorded with the numbers.  Rank 0 prints one JSON line (and writes
it to --out).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ALPHA, BETA, FB_REACH, K = 0.01, 0.5, 16, 4


def card_info(index):
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return dict(zip(["name", "power_limit", "clocks_max_sm", "clocks_sm_idle"], [x.strip() for x in r.stdout.split(",")]))
    except Exception as e:  # (reported, not guessed)
        return {"nvidia_smi_error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", default="7680x4320x4", help="WxHxLEVELS")
    ap.add_argument("--win", type=int, default=9)
    ap.add_argument("--reps", type=int, default=40, help="pairs per timed window")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    w, h, levels = (int(x) for x in args.size.split("x"))
    win = args.win

    import torch

    from bench import ClockSampler, Env, synth_pairs_torch
    from cuda_optical_flow_2_b200 import WARP_BILINEAR, Context
    from cuda_optical_flow_2_b200.dist import NativeStrips

    env = Env()
    world, rank, dev = env.world, env.rank, env.dev
    ctx = Context(env.local)
    prev, nxt, _ = synth_pairs_torch(1, w, h, dev, 4242)
    whole = ctx.flow_pairs_fb_device(prev, nxt, w, levels, win, warp_mode=WARP_BILINEAR, alpha=ALPHA, beta=BETA, want_err2=True)
    torch.cuda.synchronize()
    transport = "peer" if world > 1 else "local"
    handles = [NativeStrips(ctx, w, h, levels, win, world, rank, dev, WARP_BILINEAR, 1.0, 16, transport=transport, fb_reach=FB_REACH)
               for _ in range(K)]
    y0, y1 = handles[0].own_rows(0)
    ins = []
    for ns in handles:
        ns.set_total(False)
        pin, nin = ns.input_rows()  # the producer writes the own rows where the runner keeps them
        pin[:, :w].copy_(prev[0, y0:y1, :w])
        nin[:, :w].copy_(nxt[0, y0:y1, :w])
        ins.append((pin, nin))
    streams = [torch.cuda.Stream(dev) for _ in range(K)]

    def enqueue(kind, i, stream):
        ns, (pin, nin) = handles[i], ins[i]
        if kind == "c":
            ns.run_fb(pin, nin, ALPHA, BETA, False, stream)
        else:
            ns.run(pin, nin, stream)

    # warm-up (every kernel of both kinds), then one graph per handle and kind
    for i, st in enumerate(streams):
        with torch.cuda.stream(st):
            for kind in "pcpc":
                enqueue(kind, i, st.cuda_stream)
    env.barrier()
    for ns, st in zip(handles, streams):
        ns.check(st.cuda_stream)
    graphs, use_graph = {}, True
    try:
        for i, st in enumerate(streams):
            for kind in "pc":
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=st, capture_error_mode="thread_local"):
                    enqueue(kind, i, torch.cuda.current_stream(dev).cuda_stream)
                graphs[kind, i] = g
    except Exception as ex:
        print(f"fb_strips_bench: graph capture failed ({ex!r}); eager", file=sys.stderr)
        use_graph, graphs = False, {}
    env.barrier()

    def measure(n_handles, kind_of):
        env.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ss = streams[:n_handles]
        for st in ss:
            st.wait_stream(torch.cuda.current_stream(dev))
        e0.record()
        for st in ss:
            st.wait_event(e0)
        for i in range(args.reps):
            hi = i % n_handles
            kind, st = kind_of(i, n_handles), streams[hi]
            with torch.cuda.stream(st):
                if use_graph:
                    graphs[kind, hi].replay()
                else:
                    enqueue(kind, hi, st.cuda_stream)
        for st in ss:
            torch.cuda.current_stream(dev).wait_stream(st)
        e1.record()
        env.barrier()
        for ns, st in zip(handles[:n_handles], ss):
            ns.check(st.cuda_stream)
        return env.max_over_ranks(e0.elapsed_time(e1) / args.reps)

    configs = {"plain_1": (1, lambda i, n: "p"), "checked_1": (1, lambda i, n: "c"), "plain_4": (K, lambda i, n: "p"),
               "checked_4": (K, lambda i, n: "c"), "alternated_4": (K, lambda i, n: "pc"[(i + i // n) % 2])}
    times = {k: [] for k in configs}
    clocks = ClockSampler(env.local)
    clocks.start()
    for _ in range(args.rounds):
        for name, (n, kind_of) in configs.items():
            times[name].append(measure(n, kind_of))
    clk = clocks.stop()

    # the check kernel alone on a field of the own rows' size
    f = whole[0][:, y0:y1].contiguous()
    b = whole[1][:, y0:y1].contiguous()
    for _ in range(3):
        ctx.fb_check_device(f, b, 1.0, ALPHA, BETA)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        ctx.fb_check_device(f, b, 1.0, ALPHA, BETA)
    e1.record()
    torch.cuda.synchronize()
    check_ms = env.max_over_ranks(e0.elapsed_time(e1) / 20)

    # bit identity of a checked pair (with err2) against the whole frame, on every rank
    st0 = streams[0]
    handles[0].run_fb(ins[0][0], ins[0][1], ALPHA, BETA, True, st0.cuda_stream)
    handles[0].check(st0.cuda_stream)
    ok = True
    for got, ref in zip(handles[0].own_fb(), whole):
        ref = ref[0, y0:y1]
        if ref.dtype == torch.uint8:
            ok &= bool(torch.equal(got, ref))
        else:
            ng, nr = torch.isnan(got), torch.isnan(ref)
            ok &= bool(torch.equal(ng, nr)) and bool(torch.equal(got[~ng].view(torch.int32), ref[~nr].view(torch.int32)))
    flag = torch.tensor([1 if ok else 0], device=dev)
    if world > 1:
        env.dist.all_reduce(flag, op=env.dist.ReduceOp.MIN)
    ok = bool(flag.item())

    med = {k: statistics.median(v) for k, v in times.items()}
    rec = {"workload": f"{w}x{h} pair, {levels} levels, window {win}, row strips over {world} rank(s), fb_reach {FB_REACH}",
           "n_ranks": world, "transport": "peer" if world > 1 else None, "cuda_graph": use_graph, "reps": args.reps,
           "rounds": args.rounds, "own_rows_rank0": [y0, y1] if rank == 0 else None,
           "ms_per_pair_median": med, "ms_per_pair_rounds": times,
           "checked_over_plain": {"alone": med["checked_1"] / med["plain_1"], "in_flight_4": med["checked_4"] / med["plain_4"]},
           "check_kernel_ms_own_rows": check_ms, "bit_identical_to_whole_frame": ok,
           "card": card_info(env.local), "clocks_under_load": clk}
    env.barrier()
    for ns in handles:
        ns.close()
    if rank == 0:
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "w") as fo:
                fo.write(line + "\n")
    if world > 1:
        env.dist.destroy_process_group()
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
