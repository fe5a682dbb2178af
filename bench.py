#!/usr/bin/env python
"""bench.py -- megapixel frame-pairs/s of the dense pyramidal LK path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--pairs B] [--impl b200|reference] [--solve fast|exact]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): 1920x1080 frame pairs, 3-level Gaussian pyramid, 9x9 window.
A step is one pass of the whole path (both pyramids + 3 fused LK levels) over a batch of B synthetic
pairs per GPU (default 1024).  `value` is timed with CUDA events with every input already resident in HBM; the
batch's inputs (B x 4.1 MB) are larger than the 126 MB L2, so no step re-reads cached frames.
`e2e` is the same metric through the host-pointer C-ABI call (ofb_flow_pairs_host) with pinned host
buffers in the reference's 3-channel layout, H2D and D2H inside the timed region.
N > 1 (torchrun): pairs are sharded per GPU, no data-path collective, weak scaling.

The headline runs the tolerance-mode solve (OFB_SOLVE_FAST: exact integer sums, determinant and numerators, one float
reciprocal; |du|,|dv| <= 1e-4 px + 1e-5 |ref| per level, checked in this run: `parity`); the bit-exact solve is timed
beside it (`exact`).  Further records of the same line: `configs` (BASELINE configs[0] and [2]), `strips` (configs[4]:
one 7680x4320 pair cut into row strips over the N ranks, halo rows over NVLink peer memory), `e2e_dropin` (the
reference's own per-level entry points with host pointers), `reference_gpu` (the unmodified reference's GPU path on this
GPU, for scale), `cpu_baseline`.

`--impl reference` times the reference's own CPU implementation (cpu::gauss_pyramid +
cpu::calc_optical_flow, compiled unmodified into oracle/_ref/libofref.so) on the host cores.

`--dump-outputs DIR` writes what the headline's last timed step returned, so that two builds can be compared output for
output (the inputs depend only on the arguments): DIR/flow_level<k>.npy, float32 (pairs, H >> k, W >> k, 2), the residual
flow of level k for a fixed, seeded sample of the batch's pairs (as many whole pairs as fit in 64 MB; rank 0's batch).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W, H, LEVELS, WIN = 1920, 1080, 3, 9
METRIC = "megapixel frame-pairs/sec (1080p, 3-level, win 9)"
UNIT = "Mpx-pairs/s"
# identical in both arms (the driver compares the arms' `config`); everything run-specific lives under `run`
CONFIG = {"workload": "1920x1080 frame pair, 3-level Gaussian pyramid, 9x9 window"}
TOL_ABS, TOL_REL = 1e-4, 1e-5  # the stated per-level tolerance of the tolerance-mode solve (px on u and v)


# ----------------------------------------------------------------------------------------------
def synth_pairs_torch(n, w, h, device, seed, return_shifts=False):
    """Value-noise frames on the GPU: random 8-px grid, bilinear, next = prev shifted sub-pixel."""
    import torch

    g = torch.Generator(device="cpu").manual_seed(seed)
    cell = 8
    gw, gh = w // cell + 6, h // cell + 6
    pitch = (w + 63) // 64 * 64
    prev = torch.zeros((n, h, pitch), dtype=torch.uint8, device=device)
    nxt = torch.zeros((n, h, pitch), dtype=torch.uint8, device=device)
    xs = torch.arange(w, device=device, dtype=torch.float32)
    ys = torch.arange(h, device=device, dtype=torch.float32)
    shifts = []
    for i in range(n):
        grid = torch.randint(0, 256, (gh, gw), generator=g).to(device=device, dtype=torch.float32)
        dxy = (torch.rand(2, generator=g) * 8.0 - 4.0).tolist()  # up to +-4 px: the pyramid matters
        shifts.append(dxy)
        for dst, (dx, dy) in ((prev, (0.0, 0.0)), (nxt, dxy)):
            fx = (xs - dx) / cell + 2.5
            fy = (ys - dy) / cell + 2.5
            ix = fx.floor().clamp(0, gw - 2).long()
            iy = fy.floor().clamp(0, gh - 2).long()
            ax = (fx - ix).view(1, -1)
            ay = (fy - iy).view(-1, 1)
            g00 = grid[iy][:, ix]
            g01 = grid[iy][:, ix + 1]
            g10 = grid[iy + 1][:, ix]
            g11 = grid[iy + 1][:, ix + 1]
            v = (1 - ay) * ((1 - ax) * g00 + ax * g01) + ay * ((1 - ax) * g10 + ax * g11)
            dst[i, :, :w] = v.clamp(0, 255).to(torch.uint8)
    if return_shifts:
        return prev, nxt, pitch, shifts
    return prev, nxt, pitch


def synth_pairs_numpy(n, w, h, seed):
    """Same construction on the host (3-channel reference layout) for the CPU arms and e2e."""
    rng = np.random.default_rng(seed)
    cell = 8
    gw, gh = w // cell + 6, h // cell + 6
    prev = np.empty((n, h, w, 3), np.uint8)
    nxt = np.empty((n, h, w, 3), np.uint8)
    xs = np.arange(w, dtype=np.float32)
    ys = np.arange(h, dtype=np.float32)
    for i in range(n):
        grid = rng.integers(0, 256, (gh, gw)).astype(np.float32)
        dxy = rng.random(2) * 8.0 - 4.0
        for dst, (dx, dy) in ((prev, (0.0, 0.0)), (nxt, dxy)):
            fx = (xs - np.float32(dx)) / cell + 2.5
            fy = (ys - np.float32(dy)) / cell + 2.5
            ix = np.clip(np.floor(fx), 0, gw - 2).astype(np.int64)
            iy = np.clip(np.floor(fy), 0, gh - 2).astype(np.int64)
            ax = (fx - ix)[None, :]
            ay = (fy - iy)[:, None]
            g00, g01 = grid[iy][:, ix], grid[iy][:, ix + 1]
            g10, g11 = grid[iy + 1][:, ix], grid[iy + 1][:, ix + 1]
            v = (1 - ay) * ((1 - ax) * g00 + ax * g01) + ay * ((1 - ax) * g10 + ax * g11)
            dst[i] = np.clip(v, 0, 255).astype(np.uint8)[:, :, None]
    return prev, nxt


class ClockSampler:
    """SM clock, power and throttle reasons sampled through NVML every 5 ms while the timed region runs."""

    def __init__(self, index: int):
        self.index, self.samples, self._stop, self.err = index, [], threading.Event(), None

    def start(self):
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as ex:  # no NVML: report it instead of inventing numbers
            self.err = repr(ex)
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                clk = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.samples.append((clk, rs, pw))
            except Exception as ex:
                self.err = repr(ex)
                return
            time.sleep(0.005)

    def stop(self):
        if self.err and not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + self.err], "samples": 0}
        self._stop.set()
        self.t.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        # samples under load = the upper half by power draw (the region also covers launch gaps)
        s = sorted(self.samples, key=lambda x: x[2])
        hot = s[len(s) // 2:] if s else []
        reasons = sorted({n for n, bit in names.items() for (_, rs, _) in self.samples if rs & bit})
        return {"sm_mhz": float(np.median([c for c, _, _ in hot])) if hot else None, "sm_max_mhz": float(self.max_sm),
                "reasons": reasons, "samples": len(self.samples),
                "power_w_max": max((pw for _, _, pw in self.samples), default=None)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """DRAM bytes per launch of the level-0 kernel from the committed ncu --set full summary."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


def level_bytes(w, h, level, levels, n_pairs, cum_out):
    """Algorithmic bytes of one fused-LK launch (DESIGN.md 3.1): 1 B prev + 1 B next + 8 B flow per pixel, + 8 B per
    coarser pixel of cumulative flow in (warped levels), + 8 B per pixel of cumulative flow out where a level writes it."""
    n = (w >> level) * (h >> level)
    b = n * 10
    if level < levels - 1:
        b += (w >> (level + 1)) * (h >> (level + 1)) * 8
    if cum_out:
        b += n * 8
    return b * n_pairs


# ---------------------------------------------------------------------------------------------- reference arm
def ref_lib():
    from oracle import oracle as O  # the one place bench.py executes oracle/: the CPU baseline (and reference_gpu)

    if not O.have_ref():
        return None, O
    return O.ref(), O


def run_reference_cpu(n_pairs: int, threads: int, reps: int = 1):
    """Reference CPU path on `threads` host threads, one pair per task.  Returns (seconds per rep, cores)."""
    from concurrent.futures import ThreadPoolExecutor

    lib, O = ref_lib()
    prev, nxt = synth_pairs_numpy(min(n_pairs, 4), W, H, 7)
    kind = "reference"
    if lib is None:
        kind = "port"

    def one(i):
        p, q = prev[i % len(prev)], nxt[i % len(nxt)]
        if lib is not None:
            flows = [np.zeros((H >> k, W >> k, 2), np.float32) for k in range(LEVELS)]
            ptr = (O._f32p * LEVELS)(*[f.ctypes.data_as(O._f32p) for f in flows])
            lib.ref_cpu_flow_pair(p.ctypes.data_as(O._u8p), q.ctypes.data_as(O._u8p), W, H, LEVELS, ptr)
        else:
            O.flow_pair(np.ascontiguousarray(p[:, :, 0]), np.ascontiguousarray(q[:, :, 0]), LEVELS, WIN,
                        O.WARP_AS_WRITTEN, O.SUMS_F32_SEQUENTIAL)

    times = []
    with ThreadPoolExecutor(max_workers=threads) as ex:
        for _ in range(reps):
            t0 = time.perf_counter()
            list(ex.map(one, range(n_pairs)))
            times.append(time.perf_counter() - t0)
    return times, kind


def main_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    n_pairs = cores  # one pair per host thread per step: a bounded sample of the workload
    times, kind = run_reference_cpu(n_pairs, cores, reps=args.warmup + args.steps)
    timed = times[args.warmup:]
    total = sum(timed)
    value = (W * H / 1e6) * n_pairs * len(timed) / total
    sample = f"{n_pairs} pairs per step on {cores} threads, {len(timed)} steps"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(timed),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8->int->f64 (CPU)",
            "data": "synthetic", "config": dict(CONFIG),
            "run": {"pairs_per_step": n_pairs, "where": "host CPU", "note": "the host threads do not grow with --gpus: the "
                    "driver's ratio at N > 1 is not a scaling statement"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------- B200 arm: pieces
class Env:
    """Process-wide handles of the B200 arm."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.stream = torch.cuda.current_stream().cuda_stream

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def sum_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.item()


def timed_device_steps(env, ctx, prev, nxt, w, h, levels, win, steps, warmup, flows=None, sampler=None):
    """K steps of the device-resident path between two events, barrier + synchronize on both sides, per-level CUDA-event
    timing on.  Returns (ms per step = max over ranks, launches on this rank, [(ms, n) per level], (ms, n) pyramid, clocks)."""
    from cuda_optical_flow_2_b200 import WARP_BILINEAR, _lib

    torch = env.torch
    n = prev.shape[0]
    if flows is None:
        flows = [torch.empty((n, h >> k, w >> k, 2), dtype=torch.float32, device=env.dev) for k in range(levels)]

    def step():
        ctx.flow_pairs_device(prev, nxt, w, levels, win, warp_mode=WARP_BILINEAR, flows=flows, stream=env.stream)

    for _ in range(warmup):
        step()
    env.barrier()
    if sampler is not None:
        sampler.start()
    ctx.profile_enable(True)
    l0 = ctx.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.barrier()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    env.barrier()
    ms_total = e0.elapsed_time(e1)
    launches = ctx.launch_count - l0
    clocks = sampler.stop() if sampler is not None else None
    lvl = [ctx.profile_read(k) for k in range(levels)]
    pyr = ctx.profile_read(_lib.PROFILE_PYRAMID)
    ctx.profile_enable(False)
    return env.max_over_ranks(ms_total) / steps, launches, lvl, pyr, clocks, flows


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, flows):
    """Writes a fixed, seeded sample of whole pairs of `flows` (one (n, h, w, 2) tensor per level) to out_dir; returns the
    sampled pair indices."""
    n = flows[0].shape[0]
    per_pair = sum(f[0].numel() * f.element_size() for f in flows)
    pairs = np.sort(np.random.default_rng(0).choice(n, max(1, min(n, DUMP_BYTES // per_pair)), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for k, f in enumerate(flows):
        np.save(os.path.join(out_dir, f"flow_level{k}.npy"), f[pairs.tolist()].cpu().numpy())
    return pairs.tolist()


def roofline_of(level_ms, w, h, level, levels, n_pairs, cum_out, peak):
    ms, n = level_ms
    avg = ms / max(n, 1)
    b = level_bytes(w, h, level, levels, n_pairs, cum_out)
    ach = b / (avg * 1e-3) / 1e9 if avg > 0 else 0.0
    return {"avg_launch_ms": avg, "algorithmic_bytes_per_launch": b, "achieved": ach, "frac": ach / peak}


def parity_block(env, ctx):
    """Accuracy of what the headline measures, on 4 synthetic 1080p pairs with a known uniform shift (rank 0):
    tolerance-mode solve against the bit-exact one (per level on identical inputs = the coarsest level, and through the
    whole pipeline), end-point error of the total flow against the known shift for the three warp modes (the flow is in
    the reference's units of 15/8 px, Q1, so it is scaled by 8/15 first), and bilinear against the as-written warp."""
    from cuda_optical_flow_2_b200 import SOLVE_EXACT, SOLVE_FAST, WARP_AS_WRITTEN, WARP_BILINEAR, WARP_NEAREST

    torch = env.torch
    n = 4
    prev, nxt, _, shifts = synth_pairs_torch(n, W, H, env.dev, 99, return_shifts=True)
    sh = torch.tensor(shifts, dtype=torch.float32, device=env.dev).view(n, 1, 1, 2)
    keep = ctx.solve

    def run(mode, scale, solve):
        ctx.solve = solve
        total = torch.empty((n, H, W, 2), dtype=torch.float32, device=env.dev)
        fl = ctx.flow_pairs_device(prev, nxt, W, LEVELS, WIN, warp_mode=mode, flow_scale=scale, total_flow=total)
        torch.cuda.synchronize()
        return [f.clone() for f in fl], total

    out = {"pairs": n, "tolerance": f"|du|,|dv| <= {TOL_ABS} px + {TOL_REL} |ref| per level on identical inputs"}
    try:
        ex_f, ex_t = run(WARP_BILINEAR, 1.0, SOLVE_EXACT)
        fa_f, fa_t = run(WARP_BILINEAR, 1.0, SOLVE_FAST)
        per_level = []
        for k in range(LEVELS - 1, -1, -1):
            e, f = ex_f[k], fa_f[k]
            fe, ff = torch.isfinite(e), torch.isfinite(f)
            both = fe & ff
            d = (e - f).abs()[both]
            lim = TOL_ABS + TOL_REL * e.abs()[both]
            per_level.append({"level": k, "same_nonfinite_pixels": bool((fe == ff).all()), "max_abs_diff": d.max().item(),
                              "frac_beyond_tolerance": (d > lim).float().mean().item(),
                              "identical_inputs": k == LEVELS - 1})
        out["fast_vs_exact"] = {"per_level": per_level, "note": "the coarsest level has identical inputs in both runs (the "
                                "per-level bar); finer levels also see the warp re-quantised (1/256 px) where the coarser "
                                "flow moved by an ulp"}
        both = torch.isfinite(ex_t) & torch.isfinite(fa_t)
        out["fast_vs_exact"]["total_flow_max_abs_diff"] = (ex_t - fa_t).abs()[both].max().item()
        out["fast_vs_exact"]["coarsest_level_within_tolerance"] = per_level[0]["frac_beyond_tolerance"] == 0.0 and \
            per_level[0]["same_nonfinite_pixels"]

        def epe(total):  # px, interior (a window and a coarsest-level pixel away from the border), finite pixels
            m = 32
            t = total[:, m:-m, m:-m] * (8.0 / 15.0) - sh
            e = torch.sqrt((t * t).sum(-1))
            e = e[torch.isfinite(e)]
            return {"median_px": e.median().item(), "mean_px": e.clamp(max=100.0).mean().item(),
                    "frac_below_0.25px": (e < 0.25).float().mean().item()}

        acc = {}
        for name, mode in (("as_written", WARP_AS_WRITTEN), ("nearest", WARP_NEAREST), ("bilinear", WARP_BILINEAR)):
            for sname, scale in (("flow_scale_1", 1.0), ("flow_scale_8_15", 8.0 / 15.0)):
                _, t = run(mode, scale, SOLVE_EXACT)
                acc[f"{name}/{sname}"] = epe(t)
        acc["bilinear/flow_scale_8_15/fast_solve"] = epe(run(WARP_BILINEAR, 8.0 / 15.0, SOLVE_FAST)[1])
        out["epe_vs_known_shift"] = acc
        out["epe_note"] = ("total flow x 8/15 against the synthetic shift (|shift| <= 4 px per axis); flow_scale 1 is the "
                           "reference's behaviour (the warp over-shifts by 15/8, Q5), 8/15 warps by pixels")
        _, aw = run(WARP_AS_WRITTEN, 1.0, SOLVE_EXACT)
        d = (ex_t - aw)[:, 32:-32, 32:-32]
        e = torch.sqrt((d * d).sum(-1))
        e = e[torch.isfinite(e)]
        out["bilinear_vs_as_written"] = {"median_flow_units": e.median().item(), "mean_flow_units": e.clamp(max=100.0).mean().item(),
                                         "note": "total flow, reference units (15/8 px); quantifies the documented Q4 deviation"}
    finally:
        ctx.solve = keep
    return out


def single_pair_latency(env, ctx, prev, nxt, flows):
    from cuda_optical_flow_2_b200 import WARP_BILINEAR

    torch = env.torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f1 = [f[:1] for f in flows]

    def one(stream):
        ctx.flow_pairs_device(prev[:1], nxt[:1], W, LEVELS, WIN, warp_mode=WARP_BILINEAR, flows=f1, stream=stream)

    for _ in range(5):
        one(env.stream)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(50):
        one(env.stream)
    e1.record()
    torch.cuda.synchronize()
    one_ms, graph_ms = e0.elapsed_time(e1) / 50, None
    try:
        if env.world > 1:  # the single-GPU line carries it; no capture next to a live NCCL communicator
            raise RuntimeError("skipped at world > 1")
        side = torch.cuda.Stream(env.dev)
        side.wait_stream(torch.cuda.current_stream(env.dev))
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
            one(torch.cuda.current_stream(env.dev).cuda_stream)
        for _ in range(5):
            g.replay()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(50):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        graph_ms = e0.elapsed_time(e1) / 50
    except Exception as ex:  # reported, never fatal
        if env.world == 1:
            print(f"single-pair graph capture failed: {ex!r}", file=sys.stderr)
    return one_ms, graph_ms


class Pinned:
    """Pinned host arrays from the library's own allocator (the caller side of the C ABI)."""

    def __init__(self):
        from cuda_optical_flow_2_b200 import _lib

        self._lib, self.lib, self.ptrs = _lib, _lib.load(), []

    def array(self, shape, dtype):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        p = C.c_void_p()
        self._lib.check(self.lib.ofb_host_alloc(C.byref(p), n))
        self.ptrs.append(p)
        return np.frombuffer((C.c_uint8 * n).from_address(p.value), dtype=dtype).reshape(shape)

    def free(self):
        for p in self.ptrs:
            self.lib.ofb_host_free(p)
        self.ptrs = []


def e2e_block(env, ctx, args):
    """The metric through the host-pointer C-ABI calls, all ranks concurrently (their PCIe links share the host)."""
    from cuda_optical_flow_2_b200 import WARP_BILINEAR

    torch = env.torch
    Be = args.e2e_pairs
    hp, hn = synth_pairs_numpy(min(Be, 2), W, H, 2000 + env.rank)
    pin = Pinned()
    hprev, hnext = pin.array((Be, H, W, 3), np.uint8), pin.array((Be, H, W, 3), np.uint8)
    gprev, gnext = pin.array((Be, H, W), np.uint8), pin.array((Be, H, W), np.uint8)
    for i in range(Be):
        hprev[i], hnext[i] = hp[i % len(hp)], hn[i % len(hn)]
        gprev[i], gnext[i] = hp[i % len(hp)][:, :, 0], hn[i % len(hn)][:, :, 0]
    houts = [pin.array((Be, H >> k, W >> k, 2), np.float32) for k in range(LEVELS)]
    htotal = houts[0]  # (the lean call writes the total flow where the full call writes the level-0 residual)
    steps = max(3, min(args.steps, 10))

    def timed(fn):
        for _ in range(2):
            fn()
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        return env.max_over_ranks(time.perf_counter() - t0)

    # The reference's host images are 3-channel and its kernels read channel 0.  Headline: all three channels are uploaded
    # and the device drops two (6 B per pixel pair in, the library's default).  `host_extract`: channel 0 is taken by host
    # threads inside the call (ofb_ctx_set_host_threads) and 2 B per pixel pair cross PCIe -- no faster on the 16-vCPU
    # boxes of this pool, where the host side of the copies, not the link, is the limit.
    t_full = timed(lambda: ctx.flow_pairs_host(hprev, hnext, LEVELS, WIN, warp_mode=WARP_BILINEAR, out=houts))
    host_threads = max(1, min(8, (os.cpu_count() or 8) // max(1, env.world)))
    ctx.host_threads = host_threads
    try:
        t_hx = timed(lambda: ctx.flow_pairs_host(hprev, hnext, LEVELS, WIN, warp_mode=WARP_BILINEAR, out=houts))
    finally:
        ctx.host_threads = 0
    t_lean = timed(lambda: ctx.total_flow_pairs_host(gprev, gnext, LEVELS, WIN, warp_mode=WARP_BILINEAR, out=htotal))
    px = (W * H / 1e6) * Be * env.world * steps
    h2d, d2h = int(hprev.nbytes + hnext.nbytes), int(sum(a.nbytes for a in houts))
    h2d_l, d2h_l = int(gprev.nbytes + gnext.nbytes), int(htotal.nbytes)

    # the box's ceiling for this traffic pattern: every rank copies pinned host <-> device at once, nothing else running
    dsrc = torch.empty(d2h // 4, dtype=torch.float32, device=env.dev)
    hdst = torch.from_numpy(houts[0].reshape(-1))  # a view of pinned memory
    hsrc = torch.from_numpy(hprev.reshape(-1))
    ddst = torch.empty(hsrc.numel(), dtype=torch.uint8, device=env.dev)
    n_out = min(dsrc.numel(), hdst.numel())
    s_in, s_out = torch.cuda.Stream(env.dev), torch.cuda.Stream(env.dev)

    def copies(do_in, do_out, reps=4):
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(reps):
            if do_out:
                with torch.cuda.stream(s_out):
                    hdst[:n_out].copy_(dsrc[:n_out], non_blocking=True)
            if do_in:
                with torch.cuda.stream(s_in):
                    ddst.copy_(hsrc, non_blocking=True)
        torch.cuda.synchronize()
        dt = env.max_over_ranks(time.perf_counter() - t0)
        return (reps * n_out * 4 * env.world / dt / 1e9 if do_out else None,
                reps * hsrc.numel() * env.world / dt / 1e9 if do_in else None)

    copies(True, True, 1)
    d2h_alone, _ = copies(False, True)
    _, h2d_alone = copies(True, False)
    d2h_both, h2d_both = copies(True, True)
    pin.free()
    full = {"value": px / t_full, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "pairs_per_step": Be,
            "layout": "reference 3-channel u8 in (6 B/px), float2 residual flow of every level out (10.5 B/px)",
            "d2h_gbs_all_ranks": d2h * env.world * steps / t_full / 1e9,
            "pcie_gbs_both_directions_all_ranks": (d2h + h2d) * env.world * steps / t_full / 1e9,
            "bound": "host <-> device copies (both directions share the host side)",
            "host_extract": {"value": px / t_hx, "unit": UNIT, "host_threads": host_threads, "h2d_bytes_per_step": h2d // 3,
                             "d2h_bytes_per_step": d2h,
                             "layout": "the same 3-channel host images, channel 0 extracted by host threads inside the call "
                                       "(ofb_ctx_set_host_threads): 2 B/px uploaded"}}
    lean = {"value": px / t_lean, "unit": UNIT, "h2d_bytes_per_step": h2d_l, "d2h_bytes_per_step": d2h_l, "pairs_per_step": Be,
            "layout": "planar gray u8 in (2 B/px), total flow only out (8 B/px): ofb_flow_pairs_host_ex",
            "d2h_gbs_all_ranks": d2h_l * env.world * steps / t_lean / 1e9}
    ceiling = {"what": f"{env.world} rank(s) copying pinned host <-> device concurrently, GB/s summed over ranks",
               "d2h_alone": d2h_alone, "h2d_alone": h2d_alone, "d2h_with_h2d": d2h_both, "h2d_with_d2h": h2d_both}
    if d2h_both:
        full["frac_of_box_d2h_ceiling"] = full["d2h_gbs_all_ranks"] / d2h_both
        lean["frac_of_box_d2h_ceiling"] = lean["d2h_gbs_all_ranks"] / d2h_both
        # both directions at once: what the box moves when every rank copies in and out concurrently
        full["frac_of_box_both_directions_ceiling"] = full["pcie_gbs_both_directions_all_ranks"] / (d2h_both + h2d_both)
    full["lean"] = lean
    full["box_ceiling_gbs"] = ceiling
    return full


DROPIN_SIZES = ((640, 480, 4), (1024, 1024, 4))


def _loop_ms(pair_fn):
    pair_fn()
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        pair_fn()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts))


def _pyramids(prev, nxt, w, h, levels):
    pp = [prev.copy()] + [np.zeros((h >> k, w >> k, 3), np.uint8) for k in range(1, levels)]
    pn = [nxt.copy()] + [np.zeros((h >> k, w >> k, 3), np.uint8) for k in range(1, levels)]
    return pp, pn


def dropin_block(env, ctx):
    """The reference's own contract timed as main.cu:250-262 drives it: gpu::gauss_pyramid on both frames, then
    gpu::calc_opt_flow per level coarse to fine, host pointers, synchronous -- through the drop-in entry points
    (ofb_gauss_pyramid_host_u8c3 + ofb_calc_opt_flow_host_u8c3, defaults = the reference: window 19, warp as written).
    ms per pair, median of 5 after a warm-up pair."""
    from cuda_optical_flow_2_b200 import REFERENCE_WINDOW, WARP_AS_WRITTEN

    ours = {}
    for (w, h, levels) in DROPIN_SIZES:
        p3, n3 = synth_pairs_numpy(1, w, h, 11)

        def pair():
            pp, pn = _pyramids(p3[0], n3[0], w, h, levels)
            ctx.gauss_pyramid(pp, w, h, levels)
            ctx.gauss_pyramid(pn, w, h, levels)
            flows = [np.zeros((h >> k, w >> k, 2), np.float32) for k in range(levels)]
            for k in range(levels - 1, -1, -1):
                ctx.calc_opt_flow(pp[k], pn[k], w >> k, h >> k, flows, k, levels, win=REFERENCE_WINDOW, warp_mode=WARP_AS_WRITTEN)

        ms = _loop_ms(pair)
        ours[f"{w}x{h}x{levels}"] = {"ms_per_pair": ms, "mpx_pairs_per_s": w * h / 1e6 / (ms / 1e3)}
    ours["what"] = ("ofb_gauss_pyramid_host_u8c3 x2 + ofb_calc_opt_flow_host_u8c3 per level (main.cu:250-262), window 19, warp as "
                    "written, 3-channel host buffers, synchronous calls")
    return ours


def main_refgpu(args):
    """Child process of the B200 arm: the same loop through the UNMODIFIED reference GPU path (oracle/_ref/libofref.so:
    gpu::gauss_pyramid x2 + gpu::calc_opt_flow per level, OptFlowGpu.cu:1262, 1909) on this GPU.  Its own process, so that
    nothing the reference does to its CUDA context can touch the measured arm."""
    lib, O = ref_lib()
    if lib is None:
        print(json.dumps({"what": "oracle/_ref/libofref.so not present"}), flush=True)
        return 0
    rec = {}
    for (w, h, levels) in DROPIN_SIZES:
        p3, n3 = synth_pairs_numpy(1, w, h, 11)

        def pair():
            pp, pn = _pyramids(p3[0], n3[0], w, h, levels)
            lib.ref_gpu_gauss_pyramid(O._ptr_array(pp, O._u8p), w, h, levels)
            lib.ref_gpu_gauss_pyramid(O._ptr_array(pn, O._u8p), w, h, levels)
            flows = [np.zeros((h >> k, w >> k, 2), np.float32) for k in range(levels)]
            fp = O._ptr_array(flows, O._f32p)
            for k in range(levels - 1, -1, -1):
                lib.ref_gpu_calc_opt_flow(pp[k].ctypes.data_as(O._u8p), pn[k].ctypes.data_as(O._u8p), w >> k, h >> k, fp, k, levels)

        ms = _loop_ms(pair)
        rec[f"{w}x{h}x{levels}"] = {"ms_per_pair": ms, "mpx_pairs_per_s": w * h / 1e6 / (ms / 1e3)}
    rec["what"] = ("the unmodified reference (gpu::gauss_pyramid x2 + gpu::calc_opt_flow per level, OptFlowGpu.cu:1262,1909, window "
                   "19, its CPU warp) on this B200, driven like main.cu:250-262; timing only -- its coarse levels are not "
                   "launch-valid sizes (SURVEY Q6)")
    print(json.dumps(rec), flush=True)
    return 0


def refgpu_block():
    import subprocess

    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--refgpu-only"], capture_output=True, text=True, timeout=300,
                           cwd=ROOT)
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        if r.returncode != 0 or not lines:
            return {"error": f"rc {r.returncode}: {r.stderr[-300:]}"}
        return json.loads(lines[-1])
    except Exception as ex:
        return {"error": repr(ex)}


def config_block(env, ctx, w, h, levels, win, pairs, steps, peak):
    torch = env.torch
    prev, nxt, _ = synth_pairs_torch(min(pairs, 8), w, h, env.dev, 31)
    if pairs > prev.shape[0]:  # tile the few synthesised pairs up to the batch (the kernels do not care)
        rep = (pairs + prev.shape[0] - 1) // prev.shape[0]
        prev, nxt = prev.repeat(rep, 1, 1)[:pairs].contiguous(), nxt.repeat(rep, 1, 1)[:pairs].contiguous()
    ms, _, lvl, _, _, flows = timed_device_steps(env, ctx, prev, nxt, w, h, levels, win, steps, 3)
    rec = {"workload": f"{w}x{h}, {levels} level(s), window {win}, {pairs} pairs per step", "ms_per_step": ms,
           "value": (w * h / 1e6) * pairs * env.world / (ms / 1e3), "unit": "Mpx-pairs/s",
           "level0_roofline_frac": roofline_of(lvl[0], w, h, 0, levels, pairs, False, peak)["frac"]}
    del flows, prev, nxt
    torch.cuda.empty_cache()
    return rec


def strips_block(env, ctx, w, h, levels, win, reps):
    """BASELINE configs[4]: one large pair cut into row strips over the N ranks; halo rows pushed into the neighbours'
    memory over NVLink (CUDA IPC peer mappings), one exchange per pyramid level; every rank's result compared bit for
    bit with the whole-frame result computed on its own GPU."""
    from cuda_optical_flow_2_b200 import WARP_BILINEAR
    from cuda_optical_flow_2_b200.dist import NativeStrips, StripPlan

    torch = env.torch
    world, rank, dev = env.world, env.rank, env.dev
    prev, nxt, pitch = synth_pairs_torch(1, w, h, dev, 4242)  # the same frames on every rank
    whole = ctx.flow_pairs_device(prev, nxt, w, levels, win, warp_mode=WARP_BILINEAR)
    torch.cuda.synchronize()
    plan = StripPlan(w, h, levels, win, world, 16)
    plan.validate()
    K = 4  # handles = pairs that can be in flight at once
    handles = [NativeStrips(ctx, w, h, levels, win, world, rank, dev, WARP_BILINEAR, 1.0, 16, transport="peer") for _ in range(K)]
    ins = []
    fused = os.environ.get("OFB_STRIPS_FUSED", "1") != "0"  # (experiments: the separate copy / wait kernels instead)
    for nat in handles:
        nat.set_fused(fused)
        nat.set_total(False)
        y0, y1 = nat.own_rows(0)
        pin, nin = nat.input_rows()  # the producer writes the own rows where the runner keeps them
        pin[:, :w].copy_(prev[0, y0:y1, :w])
        nin[:, :w].copy_(nxt[0, y0:y1, :w])
        ins.append((pin, nin))
    streams = [torch.cuda.Stream(dev) for _ in range(K)]

    def identical(nat):
        ok = True
        for k in range(levels):
            y0, y1 = nat.own_rows(k)
            ref, got = whole[k][0, y0:y1], nat.own_flow(k)
            m = ~torch.isnan(ref)
            ok &= bool(torch.equal(torch.isnan(ref), torch.isnan(got)) and torch.equal(ref[m], got[m]))
        f = torch.tensor([1 if ok else 0], device=dev)
        if world > 1:
            env.dist.all_reduce(f, op=env.dist.ReduceOp.MIN)
        return bool(f.item())

    def measure(n_handles, graph):
        hs, ss = handles[:n_handles], streams[:n_handles]
        runs = []
        for nat, st, (pin, nin) in zip(hs, ss, ins):
            with torch.cuda.stream(st):
                for _ in range(2):
                    nat.run(pin, nin, st.cuda_stream)
            nat.check(st.cuda_stream)
            if graph:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=st, capture_error_mode="thread_local"):
                    nat.run(pin, nin, torch.cuda.current_stream(dev).cuda_stream)
                runs.append((st, g.replay))
            else:
                runs.append((st, (lambda nat=nat, pin=pin, nin=nin, st=st: nat.run(pin, nin, st.cuda_stream))))
        env.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for st in ss:
            st.wait_stream(torch.cuda.current_stream(dev))
        e0.record()
        for st in ss:
            st.wait_event(e0)
        for i in range(reps):
            st, fn = runs[i % n_handles]
            with torch.cuda.stream(st):
                fn()
        for st in ss:
            torch.cuda.current_stream(dev).wait_stream(st)
        e1.record()
        env.barrier()
        ms = env.max_over_ranks(e0.elapsed_time(e1) / reps)
        for nat, st in zip(hs, ss):
            nat.check(st.cuda_stream)
        return ms, all(identical(nat) for nat in hs)

    halo = sum((hi - lo) * 2 * ((w + 63) // 64 * 64) for _, lo, hi, _ in plan.halo_messages(0, rank)) + \
        sum((hi - lo) * (w >> (k + 1)) * 8 for k in range(levels) for _, lo, hi, _ in plan.cum_messages(k, rank))
    rec = {"workload": f"{w}x{h} pair, {levels} levels, window {win}, row strips over {world} rank(s)", "n_ranks": world,
           "transport": "peer" if world > 1 else None, "reps": reps,
           "halo_exchange": ("fused into the level kernels (peer stores + arrival flags from the producing kernel, flag waits in the "
                             "consuming kernel)" if fused else "separate copy / wait kernels") if world > 1 else None,
           "algorithmic_bytes_per_pair": sum(level_bytes(w, h, k, levels, 1, 0 < k < levels - 1) for k in range(levels)) +
           2 * sum((w >> (k - 1)) * (h >> (k - 1)) + (w >> k) * (h >> k) for k in range(1, levels))}
    try:
        ms, ok = measure(1, True)
        rec.update({"ms_per_pair": ms, "cuda_graph": True, "bit_identical_to_whole_frame": ok})
    except Exception as ex:
        print(f"strips: graph capture failed ({ex!r}); eager", file=sys.stderr)
        ms, ok = measure(1, False)
        rec.update({"ms_per_pair": ms, "cuda_graph": False, "bit_identical_to_whole_frame": ok})
    rec["ms_per_pair_note"] = "one pair at a time on one stream: the latency of the whole dependency chain of a pair"
    best = rec["ms_per_pair"]
    for nf in (2, 4):
        try:
            ms2, ok2 = measure(nf, rec["cuda_graph"])
            rec[f"in_flight_{nf}"] = {"ms_per_pair": ms2, "bit_identical_to_whole_frame": ok2}
            if ok2:
                best = min(best, ms2)
        except Exception as ex:
            rec[f"in_flight_{nf}"] = {"error": repr(ex)}
    rec["in_flight_note"] = ("K handles on K streams, pairs alternate (throughput of a frame sequence): the late, small levels of a "
                             "pair and its halo exchanges overlap the next pairs' early levels")
    rec["ms_per_pair_pipelined"] = best
    rec["mpx_pairs_per_s"] = w * h / 1e6 / (best / 1e3)
    rec["halo_bytes_sent_rank0_per_pair"] = int(halo)
    peak, _ = measured_peak()
    rec["frac_of_n_gpu_hbm_roofline"] = rec["algorithmic_bytes_per_pair"] / (best * 1e-3) / 1e9 / (peak * world)
    env.barrier()
    for nat in handles:
        nat.close()
    return rec


# ---------------------------------------------------------------------------------------------- B200 arm
def main_b200(args):
    import torch

    from cuda_optical_flow_2_b200 import SOLVE_EXACT, SOLVE_FAST, Context

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the B200 arm has no CPU fallback"}), flush=True)
        return 1
    env = Env()
    world, rank, dev = env.world, env.rank, env.dev
    ctx = Context(env.local)
    peak, peak_src = measured_peak()

    if args.strips_only:
        sw, sh, sl = (int(x) for x in args.strips_size.split("x"))
        ctx.solve = SOLVE_FAST if args.solve == "fast" else SOLVE_EXACT
        rec = strips_block(env, ctx, sw, sh, sl, WIN, args.strips_reps)
        if rank == 0:
            print(json.dumps({"strips": rec}), flush=True)
        if world > 1:
            env.dist.destroy_process_group()
        ctx.close()
        return 0

    B = args.pairs
    warm = max(args.warmup, 3)
    # 64 distinct synthetic pairs, tiled up to the batch: every pair has its own memory (the step streams B x 4.1 MB of
    # frames, far beyond L2), the arithmetic does not depend on the content
    prev, nxt, pitch = synth_pairs_torch(min(B, 64), W, H, dev, 1000 + rank)
    if B > prev.shape[0]:
        rep = (B + prev.shape[0] - 1) // prev.shape[0]
        prev, nxt = prev.repeat(rep, 1, 1)[:B].contiguous(), nxt.repeat(rep, 1, 1)[:B].contiguous()

    # ---- headline: device-resident batch, the solve the line names
    ctx.solve = SOLVE_FAST if args.solve == "fast" else SOLVE_EXACT
    sampler = ClockSampler(env.local) if rank == 0 else None
    ms_step, launches, lvl_ms, pyr_ms, clocks, flows = timed_device_steps(env, ctx, prev, nxt, W, H, LEVELS, WIN, args.steps, warm,
                                                                         sampler=sampler)
    launches = int(env.sum_over_ranks(launches))
    value = (W * H / 1e6) * B * world / (ms_step / 1e3)
    dumped = None
    if args.dump_outputs and rank == 0:  # before the next measurement reuses `flows`
        dumped = {"dir": args.dump_outputs, "pairs": dump_outputs(args.dump_outputs, flows)}

    # ---- the other solve, same way, fewer steps (rank-local clock is enough for a side record)
    other = SOLVE_EXACT if args.solve == "fast" else SOLVE_FAST
    ctx.solve = other
    o_steps = max(3, min(args.steps, 10))
    o_ms, _, o_lvl, _, _, _ = timed_device_steps(env, ctx, prev, nxt, W, H, LEVELS, WIN, o_steps, 3, flows=flows)
    ctx.solve = SOLVE_FAST if args.solve == "fast" else SOLVE_EXACT

    one_ms = one_graph_ms = None
    if rank == 0:
        one_ms, one_graph_ms = single_pair_latency(env, ctx, prev, nxt, flows)

    e2e = e2e_block(env, ctx, args)
    del flows
    torch.cuda.empty_cache()

    parity = dropin = refgpu = cfgs = None
    if rank == 0:
        parity = parity_block(env, ctx)
    if world == 1 and not args.quick:
        dropin = dropin_block(env, ctx)
        cfgs = {"configs[0]": config_block(env, ctx, 640, 480, 1, 5, 1024, 5, peak),
                "configs[2]": config_block(env, ctx, 3840, 2160, 4, 15, 64, 5, peak)}
    del prev, nxt
    torch.cuda.empty_cache()
    strips = None
    if not args.quick:
        try:
            strips = strips_block(env, ctx, 7680, 4320, 4, WIN, args.strips_reps)
        except Exception as ex:  # a side record never costs the headline
            strips = {"error": repr(ex)}

    if world == 1 and not args.quick:
        refgpu = refgpu_block()  # (a child process; after every measurement of this arm)
    composing = os.environ.get("OFB_NO_COMPOSE", "0") != "1"
    if rank == 0:
        n0 = W * H
        r0 = roofline_of(lvl_ms[0], W, H, 0, LEVELS, B, False, peak)
        traffic = ncu_traffic()
        total_ms = ms_step * args.steps
        # Level 1 does not write its cumulative flow: level 0 composes it from the residual flows of levels 1 and 2 (even
        # sizes, per-pixel warp: csrc/ofb_api.cu run_pairs_device; OFB_NO_COMPOSE=1 restores the old form).  The level-0
        # kernel then also reads the level-2 flow: 8 B per level-2 pixel = 0.5 B per level-0 pixel on top of SURVEY 8(d)'s 12.
        n2 = (W >> 2) * (H >> 2)
        own_bytes = r0["algorithmic_bytes_per_launch"] + (B * n2 * 8 if composing else 0)
        own_ach = own_bytes / (r0["avg_launch_ms"] * 1e-3) / 1e9 if r0["avg_launch_ms"] > 0 else 0.0
        pair_survey, pair_moved = 43027200, 43027200 - (8 * (W >> 1) * (H >> 1) - 8 * n2 if composing else 0)
        roofline = {"bound": "hbm", "kernel": f"lk_level_kernel<9, bilinear, {args.solve} solve{', composing' if composing else ''}> level 0",
                    "achieved": own_ach, "peak": peak, "unit": "GB/s", "frac": own_ach / peak, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": own_bytes, "avg_launch_ms": r0["avg_launch_ms"],
                    "bytes_note": ("every array once: 1 B prev + 1 B next + 8 B flow out per pixel, 8 B per level-1 pixel of coarser flow in"
                                   + (", 8 B per level-2 pixel of the flow it composes with (12.5 B/px; level 1 in turn writes no cumulative "
                                      "flow, 8 B per level-1 pixel less)" if composing else " (12 B/px)")),
                    "frac_at_survey_12_bytes_per_px": r0["frac"],
                    "traffic": (traffic or {}).get("dram_bytes_per_launch"),
                    "traffic_note": (traffic or {}).get("note"),
                    "other_levels": {"level_1": dict(roofline_of(lvl_ms[1], W, H, 1, LEVELS, B, not composing, peak),
                                                     writes_cumulative_flow=not composing),
                                     "level_2_coarsest": roofline_of(lvl_ms[2], W, H, 2, LEVELS, B, False, peak)},
                    "whole_step_frac": B * pair_survey / (ms_step * 1e-3) / 1e9 / peak,
                    "whole_step_frac_bytes_moved": B * pair_moved / (ms_step * 1e-3) / 1e9 / peak,
                    "whole_step_note": f"{pair_survey} B per pair by SURVEY 8(d) (the definition of the work); {pair_moved} B with the "
                                       "composition (no level-1 cumulative flow written, the level-2 flow read once more)",
                    "step_share": {"pyramid": pyr_ms[0] / total_ms if total_ms else None,
                                   **{f"lk_level_{k}": lvl_ms[k][0] / total_ms for k in range(LEVELS)}}}
        other_name = "exact" if args.solve == "fast" else "fast"
        other_rec = {"solve": other_name, "value": (n0 / 1e6) * B / (o_ms / 1e3) * world, "ms_per_step": o_ms, "steps": o_steps,
                     "level0_roofline_frac": roofline_of(o_lvl[0], W, H, 0, LEVELS, B, False, peak)["frac"],
                     "level0_avg_launch_ms": o_lvl[0][0] / max(o_lvl[0][1], 1)}
        cores = os.cpu_count() or 1
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            try:
                times, kind = run_reference_cpu(cores, cores, reps=1)
                cpu = {"value": (W * H / 1e6) * cores / times[0], "unit": UNIT, "cores": cores, "kind": kind,
                       "sample": f"{cores} pairs of the same 1080p/3-level/win-9 workload, one per host thread, "
                                 f"{times[0]:.1f} s wall"}
            except Exception as ex:  # the baseline is a report, never a reason to lose the GPU number
                cpu = {"value": None, "unit": UNIT, "cores": cores, "kind": "unavailable", "sample": repr(ex)}
        dtype = ("u8 -> exact int32 window sums -> exact int64 determinant/numerators -> f32 quotient" if args.solve == "fast"
                 else "u8 -> int32 sums -> f64 solve -> f32 flow")
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": dict(CONFIG),
                "run": {"pairs_per_gpu_per_step": B, "warp": "bilinear", "solve": args.solve,
                        "solve_note": "fast = OFB_SOLVE_FAST, tolerance-mode (see parity); exact = bit-identical to the reference's "
                                      "double-precision solve, timed in the record named `exact`/`fast` beside the headline",
                        "single_pair_latency_ms": one_ms, "single_pair_latency_ms_cuda_graph": one_graph_ms,
                        "l2": f"inputs exceed L2 ({B * 2 * pitch * H / 1e6:.0f} MB of frames per step, fresh outputs each level)",
                        "parallelism": f"frame-batch x{world}", "dumped_outputs": dumped},
                "roofline": roofline, other_name: other_rec, "parity": parity, "cpu_baseline": cpu, "e2e": e2e,
                "e2e_dropin": dropin, "reference_gpu": refgpu, "configs": cfgs, "strips": strips,
                "gpu_launches": launches, "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        env.dist.destroy_process_group()
    ctx.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=1024, help="frame pairs per GPU per step (device-resident); BASELINE configs[3] is a "
                    "batch of 4096 pairs over the GPUs")
    ap.add_argument("--e2e-pairs", type=int, default=32, help="frame pairs per GPU per end-to-end step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--solve", default="fast", choices=["fast", "exact"], help="the solve the headline is measured with")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline, parity and e2e only (no configs / drop-in / strips records)")
    ap.add_argument("--strips-only", action="store_true", help="only the row-strip record (tests, experiments)")
    ap.add_argument("--strips-size", default="7680x4320x4", help="WxHxLEVELS of the row-strip record")
    ap.add_argument("--strips-reps", type=int, default=100)
    ap.add_argument("--refgpu-only", action="store_true", help="(child of the B200 arm) time the reference's own GPU path")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the flows of the headline's last timed step (a seeded sample of "
                    "whole pairs, at most 64 MB) to DIR/flow_level<k>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.strips_only):
        ap.error("--dump-outputs applies to the B200 arm's headline (not --impl reference or --strips-only)")
    if args.refgpu_only:
        return main_refgpu(args)
    if args.impl == "reference":
        return main_reference(args)
    return main_b200(args)


if __name__ == "__main__":
    sys.exit(main())
