"""Row-strip run of one large pair over N GPUs (torchrun), BASELINE.json configs[4]:
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        scripts/run_strips.py [--w 7680 --h 4320 --levels 4 --win 9 --reps 10 --check]
Every rank generates the same synthetic frames, keeps only its own rows and solves its strip with the native runner
(csrc/strips.cu): the sender's kernels store the halo rows into the receiver's memory over NVLink (CUDA IPC) and raise
epoch flags there, one exchange per pyramid level.  --check compares every rank's own rows of every level with the
whole-frame result computed on its own GPU (bit for bit).  Prints one JSON line on rank 0."""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.distributed as dist
from bench import synth_pairs_torch
from cuda_optical_flow_2_b200 import Context, WARP_BILINEAR
from cuda_optical_flow_2_b200.dist import NativeStrips, StripPlan

ap = argparse.ArgumentParser()
ap.add_argument("--w", type=int, default=7680); ap.add_argument("--h", type=int, default=4320)
ap.add_argument("--levels", type=int, default=4); ap.add_argument("--win", type=int, default=9)
ap.add_argument("--reps", type=int, default=10); ap.add_argument("--reach", type=int, default=16)
ap.add_argument("--check", action="store_true")
ap.add_argument("--total", action="store_true", help="level 0 also writes the total flow of the pair (8 more bytes per pixel)")
ap.add_argument("--copy-in", action="store_true", help="the own rows are copied into the runner every pair instead of living there (ofb_strips_input)")
ap.add_argument("--graph", action="store_true", help="capture one pair in a CUDA graph and replay it")
a = ap.parse_args()
world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local); dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
ctx = Context(local)
prev, nxt, pitch = synth_pairs_torch(1, a.w, a.h, dev, 4242)  # same seed on every rank
plan = StripPlan(a.w, a.h, a.levels, a.win, world, a.reach); plan.validate()
nat = NativeStrips(ctx, a.w, a.h, a.levels, a.win, world, rank, dev, WARP_BILINEAR, 1.0, a.reach, transport="peer")
nat.set_total(a.total)
y0, y1 = nat.own_rows(0)
nin = (prev[0, y0:y1], nxt[0, y0:y1])
if not a.copy_in:  # the producer writes the own rows where the runner keeps them
    nin = nat.input_rows()
    nin[0][:, :a.w].copy_(prev[0, y0:y1, :a.w]); nin[1][:, :a.w].copy_(nxt[0, y0:y1, :a.w])
def one():
    nat.run(nin[0], nin[1], torch.cuda.current_stream(dev).cuda_stream)
side = torch.cuda.Stream(dev)
side.wait_stream(torch.cuda.current_stream(dev))
with torch.cuda.stream(side):
    for _ in range(3): one()
    nat.check(torch.cuda.current_stream(dev).cuda_stream)
    if a.graph:
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):  # the NCCL watchdog thread queries events
            one()
        one = g.replay
        for _ in range(2): one()
torch.cuda.current_stream(dev).wait_stream(side)
torch.cuda.synchronize()
def barrier():
    if world > 1: dist.barrier()
    torch.cuda.synchronize()
barrier(); e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(a.reps): one()
e1.record(); barrier()
t = torch.tensor([e0.elapsed_time(e1) / a.reps], dtype=torch.float64, device=dev)
if world > 1: dist.all_reduce(t, op=dist.ReduceOp.MAX)
ok = None
if a.check:
    whole = ctx.flow_pairs_device(prev, nxt, a.w, a.levels, a.win, warp_mode=WARP_BILINEAR)
    torch.cuda.synchronize()
    ok = True
    for k in range(a.levels):
        y0, y1 = nat.own_rows(k)
        ref, got = whole[k][0, y0:y1], nat.own_flow(k)
        m = ~torch.isnan(ref)
        ok &= bool(torch.equal(torch.isnan(ref), torch.isnan(got)) and torch.equal(ref[m], got[m]))
    f = torch.tensor([1 if ok else 0], device=dev)
    if world > 1: dist.all_reduce(f, op=dist.ReduceOp.MIN)
    ok = bool(f.item())
if rank == 0:
    # what rank 0 pushes per pair: its level-0 image rows (both frames) and its cumulative-flow rows of the coarser levels
    halo = sum((hi - lo) * 2 * ((a.w + 63) // 64 * 64) for _, lo, hi, _ in plan.halo_messages(0, 0)) + \
           sum((hi - lo) * (a.w >> (k + 1)) * 8 for k in range(a.levels) for _, lo, hi, _ in plan.cum_messages(k, 0))
    print(json.dumps({"mode": "row-strips", "w": a.w, "h": a.h, "levels": a.levels, "win": a.win, "n_gpus": world,
                      "ms_per_pair": t.item(), "mpx_pairs_per_s": a.w * a.h / 1e6 / (t.item() / 1e3),
                      "bit_identical_to_whole_frame": ok, "cuda_graph": bool(a.graph), "transport": "peer" if world > 1 else None,
                      "halo_bytes_sent_rank0_per_pair": halo}), flush=True)
nat.close()
if world > 1: dist.destroy_process_group()
