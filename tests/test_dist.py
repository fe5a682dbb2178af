"""Multi-GPU host logic.  CPU: batch sharding, the strip schedule's invariants, and the native runner's schedule against
StripPlan.  GPU: the native strip runner, N ranks on one device (or one per GPU), must reproduce the whole-frame flow bit
for bit, and must report a warp that reaches past the rows it holds."""
import os

import numpy as np
import pytest

from support import BIL, NEAR, reach_flag, requested_rows


def test_shard_range_partitions_the_batch():
    from cuda_optical_flow_2_b200.dist import shard_range

    for n, world in ((4096, 8), (10, 4), (3, 8), (0, 2)):
        blocks = [shard_range(n, world, r) for r in range(world)]
        assert blocks[0][0] == 0 and blocks[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(blocks, blocks[1:]))
        sizes = [hi - lo for lo, hi in blocks]
        assert max(sizes) - min(sizes) <= 1


@pytest.mark.parametrize("W,H,levels,win,world", [(7680, 4320, 4, 9, 8), (7680, 4320, 4, 9, 2), (3840, 2160, 4, 15, 4),
                                                  (640, 486, 3, 5, 3), (1920, 1080, 3, 9, 8)])
def test_strip_plan_invariants(W, H, levels, win, world):
    from cuda_optical_flow_2_b200.dist import StripPlan

    plan = StripPlan(W, H, levels, win, world, reach=8)
    plan.validate()
    r = win // 2
    for k in range(levels):
        for rk in range(world):
            s = plan.level(k, rk)
            # strips nest: a rank's rows at level k sit on its rows at level k+1
            if k + 1 < levels:
                up = plan.level(k + 1, rk)
                assert s.y0 == 2 * up.y0 and (s.y1 == 2 * up.y1 or rk == world - 1)
                # pyramid: level k+1 own rows need level k rows 2y-1 .. 2y+1, all inside the level-k buffer
                assert s.by0 <= max(0, 2 * up.y0 - 1) and 2 * (up.y1 - 1) + 1 < s.by1
                # the kernel looks up cum[(y >> 1)] for the rows of its tile
                lo, hi = max(0, s.y0 - r - 2), min(s.h - 1, s.y1 + r + 1)
                assert s.cy0 <= lo >> 1 and min(hi >> 1, (H >> (k + 1)) - 1) < s.cy1
            # stencil + window halo present (or the image border)
            assert s.by0 <= max(0, s.y0 - r - 2) and s.by1 >= min(s.h, s.y1 + r + 2)
            # every halo row is owned by exactly one sender
            got = np.zeros(s.h, int)
            got[s.y0:s.y1] += 1
            for peer in range(world):
                for dst, lo, hi, _ in plan.halo_messages(k, peer):
                    if dst == rk:
                        got[lo:hi] += 1
            assert (got[s.by0:s.by1] == 1).all() and got.sum() == s.buf_rows


# ------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("W,H,levels,win", [(640, 480, 3, 9), (322, 406, 2, 5), (1920, 1080, 4, 15)])
def test_native_strip_runner_world_one_equals_whole_frame(ctx, oracle, W, H, levels, win):
    """csrc/strips.cu on a single rank (no exchange): own-row upload, locally built pyramid, strip variants of the
    kernels -- bit for bit the whole-frame result.  (The multi-rank exchange is exercised by the peer-memory tests
    below; its schedule is the one test_strip_plan_invariants checks.)"""
    import torch

    from cuda_optical_flow_2_b200 import WARP_BILINEAR, planar_to_device
    from cuda_optical_flow_2_b200.dist import NativeStrips

    prev = oracle.make_frame(W, H, 0, 0, 8, 321)
    nxt = oracle.make_frame(W, H, 2.25, -1.5, 8, 321)
    dp, dn = planar_to_device(prev[None]), planar_to_device(nxt[None])
    whole = ctx.flow_pairs_device(dp, dn, W, levels, win, warp_mode=WARP_BILINEAR)
    ns = NativeStrips(ctx, W, H, levels, win, 1, 0, torch.device("cuda", 0), WARP_BILINEAR, 1.0, 16)
    try:
        assert ns.own_rows(0) == (0, H)
        st = torch.cuda.current_stream().cuda_stream
        ns.run(dp[0], dn[0], st)
        ns.check(st)
        for k in range(levels):
            ref, got = whole[k][0], ns.own_flow(k)
            m = ~torch.isnan(ref)
            assert torch.equal(torch.isnan(ref), torch.isnan(got)) and torch.equal(ref[m], got[m]), f"level {k}"
    finally:
        ns.close()


@pytest.mark.gpu
@pytest.mark.parametrize("W,H,levels,win,world,mode", [(640, 480, 3, 9, 2, BIL), (640, 480, 3, 9, 3, NEAR), (640, 480, 3, 9, 4, BIL),
                                                       (322, 406, 2, 5, 3, BIL), (322, 406, 2, 5, 3, NEAR),
                                                       (1920, 1080, 3, 9, 8, BIL), (1920, 1080, 4, 15, 4, BIL),
                                                       (1920, 1080, 4, 15, 4, NEAR), (512, 384, 1, 9, 4, BIL),
                                                       (7680, 4320, 4, 9, 8, BIL)])
def test_native_strips_peer_memory_transport_equals_whole_frame(ctx, oracle, W, H, levels, win, world, mode):
    """csrc/strips.cu with the peer-memory transport: `world` ranks live in this process on one GPU; the sender's copy
    kernel stores halo rows straight into the receiver's arena and raises an epoch flag, the receiver's wait kernel
    checks it.  All ranks share ONE stream and their pairs are enqueued phase by phase (run_local_sequenced), so every
    flag is raised by a kernel ahead of its waiter: kernels of different ranks never have to be co-scheduled on the one
    GPU.  Three pairs back to back (flags, epochs and the done handshake are re-used), each bit for bit the whole-frame
    result at every level and in the total flow (at one level the residual flow), in both per-pixel warp modes.  Across
    processes the same kernels run on CUDA IPC mappings, each rank enqueuing its whole pair at once
    (test_native_strips_two_processes_over_cuda_ipc, bench.py under torchrun)."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device
    from cuda_optical_flow_2_b200.dist import NativeStrips

    dev = torch.device("cuda", 0)
    ranks = [NativeStrips(ctx, W, H, levels, win, world, rk, dev, mode, 1.0, 16, transport="local") for rk in range(world)]
    streams = [torch.cuda.Stream(dev) for _ in range(world)]
    try:
        NativeStrips.connect_local(ranks)
        for trial, (dx, dy) in enumerate([(2.25, -1.5), (-3.0, 0.75), (0.5, 2.0)]):
            prev = oracle.make_frame(W, H, 0, 0, 8, 900 + trial)
            nxt = oracle.make_frame(W, H, dx, dy, 8, 900 + trial)
            dp, dn = planar_to_device(prev[None]), planar_to_device(nxt[None])
            total = torch.empty((1, H, W, 2), dtype=torch.float32, device=dev)
            whole = ctx.flow_pairs_device(dp, dn, W, levels, win, warp_mode=mode, total_flow=total)
            torch.cuda.synchronize()
            inputs = []
            for ns in ranks:
                y0, y1 = ns.own_rows(0)
                if trial == 1:  # the producer writes the own rows in place: no upload copy
                    pin, nin = ns.input_rows()
                    pin[:, :W].copy_(dp[0, y0:y1, :W])
                    nin[:, :W].copy_(dn[0, y0:y1, :W])
                    inputs.append((pin, nin))
                else:
                    inputs.append((dp[0, y0:y1], dn[0, y0:y1]))
            torch.cuda.synchronize()
            NativeStrips.run_local_sequenced(ranks, inputs, streams[0].cuda_stream)
            for ns in ranks:
                ns.check(streams[0].cuda_stream)
            for ns in ranks:
                for k in range(levels):
                    y0, y1 = ns.own_rows(k)
                    ref, got = whole[k][0, y0:y1], ns.own_flow(k)
                    m = ~torch.isnan(ref)
                    assert torch.equal(torch.isnan(ref), torch.isnan(got)) and torch.equal(ref[m], got[m]), \
                        f"pair {trial} rank {ns.rank} level {k}"
                y0, y1 = ns.own_rows(0)
                ref, got = total[0, y0:y1], ns.own_flow(0, total=True)
                m = ~torch.isnan(ref)
                assert torch.equal(torch.isnan(ref), torch.isnan(got)) and torch.equal(ref[m], got[m]), \
                    f"pair {trial} rank {ns.rank} total flow"
    finally:
        torch.cuda.synchronize()
        for ns in ranks:
            ns.close()


@pytest.mark.gpu
def test_native_strip_reach_overflow_is_reported(ctx, oracle):
    """A warp that reaches past the rows a rank holds must raise, not silently change the numbers.  With reach=1 a middle
    rank of this 320x480 pair (3 levels, window 9, 4 ranks) holds its own rows plus 39 above and 36 below at level 0, 19
    and 18 at level 1: the halo and the rows the coarser levels' halo rows are rebuilt from.  On these frames the flow of
    the coarsest level, which the strips compute exactly, makes rank 1's level-1 warp ask for rows past those (the rule of
    support.requested_rows), so its flag is certain.  With the default reach=16 no rank asks for a row it does not
    hold, and the strips equal the whole frame bit for bit."""
    import ctypes as C

    import torch

    from cuda_optical_flow_2_b200 import _lib, planar_to_device
    from cuda_optical_flow_2_b200.dist import NativeStrips

    W, H, levels, win, world = 320, 480, 3, 9, 4
    prev = oracle.make_frame(W, H, 0, 0, 16, 5)
    nxt = oracle.make_frame(W, H, 0.0, 20.0, 16, 5)  # large vertical motion
    _, cums = oracle.flow_pair(prev, nxt, levels, win, BIL, oracle.SUMS_EXACT, want_cum=True)
    lib, out = _lib.load(), (C.c_int * 8)()

    def flagged(reach):
        """(rank, level) whose warp, on the whole frame's coarser flow, asks for a row outside the rows the rank holds."""
        got = []
        for rk in range(world):
            for k in range(levels - 1):
                _lib.check(lib.ofb_strips_plan_query(W, H, levels, win, world, rk, reach, k, out))
                y0, y1, _, _, cy0, cy1, eb0, eb1 = list(out)
                if reach_flag(requested_rows(cums[k + 1], W >> k, H >> k, BIL, y0, y1, win), eb0, eb1 - eb0, cy0, cy1 - cy0):
                    got.append((rk, k))
        return got

    assert (1, 1) in flagged(1) and flagged(16) == []
    dev = torch.device("cuda", 0)
    dp, dn = planar_to_device(prev[None]), planar_to_device(nxt[None])
    whole = ctx.flow_pairs_device(dp, dn, W, levels, win, warp_mode=BIL)
    torch.cuda.synchronize()
    for reach in (1, 16):
        ranks = [NativeStrips(ctx, W, H, levels, win, world, rk, dev, BIL, 1.0, reach, transport="local") for rk in range(world)]
        try:
            NativeStrips.connect_local(ranks)
            st = torch.cuda.current_stream().cuda_stream
            inputs = [(dp[0, y0:y1], dn[0, y0:y1]) for y0, y1 in (ns.own_rows(0) for ns in ranks)]
            NativeStrips.run_local_sequenced(ranks, inputs, st)
            if reach == 1:
                with pytest.raises(RuntimeError, match="raise `reach`"):
                    ranks[1].check(st)
                continue
            for ns in ranks:
                ns.check(st)
                for k in range(levels):
                    y0, y1 = ns.own_rows(k)
                    ref, got = whole[k][0, y0:y1], ns.own_flow(k)
                    m = ~torch.isnan(ref)
                    assert torch.equal(torch.isnan(ref), torch.isnan(got)) and torch.equal(ref[m], got[m]), f"rank {ns.rank} level {k}"
        finally:
            torch.cuda.synchronize()
            for ns in ranks:
                ns.close()


@pytest.mark.gpu
def test_native_strips_peer_memory_pair_replays_as_cuda_graph(ctx, oracle):
    """The peer-memory transport has no host-side state per pair (the epoch lives in device memory), so a pair is
    capturable as a CUDA graph; the replays stay bit for bit the whole-frame result.  (Both ranks of this one-GPU test
    are captured into one graph, phase by phase; across GPUs each rank captures its own run().)"""
    import torch

    from cuda_optical_flow_2_b200 import WARP_BILINEAR, planar_to_device
    from cuda_optical_flow_2_b200.dist import NativeStrips

    W, H, levels, win, world = 1280, 720, 3, 9, 2
    dev = torch.device("cuda", 0)
    ranks = [NativeStrips(ctx, W, H, levels, win, world, rk, dev, WARP_BILINEAR, 1.0, 16, transport="local") for rk in range(world)]
    streams = [torch.cuda.Stream(dev) for _ in range(world)]
    try:
        NativeStrips.connect_local(ranks)
        ins = [ns.input_rows() for ns in ranks]

        def load(seed, dx, dy):
            prev = oracle.make_frame(W, H, 0, 0, 8, seed)
            nxt = oracle.make_frame(W, H, dx, dy, 8, seed)
            dp, dn = planar_to_device(prev[None]), planar_to_device(nxt[None])
            for ns, (pin, nin) in zip(ranks, ins):
                y0, y1 = ns.own_rows(0)
                pin[:, :W].copy_(dp[0, y0:y1, :W])
                nin[:, :W].copy_(dn[0, y0:y1, :W])
            whole = ctx.flow_pairs_device(dp, dn, W, levels, win, warp_mode=WARP_BILINEAR)
            torch.cuda.synchronize()
            return whole

        load(11, 1.0, 1.0)
        NativeStrips.run_local_sequenced(ranks, ins, streams[0].cuda_stream)  # warm-up pair, eager
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=streams[0], capture_error_mode="thread_local"):
            NativeStrips.run_local_sequenced(ranks, ins, torch.cuda.current_stream(dev).cuda_stream)
        for trial, (dx, dy) in enumerate([(2.25, -1.5), (-3.0, 0.75)]):
            whole = load(20 + trial, dx, dy)
            with torch.cuda.stream(streams[0]):
                g.replay()
            torch.cuda.synchronize()
            for ns in ranks:
                ns.check(0)
                for k in range(levels):
                    y0, y1 = ns.own_rows(k)
                    ref, got = whole[k][0, y0:y1], ns.own_flow(k)
                    m = ~torch.isnan(ref)
                    assert torch.equal(torch.isnan(ref), torch.isnan(got)) and torch.equal(ref[m], got[m]), \
                        f"replay {trial} rank {ns.rank} level {k}"
    finally:
        torch.cuda.synchronize()
        for ns in ranks:
            ns.close()


@pytest.mark.gpu
def test_native_strips_two_processes_over_cuda_ipc():
    """Two PROCESSES, one GPU each, connected over CUDA IPC (the peer-memory transport as bench.py runs it under
    torchrun): rows pushed into the neighbour's arena over NVLink, two pairs in flight, bit for bit the whole-frame
    result.  Skipped on a one-GPU box."""
    import json
    import socket
    import subprocess
    import sys

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(root, "bench.py"), "--strips-only", "--strips-size", "1920x1080x3",
           "--strips-reps", "6"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    rec = line["strips"]
    assert rec["n_ranks"] == 2 and rec["transport"] == "peer"
    assert rec["bit_identical_to_whole_frame"] is True
    assert rec["in_flight_2"]["bit_identical_to_whole_frame"] is True


def test_native_strip_plan_matches_python_plan():
    """The schedule exists twice -- StripPlan here (the Python restatement, checked by test_strip_plan_invariants) and in
    csrc/strips.cu (the runner): own rows, kernel rows and coarse-flow rows must agree for every rank and level; the
    native image buffers may only be larger (they also hold the rows from which the coarser levels' halo rows are
    rebuilt locally)."""
    import ctypes as C

    from cuda_optical_flow_2_b200 import _lib
    from cuda_optical_flow_2_b200.dist import StripPlan

    lib = _lib.load()
    out = (C.c_int * 8)()
    n = 0
    for (W, H, levels, win, reach) in [(7680, 4320, 4, 9, 16), (1920, 1080, 3, 9, 16), (3840, 2160, 4, 15, 8), (322, 406, 2, 5, 16),
                                       (640, 480, 1, 5, 4), (1001, 777, 3, 19, 2)]:
        for world in (1, 2, 3, 4, 8):
            if (H >> (levels - 1)) < world:
                continue
            plan = StripPlan(W, H, levels, win, world, reach)
            plan.validate()
            for rank in range(world):
                for k in range(levels):
                    _lib.check(lib.ofb_strips_plan_query(W, H, levels, win, world, rank, reach, k, out))
                    y0, y1, by0, by1, cy0, cy1, eb0, eb1 = list(out)
                    s = plan.level(k, rank)
                    assert (y0, y1, by0, by1, cy0, cy1) == (s.y0, s.y1, s.by0, s.by1, s.cy0, s.cy1), (W, H, levels, win, world, rank, k)
                    assert eb0 <= by0 and eb1 >= by1 and 0 <= eb0 and eb1 <= (H >> k)
                    if k + 1 < levels:  # every buffer row of the next level can be built from this level's buffer
                        _lib.check(lib.ofb_strips_plan_query(W, H, levels, win, world, rank, reach, k + 1, out))
                        ceb0, ceb1 = out[6], out[7]
                        assert eb0 <= max(0, 2 * ceb0 - 1) and eb1 >= min(H >> k, 2 * (ceb1 - 1) + 2)
                    n += 1
    assert n > 100
    assert lib.ofb_strips_plan_query(640, 480, 3, 9, 500, 0, 16, 0, out) != 0  # more strips than coarsest rows
