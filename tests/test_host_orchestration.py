"""Host orchestration shared by the entry points: the frame stream's plain push on the whole-frame level loop, and the
native row-strip runner across processes.

- A push without a total flow composes the cumulative flow at level 0 (at least 3 levels, even sizes, a per-pixel warp
  mode), like every other whole-frame entry point.  Its flow must equal a push with the total, bit for bit, and the
  pairwise oracle on the preprocessed frames.
- A plain push launches grayscale, the optional bilateral filter (range table + filter), the pyramid and one kernel per
  level, with or without the total.
- With profiling on, a push records one pyramid record and, from the second frame on, one record per level.
- The native strip runner over peer memory (scripts/run_strips.py under torchrun, CUDA IPC between the processes)
  equals the whole frame bit for bit on 2 and 3 processes.
"""
from __future__ import annotations

import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from support import BIL, NEAR, assert_same_bytes, bgr_sequence, pyramid_launches

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,levels,win,mode", [(160, 120, 3, 9, BIL), (192, 128, 4, 7, NEAR), (256, 144, 4, 9, BIL)])
def test_stream_push_without_total_composes_bit_identically(ctx, oracle, w, h, levels, win, mode):
    frames = bgr_sequence(oracle, w, h, seed=83)
    lean = ctx.open_stream(w, h, levels, win, warp_mode=mode)
    full = ctx.open_stream(w, h, levels, win, warp_mode=mode)
    try:
        assert lean.push(frames[0]) is None and full.push(frames[0], want_total=True) is None
        prev = oracle.grayscale_c3(frames[0])[:, :, 0]
        for t in range(1, len(frames)):
            flows, total = lean.push(frames[t])
            ref_flows, ref_total = full.push(frames[t], want_total=True)
            assert total is None and ref_total is not None
            cur = oracle.grayscale_c3(frames[t])[:, :, 0]
            ref = oracle.flow_pair(np.ascontiguousarray(prev), np.ascontiguousarray(cur), levels, win, mode, oracle.SUMS_EXACT)
            for k in range(levels):
                assert_same_bytes(flows[k], ref_flows[k], f"push {t} level {k} against the push with the total")
                r = np.asarray(ref[k]).reshape(flows[k].shape)
                assert np.array_equal(np.isnan(flows[k]), np.isnan(r)), f"push {t} level {k}: NaN masks differ from the oracle"
                m = ~np.isnan(r)
                assert np.array_equal(flows[k][m], r[m]), f"push {t} level {k} differs from the oracle"
            prev = cur
    finally:
        lean.close()
        full.close()


@pytest.mark.gpu
@pytest.mark.parametrize("levels", [1, 2, 3, 4])
@pytest.mark.parametrize("bil", [0, 5])
@pytest.mark.parametrize("want_total", [False, True])
def test_stream_push_launch_count(ctx, oracle, levels, bil, want_total):
    w, h = 96, 64
    frames = bgr_sequence(oracle, w, h, seed=5)[:3]
    s = ctx.open_stream(w, h, levels, 9, bil_win=bil)
    try:
        for t, f in enumerate(frames):
            c0 = ctx.launch_count
            s.push(f, want_total=want_total)
            pre = 1 + (2 if bil else 0) + pyramid_launches(levels)
            assert ctx.launch_count - c0 == pre + (levels if t else 0), f"push {t}"
    finally:
        s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("levels", [1, 3, 4])
def test_stream_push_profile_records(ctx, oracle, levels):
    from cuda_optical_flow_2_b200 import PROFILE_PYRAMID

    w, h, pushes = 96, 64, 3
    frames = bgr_sequence(oracle, w, h, seed=7)[:pushes]
    s = ctx.open_stream(w, h, levels, 9)
    ctx.profile_enable(True)
    try:
        for f in frames:
            s.push(f)
        pyr = ctx.profile_read(PROFILE_PYRAMID)
        lv = [ctx.profile_read(k) for k in range(levels)]
    finally:
        ctx.profile_enable(False)
        s.close()
    assert pyr[1] == (pushes if levels > 1 else 0)
    for k in range(levels):
        assert lv[k][1] == pushes - 1, f"level {k}"


@pytest.mark.gpu
@pytest.mark.parametrize("nproc", [2, 3])
def test_native_strips_over_peer_memory(nproc):
    """One process per GPU, halo rows stored by the sender's kernels into the receiver's memory over CUDA IPC
    (csrc/strips.cu), three levels of a 1080p pair; every rank's own rows of every level equal the whole frame.  Skipped
    with fewer GPUs than processes."""
    import torch

    if torch.cuda.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "scripts", "run_strips.py"), "--check",
           "--w", "1920", "--h", "1080", "--levels", "3", "--reps", "4"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    rec = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert rec["n_gpus"] == nproc and rec["transport"] == "peer"
    assert rec["bit_identical_to_whole_frame"] is True
