"""Forward-backward consistency check on row strips (ofb_strips_create_fb / ofb_strips_run_fb_device, dist.NativeStrips).

A checked pair runs both directions on one pyramid build per rank, fetches the neighbours' backward total rows its check
samples and checks its own rows.  Every output must be bit-identical to rows [y0, y1) of ofb_flow_pairs_fb_device on the
whole frame, except pixels whose check needs a backward tap outside the rows the rank holds: those are FB_UNCHECKED.

CPU: the UNCHECKED rule in numpy against the whole-frame status of the C restatement (orc_fb_check), on fields that put
targets on the held-row bounds, one row either side and on zero-weight taps.
GPU: ranks live in this process on one device (connect_local), their phases interleaved on one stream
(run_local_sequenced_fb): equivalence to the whole frame, motion beyond fb_reach, plain and checked pairs alternating,
CUDA graph replay, refusals; and two processes over CUDA IPC under torchrun (skipped on a one-GPU box).
"""
import os

import numpy as np
import pytest

from support import (F32, FB_BWD_NONFINITE, FB_CONSISTENT, FB_FWD_NONFINITE, FB_INCONSISTENT, FB_OUTSIDE, FB_UNCHECKED, S815,
                     assert_equals_whole, assert_same_bits, assert_status_equal, fbo, held_rows, np_fb_check, solve,
                     tap_rows_outside)  # noqa: F401 (fbo is a fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------ numpy restatement of the strip rule
def np_fb_check_strip(fwd_own, bwd_held, y0, h, b0, b1, s, alpha=0.01, beta=0.5):
    """The strip check from what a rank holds: its own forward rows and backward rows [b0, b1)."""
    rows, w = fwd_own.shape[:2]
    fwd = np.full((h, w, 2), np.nan, F32)
    fwd[y0:y0 + rows] = fwd_own
    bwd = np.zeros((h, w, 2), F32)  # rows outside [b0, b1) are never read by a pixel that is not UNCHECKED
    bwd[b0:b1] = bwd_held
    status, err2 = np_fb_check(fwd, bwd, s, alpha, beta)
    status, err2 = status[y0:y0 + rows], err2[y0:y0 + rows]
    _, out = tap_rows_outside(fwd_own, y0, h, b0, b1, s)
    status[out] = FB_UNCHECKED
    err2[out] = np.nan
    return status, err2


def _bound_field(w=16, h=40, y0=16, y1=24, fb_reach=3):
    """Own rows [y0, y1); held rows [y0 - fb_reach, y1 + fb_reach + 1) = [13, 28).  Column j of every own row gets a vertical
    displacement that puts its target on, or one row either side of, a held-row bound, with and without a zero-weight
    second tap; the last columns are NaN forward flow, a target outside the frame and a horizontal-only move."""
    b0, b1 = held_rows(y0, y1, h, fb_reach)
    rng = np.random.default_rng(7)
    fwd = rng.normal(0, 0.3, (h, w, 2)).astype(F32)
    bwd = (-fwd + rng.normal(0, 0.05, (h, w, 2))).astype(F32)
    targets = [b0 - 1, b0 - 1 + 0.5, b0, b0 + 0.25, b0 + 1,  # the top bound: outside, straddling, on it (zero weight), inside
               b1 - 2, b1 - 2 + 0.5, b1 - 1, b1 - 1 + 0.5, b1, b1 + 1]  # the bottom bound: inside, on it, straddling, outside
    for i in range(y0, y1):
        for j, t in enumerate(targets):
            fwd[i, j] = (F32(0.25), F32(t - i))
        fwd[i, len(targets), :] = np.nan
        fwd[i, len(targets) + 1, 1] = F32(h + 5 - i)  # leaves the frame: OUTSIDE, reads nothing
        fwd[i, len(targets) + 2] = (F32(1.5), F32(0))
    bwd[b1 - 1, 7, 0] = np.nan  # held, read by column 7 (target row b1 - 1 exactly): BWD_NONFINITE stays; column 8 also
    bwd[b1 - 1, 8, 1] = np.nan  # reads it, but its second tap row b1 is not held: UNCHECKED takes precedence
    bwd[b1, 9, 0] = np.nan      # not held: its reader (column 9) is UNCHECKED, never BWD_NONFINITE
    return fwd, bwd, y0, y1, b0, b1, len(targets)


@pytest.mark.parametrize("flow_scale", [1.0, S815])
def test_unchecked_rule_against_whole_frame_oracle(fbo, flow_scale):
    w, h = 16, 40
    fwd, bwd, y0, y1, b0, b1, nt = _bound_field(w, h)
    # the rule is stated in pixels: scale the crafted displacements back to flow units
    fwd = (fwd / F32(flow_scale)).astype(F32)
    whole_st, whole_e2 = fbo.fb_check(fwd, bwd, flow_scale)
    st, e2 = np_fb_check_strip(fwd[y0:y1], bwd[b0:b1], y0, h, b0, b1, flow_scale)
    ref_st, ref_e2 = whole_st[y0:y1], whole_e2[y0:y1]
    unchecked = st == FB_UNCHECKED
    # only pixels that read taps are replaced; every other pixel is the whole-frame result, bit for bit
    assert np.isin(ref_st[unchecked], [FB_CONSISTENT, FB_INCONSISTENT, FB_BWD_NONFINITE]).all()
    assert_status_equal(st[~unchecked], ref_st[~unchecked])
    assert_same_bits(e2[~unchecked], ref_e2[~unchecked], "err2 of checked pixels")
    assert np.isnan(e2[unchecked]).all()
    assert (st[ref_st == FB_FWD_NONFINITE] == FB_FWD_NONFINITE).all()
    assert (st[ref_st == FB_OUTSIDE] == FB_OUTSIDE).all()
    # the crafted columns: which targets are UNCHECKED, row by row (with flow_scale 8/15 the rounding to 1/256 px can move
    # a target by one step, so only the exact scale pins the columns)
    if flow_scale == 1.0:
        expect = np.array([True, True, False, False, False, False, False, False, True, True, True])
        for r in range(y1 - y0):
            assert np.array_equal(unchecked[r, :nt], expect), f"row {y0 + r}: {unchecked[r, :nt]}"
        assert (st[:, nt] == FB_FWD_NONFINITE).all() and (st[:, nt + 1] == FB_OUTSIDE).all()
        assert (st[:, nt + 2] != FB_UNCHECKED).all()
        assert (st[:, 7] == FB_BWD_NONFINITE).all()
        assert (ref_st[:, 8] == FB_BWD_NONFINITE).all() and (ref_st[:, 9] == FB_BWD_NONFINITE).all()


def test_unchecked_rule_on_random_fields(fbo):
    """Random flow with large vertical motion on every split of a frame: the numpy strip rule agrees with the whole-frame
    oracle on every checked pixel, and a pixel is UNCHECKED exactly when it reads a tap outside the held rows."""
    rng = np.random.default_rng(11)
    w, h = 24, 60
    fwd = np.stack([rng.normal(0, 2, (h, w)), rng.normal(0, 6, (h, w))], -1).astype(F32)
    bwd = (-np.roll(fwd, 1, 0) + rng.normal(0, 0.5, (h, w, 2))).astype(F32)
    whole_st, whole_e2 = fbo.fb_check(fwd, bwd, 1.0)
    seen = 0
    for y0, y1 in ((0, 20), (20, 40), (40, 60), (13, 31)):
        for fb_reach in (0, 2, 5, 40):
            b0, b1 = held_rows(y0, y1, h, fb_reach)
            st, e2 = np_fb_check_strip(fwd[y0:y1], bwd[b0:b1], y0, h, b0, b1, 1.0)
            reads, out = tap_rows_outside(fwd[y0:y1], y0, h, b0, b1, 1.0)
            assert np.array_equal(st == FB_UNCHECKED, out)
            assert np.array_equal(reads, np.isin(whole_st[y0:y1], [FB_CONSISTENT, FB_INCONSISTENT, FB_BWD_NONFINITE]))
            assert_status_equal(st[~out], whole_st[y0:y1][~out])
            assert_same_bits(e2[~out], whole_e2[y0:y1][~out])
            seen += int(out.sum())
    assert seen > 100


def test_package_exports_unchecked():
    import cuda_optical_flow_2_b200 as pkg

    assert pkg.FB_UNCHECKED == FB_UNCHECKED and "FB_UNCHECKED" in pkg.__all__


# ------------------------------------------------------------------------------------------------------------------- GPU
def _make_ranks(ctx, W, H, levels, win, world, warp_mode, fb_reach, reach=16, flow_scale=1.0):
    import torch

    from cuda_optical_flow_2_b200.dist import NativeStrips

    dev = torch.device("cuda", 0)
    ranks = [NativeStrips(ctx, W, H, levels, win, world, rk, dev, warp_mode, flow_scale, reach, transport="local", fb_reach=fb_reach)
             for rk in range(world)]
    NativeStrips.connect_local(ranks)
    return ranks


def _close(ranks):
    import torch

    torch.cuda.synchronize()
    for ns in ranks:
        ns.close()


def _frames(oracle, W, H, seed, dx, dy):
    from cuda_optical_flow_2_b200 import planar_to_device

    prev = oracle.make_frame(W, H, 0, 0, 8, seed)
    nxt = oracle.make_frame(W, H, dx, dy, 8, seed)
    return planar_to_device(prev[None]), planar_to_device(nxt[None])


def _inputs(ranks, dp, dn):
    out = []
    for ns in ranks:
        y0, y1 = ns.own_rows(0)
        out.append((dp[0, y0:y1], dn[0, y0:y1]))
    return out


EQUIV = [(640, 480, 3, 9, 1, 2), (640, 480, 3, 9, 2, 1), (640, 480, 3, 5, 4, 2), (640, 480, 1, 9, 3, 2), (322, 406, 2, 5, 3, 2),
         (322, 406, 2, 15, 2, 1), (322, 406, 3, 9, 4, 2), (1920, 1080, 3, 9, 8, 2), (1920, 1080, 4, 15, 4, 1),
         (7680, 4320, 4, 9, 8, 2), (7680, 4320, 4, 9, 2, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("kind", ["exact", "fast"])
@pytest.mark.parametrize("W,H,levels,win,world,mode", EQUIV)
def test_checked_pair_equals_whole_frame(ctx, oracle, W, H, levels, win, world, mode, kind, fused):
    """Three checked pairs back to back on the same handles (err2 on, off, on), every output bit-identical to the
    whole-frame ofb_flow_pairs_fb_device rows, NaN positions included."""
    import torch

    from cuda_optical_flow_2_b200 import SOLVE_EXACT, SOLVE_FAST
    from cuda_optical_flow_2_b200.dist import NativeStrips

    with solve(ctx, SOLVE_FAST if kind == "fast" else SOLVE_EXACT):
        ranks = _make_ranks(ctx, W, H, levels, win, world, mode, fb_reach=16)
        try:
            for ns in ranks:
                ns.set_fused(fused)
            for trial, (dx, dy) in enumerate([(2.25, -1.5), (-3.0, 0.75), (0.5, 2.0)]):
                want_err2 = trial != 1
                dp, dn = _frames(oracle, W, H, 700 + trial, dx, dy)
                whole = ctx.flow_pairs_fb_device(dp, dn, W, levels, win, warp_mode=mode, want_err2=want_err2)
                torch.cuda.synchronize()
                NativeStrips.run_local_sequenced_fb(ranks, _inputs(ranks, dp, dn), want_err2=want_err2,
                                                    stream=torch.cuda.current_stream().cuda_stream)
                assert_equals_whole(ranks, whole, want_err2, f"pair {trial}")
        finally:
            _close(ranks)


@pytest.mark.gpu
@pytest.mark.parametrize("flow_scale", [1.0, S815])
def test_motion_beyond_fb_reach_is_unchecked(ctx, oracle, flow_scale):
    """A vertical motion larger than fb_reach (reach large enough that no warp overflows): bit 2 is raised on the ranks
    concerned, the UNCHECKED pixels are exactly those the whole-frame forward total sends outside the held rows, and every
    other output equals the whole frame."""
    import torch

    from cuda_optical_flow_2_b200.dist import NativeStrips

    W, H, levels, win, world, fb_reach = 640, 480, 3, 9, 4, 2
    ranks = _make_ranks(ctx, W, H, levels, win, world, 2, fb_reach=fb_reach, reach=24, flow_scale=flow_scale)
    try:
        dp, dn = _frames(oracle, W, H, 41, 1.0, 6.0 / flow_scale)
        fwd, bwd, st, e2 = ctx.flow_pairs_fb_device(dp, dn, W, levels, win, flow_scale=flow_scale, want_err2=True)
        torch.cuda.synchronize()
        NativeStrips.run_local_sequenced_fb(ranks, _inputs(ranks, dp, dn), want_err2=True)
        total = 0
        for ns in ranks:
            y0, y1 = ns.own_rows(0)
            b0, b1 = held_rows(y0, y1, H, fb_reach)
            _, out = tap_rows_outside(fwd[0, y0:y1].cpu().numpy(), y0, H, b0, b1, flow_scale)
            if out.any():
                with pytest.raises(RuntimeError, match="fb_reach"):
                    ns.check()
            else:
                ns.check()
            gf, gb, gs, ge = (t.cpu().numpy() for t in ns.own_fb())
            assert np.array_equal(gs == FB_UNCHECKED, out), f"rank {ns.rank}"
            ref_st, ref_e2 = st[0, y0:y1].cpu().numpy(), e2[0, y0:y1].cpu().numpy()
            assert_status_equal(gs[~out], ref_st[~out], f"rank {ns.rank}")
            assert_same_bits(ge[~out], ref_e2[~out], f"rank {ns.rank} err2")
            assert np.isnan(ge[out]).all()
            assert_same_bits(gf, fwd[0, y0:y1].cpu().numpy(), "forward total")
            assert_same_bits(gb, bwd[0, y0:y1].cpu().numpy(), "backward total")
            total += int(out.sum())
        assert total > 1000
        for ns in ranks:
            ns.check()  # the flag is sticky until read, then clear
    finally:
        _close(ranks)


@pytest.mark.gpu
@pytest.mark.parametrize("world,fb_reach", [(2, 8), (3, 170), (4, 130)])
def test_plain_and_checked_pairs_alternate(ctx, oracle, world, fb_reach):
    """Plain and checked pairs alternate on one set of check-capable handles.  fb_reach 170 (3 strips of 160 rows) and 130
    (4 of 120): ranks that are not adjacent push check rows -- through the level kernel's two slots, or with more targets
    through the copy kernel -- and must be acknowledged by plain pairs too.  Plain pairs give the bytes and the launch count
    of plain handles; checked pairs the whole frame."""
    import torch

    from cuda_optical_flow_2_b200.dist import NativeStrips

    W, H, levels, win = 640, 480, 3, 9
    fb = _make_ranks(ctx, W, H, levels, win, world, 2, fb_reach=fb_reach)
    plain = _make_ranks(ctx, W, H, levels, win, world, 2, fb_reach=None)
    try:
        for step, kind in enumerate("pcppccp"):
            dp, dn = _frames(oracle, W, H, 300 + step, 1.5 - step * 0.5, 0.75)
            torch.cuda.synchronize()
            if kind == "c":
                whole = ctx.flow_pairs_fb_device(dp, dn, W, levels, win, want_err2=True)
                NativeStrips.run_local_sequenced_fb(fb, _inputs(fb, dp, dn), want_err2=True)
                assert_equals_whole(fb, whole, True, f"step {step}")
                continue
            n0 = ctx.launch_count
            NativeStrips.run_local_sequenced(plain, _inputs(plain, dp, dn))
            n1 = ctx.launch_count
            NativeStrips.run_local_sequenced(fb, _inputs(fb, dp, dn))
            n2 = ctx.launch_count
            assert n2 - n1 == n1 - n0, f"step {step}: launches {n2 - n1} on check-capable handles, {n1 - n0} on plain ones"
            for a, b in zip(plain, fb):
                a.check()
                b.check()
                for k in range(levels):
                    assert_same_bits(b.own_flow(k), a.own_flow(k), f"step {step} rank {a.rank} level {k}")
                assert_same_bits(b.own_flow(0, total=True), a.own_flow(0, total=True), f"step {step} rank {a.rank} total")
    finally:
        _close(fb + plain)


@pytest.mark.gpu
def test_checked_pair_replays_as_cuda_graph(ctx, oracle):
    import torch

    from cuda_optical_flow_2_b200.dist import NativeStrips

    W, H, levels, win, world = 1280, 720, 3, 9, 2
    dev = torch.device("cuda", 0)
    ranks = _make_ranks(ctx, W, H, levels, win, world, 2, fb_reach=16)
    side = torch.cuda.Stream(dev)
    try:
        ins = [ns.input_rows() for ns in ranks]

        def load(seed, dx, dy):
            dp, dn = _frames(oracle, W, H, seed, dx, dy)
            for ns, (pin, nin) in zip(ranks, ins):
                y0, y1 = ns.own_rows(0)
                pin[:, :W].copy_(dp[0, y0:y1, :W])
                nin[:, :W].copy_(dn[0, y0:y1, :W])
            whole = ctx.flow_pairs_fb_device(dp, dn, W, levels, win, want_err2=True)
            torch.cuda.synchronize()
            return whole

        load(11, 1.0, 1.0)
        NativeStrips.run_local_sequenced_fb(ranks, ins, want_err2=True, stream=side.cuda_stream)  # warm-up pair, eager
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
            NativeStrips.run_local_sequenced_fb(ranks, ins, want_err2=True, stream=torch.cuda.current_stream(dev).cuda_stream)
        for trial, (dx, dy) in enumerate([(2.25, -1.5), (-3.0, 0.75)]):
            whole = load(20 + trial, dx, dy)
            with torch.cuda.stream(side):
                g.replay()
            torch.cuda.synchronize()
            assert_equals_whole(ranks, whole, True, f"replay {trial}")
    finally:
        _close(ranks)


@pytest.mark.gpu
def test_checked_strip_refusals_enqueue_nothing(ctx, oracle):
    import ctypes as C

    import torch

    from cuda_optical_flow_2_b200 import OfbError, _lib
    from cuda_optical_flow_2_b200.dist import NativeStrips

    lib = _lib.load()
    h = C.c_void_p()
    W, H = 640, 480
    for scale in (0.0, -1.0, float("nan")):
        assert lib.ofb_strips_create_fb(ctx._h, W, H, 3, 9, 2, C.c_float(scale), 1, 0, 16, 8, C.byref(h)) == _lib.OFB_ERR_INVALID
    assert lib.ofb_strips_create_fb(ctx._h, W, H, 3, 9, 2, C.c_float(1.0), 1, 0, 16, -1, C.byref(h)) == _lib.OFB_ERR_INVALID
    assert lib.ofb_strips_create_fb(ctx._h, W, H, 3, 9, 0, C.c_float(1.0), 1, 0, 16, 8, C.byref(h)) == \
        _lib.OFB_ERR_UNSUPPORTED  # OFB_WARP_AS_WRITTEN, as ofb_strips_create
    ranks = _make_ranks(ctx, W, H, 3, 9, 2, 2, fb_reach=8)
    plain = _make_ranks(ctx, W, H, 3, 9, 2, 2, fb_reach=None)
    try:
        dp, dn = _frames(oracle, W, H, 5, 1.0, 1.0)
        pin, nin = _inputs(ranks, dp, dn)[0]
        torch.cuda.synchronize()
        n0 = ctx.launch_count
        for alpha, beta in ((-0.01, 0.5), (0.01, -1.0), (float("nan"), 0.5), (0.01, float("inf"))):
            with pytest.raises(OfbError):
                ranks[0].run_fb(pin, nin, alpha, beta)
        with pytest.raises(OfbError):
            ranks[0].run_fb_phase(pin, nin, 4 * 3 + 1)
        with pytest.raises(OfbError):
            plain[0].run_fb(pin, nin)
        with pytest.raises(OfbError):
            plain[0].own_fb()
        torch.cuda.synchronize()
        assert ctx.launch_count == n0
        for ns in ranks + plain:
            ns.check()
    finally:
        _close(ranks + plain)


@pytest.mark.gpu
def test_checked_pairs_two_processes_over_cuda_ipc():
    """Two PROCESSES, one GPU each, over CUDA IPC: scripts/fb_strips_bench.py under torchrun runs plain and checked pairs
    (alone, in flight, graph-replayed, alternated) and reports bit-identity to the whole frame.  Skipped on a one-GPU box."""
    import json
    import socket
    import subprocess
    import sys

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "scripts", "fb_strips_bench.py"), "--size", "1920x1080x3", "--reps", "4"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    rec = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert rec["n_ranks"] == 2 and rec["transport"] == "peer"
    assert rec["bit_identical_to_whole_frame"] is True
