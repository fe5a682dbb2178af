"""Sparse pyramidal Lucas-Kanade (ofb_track_points_device): a list of sub-pixel points tracked through the pyramid.

The tracker's arithmetic is pinned (include/ofb200.h): 8.8 fixed-point positions, exact integer fields and window sums, the
dense path's double-precision solve.  So the CUDA kernel (csrc/track.cu) and the C restatement in tests/track_oracle.c
(compiled here into a temporary directory, on the pyramid levels of the pinned oracle.gauss_pyramid) must agree bit for bit.

CPU tests (no mark): the restatement against the pinned dense oracle (oracle.lk_level) where the rule says they coincide,
crafted inputs that reach every branch, and the tracker's meaning on frames with a known sub-pixel shift.
GPU tests: the kernel against the restatement over windows, levels, sizes, batch shapes, iteration counts, thresholds and
flow scales; against the dense path itself; CUDA graph replay; argument refusals.
"""
import ctypes as C

import numpy as np
import pytest

from support import (F32, PT_LOW_TEXTURE, PT_NONFINITE, PT_OUTSIDE, PT_TRACKED, S815, assert_same_bits, assert_status_equal,
                     assert_values_equal, border_points, random_points, solve, to_device, tro)  # noqa: F401 (tro is a fixture)


def frames(oracle, w, h, dx=1.5, dy=-0.75, cell=4, seed=1234):
    return oracle.make_frame(w, h, 0, 0, cell, seed), oracle.make_frame(w, h, dx, dy, cell, seed)


# ------------------------------------------------------------------------------------ CPU: the tie to the pinned oracle
@pytest.mark.parametrize("win", list(range(3, 20, 2)))
def test_single_level_single_iteration_is_the_dense_oracle(tro, oracle, win):
    """levels = 1, iters = 1, integer points, min_eig = 0: every sample is the field value and the solve is the dense one, so
    the flow of a point is oracle.lk_level at its pixel; on every border pixel and corner of an odd-sized frame."""
    w, h = 37, 29
    prev, nxt = frames(oracle, w, h, 1.3, -0.6)
    pts = np.concatenate([border_points(w, h), np.array([[w // 2, h // 2], [5, 7], [30, 20]], F32)])
    flow, st = tro.track(prev, nxt, 1, win, pts, 1.0, iters=1, eps=0.0)
    dense = oracle.lk_level(prev, nxt, win)
    ref = dense[pts[:, 1].astype(int), pts[:, 0].astype(int)]
    assert_values_equal(flow, ref, f"win {win}")
    fin = np.isfinite(flow).all(1)
    assert (st[~fin] == PT_NONFINITE).all() and np.isin(st[fin], [PT_TRACKED, PT_OUTSIDE]).all()


# ------------------------------------------------------------------------------------ CPU: every branch
def test_starts(tro, oracle):
    """NaN, inf and outside starts are OUTSIDE with NaN flow; x = w-1 and y = h-1 exactly are tracked."""
    w, h = 40, 30
    prev, nxt = frames(oracle, w, h)
    pts = np.array([[np.nan, 5], [5, np.inf], [-1e-3, 5], [5, -0.5], [w - 1 + 1 / 256, 5], [5, h - 1 + 1e-3],
                    [w - 1, 5], [5, h - 1], [w - 1, h - 1], [0, 0]], F32)
    flow, st = tro.track(prev, nxt, 2, 7, pts)
    assert (st[:6] == PT_OUTSIDE).all() and np.isnan(flow[:6]).all()
    assert not np.isnan(flow[6:]).any()


def test_half_to_even_positions(tro, oracle):
    """x * 256 exactly at n + 0.5 rounds to the even neighbour: a tie tracks exactly like the point at the even position
    and unlike the one at the odd position (one level, where the position is x * 256; the GPU tests also start points on
    ties of levels 1..3)."""
    w, h = 64, 48
    prev, nxt = frames(oracle, w, h, 0.7, 0.4)
    n = np.array([5000, 5001, 3333], F32)  # ties n + 0.5: 5000.5 -> 5000, 5001.5 -> 5002, 3333.5 -> 3334
    x = (n + F32(0.5)) / F32(256)
    even = np.where(n % 2 == 0, n, n + 1) / F32(256)
    odd = np.where(n % 2 == 0, n + 1, n) / F32(256)
    y = np.full(3, 20.25, F32)
    run = lambda xs: tro.track(prev, nxt, 1, 9, np.stack([xs, y], 1), S815, iters=5, eps=0)
    ft, st = run(x)
    fe, se = run(even)
    fo, _ = run(odd)
    assert_same_bits(ft, fe)
    assert_status_equal(st, se)
    assert (ft != fo).any(1).all()


def test_flat_patch_is_nonfinite(tro, oracle):
    """A constant block in both frames: det == 0 (Q3) at the coarsest level, flow non-finite."""
    w, h = 160, 160
    prev, nxt = frames(oracle, w, h)
    prev[32:128, 32:128] = 77
    nxt[32:128, 32:128] = 77
    flow, st = tro.track(prev, nxt, 3, 9, np.array([[80, 80], [79.3, 81.6]], F32))
    assert (st == PT_NONFINITE).all() and not np.isfinite(flow).all(1).any()


def test_min_eig_threshold(tro, oracle):
    """A weak-gradient patch (values 100..103): min_eig 0.1 % above the window's lam is LOW_TEXTURE (flow 0), 0.1 % below
    is tracked; lam from the pinned oracle's exact window sums (integer point, one level: samples are field values)."""
    w, h, win = 48, 40, 9
    rng = np.random.default_rng(3)
    prev = (100 + rng.integers(0, 4, (h, w))).astype(np.uint8)
    nxt = np.roll(prev, 1, 1)
    x, y = 20, 17
    a, d, b = (int(s[y, x]) for s in oracle.lk_level_sums(prev, nxt, win)[:3])
    lam = ((a + d) - np.sqrt(float((a - d) ** 2 + 4 * b * b))) / (2 * win * win)
    assert 0 < lam < 50  # weak
    pt = np.array([[x, y]], F32)
    f_hi, s_hi = tro.track(prev, nxt, 1, win, pt, min_eig=lam * 1.001)
    f_lo, s_lo = tro.track(prev, nxt, 1, win, pt, min_eig=lam * 0.999)
    assert s_hi[0] == PT_LOW_TEXTURE and (f_hi == 0).all()
    assert s_lo[0] != PT_LOW_TEXTURE and np.isfinite(f_lo).all()


def test_point_driven_off_the_frame(tro, oracle):
    """Points on the last column and the last row, one level, one iteration: any update that moves the target right /
    down drives it off the frame.  Exactly those points are OUTSIDE, with their (finite) flow kept; the others are
    TRACKED."""
    w, h = 53, 41
    prev, nxt = frames(oracle, w, h, 1.7, 1.1)
    pts = np.concatenate([np.stack([np.full(h - 2, w - 1), np.arange(1, h - 1)], 1),
                          np.stack([np.arange(1, w - 1), np.full(w - 2, h - 1)], 1)]).astype(F32)
    flow, st = tro.track(prev, nxt, 1, 9, pts, S815, iters=1, eps=0)
    fin = np.isfinite(flow).all(1)
    U = np.rint(flow[fin] * F32(S815 * 256)).astype(np.int64)
    T = pts[fin].astype(np.int64) * 256 + U
    off = (T[:, 0] > (w - 1) * 256) | (T[:, 1] > (h - 1) * 256) | (T < 0).any(1)
    assert np.array_equal(st[fin] == PT_OUTSIDE, off) and off.any() and (~off).any()
    assert (st[fin][~off] == PT_TRACKED).all()


def test_32768_px_guard(tro, oracle):
    """flow_scale 1e6: after the first update |s*d| >= 32768 px, so the second iteration of level 1 stops the point OUTSIDE
    and reports 2 d.  With one iteration per level the guard stops it at the start of level 0 with the same 2 d."""
    w, h = 64, 48
    prev, nxt = frames(oracle, w, h)
    pts = np.array([[20, 20], [33.3, 17.8], [40, 30]], F32)
    flow, st = tro.track(prev, nxt, 2, 9, pts, 1e6, iters=5, eps=0)
    assert (st == PT_OUTSIDE).all() and (np.abs(F32(1e6) * flow).max(1) >= 32768).all()
    f1, st1 = tro.track(prev, nxt, 2, 9, pts, 1e6, iters=1, eps=0)
    assert (st1 == PT_OUTSIDE).all()
    assert_same_bits(flow, f1)


def test_eps_early_stop(tro, oracle):
    """eps so large that every level stops after its first update equals iters = 1 bit for bit; eps = 0.01 stops some
    levels early, so it differs from 30 fixed iterations on some points."""
    w, h = 96, 80
    prev, nxt = frames(oracle, w, h, 2.3, -1.2)
    pts = random_points(w, h, 64, 11, margin=-8)
    f1, s1 = tro.track(prev, nxt, 3, 9, pts, S815, iters=1, eps=0)
    fb, sb = tro.track(prev, nxt, 3, 9, pts, S815, iters=30, eps=1e9)
    assert_same_bits(fb, f1)
    assert_status_equal(sb, s1)
    fe, _ = tro.track(prev, nxt, 3, 9, pts, S815, iters=30, eps=0.01)
    f0, _ = tro.track(prev, nxt, 3, 9, pts, S815, iters=30, eps=0)
    ok = np.isfinite(fe).all(1) & np.isfinite(f0).all(1)
    assert (fe[ok] != f0[ok]).any(1).sum() > 0


def test_every_status_is_reached(tro, oracle):
    w, h = 160, 160
    prev, nxt = frames(oracle, w, h)
    prev[32:128, 32:128] = 77
    nxt[32:128, 32:128] = 77
    pts = np.array([[80, 80], [10, 10], [np.nan, 1], [w - 2, 150]], F32)
    _, st = tro.track(prev, nxt, 3, 9, pts, S815, min_eig=0)
    _, st_low = tro.track(prev, nxt, 3, 9, pts[1:2], S815, min_eig=1e6)
    assert set(st.tolist()) | set(st_low.tolist()) == {PT_TRACKED, PT_NONFINITE, PT_LOW_TEXTURE, PT_OUTSIDE}


# ------------------------------------------------------------------------------------ CPU: meaning
SHIFTS = [(-3.4, 2.6), (4.25, -3.75), (6.6, 1.2)]


def position_errors(tro, oracle, iters):
    """Median |s*flow - shift| (px) of TRACKED points, per shift, 3 levels, window 9, flow_scale 8/15, eps 0."""
    w, h = 192, 144
    pts = random_points(w, h, 200, 21, margin=-20)[11:]
    med = []
    for i, (dx, dy) in enumerate(SHIFTS):
        prev, nxt = frames(oracle, w, h, dx, dy, cell=4, seed=300)
        flow, st = tro.track(prev, nxt, 3, 9, pts, S815, iters=iters, eps=0.0)
        ok = st == PT_TRACKED
        assert ok.mean() > 0.9
        err = np.hypot(S815 * flow[ok, 0] - dx, S815 * flow[ok, 1] - dy)
        med.append(float(np.median(err)))
    return np.array(med)


def test_iterations_reduce_the_position_error(tro, oracle):
    """Sub-pixel shifts of 4.3, 5.6 and 6.7 px, 3 levels, window 9.  Measured with the restatement: median error 0.07,
    0.26 and 0.80 px with one iteration per level, 0.028, 0.023 and 0.026 px with 30.  The bar: 30 iterations at most half
    the one-iteration error, and at most 0.05 px."""
    e1 = position_errors(tro, oracle, 1)
    e30 = position_errors(tro, oracle, 30)
    assert (e30 <= 0.5 * e1).all(), (e1, e30)
    assert (e30 <= 0.05).all(), e30


# ------------------------------------------------------------------------------------ CPU: ABI
def test_null_context_is_rejected():
    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    p = _lib.OfbParams(64, 64, 1, 9, 2, 1.0, 1)
    assert lib.ofb_track_points_device(None, C.byref(p), None, None, 64, 4096, None, 1, 30, 0.01, 0.0, None, None,
                                       None) == _lib.OFB_ERR_INVALID
    assert b"NULL" in lib.ofb_last_error()


# ------------------------------------------------------------------------------------ GPU
def _batch(oracle, w, h, n, seed):
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 4, seed + i) for i in range(n)])
    nexts = np.stack([oracle.make_frame(w, h, 1.2 + 0.37 * (i % 7), -0.8 + 0.21 * (i % 5), 4, seed + i) for i in range(n)])
    return prevs, nexts


def _run_gpu(ctx, prevs, nexts, w, levels, win, pts, **kw):
    from cuda_optical_flow_2_b200 import planar_to_device

    flow, st = ctx.track_points_device(planar_to_device(prevs), planar_to_device(nexts), w, levels, win, to_device(pts), **kw)
    return flow.cpu().numpy(), st.cpu().numpy()


def _check_pairs(ctx, tro, prevs, nexts, w, levels, win, pts, check=None, **kw):
    flow, st = _run_gpu(ctx, prevs, nexts, w, levels, win, pts, **kw)
    pairs = range(len(prevs)) if check is None else check
    for i in pairs:
        rf, rs = tro.track(prevs[i], nexts[i], levels, win, pts[i], **kw)
        assert_same_bits(flow[i], rf, f"pair {i} flow")
        assert_status_equal(st[i], rs, f"pair {i} status")
    return flow, st


@pytest.mark.gpu
@pytest.mark.parametrize("iters,eps", [(1, 0.0), (1, 0.01), (5, 0.0), (5, 0.01), (30, 0.0), (30, 0.01)])
@pytest.mark.parametrize("win,w,h,levels,flow_scale,min_eig", [
    (3, 67, 45, 1, 1.0, 0.0), (5, 96, 64, 2, S815, 0.0), (7, 101, 77, 3, S815, 1e4), (9, 160, 120, 3, S815, 0.0),
    (11, 133, 95, 4, 1.0, 0.0), (13, 128, 96, 2, S815, 1e4), (15, 99, 81, 3, 1.0, 0.0), (17, 150, 110, 4, S815, 0.0),
    (19, 141, 117, 3, S815, 1e4),
])
def test_kernel_equals_restatement(ctx, tro, oracle, win, w, h, levels, flow_scale, min_eig, iters, eps):
    """Odd sizes, 3 pairs, 37 points each (not a multiple of the 4 points per CTA), sub-pixel, border, outside and
    half-to-even starts.  min_eig 1e4 lies inside the range of these frames' lam: some points are LOW_TEXTURE, some not."""
    prevs, nexts = _batch(oracle, w, h, 3, 40 + win)
    pts = np.stack([random_points(w, h, 37, 1000 * win + i) for i in range(3)])
    _, st = _check_pairs(ctx, tro, prevs, nexts, w, levels, win, pts, flow_scale=flow_scale, iters=iters, eps=eps,
                         min_eig=min_eig)
    assert (st == PT_TRACKED).any() and (st == PT_OUTSIDE).any()
    assert (st == PT_LOW_TEXTURE).any() == (min_eig > 0)


def crafted_cases(oracle):
    """(name, prev, next, levels, win, points, kwargs, statuses the case must produce): the CPU branch tests' inputs."""
    cases = []
    w, h = 160, 160
    prev, nxt = frames(oracle, w, h)
    prev[32:128, 32:128] = 77
    nxt[32:128, 32:128] = 77
    cases.append(("flat_block", prev, nxt, 3, 9, np.array([[80, 80], [79.3, 81.6], [10, 10]], F32), dict(flow_scale=S815),
                  {PT_NONFINITE, PT_TRACKED}))
    w, h, win = 48, 40, 9
    rng = np.random.default_rng(3)
    weak = (100 + rng.integers(0, 4, (h, w))).astype(np.uint8)
    weak_next = np.roll(weak, 1, 1)
    x, y = 20, 17
    a, d, b = (int(s[y, x]) for s in oracle.lk_level_sums(weak, weak_next, win)[:3])
    lam = ((a + d) - np.sqrt(float((a - d) ** 2 + 4 * b * b))) / (2 * win * win)
    for f, want in ((1.001, PT_LOW_TEXTURE), (0.999, PT_TRACKED)):
        cases.append((f"min_eig_lam_x{f}", weak, weak_next, 1, win, np.array([[x, y]], F32), dict(min_eig=lam * f), {want}))
    w, h = 64, 48
    prev, nxt = frames(oracle, w, h)
    cases.append(("guard_32768px", prev, nxt, 2, 9, np.array([[20, 20], [33.3, 17.8], [40, 30]], F32),
                  dict(flow_scale=1e6, iters=5, eps=0), {PT_OUTSIDE}))
    w, h = 53, 41
    prev, nxt = frames(oracle, w, h, 1.7, 1.1)
    edge = np.concatenate([np.stack([np.full(h - 2, w - 1), np.arange(1, h - 1)], 1),
                           np.stack([np.arange(1, w - 1), np.full(w - 2, h - 1)], 1)]).astype(F32)
    cases.append(("final_target_off_frame", prev, nxt, 1, 9, edge, dict(flow_scale=S815, iters=1, eps=0),
                  {PT_OUTSIDE, PT_TRACKED}))
    w, h = 40, 30
    prev, nxt = frames(oracle, w, h)
    starts = np.array([[np.nan, 5], [5, np.inf], [-1e-3, 5], [w - 1 + 1 / 256, 5], [w - 1, 5], [5, h - 1]], F32)
    cases.append(("starts", prev, nxt, 2, 7, starts, {}, {PT_OUTSIDE}))
    return cases


@pytest.mark.gpu
def test_kernel_equals_restatement_on_every_status(ctx, tro, oracle):
    """The CPU branch tests' crafted inputs through the kernel: a flat block (NONFINITE), a weak-gradient patch with min_eig
    0.1 % above / below its lam (LOW_TEXTURE / not), flow_scale 1e6 (the 32768 px guard), targets driven off the frame and
    outside starts.  Every case is bit-identical to the restatement and yields its statuses, and all four statuses occur
    among the points compared."""
    seen = set()
    for name, prev, nxt, levels, win, pts, kw, want in crafted_cases(oracle):
        h, w = prev.shape
        flow, st = _check_pairs(ctx, tro, prev[None], nxt[None], w, levels, win, pts[None], **kw)
        got = set(np.unique(st).tolist())
        assert want <= got, (name, want, got)
        seen |= got
    assert seen == {PT_TRACKED, PT_NONFINITE, PT_LOW_TEXTURE, PT_OUTSIDE}


@pytest.mark.gpu
def test_kernel_equals_restatement_batch_shapes(ctx, tro, oracle):
    """One point on one pair; 257 pairs of 5 points; 100 k points on one pair (a random 3000 of them checked)."""
    w, h = 75, 53
    prevs, nexts = _batch(oracle, w, h, 1, 7)
    _check_pairs(ctx, tro, prevs, nexts, w, 2, 9, np.array([[[30.3, 21.7]]], F32), flow_scale=S815)
    prevs, nexts = _batch(oracle, w, h, 257, 11)
    pts = np.stack([random_points(w, h, 5, i) for i in range(257)])
    _check_pairs(ctx, tro, prevs, nexts, w, 3, 5, pts, check=[0, 1, 128, 255, 256], flow_scale=S815, iters=5)
    w, h = 320, 240
    prevs, nexts = _batch(oracle, w, h, 1, 3)
    pts = random_points(w, h, 100_000, 5)[None]
    flow, st = _run_gpu(ctx, prevs, nexts, w, 3, 7, pts, flow_scale=S815, iters=5)
    sel = np.sort(np.random.default_rng(0).choice(100_000, 3000, replace=False))
    rf, rs = tro.track(prevs[0], nexts[0], 3, 7, pts[0, sel], flow_scale=S815, iters=5)
    assert_same_bits(flow[0, sel], rf, "100k flow")
    assert_status_equal(st[0, sel], rs, "100k status")


@pytest.mark.gpu
@pytest.mark.parametrize("win", [3, 9, 19])
def test_single_level_single_iteration_is_the_dense_path(ctx, oracle, win):
    """levels = 1, iters = 1, integer points: the flow is flow_pairs_device's (EXACT solve) at those pixels, compared with no
    restatement in between; setting the context to SOLVE_FAST changes nothing in the tracker."""
    from cuda_optical_flow_2_b200 import SOLVE_EXACT, SOLVE_FAST, planar_to_device
    w, h, n = 83, 61, 2
    prevs, nexts = _batch(oracle, w, h, n, 50 + win)
    p, q = planar_to_device(prevs), planar_to_device(nexts)
    assert ctx.solve == SOLVE_EXACT
    dense = ctx.flow_pairs_device(p, q, w, 1, win)[0].cpu().numpy()
    rng = np.random.default_rng(win)
    pts = np.stack([np.concatenate([border_points(w, h), np.stack([rng.integers(0, w, 200), rng.integers(0, h, 200)], 1)])
                    for _ in range(n)]).astype(F32)
    flow, st = ctx.track_points_device(p, q, w, 1, win, to_device(pts), iters=1, eps=0.0)
    flow = flow.cpu().numpy()
    for i in range(n):
        ref = dense[i][pts[i, :, 1].astype(int), pts[i, :, 0].astype(int)]
        assert_values_equal(flow[i], ref, f"pair {i}")
    with solve(ctx, SOLVE_FAST):
        f2, s2 = ctx.track_points_device(p, q, w, 1, win, to_device(pts), iters=1, eps=0.0)
        f3, s3 = ctx.track_points_device(p, q, w, 3, win, to_device(pts), flow_scale=S815)
    f4, s4 = ctx.track_points_device(p, q, w, 3, win, to_device(pts), flow_scale=S815)
    assert_same_bits(f2.cpu().numpy(), flow)
    assert np.array_equal(s2.cpu().numpy(), st.cpu().numpy())
    assert_same_bits(f3.cpu().numpy(), f4.cpu().numpy())
    assert np.array_equal(s3.cpu().numpy(), s4.cpu().numpy())


@pytest.mark.gpu
def test_cuda_graph_replay(ctx, oracle):
    """After reserve_pairs with the same parameters, a captured call replays bit-identically on new frames and points
    written into the captured input buffers."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, levels, win, n, m = 160, 96, 3, 9, 2, 500
    ctx.reserve_pairs(w, h, levels, win, n)
    rounds = [(_batch(oracle, w, h, n, 900 + 10 * r), np.stack([random_points(w, h, m, 77 * r + i) for i in range(n)]))
              for r in range(3)]
    (p0, q0), pts0 = rounds[0]
    p, q, pts = planar_to_device(p0), planar_to_device(q0), to_device(pts0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        ctx.track_points_device(p, q, w, levels, win, pts, S815, stream=side.cuda_stream)  # warm-up
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = ctx.track_points_device(p, q, w, levels, win, pts, S815, stream=torch.cuda.current_stream().cuda_stream)
    for (prevs, nexts), pr in rounds[1:]:
        p.copy_(planar_to_device(prevs))
        q.copy_(planar_to_device(nexts))
        pts.copy_(to_device(pr))
        g.replay()
        torch.cuda.synchronize()
        eager = ctx.track_points_device(planar_to_device(prevs), planar_to_device(nexts), w, levels, win, to_device(pr), S815)
        torch.cuda.synchronize()
        for got, ref in zip(out, eager):
            assert np.array_equal(got.cpu().numpy().view(np.uint8), ref.cpu().numpy().view(np.uint8))


@pytest.mark.gpu
def test_profile_record_around_the_tracker(ctx, oracle):
    from cuda_optical_flow_2_b200 import PROFILE_PYRAMID, PROFILE_TRACK

    w, h = 96, 64
    prevs, nexts = _batch(oracle, w, h, 1, 5)
    ctx.profile_enable(True)
    try:
        _run_gpu(ctx, prevs, nexts, w, 3, 9, random_points(w, h, 100, 1)[None])
        ms, n = ctx.profile_read(PROFILE_TRACK)
        _, n_pyr = ctx.profile_read(PROFILE_PYRAMID)
    finally:
        ctx.profile_enable(False)
    assert n == 1 and ms > 0 and n_pyr == 1


@pytest.mark.gpu
def test_refusals_enqueue_nothing(ctx):
    import torch

    from cuda_optical_flow_2_b200 import WARP_AS_WRITTEN, WARP_NEAREST, OfbError, _lib, planar_to_device

    lib = _lib.load()
    w, h, n, m = 64, 48, 2, 10
    frame = planar_to_device(np.zeros((n, h, w), np.uint8))
    pts = torch.zeros((n, m, 2), dtype=torch.float32, device="cuda")
    flow = torch.zeros((n, m, 2), dtype=torch.float32, device="cuda")
    st = torch.zeros((n, m), dtype=torch.uint8, device="cuda")
    inv = _lib.OFB_ERR_INVALID

    def call(warp=2, levels=3, win=9, pairs=n, fs=1.0, prev=frame.data_ptr(), nxt=frame.data_ptr(), pitch=64,
             points=pts.data_ptr(), n_points=m, iters=30, eps=0.01, min_eig=0.0, fl=flow.data_ptr(), status=st.data_ptr()):
        p = _lib.OfbParams(w, h, levels, win, warp, fs, pairs)
        return lib.ofb_track_points_device(ctx._h, C.byref(p), prev, nxt, pitch, pitch * h, points, n_points, iters, eps,
                                           min_eig, fl, status, None)

    assert call() == 0
    torch.cuda.synchronize()
    before = ctx.launch_count
    bad = [dict(warp=WARP_AS_WRITTEN), dict(warp=WARP_NEAREST), dict(n_points=0), dict(n_points=(1 << 24) + 1),
           dict(iters=0), dict(iters=65), dict(eps=-0.01), dict(eps=float("nan")), dict(min_eig=-1.0),
           dict(min_eig=float("inf")), dict(prev=None), dict(nxt=None), dict(points=None), dict(fl=None), dict(status=None),
           dict(points=pts.data_ptr() + 4), dict(fl=flow.data_ptr() + 4), dict(fs=0.0), dict(fs=float("nan")), dict(fs=2e36),
           dict(pairs=65536), dict(pitch=32), dict(levels=0), dict(win=8)]
    for kw in bad:
        assert call(**kw) != 0, kw
        assert ctx.launch_count == before, kw
    assert call(n_points=0) == inv and b"n_points" in lib.ofb_last_error()
    with pytest.raises(OfbError, match="warp mode"):
        lib_p = _lib.OfbParams(w, h, 3, 9, WARP_NEAREST, 1.0, n)
        _lib.check(lib.ofb_track_points_device(ctx._h, C.byref(lib_p), frame.data_ptr(), frame.data_ptr(), 64, 64 * h,
                                               pts.data_ptr(), m, 30, 0.01, 0.0, flow.data_ptr(), st.data_ptr(), None))
    with pytest.raises(ValueError, match="points"):
        ctx.track_points_device(frame, frame, w, 3, 9, pts[:1])
    with pytest.raises(ValueError, match="points"):
        ctx.track_points_device(frame, frame, w, 3, 9, pts.cpu())  # a host tensor is refused, not dereferenced
    with pytest.raises(ValueError, match="CUDA"):
        ctx.track_points_device(frame.cpu(), frame.cpu(), w, 3, 9, pts)
    assert call(fs=2e36) == inv and b"flow_scale" in lib.ofb_last_error()
    assert ctx.launch_count == before
