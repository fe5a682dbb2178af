"""Forward-backward consistency check: ofb_fb_check_device, ofb_flow_pairs_fb_device and the oracle's orc_fb_check.

The check's arithmetic is pinned (include/ofb200.h): every multiply and add rounded on its own, no fma, the displacement
rounded to 1/256 px as the bilinear warp does.  So three implementations must agree bit for bit: the CUDA kernel
(csrc/fb_check.cu), the C restatement in tests/fb_oracle.c (compiled into a temporary directory) and the numpy
float32 restatement support.np_fb_check.  The flow both directions are checked on comes from the pinned oracle's oracle.flow_pair.

CPU tests (no mark): the oracle against numpy on inputs that reach every branch, the check's semantics on the oracle's
flow (the GPU path is pinned to the oracle, so the thresholds are set here), and the ABI's NULL-context checks.
GPU tests: the kernel and the two-direction entry point against the oracle, the shared pyramids against two
ofb_flow_pairs_device calls, symmetry, adversarial content, CUDA graph replay and argument checks.
"""
import ctypes as C

import numpy as np
import pytest

from support import (F32, FB_BWD_NONFINITE, FB_CONSISTENT, FB_FWD_NONFINITE, FB_INCONSISTENT, FB_OUTSIDE, PAIRS, S815,
                     assert_same_bits, assert_status_equal, assert_values_equal, fbo, np_fb_check, solve, to_device)  # noqa: F401


# ------------------------------------------------------------------------------------ the pin's inputs
def _random(w, h, seed):
    rng = np.random.default_rng(seed)
    fwd = (rng.normal(0, 3, (h, w, 2)) + rng.normal(0, 2, 2)).astype(F32)
    bwd = (-np.roll(fwd, (1, -2), (0, 1)) + rng.normal(0, 0.4, (h, w, 2))).astype(F32)
    return fwd, bwd


def _every_status(w=16, h=12):
    """Rows of the crafted field, top to bottom: consistent, inconsistent, outside, forward NaN / inf, backward NaN."""
    fwd = np.zeros((h, w, 2), F32)
    bwd = np.zeros((h, w, 2), F32)
    fwd[0, :, 0] = 0.5
    bwd[0, :, 0] = -0.5  # cancels: consistent
    fwd[1, :, 0] = 1.0
    bwd[1:3, :, 0] = 1.0  # same direction: |f + b|^2 = 4 > 0.01 * 2 + 0.5
    fwd[2, :, 0] = -np.arange(w, dtype=F32) - 1  # one pixel left of column 0
    fwd[3, ::2, 0] = np.nan
    fwd[3, 1::2, 1] = -np.inf
    fwd[4, :, 1] = 1.25
    bwd[5, ::3, 1] = np.nan  # read by row 4 (wy = 64)
    bwd[5, 1::3, 0] = np.inf
    fwd[6, :, 1] = 40000.0  # |dv| >= 32768
    fwd[7, :, 0] = 3e38  # s*u overflows to inf: outside
    return fwd, bwd


def _last_row_and_column(w=9, h=7):
    """Targets exactly on X == (w-1)*256 / Y == (h-1)*256 (inside), and 1/256 px beyond (outside)."""
    ii, jj = np.meshgrid(np.arange(h), np.arange(w), indexing="ij")
    fwd = np.stack([(w - 1 - jj), (h - 1 - ii)], -1).astype(F32)
    fwd[::2, :, 0] += F32(1 / 256)
    fwd[:, ::3, 1] += F32(1 / 256)
    rng = np.random.default_rng(5)
    bwd = rng.normal(0, 2, (h, w, 2)).astype(F32)
    bwd[h - 1, w - 1] = -fwd[1, 1]  # every unshifted pixel reads only the corner
    return fwd, bwd


def _half_to_even(w=12, h=10):
    """du*256 exactly at k + 0.5 for k = -6..5 (round half to even picks the even neighbour), u and v."""
    ks = np.arange(-6, 6, dtype=F32)
    fwd = np.zeros((h, w, 2), F32)
    fwd[..., 0] = ((ks + F32(0.5)) / F32(256))[None, :w]
    fwd[..., 1] = ((np.arange(h, dtype=F32) - 5 + F32(0.5)) / F32(256))[:, None]
    bwd = np.random.default_rng(9).normal(0, 0.01, (h, w, 2)).astype(F32)
    bwd[:, 1::2] = np.inf  # read or not, depending on where the rounding lands
    return fwd, bwd


def _range_limit(w=8, h=6):
    """|du| just below 32768 and at 32768, both signs, u and v (all outside: the frame is small, the branch differs)."""
    fwd = np.zeros((h, w, 2), F32)
    below = np.nextafter(F32(32768), F32(0))
    vals = np.array([below, F32(32768), -below, F32(-32768)], F32)
    fwd[0, :4, 0] = vals
    fwd[1, :4, 1] = vals
    fwd[2, :4, 0] = vals / F32(256)  # 128 px: outside through the bounds test
    return fwd, np.zeros((h, w, 2), F32)


def _bwd_specials(w=10, h=8):
    """inf / NaN / +-huge finite values in bwd on a zero-weight tap and on a read tap."""
    fwd = np.zeros((h, w, 2), F32)
    bwd = np.zeros((h, w, 2), F32)
    specials = [np.inf, -np.inf, np.nan, F32(3e38), F32(-3e38)]
    for r, val in enumerate(specials):
        # even columns: integer target (wx = 0), the special value one pixel right is never read; odd: wx = 128 reads it
        fwd[r, 1::2, 0] = 0.5
        bwd[r, 1::2, 0] = val
    fwd[5:, :, 0] = 0.25
    bwd[5:, :, 0] = F32(3e38)  # uniform huge backward flow: err2 = inf and mag2 = inf
    bwd[7, :, 1] = F32(-3e38)
    return fwd, bwd


def pin_cases():
    """(name, fwd, bwd, flow_scale, alpha, beta), every shape once with each flow_scale."""
    base = [("random_37x23", *_random(37, 23, 1)), ("random_64x16", *_random(64, 16, 2)), ("every_status", *_every_status()),
            ("last_row_col", *_last_row_and_column()), ("half_to_even", *_half_to_even()), ("range_limit", *_range_limit()),
            ("bwd_specials", *_bwd_specials()), ("w2", *_random(2, 9, 3)), ("h2", *_random(11, 2, 4)),
            ("2x2", *_random(2, 2, 5)), ("odd_33x17", *_random(33, 17, 6))]
    out = []
    for name, f, b in base:
        out.append((name + "_s1", f, b, 1.0, 0.01, 0.5))
        out.append((name + "_s8/15", f, b, S815, 0.01, 0.5))
    out.append(("random_alpha0_beta0", *_random(21, 13, 7), 1.0, 0.0, 0.0))
    return out


CASES = pin_cases()
CASE_IDS = [c[0] for c in CASES]


# ------------------------------------------------------------------------------------ CPU: the pin
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_oracle_equals_numpy_restatement(fbo, case):
    _, fwd, bwd, s, alpha, beta = case
    st, e2 = fbo.fb_check(fwd, bwd, s, alpha, beta)
    nst, ne2 = np_fb_check(fwd, bwd, s, alpha, beta)
    assert_status_equal(st, nst)
    assert_same_bits(e2, ne2, "err2")


def test_pin_inputs_reach_every_branch(fbo):
    """The crafted inputs take every status, the zero-weight tap rule, both half-to-even neighbours and err2 = inf."""
    seen = set()
    for _, fwd, bwd, s, alpha, beta in CASES:
        seen |= set(np.unique(fbo.fb_check(fwd, bwd, s, alpha, beta)[0]).tolist())
    assert seen == {0, 1, 2, 3, 4}
    f, b = _bwd_specials()
    st, e2 = fbo.fb_check(f, b, 1.0)
    assert (st[:5, 0::2] == FB_CONSISTENT).all()  # the special value sits on a zero-weight tap
    assert (st[:3, 1:-1:2] == FB_BWD_NONFINITE).all()  # inf / NaN read (the last column's target leaves the frame)
    assert (st[3:5, 1:-1:2] == FB_INCONSISTENT).all()  # huge finite read: err2 overflows
    assert np.isinf(e2[5:, :-1]).all() and (st[5:, :-1] == FB_INCONSISTENT).all()  # inf <= alpha*inf + beta does not pass
    f, b = _last_row_and_column()
    st, _ = fbo.fb_check(f, b, 1.0)
    assert st[1, 1] == FB_CONSISTENT and (st[::2] == FB_OUTSIDE).all() and (st[:, ::3] == FB_OUTSIDE).all()
    assert (st[1::2][:, [j for j in range(f.shape[1]) if j % 3]] != FB_OUTSIDE).all()
    f, _ = _half_to_even()
    U = np.rint(f[0, :, 0] * F32(256)).astype(int)  # k + 0.5 -> the even one of k, k + 1
    assert (U % 2 == 0).all() and set((U - np.arange(-6, 6)).tolist()) == {0, 1}


# ------------------------------------------------------------------------------------ CPU: semantics on the oracle
W_S, H_S = 256, 192


def square_scene(shift=6):
    """Static textured background, a differently textured 64x64 square that moves `shift` px to the right."""
    from oracle import oracle as O

    bg = O.make_frame(W_S, H_S, 0, 0, 8, 101)
    sq = O.make_frame(64, 64, 0, 0, 4, 202)
    x0, y0 = 96, 64
    prev, nxt = bg.copy(), bg.copy()
    prev[y0:y0 + 64, x0:x0 + 64] = sq
    nxt[y0:y0 + 64, x0 + shift:x0 + shift + 64] = sq
    return prev, nxt, x0, y0


def test_moving_square_marks_its_edges(oracle, fbo):
    """3 levels, window 9, bilinear warp, flow_scale 8/15.  Measured: background more than 16 px from the square 100 %
    CONSISTENT (0 % INCONSISTENT); the band from 6 px before to 12 px after each vertical edge of the square 73 %
    INCONSISTENT."""
    shift = 6
    prev, nxt, x0, y0 = square_scene(shift)
    _, _, st, _ = fbo.fb_pair(prev, nxt, 3, 9, oracle.WARP_BILINEAR, S815, 0.01, 0.5)
    ii, jj = np.meshgrid(np.arange(H_S), np.arange(W_S), indexing="ij")
    dx = np.maximum(np.maximum(x0 - jj, jj - (x0 + shift + 63)), 0)
    dy = np.maximum(np.maximum(y0 - ii, ii - (y0 + 63)), 0)
    far = np.maximum(dx, dy) > 16
    rows = (ii >= y0) & (ii < y0 + 64)
    band = rows & (((jj >= x0 - 6) & (jj < x0 + 12)) | ((jj >= x0 + 58) & (jj < x0 + 76)))
    assert (st[far] == FB_CONSISTENT).mean() >= 0.98
    assert (st[far] == FB_INCONSISTENT).mean() <= 0.02
    assert (st[band] == FB_INCONSISTENT).mean() >= 0.5


def test_flat_region_is_forward_nonfinite(oracle, fbo):
    """A constant 64x64 block in both frames: every window that sees only the block has det == 0 (Q3), so the total flow
    is NaN there.  Measured: all pixels 6 or more px inside the block (window 9 plus the 3x3 stencil) FWD_NONFINITE."""
    prev = oracle.make_frame(W_S, H_S, 0, 0, 8, 303)
    nxt = oracle.make_frame(W_S, H_S, 1.5, 0.5, 8, 303)
    prev[64:128, 64:128] = 77
    nxt[64:128, 64:128] = 77
    _, _, st, e2 = fbo.fb_pair(prev, nxt, 3, 9, oracle.WARP_BILINEAR, 1.0)
    assert (st[70:122, 70:122] == FB_FWD_NONFINITE).all()
    assert np.isnan(e2[70:122, 70:122]).all()


def test_global_shift_pushes_edge_columns_outside(oracle, fbo):
    """Everything moves 8 px right (4 levels, window 9, bilinear, flow_scale 8/15; measured median flow 8.0 px): the
    targets of the last columns leave the frame.  Measured: last 4 columns 85 % OUTSIDE, columns 16 .. w-16 0.4 %."""
    shift = 8
    prev = oracle.make_frame(W_S, H_S, 0, 0, 16, 404)
    nxt = oracle.make_frame(W_S, H_S, shift, 0, 16, 404)
    fwd, _, st, _ = fbo.fb_pair(prev, nxt, 4, 9, oracle.WARP_BILINEAR, S815)
    assert abs(np.nanmedian(fwd[:, 16:-32, 0]) * S815 - shift) < 0.25
    assert (st[:, W_S - shift // 2:] == FB_OUTSIDE).mean() >= 0.75
    assert (st[:, 16:W_S - 2 * shift] == FB_OUTSIDE).mean() <= 0.02


# ------------------------------------------------------------------------------------ CPU: ABI
def test_null_context_is_rejected_by_the_fb_entry_points():
    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    p = _lib.OfbParams(64, 64, 1, 9, 2, 1.0, 1)
    assert lib.ofb_fb_check_device(None, None, None, 64, 64, 1, 1.0, 0.01, 0.5, None, None, None) == _lib.OFB_ERR_INVALID
    assert b"NULL" in lib.ofb_last_error()
    assert lib.ofb_flow_pairs_fb_device(None, C.byref(p), None, None, 64, 4096, 0.01, 0.5, None, None, None, None,
                                        None) == _lib.OFB_ERR_INVALID
    assert lib.ofb_ctx_reserve_pairs_fb(None, C.byref(p)) == _lib.OFB_ERR_INVALID


# ------------------------------------------------------------------------------------ GPU
@pytest.fixture
def exact_ctx(ctx):
    from cuda_optical_flow_2_b200 import SOLVE_EXACT

    with solve(ctx, SOLVE_EXACT):
        yield ctx


@pytest.mark.gpu
@pytest.mark.parametrize("want_err2", [False, True])
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_fb_check_device_equals_oracle(ctx, fbo, case, want_err2):
    _, fwd, bwd, s, alpha, beta = case
    st, e2 = ctx.fb_check_device(to_device(fwd[None]), to_device(bwd[None]), s, alpha, beta, want_err2=want_err2)
    rst, re2 = fbo.fb_check(fwd, bwd, s, alpha, beta)
    assert_status_equal(st[0].cpu().numpy(), rst)
    if want_err2:
        assert_same_bits(e2[0].cpu().numpy(), re2, "err2")
    else:
        assert e2 is None


@pytest.mark.gpu
@pytest.mark.parametrize("want_err2", [False, True])
@pytest.mark.parametrize("w,h,n", [(37, 23, 3), (61, 17, 5), (64, 16, 4), (130, 7, 2)])
def test_fb_check_device_batch(ctx, fbo, w, h, n, want_err2):
    """Several pairs per launch; odd widths put rows off the 16-byte grid (the per-pixel path), w % 4 == 0 takes the
    wide loads and stores everywhere."""
    pairs = [_random(w, h, 100 + i) for i in range(n)]
    fwd = np.stack([p[0] for p in pairs])
    bwd = np.stack([p[1] for p in pairs])
    fwd[1, 0, :3] = np.nan
    bwd[-1, 1:3, 2:5] = np.inf
    st, e2 = ctx.fb_check_device(to_device(fwd), to_device(bwd), S815, want_err2=want_err2)
    rst, re2 = fbo.fb_check(fwd, bwd, S815)
    assert_status_equal(st.cpu().numpy(), rst)
    if want_err2:
        assert_same_bits(e2.cpu().numpy(), re2, "err2")


def _frames(oracle, w, h, n, seed=1234, dx=1.5, dy=-0.75):
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 4, seed + i) for i in range(n)])
    nexts = np.stack([oracle.make_frame(w, h, dx + 0.5 * i, dy, 4, seed + i) for i in range(n)])
    return prevs, nexts


@pytest.mark.gpu
@pytest.mark.parametrize("flow_scale", [1.0, S815])
@pytest.mark.parametrize("mode,w,h,levels,win,n", [
    (0, 96, 64, 3, 9, 2), (1, 96, 64, 3, 9, 2), (2, 96, 64, 3, 9, 2),
    (2, 101, 67, 1, 3, 2), (1, 75, 53, 3, 19, 1), (2, 128, 96, 4, 19, 1), (0, 133, 71, 4, 3, 1),
    (2, 160, 120, 3, 9, 3),  # even sizes: the shape on which ofb_flow_pairs_device composes level 0 on the fly
    (2, 203, 117, 3, 9, 2),
])
def test_flow_pairs_fb_device_equals_oracle(exact_ctx, oracle, fbo, mode, w, h, levels, win, n, flow_scale):
    from cuda_optical_flow_2_b200 import planar_to_device

    prevs, nexts = _frames(oracle, w, h, n)
    fwd, bwd, st, e2 = exact_ctx.flow_pairs_fb_device(planar_to_device(prevs), planar_to_device(nexts), w, levels, win,
                                                      warp_mode=mode, flow_scale=flow_scale, want_err2=True)
    fwd, bwd, st, e2 = (t.cpu().numpy() for t in (fwd, bwd, st, e2))
    for i in range(n):
        rf, rb, rst, re2 = fbo.fb_pair(prevs[i], nexts[i], levels, win, mode, flow_scale, 0.01, 0.5)
        assert_values_equal(fwd[i], rf, f"pair {i} forward total")
        assert_values_equal(bwd[i], rb, f"pair {i} backward total")
        assert_status_equal(st[i], rst, f"pair {i}")
        assert_same_bits(e2[i], re2, f"pair {i} err2")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["exact", "fast"])
@pytest.mark.parametrize("w,h,levels,win,n", [(160, 120, 3, 9, 3), (203, 117, 4, 15, 2), (96, 64, 1, 5, 2)])
def test_shared_pyramids_change_nothing(ctx, oracle, fbo, kind, w, h, levels, win, n):
    """Both totals are bit-identical to two ofb_flow_pairs_device calls (prev, next) and (next, prev), in both solve
    modes (SOLVE_FAST has no bit-exact oracle across levels); the status is the oracle's check of those totals."""
    import torch

    from cuda_optical_flow_2_b200 import SOLVE_EXACT, SOLVE_FAST, planar_to_device

    prevs, nexts = _frames(oracle, w, h, n, seed=77)
    p, q = planar_to_device(prevs), planar_to_device(nexts)
    with solve(ctx, SOLVE_FAST if kind == "fast" else SOLVE_EXACT):
        fwd, bwd, st, _ = ctx.flow_pairs_fb_device(p, q, w, levels, win, flow_scale=S815)
        ref_f = torch.empty((n, h, w, 2), dtype=torch.float32, device="cuda")
        ref_b = torch.empty_like(ref_f)
        ctx.flow_pairs_device(p, q, w, levels, win, flow_scale=S815, total_flow=ref_f)
        ctx.flow_pairs_device(q, p, w, levels, win, flow_scale=S815, total_flow=ref_b)
    ref_f, ref_b = ref_f.cpu().numpy(), ref_b.cpu().numpy()
    assert_values_equal(fwd.cpu().numpy(), ref_f, "forward total")
    assert_values_equal(bwd.cpu().numpy(), ref_b, "backward total")
    assert_status_equal(st.cpu().numpy(), fbo.fb_check(ref_f, ref_b, S815)[0])


@pytest.mark.gpu
def test_swapping_the_frames_swaps_the_totals(exact_ctx, oracle):
    from cuda_optical_flow_2_b200 import planar_to_device

    w, h = 141, 90
    prevs, nexts = _frames(oracle, w, h, 2, seed=5)
    p, q = planar_to_device(prevs), planar_to_device(nexts)
    f1, b1, _, _ = exact_ctx.flow_pairs_fb_device(p, q, w, 3, 9)
    f2, b2, _, _ = exact_ctx.flow_pairs_fb_device(q, p, w, 3, 9)
    for a, b in ((f1, b2), (b1, f2)):
        assert np.array_equal(a.cpu().numpy().view(np.uint32), b.cpu().numpy().view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["zero_to_full", "zeros", "full"])
@pytest.mark.parametrize("w,h,levels,win", [(96, 64, 3, 9), (67, 45, 2, 19)])
def test_adversarial_content_status(exact_ctx, oracle, fbo, name, w, h, levels, win):
    """The pair 0 -> 255 and flat frames (det == 0 everywhere: every total flow NaN) give the oracle's status."""
    from cuda_optical_flow_2_b200 import planar_to_device

    prev, nxt = PAIRS[name](w, h)
    fwd, bwd, st, e2 = exact_ctx.flow_pairs_fb_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, levels,
                                                      win, want_err2=True)
    rf, rb, rst, re2 = fbo.fb_pair(prev, nxt, levels, win, oracle.WARP_BILINEAR, 1.0, 0.01, 0.5)
    assert_status_equal(st[0].cpu().numpy(), rst)
    assert_same_bits(e2[0].cpu().numpy(), re2, "err2")


@pytest.mark.gpu
def test_cuda_graph_replay(exact_ctx, oracle):
    """After reserve_pairs_fb, one captured flow_pairs_fb_device call replays on new frames written into the same input
    buffers and gives the eager result."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, levels, win, n = 160, 96, 3, 9, 2
    exact_ctx.reserve_pairs_fb(w, h, levels, win, n)
    frames = [_frames(oracle, w, h, n, seed=900 + 10 * r, dx=0.5 + r) for r in range(3)]
    p, q = planar_to_device(frames[0][0]), planar_to_device(frames[0][1])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        exact_ctx.flow_pairs_fb_device(p, q, w, levels, win, want_err2=True, stream=side.cuda_stream)  # warm-up
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = exact_ctx.flow_pairs_fb_device(p, q, w, levels, win, want_err2=True,
                                             stream=torch.cuda.current_stream().cuda_stream)
    for prevs, nexts in frames[1:]:
        p.copy_(planar_to_device(prevs))
        q.copy_(planar_to_device(nexts))
        g.replay()
        torch.cuda.synchronize()
        eager = exact_ctx.flow_pairs_fb_device(planar_to_device(prevs), planar_to_device(nexts), w, levels, win, want_err2=True)
        torch.cuda.synchronize()
        for got, ref in zip(out, eager):
            g_np, r_np = got.cpu().numpy(), ref.cpu().numpy()
            assert np.array_equal(g_np.view(np.uint8), r_np.view(np.uint8))


@pytest.mark.gpu
def test_profile_record_around_the_check(ctx):
    from cuda_optical_flow_2_b200 import PROFILE_FB_CHECK

    fwd, bwd = _random(64, 32, 3)
    ctx.profile_enable(True)
    try:
        ctx.fb_check_device(to_device(fwd[None]), to_device(bwd[None]))
        ms, n = ctx.profile_read(PROFILE_FB_CHECK)
    finally:
        ctx.profile_enable(False)
    assert n == 1 and ms > 0


@pytest.mark.gpu
def test_bad_arguments_are_rejected(ctx):
    import torch

    from cuda_optical_flow_2_b200 import OfbError, _lib, planar_to_device

    lib = _lib.load()
    w, h, n = 64, 48, 1
    f = torch.zeros((n, h, w, 2), dtype=torch.float32, device="cuda")
    st = torch.zeros((n, h, w), dtype=torch.uint8, device="cuda")
    with pytest.raises(OfbError, match="alpha"):
        ctx.fb_check_device(f, f, alpha=-0.01)
    with pytest.raises(OfbError, match="beta"):
        ctx.fb_check_device(f, f, beta=float("nan"))
    for s in (0.0, -1.0, float("inf")):
        with pytest.raises(OfbError, match="flow_scale"):
            ctx.fb_check_device(f, f, flow_scale=s)
    inv = _lib.OFB_ERR_INVALID
    call = lambda fw, bw, status, err2=None: lib.ofb_fb_check_device(ctx._h, fw, bw, w, h, n, 1.0, 0.01, 0.5, status, err2, None)
    assert call(f.data_ptr(), f.data_ptr(), None) == inv
    assert call(f.data_ptr() + 4, f.data_ptr(), st.data_ptr()) == inv  # fwd 4-byte aligned only
    assert call(f.data_ptr(), f.data_ptr() + 4, st.data_ptr()) == inv
    assert call(f.data_ptr(), f.data_ptr(), st.data_ptr(), f.data_ptr() + 2) == inv  # err2 misaligned
    assert call(None, f.data_ptr(), st.data_ptr()) == inv
    frame = planar_to_device(np.zeros((n, h, w), np.uint8))
    for s in (0.0, -1.0):
        with pytest.raises(OfbError, match="flow_scale"):
            ctx.flow_pairs_fb_device(frame, frame, w, 3, 9, flow_scale=s)
    with pytest.raises(OfbError, match="alpha"):
        ctx.flow_pairs_fb_device(frame, frame, w, 3, 9, alpha=-1.0)
    p = _lib.OfbParams(w, h, 3, 9, 2, 1.0, n)
    fb = lambda fw, bw, status: lib.ofb_flow_pairs_fb_device(ctx._h, C.byref(p), frame.data_ptr(), frame.data_ptr(), 64, 64 * h,
                                                             0.01, 0.5, fw, bw, status, None, None)
    assert fb(f.data_ptr(), f.data_ptr(), None) == inv
    assert fb(None, f.data_ptr(), st.data_ptr()) == inv
    assert fb(f.data_ptr() + 4, f.data_ptr(), st.data_ptr()) == inv
    torch.cuda.synchronize()
