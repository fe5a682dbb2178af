"""Shi-Tomasi corners for the point tracker (ofb_min_eig_map_device, ofb_detect_corners_device).

The rule is pinned in include/ofb200.h: exact int32 structure-tensor sums of the tracker's Sobel fields, the smaller
eigenvalue in double with every operation rounded on its own, the strict key-order local maximum and OpenCV's sequential
greedy selection.  So the CUDA kernels (csrc/corners.cu) and the C restatement in tests/corner_oracle.c (compiled here into a
temporary directory) must agree bit for bit.

CPU tests (no mark): the restatement's score against exact arithmetic (numpy/scipy sums, 50-digit decimal eigenvalue), its
selection against a plain-Python greedy on crafted maps, its meaning on bright rectangles, and the tie to the tracker's
LOW_TEXTURE decision (tests/track_oracle.c).
GPU tests: the kernels against the restatement over windows, sizes, layouts, batches, content and parameters; CUDA graph
capture of detection followed by tracking; detect-then-track end to end; argument refusals; the profile record.
"""
import decimal
import math

import numpy as np
import pytest

from cuda_optical_flow_2_b200 import align_up
from support import (F32, PT_LOW_TEXTURE, PT_OUTSIDE, PT_TRACKED, S815, assert_same_bits, content, cro, device_frames,  # noqa: F401
                     exact_sums, plain_greedy, tro)

WINS = list(range(3, 20, 2))


# ------------------------------------------------------------------------------------ CPU: score vs exact arithmetic
@pytest.mark.parametrize("win", WINS)
@pytest.mark.parametrize("kind", ["textured", "stripes", "isotropic", "noise"])
def test_score_is_l1_over_win2_within_one_ulp(cro, win, kind):
    w, h = 31, 23
    img = content(kind, w, h, win)
    got = cro.score(img, win)
    A, D, B = exact_sums(img, win)
    assert max(A.max(), D.max(), np.abs(B).max()) < 2 ** 31
    decimal.getcontext().prec = 50
    n2 = decimal.Decimal(win * win)
    for y in range(h):
        for x in range(w):
            a, d, b = int(A[y, x]), int(D[y, x]), int(B[y, x])
            s = decimal.Decimal(a + d)
            disc = decimal.Decimal((a - d) ** 2 + 4 * b * b)
            lam = (s - disc.sqrt()) / 2 / n2
            ref = float(lam)
            g = float(got[y, x])
            if a * d - b * b == 0:
                assert g == 0.0, (x, y, g)
                continue
            ulp = float(np.spacing(F32(ref)))
            assert abs(g - ref) <= ulp, (x, y, g, ref)
    if kind == "stripes":  # the zero padding makes gy at the top and bottom rows; inside, every window is one-dimensional
        m = win // 2 + 1
        assert (got[m:h - m, m:w - m] == 0).all()


# ------------------------------------------------------------------------------------ CPU: selection vs a plain greedy
def assert_selection(got, acc, max_corners):
    corners, scores, n = got
    assert n == len(acc)
    if n:
        assert np.array_equal(corners[:n], np.array([(x, y) for x, y, _ in acc], F32))
        assert np.array_equal(scores[:n].view(np.uint32), np.array([s for _, _, s in acc], F32).view(np.uint32))
    assert np.isnan(corners[n:]).all() and np.isnan(scores[n:]).all()


def crafted_maps():
    """(name, map, win): a period-2 checkerboard plateau (the densest candidates), equal-score ties, random maps."""
    rng = np.random.default_rng(5)
    maps = []
    yy, xx = np.mgrid[0:40, 0:52]
    maps.append(("checker_plateau", np.where((xx + yy) % 2 == 0, F32(3.0), F32(1.0)), 3))
    maps.append(("flat_plateau", np.full((30, 33), F32(2.5)), 5))
    maps.append(("ties", rng.integers(1, 4, (37, 41)).astype(F32), 3))
    maps.append(("random", rng.random((45, 38)).astype(F32), 7))
    maps.append(("sparse", (rng.random((50, 60)) * (rng.random((50, 60)) < 0.2)).astype(F32), 3))
    return maps


SELECT_CASES = [dict(max_corners=10_000, quality_level=0.0, min_distance=d) for d in
                (0.0, 1.0, float(F32(math.sqrt(2))), 1.5, 10.0, 500.0)] + [
    dict(max_corners=7, quality_level=0.01, min_distance=2.0), dict(max_corners=1, quality_level=0.0, min_distance=0.0),
    dict(max_corners=10_000, quality_level=1.0, min_distance=0.0), dict(max_corners=10_000, quality_level=0.5, min_distance=3.0),
    dict(max_corners=50, quality_level=0.0, min_distance=2.5, min_score=0.3), dict(max_corners=50, quality_level=0.0,
                                                                                  min_distance=0.0, min_score=1e9)]


@pytest.mark.parametrize("case", range(len(SELECT_CASES)))
def test_selection_equals_plain_greedy(cro, case):
    kw = SELECT_CASES[case]
    for name, score, win in crafted_maps():
        got = cro.select(score, win, **kw)
        assert_selection(got, plain_greedy(score, win, kw["max_corners"], kw["quality_level"], kw["min_distance"],
                                           kw.get("min_score", 0.0)), kw["max_corners"])
        if kw.get("min_score", 0.0) > 1e6:
            assert got[2] == 0


def test_selection_boundaries(cro):
    """Frames of size 2m (no interior: 0 corners) and 2m+1 (one interior pixel); the checkerboard plateau's candidates are
    never 8-adjacent, and their number stays within the bound that sizes the workspace."""
    win = 5
    m = win // 2 + 1
    for size, want in ((2 * m, 0), (2 * m + 1, 1)):
        score = np.ones((size, size), F32)
        c, s, n = cro.select(score, win, 4, quality_level=0.0, min_distance=0.0)
        assert n == want and np.isnan(c[n:]).all() and np.isnan(s[n:]).all()
    yy, xx = np.mgrid[0:40, 0:52]
    score = np.where((xx + yy) % 2 == 0, F32(3.0), F32(1.0))
    c, _, n = cro.select(score, 3, 10_000, quality_level=0.0, min_distance=0.0)
    pts = c[:n].astype(int)
    d = np.abs(pts[:, None] - pts[None]).max(-1)
    np.fill_diagonal(d, 99)
    assert d.min() >= 2  # no two candidates are 8-adjacent
    iw, ih = 52 - 2 * 2, 40 - 2 * 2
    assert n <= ((iw + 1) // 2) * ((ih + 1) // 2)


# ------------------------------------------------------------------------------------ CPU: meaning
def rectangles(w=160, h=120):
    img = np.full((h, w), 20, np.uint8)
    rects = [(20, 15, 55, 45), (80, 20, 130, 60), (30, 70, 70, 105), (95, 75, 140, 100)]  # x0, y0, x1, y1 (exclusive)
    for x0, y0, x1, y1 in rects:
        img[y0:y1, x0:x1] = 220
    corners = [(x, y) for x0, y0, x1, y1 in rects for x, y in ((x0, y0), (x1 - 1, y0), (x0, y1 - 1), (x1 - 1, y1 - 1))]
    return img, np.array(corners, float)


@pytest.mark.parametrize("win,tol", [(3, 1), (5, 1), (9, 3)])
def test_rectangle_corners_are_found_and_nothing_else(cro, win, tol):
    """Every corner pixel of a bright rectangle is found within 1 px (Chebyshev) at windows 3 and 5, and nothing else is
    found.  A larger window moves the maximum of the smaller eigenvalue inside the rectangle, along the diagonal: 3 px at
    window 9 (as in any Shi-Tomasi detector)."""
    img, truth = rectangles()
    c, _, n = cro.detect(img, win, 100, quality_level=0.05, min_distance=5.0)
    pts = c[:n].astype(float)
    d = np.abs(pts[:, None] - truth[None]).max(-1)  # Chebyshev distance, detections x true corners
    assert (d.min(0) <= tol).all(), d.min(0)  # every rectangle corner found
    assert (d.min(1) <= tol).all(), pts[d.min(1) > tol]  # nothing on an edge or a flat area
    assert n == len(truth)


# ------------------------------------------------------------------------------------ CPU: the tie to the tracker
@pytest.mark.parametrize("win", [3, 9, 19])
def test_score_is_the_trackers_low_texture_threshold(cro, tro, oracle, win):
    """levels = 1, iters = 1, integer points at every interior pixel with score > 0: min_eig = score * (1 - 1e-5) never
    gives LOW_TEXTURE, score * (1 + 1e-5) always does."""
    w, h = 34, 28
    img = content("natural", w, h, win)
    nxt = np.roll(img, 1, 1)
    score = cro.score(img, win)
    m = win // 2 + 1
    checked = 0
    for y in range(m, h - m):
        for x in range(m, w - m):
            s = float(score[y, x])
            if s <= 0:
                continue
            pt = np.array([[x, y]], F32)
            _, lo = tro.track(img, nxt, 1, win, pt, iters=1, eps=0.0, min_eig=s * (1 - 1e-5))
            _, hi = tro.track(img, nxt, 1, win, pt, iters=1, eps=0.0, min_eig=s * (1 + 1e-5))
            assert lo[0] != PT_LOW_TEXTURE and hi[0] == PT_LOW_TEXTURE, (x, y, s, lo, hi)
            checked += 1
    assert checked > 50


# ------------------------------------------------------------------------------------ CPU: ABI
def test_null_context_is_rejected():
    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    assert lib.ofb_min_eig_map_device(None, None, 64, 4096, 64, 64, 1, 3, None, None) == _lib.OFB_ERR_INVALID
    assert lib.ofb_detect_corners_device(None, None, 64, 4096, 64, 64, 1, 3, 10, 0.01, 10.0, 0.0, None, None, None,
                                         None) == _lib.OFB_ERR_INVALID
    assert lib.ofb_ctx_reserve_corners(None, 64, 64, 1, 3, 10) == _lib.OFB_ERR_INVALID
    assert b"NULL" in lib.ofb_last_error()


# ------------------------------------------------------------------------------------ GPU
def _map(ctx, frames, imgs, win):
    import torch

    from cuda_optical_flow_2_b200 import _lib

    (dev, pitch, stride), (n, h, w) = frames, imgs.shape
    out = torch.empty((n, h, w), dtype=torch.float32, device=dev.device)
    _lib.check(_lib.load().ofb_min_eig_map_device(ctx._h, dev.data_ptr(), pitch, stride, w, h, n, win, out.data_ptr(), None))
    return out.cpu().numpy()


def _detect(ctx, frames, imgs, win, max_corners, quality_level=0.01, min_distance=10.0, min_score=0.0):
    import torch

    from cuda_optical_flow_2_b200 import _lib

    (dev, pitch, stride), (n, h, w) = frames, imgs.shape
    corners = torch.empty((n, max_corners, 2), dtype=torch.float32, device=dev.device)
    scores = torch.empty((n, max_corners), dtype=torch.float32, device=dev.device)
    counts = torch.empty((n,), dtype=torch.int32, device=dev.device)
    _lib.check(_lib.load().ofb_detect_corners_device(ctx._h, dev.data_ptr(), pitch, stride, w, h, n, win, max_corners,
                                                     quality_level, min_distance, min_score, corners.data_ptr(),
                                                     scores.data_ptr(), counts.data_ptr(), None))
    return corners.cpu().numpy(), scores.cpu().numpy(), counts.cpu().numpy()


def _check_detect(cro, imgs, got, win, max_corners, **kw):
    corners, scores, counts = got
    for i, img in enumerate(imgs):
        rc, rs, rn = cro.detect(img, win, max_corners, **kw)
        assert counts[i] == rn, (i, counts[i], rn)
        assert_same_bits(corners[i], rc, f"image {i} corners")
        assert_same_bits(scores[i], rs, f"image {i} scores")


KINDS = ["zeros", "full", "checker", "stripes", "noise", "natural", "textured", "isotropic"]


@pytest.mark.gpu
@pytest.mark.parametrize("win", WINS)
def test_kernel_equals_restatement_windows_and_content(ctx, cro, win):
    """Every content kind on an odd-sized frame, in one batch with pitch > w, image stride > h * pitch and 0xFF padding
    around every image."""
    w, h = 67, 45
    imgs = np.stack([content(k, w, h, i) for i, k in enumerate(KINDS)])
    dev = device_frames(imgs, 96, 96 * (h + 3), 0xFF)
    got = _map(ctx, dev, imgs, win)
    for i in range(len(imgs)):
        assert_same_bits(got[i], cro.score(imgs[i], win), f"{KINDS[i]} map")
    for kw in (dict(quality_level=0.01, min_distance=10.0), dict(quality_level=0.0, min_distance=0.0),
               dict(quality_level=0.0, min_distance=1.5)):
        _check_detect(cro, imgs, _detect(ctx, dev, imgs, win, 300, **kw), win, 300, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 1), (2, 3), (7, 7), (8, 9), (33, 1), (1, 40), (100, 13), (257, 131), (1921, 1081)])
def test_kernel_equals_restatement_sizes(ctx, cro, w, h):
    """Sizes around the 32 x 32 tile and the interior limit 2m+1, windows 3 and 9 (the large one at window 3 only)."""
    for win in ([3, 9] if w * h < 100_000 else [3]):
        imgs = np.stack([content("natural", w, h, 3), content("noise", w, h, 4)])
        dev = device_frames(imgs, align_up(w, 16))
        got = _map(ctx, dev, imgs, win)
        for i in range(2):
            assert_same_bits(got[i], cro.score(imgs[i], win), f"{w}x{h} win {win} map")
        _check_detect(cro, imgs, _detect(ctx, dev, imgs, win, 500, quality_level=0.0, min_distance=3.0), win, 500,
                      quality_level=0.0, min_distance=3.0)


@pytest.mark.gpu
def test_kernel_equals_restatement_4k(ctx, cro):
    w, h, win = 3840, 2160, 3
    img = content("textured", w, h, 7)[None]
    dev = device_frames(img, align_up(w, 16))
    assert_same_bits(_map(ctx, dev, img, win)[0], cro.score(img[0], win), "4K map")
    for kw in (dict(quality_level=0.01, min_distance=10.0), dict(quality_level=0.0, min_distance=0.0)):
        _check_detect(cro, img, _detect(ctx, dev, img, win, 16384, **kw), win, 16384, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 3, 64, 65535])
def test_kernel_equals_restatement_batches(ctx, cro, n):
    w, h, win = 24, 19, 5
    base = np.stack([content(k, w, h, i) for i, k in enumerate(KINDS)])
    imgs = np.stack([np.roll(base[i % len(base)], i // len(base), 1) for i in range(n)])
    dev = device_frames(imgs, align_up(w, 16))
    check = sorted(set([0, n // 2, n - 1] + list(range(min(n, 16)))))
    got_map = _map(ctx, dev, imgs, win)
    got = _detect(ctx, dev, imgs, win, 40, quality_level=0.0, min_distance=2.0)
    for i in check:
        assert_same_bits(got_map[i], cro.score(imgs[i], win), f"image {i} map")
    _check_detect(cro, imgs[check], tuple(g[check] for g in got), win, 40, quality_level=0.0, min_distance=2.0)


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(SELECT_CASES)))
def test_kernel_equals_restatement_parameters(ctx, cro, case):
    """Every parameter case of the CPU selection tests, on images (the map is the kernel's, compared first)."""
    kw = dict(SELECT_CASES[case])
    mc = kw.pop("max_corners")
    w, h = 90, 70
    imgs = np.stack([content("checker", w, h), content("natural", w, h, 1), content("textured", w, h, 2),
                     content("noise", w, h, 3)])
    dev = device_frames(imgs, align_up(w, 16))
    _check_detect(cro, imgs, _detect(ctx, dev, imgs, 3, mc, **kw), 3, mc, **kw)


@pytest.mark.gpu
def test_conflict_chains(ctx, cro):
    """Candidates on a line 2 px apart with decreasing score and min_distance 2.5: each conflicts with the next, so the
    in-chunk resolution is one round per link (the sequential worst case), and only every other one is kept."""
    import torch

    w, h, win = 1200, 12, 3
    img = np.zeros((h, w), np.uint8)
    img[6, 4:w - 4:2] = 255  # isolated bright pixels along a row
    dev = device_frames(img[None], align_up(w, 16))
    got = _detect(ctx, dev, img[None], win, 4000, quality_level=0.0, min_distance=2.5)
    _check_detect(cro, img[None], got, win, 4000, quality_level=0.0, min_distance=2.5)
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_cuda_graph_detect_then_track(ctx, cro, oracle):
    """After reserve_corners and reserve_pairs, detection followed by tracking of the detected corners is captured as one
    graph; replays on new frames written into the captured buffers equal eager calls."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, n, win, mc, levels = 160, 120, 2, 7, 200, 3
    ctx.reserve_corners(w, h, n, win, mc)
    ctx.reserve_pairs(w, h, levels, 9, n)
    frames = [(np.stack([oracle.make_frame(w, h, 0, 0, 4, 50 * r + i) for i in range(n)]),
               np.stack([oracle.make_frame(w, h, 0.7, -0.4, 4, 50 * r + i) for i in range(n)])) for r in range(3)]
    p, q = planar_to_device(frames[0][0]), planar_to_device(frames[0][1])

    def step(stream):
        c, s, k = ctx.detect_corners_device(p, w, win, mc, 0.01, 5.0, stream=stream)
        f, st = ctx.track_points_device(p, q, w, levels, 9, c, S815, stream=stream)
        return c, s, k, f, st

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step(side.cuda_stream)  # warm-up
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = step(torch.cuda.current_stream().cuda_stream)
    for prevs, nexts in frames[1:]:
        p.copy_(planar_to_device(prevs))
        q.copy_(planar_to_device(nexts))
        g.replay()
        torch.cuda.synchronize()
        eager = step(0)
        torch.cuda.synchronize()
        for got, ref in zip(out, eager):
            assert np.array_equal(got.cpu().numpy().view(np.uint8), ref.cpu().numpy().view(np.uint8))
        c, s, k = (t.cpu().numpy() for t in out[:3])
        _check_detect(cro, prevs, (c, s, k), win, mc, quality_level=0.01, min_distance=5.0)


@pytest.mark.gpu
def test_detect_then_track_end_to_end(ctx, oracle):
    """Detect on prev, track to a sub-pixel shift of it: at least 99 % of the detected points TRACKED, median error below
    0.05 px, every padding slot OUTSIDE."""
    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, dx, dy = 320, 240, 1.37, -0.62
    prev = oracle.make_frame(w, h, 0, 0, 4, 77)
    nxt = oracle.make_frame(w, h, dx, dy, 4, 77)
    p, q = planar_to_device(prev[None]), planar_to_device(nxt[None])
    corners, _, counts = ctx.detect_corners_device(p, w, 9, 2000, 0.01, 6.0)
    flow, st = ctx.track_points_device(p, q, w, 3, 9, corners, S815, iters=30, eps=0.0)
    k = int(counts.cpu()[0])
    flow, st = flow.cpu().numpy()[0], st.cpu().numpy()[0]
    assert 100 < k < 2000
    assert (st[k:] == PT_OUTSIDE).all()
    ok = st[:k] == PT_TRACKED
    assert ok.mean() >= 0.99, ok.mean()
    err = np.hypot(S815 * flow[:k][ok, 0] - dx, S815 * flow[:k][ok, 1] - dy)
    assert np.median(err) < 0.05, np.median(err)


@pytest.mark.gpu
def test_profile_record(ctx):
    from cuda_optical_flow_2_b200 import PROFILE_CORNERS, planar_to_device

    dev = planar_to_device(content("natural", 96, 64, 1)[None])
    ctx.profile_enable(True)
    try:
        ctx.detect_corners_device(dev, 96, 5, 100)
        ctx.min_eig_map_device(dev, 96, 5)
        ms, n = ctx.profile_read(PROFILE_CORNERS)
    finally:
        ctx.profile_enable(False)
    assert n == 2 and ms > 0


@pytest.mark.gpu
def test_refusals_leave_outputs_untouched(ctx):
    import torch

    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    w, h, n, mc = 64, 48, 2, 10
    img = torch.zeros((n, h, 64), dtype=torch.uint8, device="cuda")
    corners = torch.full((n, mc, 2), 7.0, dtype=torch.float32, device="cuda")
    scores = torch.full((n, mc), 7.0, dtype=torch.float32, device="cuda")
    counts = torch.full((n,), 7, dtype=torch.int32, device="cuda")
    smap = torch.full((n, h, w), 7.0, dtype=torch.float32, device="cuda")
    inv, uns = _lib.OFB_ERR_INVALID, _lib.OFB_ERR_UNSUPPORTED

    def detect(im=img.data_ptr(), pitch=64, stride=64 * h, ww=w, hh=h, nn=n, win=5, max_corners=mc, ql=0.01, md=10.0, ms=0.0,
               c=corners.data_ptr(), s=scores.data_ptr(), k=counts.data_ptr()):
        return lib.ofb_detect_corners_device(ctx._h, im, pitch, stride, ww, hh, nn, win, max_corners, ql, md, ms, c, s, k, None)

    def score_map(im=img.data_ptr(), pitch=64, stride=64 * h, ww=w, hh=h, nn=n, win=5, out=smap.data_ptr()):
        return lib.ofb_min_eig_map_device(ctx._h, im, pitch, stride, ww, hh, nn, win, out, None)

    torch.cuda.synchronize()
    before = ctx.launch_count
    nan, inf = float("nan"), float("inf")
    bad = [(dict(max_corners=0), inv), (dict(max_corners=(1 << 20) + 1), inv), (dict(ql=-0.01), inv), (dict(ql=1.01), inv),
           (dict(ql=nan), inv), (dict(md=-1.0), inv), (dict(md=inf), inv), (dict(md=nan), inv), (dict(ms=-1.0), inv),
           (dict(ms=inf), inv), (dict(nn=0), inv), (dict(nn=65536), inv), (dict(ww=0), inv), (dict(hh=0), inv),
           (dict(ww=65536, hh=32768, pitch=65536, stride=65536 * 32768), inv), (dict(win=4), uns), (dict(win=21), uns),
           (dict(win=1), uns), (dict(im=None), inv), (dict(c=None), inv), (dict(k=None), inv), (dict(pitch=32), inv),
           (dict(stride=64 * h - 16), inv), (dict(c=corners.data_ptr() + 4), inv), (dict(s=scores.data_ptr() + 2), inv),
           (dict(k=counts.data_ptr() + 2), inv)]
    for kw, code in bad:
        assert detect(**kw) == code, (kw, lib.ofb_last_error())
    for kw, code in [(dict(nn=0), inv), (dict(nn=65536), inv), (dict(win=8), uns), (dict(im=None), inv), (dict(out=None), inv),
                     (dict(out=smap.data_ptr() + 2), inv), (dict(pitch=32), inv), (dict(ww=65536, hh=32768), inv)]:
        assert score_map(**kw) == code, (kw, lib.ofb_last_error())
    torch.cuda.synchronize()
    assert ctx.launch_count == before
    assert (corners == 7.0).all() and (scores == 7.0).all() and (counts == 7).all() and (smap == 7.0).all()
    assert lib.ofb_ctx_reserve_corners(ctx._h, w, h, 0, 5, mc) == inv
    assert lib.ofb_ctx_reserve_corners(ctx._h, w, h, n, 5, 0) == inv
    assert detect(max_corners=0) == inv and b"max_corners" in lib.ofb_last_error()
    assert detect(s=None) == 0  # scores are optional
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="imgs"):
        ctx.detect_corners_device(img.cpu(), w, 5, mc)
