"""The point tracker (ofb_track_points_device, csrc/track.cu) against references that do not restate its fixed-point rule,
on worst-case content, on caller frame layouts and at the argument limits of include/ofb200.h.

test_track_points.py ties the kernel to tests/track_oracle.c, a C restatement of the same pinned rule: a misunderstanding
shared by both would pass there.  Here:
  * an independent float64 KLT (numpy / scipy): textbook pyramidal Lucas-Kanade on the same pyramid, with the level-k
    position x / 2^k, exact bilinear sampling, float64 sums and solve and a real square root.  The pinned rule (restatement
    on the CPU, kernel on the GPU) must agree with it on converged, well-textured points within 0.01 px at flow_scale
    8/15 and 0.02 px at flow_scale 1;
  * numpy int64 window sums at the points of the worst-case content of test_adversarial_content (the header's "exact in
    int32" claim, and that the content really comes near 2^31);
  * an exact model of lam < min_eig (Python integers and fractions.Fraction) against the pinned eigenvalue test;
  * the kernel on caller frames with 16-byte pitch, a larger image stride and 0xFF padding, at levels 5-8, 64 iterations,
    flow scales 3 and 0.01, 2^24 points and 65535 pairs.
"""
import ctypes as C
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest
from scipy.ndimage import map_coordinates

from test_adversarial_content import PAIRS, vertical_stripes
from test_track_points import (F32, PT_LOW_TEXTURE, PT_NONFINITE, PT_OUTSIDE, PT_TRACKED, S815, TrackOracle,
                               assert_same_bits, assert_status_equal, border_points, random_points)

WINDOWS = [3, 5, 7, 9, 11, 13, 15, 17, 19]
I32 = 2 ** 31


@pytest.fixture(scope="session")
def tro(oracle, tmp_path_factory):
    so = str(tmp_path_factory.mktemp("track_oracle_ref") / "libtrackoracle.so")
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "track_oracle.c")
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra",
                           "-shared", "-o", so, src, "-lm"])
    return TrackOracle(so, oracle)


# ------------------------------------------------------------------------------------ references
def fields(img, dtype=np.float64):
    """Dx, Dy and Dt = [1 2 1; 2 3 2; 1 2 1] (*) img as correlations with zero padding."""
    h, w = img.shape
    p = np.pad(img.astype(dtype), 1)

    def c(dy, dx):
        return p[1 + dy:1 + dy + h, 1 + dx:1 + dx + w]

    ix = (c(-1, 1) + 2 * c(0, 1) + c(1, 1)) - (c(-1, -1) + 2 * c(0, -1) + c(1, -1))
    iy = (c(1, -1) + 2 * c(1, 0) + c(1, 1)) - (c(-1, -1) + 2 * c(-1, 0) + c(-1, 1))
    dt = (c(-1, -1) + c(-1, 1) + c(1, -1) + c(1, 1)) + 2 * (c(-1, 0) + c(0, -1) + c(0, 1) + c(1, 0)) + 3 * c(0, 0)
    return ix, iy, dt


def bilinear64(F, X, Y):
    """Exact bilinear interpolation of F at (X, Y), F = 0 outside."""
    return map_coordinates(np.pad(F, 2), [Y + 2, X + 2], order=1, mode="constant", cval=0.0, prefilter=False)


def klt64(oracle, prev, nxt, levels, win, pts, s, iters=30, eps=0.0):
    """Textbook pyramidal LK in float64 on oracle.gauss_pyramid's levels.  Returns (flow (m, 2), lam (m,) of the level-0
    window, last |s * update| px (m,)); NaN flow for starts outside the frame and for det == 0."""
    pp, pn = oracle.gauss_pyramid(prev, levels), oracle.gauss_pyramid(nxt, levels)
    h, w = prev.shape
    R = win // 2
    oy, ox = (o.ravel() for o in np.mgrid[-R:R + 1, -R:R + 1].astype(np.float64))
    x, y = pts[:, 0].astype(np.float64), pts[:, 1].astype(np.float64)
    live = np.isfinite(x) & np.isfinite(y) & (x >= 0) & (x <= w - 1) & (y >= 0) & (y <= h - 1)
    d = np.zeros((len(pts), 2))
    last = np.full(len(pts), np.inf)
    for k in range(levels - 1, -1, -1):
        ix, iy, sp = fields(pp[k])
        sn = fields(pn[k])[2]
        X, Y = x[live, None] / 2 ** k + ox, y[live, None] / 2 ** k + oy
        gx, gy, s0 = (bilinear64(f, X, Y).reshape(X.shape) for f in (ix, iy, sp))
        a, dd, b = (gx * gx).sum(1), (gy * gy).sum(1), (gx * gy).sum(1)
        det = a * dd - b * b
        dl = d[live]
        run = np.ones(len(dl), bool)
        with np.errstate(divide="ignore", invalid="ignore"):
            for _ in range(iters):
                if not run.any():
                    break
                It = bilinear64(sn, X[run] + s * dl[run, :1], Y[run] + s * dl[run, 1:]).reshape(-1, win * win) - s0[run]
                tx, ty = (gx[run] * It).sum(1), (gy[run] * It).sum(1)
                u = (b[run] * ty - dd[run] * tx) / det[run]
                v = (b[run] * tx - a[run] * ty) / det[run]
                dl[run] += np.stack([u, v], 1)
                step = np.maximum(np.abs(s * u), np.abs(s * v))
                lr = last[live]
                lr[run] = step
                last[live] = lr
                run[run] = np.isfinite(step) & ~(step < eps)
        d[live] = dl
        if k:
            d *= 2
    lam = np.full(len(pts), np.nan)
    lam[live] = ((a + dd) - np.sqrt((a - dd) ** 2 + 4 * b * b)) / (2 * win * win)
    d[~live] = np.nan
    return d, lam, last


def render_affine(w, h, A, t, seed, cell=4):
    """Smooth random texture (bilinear over a random grid of cell px) sampled at A (x, y) + t, rounded to u8."""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 256, (h // cell + 60, w // cell + 60)).astype(np.float64)
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float64)
    X, Y = A[0, 0] * xs + A[0, 1] * ys + t[0], A[1, 0] * xs + A[1, 1] * ys + t[1]
    v = map_coordinates(g, [Y / cell + 30, X / cell + 30], order=1, prefilter=False)
    return np.clip(np.rint(v), 0, 255).astype(np.uint8)


def affine_pair(w, h, M, seed):
    """prev, next whose content moves by the linear map M about the frame centre: next(x) = prev(M^-1 (x - c) + c)."""
    c = np.array([w / 2, h / 2])
    Minv = np.linalg.inv(M)
    return render_affine(w, h, np.eye(2), np.zeros(2), seed), render_affine(w, h, Minv, c - Minv @ c, seed)


def rotzoom(deg, zoom):
    th = np.deg2rad(deg)
    return zoom * np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])


def motion_pair(oracle, motion, w, h, amount, seed):
    if motion == "shift":
        return oracle.make_frame(w, h, 0, 0, 4, seed), oracle.make_frame(w, h, *amount, 4, seed)
    return affine_pair(w, h, motion_matrix(motion, amount), seed)


def motion_matrix(motion, amount):
    return rotzoom(*amount) if motion == "rotzoom" else np.array([[1.0, amount], [0.0, 1.0]])  # shear: x += a (y - cy)


def true_motion(motion, amount, w, h, pts):
    """The displacement, px, the frames were rendered with at each point."""
    if motion == "shift":
        return np.broadcast_to(np.array(amount, np.float64), pts.shape)
    c = np.array([w / 2, h / 2])
    return (pts.astype(np.float64) - c) @ (motion_matrix(motion, amount) - np.eye(2)).T


# (levels, win, flow_scale, motion, amount, w, h): every window, levels 1-4 and 6, both flow scales, three motions.
# One level only sees motions below a pixel or so; the amounts grow with the pyramid.
KLT_CASES = [
    (1, 3, S815, "shift", (0.6, -0.45), 96, 72), (1, 7, 1.0, "rotzoom", (0.5, 1.01), 96, 72),
    (1, 19, 1.0, "shear", 0.012, 96, 72),
    (2, 5, S815, "shift", (2.6, -1.9), 128, 96), (2, 11, 1.0, "rotzoom", (1.0, 1.02), 128, 96),
    (2, 17, S815, "shear", 0.03, 128, 96),
    (3, 9, S815, "shift", (4.25, -3.75), 192, 144), (3, 9, S815, "rotzoom", (2.0, 1.03), 192, 144),
    (3, 13, 1.0, "shear", 0.04, 192, 144),
    (4, 15, 1.0, "shift", (3.3, 2.1), 192, 144), (4, 17, S815, "rotzoom", (2.0, 1.03), 192, 144),
    (4, 3, S815, "shear", 0.05, 192, 144),
    (6, 9, S815, "shift", (11.5, -9.25), 256, 192), (6, 19, 1.0, "rotzoom", (3.0, 1.04), 256, 192),
    (6, 5, S815, "shear", 0.06, 256, 192),
]
KLT_IDS = [f"L{c[0]}-w{c[1]}-s{'1' if c[2] == 1 else '8/15'}-{c[3]}" for c in KLT_CASES]
# Points compared with the float64 reference: its level-0 window has win^2 * lam >= LAM_FLOOR_G, its last update was
# below CONVERGED px (eps 0) or below eps, and it lies within FOUND px of the true motion.  The bar, px: BAR at
# flow_scale 8/15, twice that at flow_scale 1, plus eps.  See test_restatement_within_bar_of_float64 for where these
# come from.
LAM_FLOOR_G = 12000.0
CONVERGED = 0.005
FOUND = 0.25
BAR = 0.01


def klt_inputs(oracle, case, seed=7):
    levels, win, fs, motion, amount, w, h = case
    prev, nxt = motion_pair(oracle, motion, w, h, amount, seed)
    pts = random_points(w, h, 160, 100 * levels + win, margin=-(win // 2 + 4))[11:]
    return prev, nxt, pts


def klt_bar(fs, eps):
    return BAR * (1 if fs < 1 else 2) + eps


def float64_error(oracle, case, flow, status, eps):
    """Worst s * |flow - float64| px over the compared points (TRACKED in `status`; in float64 above the floor, converged
    and on the true motion); at least 60 % of the points must be compared."""
    levels, win, fs, motion, amount, w, h = case
    prev, nxt, pts = klt_inputs(oracle, case)
    ref, lam, last = klt64(oracle, prev, nxt, levels, win, pts, fs, 30, eps)
    with np.errstate(invalid="ignore"):
        found = np.hypot(*(fs * ref - true_motion(motion, amount, w, h, pts)).T) < FOUND
    cmp = (status == PT_TRACKED) & (win * win * lam >= LAM_FLOOR_G) & found & (last < (eps if eps > 0 else CONVERGED))
    assert cmp.sum() >= 0.6 * len(pts), (cmp.sum(), len(pts))
    return float((fs * np.hypot(*(flow[cmp].astype(np.float64) - ref[cmp]).T)).max())


# ------------------------------------------------------------------------------------ CPU: the pinned rule vs float64
@pytest.mark.parametrize("case", KLT_CASES, ids=KLT_IDS)
def test_restatement_within_bar_of_float64(tro, oracle, case):
    """The restatement (eps 0 and 0.01, 30 iterations) against klt64 on translations, a rotation with zoom and a shear.

    Where the rule differs: positions and targets on the 1/256 px grid, and every sample rounded to an integer (each It
    carries two roundings, sigma = sqrt(2/12) = 0.41).  For a Newton step (flow_scale 8/15 = Sobel gain 8 over Dt gain
    15) that noise moves the converged flow by about s * 0.41 / sqrt(l1) px along the weak direction, l1 = win^2 * lam
    the structure tensor's smaller eigenvalue; 0.01 px at 5 sigma needs l1 >= (5 * 0.533 * 0.41 / 0.01)^2 = 11900: the
    floor LAM_FLOOR_G.  At flow_scale 1 the step is 15/8 of the Newton step: the iteration overshoots and oscillates
    (factor -7/8 per step), which amplifies the same noise (measured 2-4x the 8/15 error on the same frames): bar 0.02 px.
    With eps 0.01 the two may stop one step apart, and that step is below eps: the bar grows by eps.  Only points on
    which float64 converged to the true motion are compared (a non-converged or diverging iteration separates any two
    implementations); they must be at least 60 % of the points.

    Worst s * |rule - float64| px measured, eps 0 / 0.01: L1 w3 shift 0.0052 / 0.0065, L1 w7 s1 rotzoom 0.0122 / 0.0109,
    L1 w19 s1 shear 0.0110 / 0.0129, L2 w5 shift 0.0041 / 0.0040, L2 w11 s1 rotzoom 0.0086 / 0.0115, L2 w17 shear
    0.0026 / 0.0030, L3 w9 shift 0.0028 / 0.0044, L3 w9 rotzoom 0.0028 / 0.0031, L3 w13 s1 shear 0.0126 / 0.0123, L4
    w15 s1 shift 0.0105 / 0.0111, L4 w17 rotzoom 0.0026 / 0.0028, L4 w3 shear 0.0048 / 0.0059, L6 w9 shift 0.0032 /
    0.0037, L6 w19 s1 rotzoom 0.0070 / 0.0102, L6 w5 shear 0.0037 / 0.0054."""
    levels, win, fs = case[:3]
    prev, nxt, pts = klt_inputs(oracle, case)
    for eps in (0.0, 0.01):
        flow, st = tro.track(prev, nxt, levels, win, pts, fs, iters=30, eps=eps)
        err = float64_error(oracle, case, flow, st, eps)
        assert err <= klt_bar(fs, eps), (eps, err)


def test_float64_reference_finds_the_motion(oracle):
    """klt64 itself: on the 3-level shift and rotation-with-zoom cases the median error against the rendered motion is
    below 0.1 px (a reference that missed the motion would make the comparisons above meaningless).  Measured 0.024 px
    for the shift and 0.072 px for the rotation with zoom, which a window translation can only approximate."""
    for case in (KLT_CASES[6], KLT_CASES[7]):
        levels, win, fs, motion, amount, w, h = case
        prev, nxt, pts = klt_inputs(oracle, case)
        ref, _, _ = klt64(oracle, prev, nxt, levels, win, pts, fs)
        err = np.hypot(*(fs * ref - true_motion(motion, amount, w, h, pts)).T)
        assert np.nanmedian(err) < 0.1, (case, np.nanmedian(err))


# ------------------------------------------------------------------------------------ worst-case content
CONTENT_NAMES = ["zeros", "full", "zero_to_full", "binary_noise", "checker1", "checker2", "vstripes4", "diag4", "diag6",
                 "diag8", "impulses", "step_x", "step_y"]
CONTENT_W, CONTENT_H = 67, 45


def content_pair(name, w=CONTENT_W, h=CONTENT_H):
    """PAIRS of test_adversarial_content, plus period-4 stripes whose next is shifted 2 and 3 columns (vstripes4: 1)."""
    if name.startswith("vstripes4_shift"):
        prev = vertical_stripes(w, h, 4)
        return prev, np.ascontiguousarray(np.roll(prev, int(name[-1]), 1))
    return PAIRS[name](w, h)


CONTENT = CONTENT_NAMES + ["vstripes4_shift2", "vstripes4_shift3"]


def content_points(w, h, seed=5):
    """Every border pixel, integer and sub-pixel interior positions, and random_points (corners, last row / column,
    1/256 px past the last column, NaN / inf, half-to-even ties)."""
    rng = np.random.default_rng(seed)
    gy, gx = np.mgrid[2:h - 2:5, 3:w - 3:5]
    grid = np.stack([gx.ravel(), gy.ravel()], 1).astype(F32)
    sub = (grid + rng.uniform(0, 1, grid.shape)).astype(F32)
    return np.concatenate([random_points(w, h, 40, seed), border_points(w, h), grid, sub]).astype(F32)


def sample88(F, X, Y):
    """The 8.8 bilinear rule of include/ofb200.h on the int64 field F at (X, Y) in 1/256 px, F = 0 outside."""
    h, w = F.shape
    x0, y0, wx, wy = X >> 8, Y >> 8, X & 255, Y & 255

    def tap(x, y):
        inside = (x >= 0) & (x < w) & (y >= 0) & (y < h)
        return np.where(inside, F[np.clip(y, 0, h - 1), np.clip(x, 0, w - 1)], 0)

    return ((256 - wy) * ((256 - wx) * tap(x0, y0) + wx * tap(x0 + 1, y0)) +
            wy * ((256 - wx) * tap(x0, y0 + 1) + wx * tap(x0 + 1, y0 + 1)) + 32768) >> 16


TARGETS = [(0, 0), (256, 0), (-256, 0), (0, 256), (77, -130), (-383, 129)]  # (U, V), 1/256 px


def window_sums64(prev, nxt, win, pts):
    """int64 (a, dd, b) and the largest |tx|, |ty| over the TARGETS, level 0, at the points that start inside."""
    ix, iy, sp = fields(prev, np.int64)
    sn = fields(nxt, np.int64)[2]
    R = win // 2
    oy, ox = (o.ravel() for o in np.mgrid[-R:R + 1, -R:R + 1])
    PX = np.rint(pts[:, 0] * F32(256)).astype(np.int64)[:, None]
    PY = np.rint(pts[:, 1] * F32(256)).astype(np.int64)[:, None]
    X, Y = PX + 256 * ox, PY + 256 * oy
    gx, gy, s0 = sample88(ix, X, Y), sample88(iy, X, Y), sample88(sp, X, Y)
    a, dd, b = (gx * gx).sum(1), (gy * gy).sum(1), (gx * gy).sum(1)
    tx = ty = np.zeros(len(pts), np.int64)
    for U, V in TARGETS:
        It = sample88(sn, X + U, Y + V) - s0
        tx = np.maximum(tx, np.abs((gx * It).sum(1)))
        ty = np.maximum(ty, np.abs((gy * It).sum(1)))
    return a, dd, b, tx, ty


def inside_points(w, h):
    p = content_points(w, h)
    ok = np.isfinite(p).all(1) & (p[:, 0] >= 0) & (p[:, 0] <= w - 1) & (p[:, 1] >= 0) & (p[:, 1] <= h - 1)
    return p[ok]


def test_window_sums_fit_int32_and_come_near_it():
    """int64 window sums at every inside start of content_points, every window, every content pair: a, dd, |b|, |tx|,
    |ty| stay below 2^31; at window 19 the content pushes a to >= 0.17 * 2^31 and |tx| to >= 0.15 * 2^31.  Measured,
    fraction of 2^31: a 0.175 (vstripes4), dd and |b| 0.066 (diag6), |tx| 0.161 (vstripes4, stripes shifted one
    column), |ty| 0.121 (diag8)."""
    w, h = CONTENT_W, CONTENT_H
    pts = inside_points(w, h)
    top = {}
    for name in CONTENT:
        prev, nxt = content_pair(name)
        for win in WINDOWS:
            for key, v in zip(("a", "dd", "b", "tx", "ty"), window_sums64(prev, nxt, win, pts)):
                m = int(np.abs(v).max())
                assert m < I32, (name, win, key, m)
                if win == 19:
                    top[key] = max(top.get(key, (0, ""))[0], m), name
    assert top["a"][0] >= 0.17 * I32 and top["tx"][0] >= 0.15 * I32, top


def exact_below(a, dd, b, win, min_eig):
    """lam < min_eig exactly: l1 = (S - sqrt(disc)) / 2 < mu = win^2 * min_eig  <=>  S - 2 mu < sqrt(disc)."""
    mu = Fraction(float(np.float32(min_eig))) * win * win
    T = a + dd - 2 * mu
    return T < 0 or T * T < (a - dd) ** 2 + 4 * b * b


def lam_of(a, dd, b, win):
    """lam in float64 without cancellation: l1 = 2 det / (S + sqrt(disc))."""
    a, dd, b = int(a), int(dd), int(b)
    det, S = a * dd - b * b, a + dd
    return 0.0 if S == 0 else 2.0 * det / (S + np.sqrt(float((a - dd) ** 2 + 4 * b * b))) / (win * win)


def test_min_eig_decision_is_the_exact_one(tro, oracle):
    """Every window of the content pairs (one level, inside starts): the restatement's LOW_TEXTURE decision equals the
    exact lam < min_eig for min_eig = 1e-45, 1e-12, 1, 1e6 and, on a seeded 16 points per pair and window, lam * (1 +-
    1e-6); the only exception allowed is |lam - min_eig| <= 1e-9 max(lam, min_eig).  Windows with lam = 0 (flat frames,
    stripes, steps) occur, as do windows with lam > 1e-6 * 2^31."""
    w, h = CONTENT_W, CONTENT_H
    pts = inside_points(w, h)
    rng = np.random.default_rng(9)
    n_zero = n_pos = 0
    for name in CONTENT:
        prev, nxt = content_pair(name)
        for win in WINDOWS:
            a, dd, b, _, _ = window_sums64(prev, nxt, win, pts)
            lams = np.array([lam_of(*s, win) for s in zip(a, dd, b)])
            n_zero += int((a * dd == b * b).sum())
            n_pos += int((lams > 1e-6 * I32).sum())

            def check(i, me, st):
                want = exact_below(int(a[i]), int(dd[i]), int(b[i]), win, me)
                lam, me32 = lams[i], float(np.float32(me))
                assert (st == PT_LOW_TEXTURE) == want or abs(lam - me32) <= 1e-9 * max(lam, me32), \
                    (name, win, pts[i].tolist(), int(a[i]), int(dd[i]), int(b[i]), me32, st)

            for me in (1e-45, 1e-12, 1.0, 1e6):
                _, st = tro.track(prev, nxt, 1, win, pts, iters=1, eps=0.0, min_eig=me)
                for i in range(len(pts)):
                    check(i, me, st[i])
            for i in rng.choice(len(pts), 16, replace=False):
                for f in (1 - 1e-6, 1 + 1e-6):
                    if lams[i] > 0:
                        _, st = tro.track(prev, nxt, 1, win, pts[i:i + 1], iters=1, eps=0.0, min_eig=lams[i] * f)
                        check(i, lams[i] * f, st[0])
    assert n_zero > 0 and n_pos > 0, (n_zero, n_pos)


LAM0_MIN_EIG = [1e-4, 1e-8, 1e-10, 1e-12, 1e-20, 1e-30, 1e-45]


def test_one_dimensional_window_is_low_texture_at_any_min_eig(tro, oracle):
    """Period-4 vertical stripes (0, 0, 255, 255): Iy = 0, so dd = b = 0 and lam = 0 exactly.  Every min_eig > 0 down to
    the smallest subnormal float marks the point LOW_TEXTURE with flow 0, at every window and at integer and sub-pixel
    points; min_eig = 0 runs the solve, which meets det == 0 (NONFINITE)."""
    w, h = 64, 48
    prev = vertical_stripes(w, h, 4)
    nxt = np.ascontiguousarray(np.roll(prev, 1, 1))
    pts = np.array([[30, 20], [30.5, 20.25], [17.3, 33.9]], F32)
    for win in WINDOWS:
        for me in LAM0_MIN_EIG:
            flow, st = tro.track(prev, nxt, 1, win, pts, min_eig=me)
            assert (st == PT_LOW_TEXTURE).all() and (flow == 0).all(), (win, me, st.tolist())
        _, st = tro.track(prev, nxt, 1, win, pts, min_eig=0.0)
        assert (st == PT_NONFINITE).all(), (win, st.tolist())


# ------------------------------------------------------------------------------------ GPU
def _dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _track(ctx, prevs, nexts, w, levels, win, pts, **kw):
    """The kernel through Context.track_points_device on planar_to_device frames (64-byte pitch, zero padding)."""
    from cuda_optical_flow_2_b200 import planar_to_device

    flow, st = ctx.track_points_device(planar_to_device(prevs), planar_to_device(nexts), w, levels, win, _dev(pts), **kw)
    return flow.cpu().numpy(), st.cpu().numpy()


def _same_as_restatement(tro, flow, st, prev, nxt, levels, win, pts, what, **kw):
    rf, rs = tro.track(prev, nxt, levels, win, pts, **kw)
    assert_same_bits(flow, rf, f"{what} flow")
    assert_status_equal(st, rs, f"{what} status")


@pytest.mark.gpu
@pytest.mark.parametrize("case", KLT_CASES, ids=KLT_IDS)
def test_kernel_within_bar_of_float64(ctx, tro, oracle, case):
    """The kernel on the float64 cases: bit-identical to the restatement, and within the bar of klt64 directly (the
    second assertion does not go through the restatement)."""
    levels, win, fs, _, _, w, _ = case
    prev, nxt, pts = klt_inputs(oracle, case)
    for eps in (0.0, 0.01):
        flow, st = _track(ctx, prev[None], nxt[None], w, levels, win, pts[None], flow_scale=fs, iters=30, eps=eps)
        _same_as_restatement(tro, flow[0], st[0], prev, nxt, levels, win, pts, f"eps {eps}", flow_scale=fs, iters=30,
                             eps=eps)
        err = float64_error(oracle, case, flow[0], st[0], eps)
        assert err <= klt_bar(fs, eps), (eps, err)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CONTENT)
def test_kernel_on_worst_case_content(ctx, tro, oracle, name):
    """Every window at levels 1 and 3 on the content pairs, points over the whole frame, its border and outside: the
    kernel equals the restatement bit for bit with equal statuses (5 iterations, eps 0, flow_scale 8/15); one more run at
    one level with min_eig 1e-30.  The all-zero pair is NONFINITE wherever a point starts inside; stripe windows clear of
    the zero padding above and below are one-dimensional and LOW_TEXTURE at min_eig 1e-30."""
    w, h = CONTENT_W, CONTENT_H
    prev, nxt = content_pair(name)
    pts = content_points(w, h)
    inside = np.isfinite(pts).all(1) & (pts[:, 0] >= 0) & (pts[:, 0] <= w - 1) & (pts[:, 1] >= 0) & (pts[:, 1] <= h - 1)
    for win in WINDOWS:
        for levels, me in ((1, 0.0), (3, 0.0), (1, 1e-30)):
            kw = dict(flow_scale=S815, iters=5, eps=0.0, min_eig=me)
            flow, st = _track(ctx, prev[None], nxt[None], w, levels, win, pts[None], **kw)
            _same_as_restatement(tro, flow[0], st[0], prev, nxt, levels, win, pts, f"{name} win {win} L{levels} {me}", **kw)
            assert (st[0][~inside] == PT_OUTSIDE).all()
            if name == "zeros" and me == 0:
                assert (st[0][inside] == PT_NONFINITE).all()
            if name.startswith("vstripes4") and me > 0:  # rows whose window misses the zero padding above and below
                rows = inside & (pts[:, 1] >= win // 2 + 2) & (pts[:, 1] <= h - 3 - win // 2)
                assert rows.any() and (st[0][rows] == PT_LOW_TEXTURE).all()


@pytest.mark.gpu
def test_kernel_one_dimensional_window_is_low_texture_at_any_min_eig(ctx):
    """The kernel on period-4 stripes (lam = 0 exactly): LOW_TEXTURE with flow 0 at every window and every min_eig down to
    the smallest subnormal float."""
    w, h = 64, 48
    prev = vertical_stripes(w, h, 4)
    nxt = np.ascontiguousarray(np.roll(prev, 1, 1))
    pts = np.array([[[30, 20], [30.5, 20.25], [17.3, 33.9]]], F32)
    for win in WINDOWS:
        for me in LAM0_MIN_EIG:
            flow, st = _track(ctx, prev[None], nxt[None], w, 1, win, pts, min_eig=me)
            assert (st == PT_LOW_TEXTURE).all() and (flow == 0).all(), (win, me, st.tolist())


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(262, 150), (256, 160), (101, 77)])
@pytest.mark.parametrize("levels", [1, 3])
def test_caller_frame_layouts(ctx, tro, oracle, w, h, levels):
    """Caller frames through the C ABI: pitch align_up(w, 16) (w + 16 where w is a multiple of 16), image stride
    pitch * (h + 3) + 16, every byte outside the frames 0xFF.  At one level the kernel reads nothing but the caller's
    memory.  Bit-identical to the zero-padded 64-byte layout and to the restatement."""
    import torch

    from cuda_optical_flow_2_b200 import OfbParams
    from cuda_optical_flow_2_b200.api import align_up
    from cuda_optical_flow_2_b200._lib import check
    from test_adversarial_content import _padded_device

    win, fs = 9, S815
    pitch = align_up(w, 16) if w % 16 else w + 16
    stride = pitch * (h + 3) + 16
    sm = oracle.make_frame(w, h, 0, 0, 4, 77), oracle.make_frame(w, h, 1.6, -0.9, 4, 77)
    pairs = [PAIRS["binary_noise"](w, h), sm, PAIRS["diag6"](w, h)]
    prevs, nexts = np.stack([p for p, _ in pairs]), np.stack([q for _, q in pairs])
    n = len(pairs)
    pts = np.stack([np.concatenate([random_points(w, h, 100, 60 + i), border_points(w, h)]) for i in range(n)])
    plain_f, plain_s = _track(ctx, prevs, nexts, w, levels, win, pts, flow_scale=fs, iters=5, eps=0.0)
    bp, bn = _padded_device(prevs, pitch, stride), _padded_device(nexts, pitch, stride)
    dpts = _dev(pts)
    flow = torch.empty(pts.shape, dtype=torch.float32, device="cuda")
    st = torch.empty(pts.shape[:2], dtype=torch.uint8, device="cuda")
    p = OfbParams(w, h, levels, win, 2, fs, n)
    check(ctx._lib.ofb_track_points_device(ctx._h, C.byref(p), bp.data_ptr(), bn.data_ptr(), pitch, stride, dpts.data_ptr(),
                                           pts.shape[1], 5, 0.0, 0.0, flow.data_ptr(), st.data_ptr(), None))
    flow, st = flow.cpu().numpy(), st.cpu().numpy()
    assert_same_bits(flow, plain_f, "caller layout vs 64-byte layout")
    assert_status_equal(st, plain_s, "caller layout vs 64-byte layout")
    for i in range(n):
        _same_as_restatement(tro, flow[i], st[i], prevs[i], nexts[i], levels, win, pts[i], f"pair {i}", flow_scale=fs,
                             iters=5, eps=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,levels,win", [(160, 128, 5, 11), (200, 150, 6, 7), (515, 387, 7, 3), (515, 387, 7, 19),
                                            (300, 260, 8, 3), (300, 260, 8, 19)])
def test_levels_up_to_eight(ctx, tro, oracle, w, h, levels, win):
    """Levels 5-8 (300x260 at 8 levels has a 2x2 coarsest level, far smaller than the window): bit-identical to the
    restatement, with min_eig 0 (TRACKED points) and 1e4 (LOW_TEXTURE points, stopped at a coarse level)."""
    prev, nxt = oracle.make_frame(w, h, 0, 0, 4, 3), oracle.make_frame(w, h, 9.3, -6.1, 4, 3)
    pts = random_points(w, h, 80, levels * 100 + win)
    for me in (0.0, 1e4):
        kw = dict(flow_scale=S815, iters=10, eps=0.01, min_eig=me)
        flow, st = _track(ctx, prev[None], nxt[None], w, levels, win, pts[None], **kw)
        _same_as_restatement(tro, flow[0], st[0], prev, nxt, levels, win, pts, f"min_eig {me}", **kw)
        assert (st == (PT_LOW_TEXTURE if me > 0 else PT_TRACKED)).any()


@pytest.mark.gpu
def test_64_iterations_and_extreme_flow_scales(ctx, tro, oracle):
    """iters = 64 with eps 0 and 0.01; flow_scale 3 and 0.01 (s256 = 2.56, U = rint(d * 2.56)): bit-identical to the
    restatement."""
    w, h = 131, 97
    prev, nxt = oracle.make_frame(w, h, 0, 0, 4, 8), oracle.make_frame(w, h, 3.4, 2.2, 4, 8)
    pts = random_points(w, h, 120, 13)
    for kw in (dict(iters=64, eps=0.0), dict(iters=64, eps=0.01), dict(flow_scale=3.0, iters=30, eps=0.0),
               dict(flow_scale=0.01, iters=30, eps=0.0), dict(flow_scale=0.01, iters=64, eps=0.01)):
        kw = dict(dict(flow_scale=S815, min_eig=0.0), **kw)
        flow, st = _track(ctx, prev[None], nxt[None], w, 3, 9, pts[None], **kw)
        _same_as_restatement(tro, flow[0], st[0], prev, nxt, 3, 9, pts, str(kw), **kw)
        assert (st == PT_TRACKED).any(), kw


@pytest.mark.gpu
def test_two_to_the_24_points(ctx, tro, oracle):
    """2^24 points on one pair (the largest n_points): the first and last point, the last CTA and a seeded 3000 of the
    rest equal the restatement; 2^24 + 1 points are refused with nothing launched."""
    import torch

    from cuda_optical_flow_2_b200 import OfbError

    w, h, levels, win, kw = 96, 64, 2, 5, dict(flow_scale=S815, iters=3, eps=0.0)
    prev, nxt = oracle.make_frame(w, h, 0, 0, 4, 21), oracle.make_frame(w, h, 1.3, 0.8, 4, 21)
    n = 1 << 24
    rng = np.random.default_rng(24)
    pts = np.stack([rng.uniform(-1, w, n), rng.uniform(-1, h, n)], 1).astype(F32)
    flow, st = _track(ctx, prev[None], nxt[None], w, levels, win, pts[None], **kw)
    sel = np.unique(np.concatenate([[0, 1], np.arange(n - 4, n), rng.choice(n, 3000, replace=False)]))
    _same_as_restatement(tro, flow[0, sel], st[0, sel], prev, nxt, levels, win, pts[sel], "2^24 points", **kw)
    torch.cuda.synchronize()
    before = ctx.launch_count
    from cuda_optical_flow_2_b200 import planar_to_device

    with pytest.raises(OfbError, match="n_points"):
        ctx.track_points_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, levels, win,
                                torch.zeros((1, n + 1, 2), dtype=torch.float32, device="cuda"), **kw)
    assert ctx.launch_count == before


@pytest.mark.gpu
def test_65535_pairs(ctx, tro):
    """65535 pairs of 16x12 frames with 3 points each (grid.z at its limit): pairs 0, 1, 32767, 65533 and 65534 equal the
    restatement."""
    n, w, h, levels, win, kw = 65535, 16, 12, 2, 5, dict(flow_scale=S815, iters=5, eps=0.0)
    rng = np.random.default_rng(65535)
    prevs = rng.integers(0, 256, (n, h, w), dtype=np.uint8)
    nexts = np.ascontiguousarray(np.roll(prevs, 1, 2))
    pts = np.stack([rng.uniform(0, w - 1, (n, 3)), rng.uniform(0, h - 1, (n, 3))], 2).astype(F32)
    flow, st = _track(ctx, prevs, nexts, w, levels, win, pts, **kw)
    for i in (0, 1, 32767, 65533, 65534):
        _same_as_restatement(tro, flow[i], st[i], prevs[i], nexts[i], levels, win, pts[i], f"pair {i}", **kw)
