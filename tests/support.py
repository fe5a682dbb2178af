"""What the test modules share: the C restatements, the comparison bars, device helpers, solve-mode switching, content
generators, models and point sets.  A plain module (tests/ is on sys.path), so that a test module never imports another.
"""
import contextlib
import ctypes as C
import functools
import os
import subprocess
import tempfile

import numpy as np
import pytest

F32 = np.float32
S815 = 8 / 15  # px per flow unit of the reference's masks (Sobel gain 8, Dt gain 15); its products are not exact
ASW, NEAR, BIL = 0, 1, 2  # OFB_WARP_AS_WRITTEN, _NEAREST, _BILINEAR
PT_TRACKED, PT_NONFINITE, PT_LOW_TEXTURE, PT_OUTSIDE = 0, 1, 2, 3
FB_CONSISTENT, FB_INCONSISTENT, FB_OUTSIDE, FB_FWD_NONFINITE, FB_BWD_NONFINITE = 0, 1, 2, 3, 4
TOL_ABS = 1e-4  # px, stated tolerance of the tolerance-mode solve on u and v (and so on end-point error up to sqrt(2))
TOL_REL = 1e-5

TESTS = os.path.dirname(os.path.abspath(__file__))


# ------------------------------------------------------------------------------------ the C restatements
@functools.cache
def _build_dir():
    return tempfile.TemporaryDirectory(prefix="ofb-restatements-")


@functools.cache
def c_library(name):
    """tests/<name>.c as a shared library, compiled once per session.  The flags are part of the pin: without contraction
    and fast math every operation of the restatement rounds on its own, as the rule of include/ofb200.h states."""
    so = os.path.join(_build_dir().name, f"lib{name}.so")
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra",
                           "-shared", "-o", so, os.path.join(TESTS, f"{name}.c"), "-lm"])
    return so


class TrackOracle:
    """tests/track_oracle.c (orc_track_points) through ctypes, on oracle.gauss_pyramid levels."""

    def __init__(self, so_path, oracle):
        self._lib = C.CDLL(so_path)
        self._lib.orc_track_points.restype = None
        self._lib.orc_track_points.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p,
                                               C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
        self.O = oracle

    def track(self, prev, nxt, levels, win, points, flow_scale=1.0, iters=30, eps=0.01, min_eig=0.0):
        """One pair: prev / next (h, w) uint8, points (m, 2) float32 -> (flow (m, 2) float32, status (m,) uint8)."""
        h, w = prev.shape
        pp = self.O.gauss_pyramid(prev, levels)
        pn = self.O.gauss_pyramid(nxt, levels)
        arr = lambda lv: (C.c_void_p * levels)(*[a.ctypes.data for a in lv])
        pts = np.ascontiguousarray(points, F32).reshape(-1, 2)
        flow = np.empty_like(pts)
        status = np.empty(len(pts), np.uint8)
        self._lib.orc_track_points(arr(pp), arr(pn), w, h, levels, win, flow_scale, pts.ctypes.data, len(pts), iters, eps,
                                   min_eig, flow.ctypes.data, status.ctypes.data)
        return flow, status


class CornerOracle:
    """tests/corner_oracle.c through ctypes."""

    def __init__(self, so_path):
        self._lib = C.CDLL(so_path)
        self._lib.orc_min_eig_map.restype = None
        self._lib.orc_min_eig_map.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_void_p]
        self._lib.orc_detect_corners.restype = C.c_int
        self._lib.orc_detect_corners.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float,
                                                 C.c_void_p, C.c_void_p]

    def score(self, img, win):
        img = np.ascontiguousarray(img, np.uint8)
        h, w = img.shape
        out = np.empty((h, w), F32)
        self._lib.orc_min_eig_map(img.ctypes.data, w, w, h, win, out.ctypes.data)
        return out

    def select(self, score, win, max_corners, quality_level=0.01, min_distance=10.0, min_score=0.0):
        score = np.ascontiguousarray(score, F32)
        h, w = score.shape
        corners = np.empty((max_corners, 2), F32)
        scores = np.empty(max_corners, F32)
        n = self._lib.orc_detect_corners(score.ctypes.data, w, h, win, max_corners, quality_level, min_distance, min_score,
                                         corners.ctypes.data, scores.ctypes.data)
        return corners, scores, n

    def detect(self, img, win, max_corners, **kw):
        return self.select(self.score(img, win), win, max_corners, **kw)


class FbOracle:
    """tests/fb_oracle.c (orc_fb_check) through ctypes, plus the pinned oracle's flow in both directions."""

    def __init__(self, so_path, oracle):
        self._lib = C.CDLL(so_path)
        self._lib.orc_fb_check.restype = None
        self._lib.orc_fb_check.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float,
                                           C.c_void_p, C.c_void_p]
        self.O = oracle

    def fb_check(self, fwd, bwd, flow_scale=1.0, alpha=0.01, beta=0.5):
        """(h, w, 2) or (n, h, w, 2) float32 totals -> (status uint8, err2 float32), shaped like the flow without its last
        axis."""
        fwd = np.ascontiguousarray(fwd, F32)
        bwd = np.ascontiguousarray(bwd, F32)
        assert fwd.shape == bwd.shape and fwd.shape[-1] == 2 and fwd.ndim in (3, 4)
        h, w = fwd.shape[-3:-1]
        f3, b3 = fwd.reshape(-1, h, w, 2), bwd.reshape(-1, h, w, 2)
        status = np.empty(f3.shape[:3], np.uint8)
        err2 = np.empty(f3.shape[:3], F32)
        for i in range(f3.shape[0]):
            self._lib.orc_fb_check(f3[i].ctypes.data, b3[i].ctypes.data, w, h, flow_scale, alpha, beta, err2[i].ctypes.data,
                                   status[i].ctypes.data)
        return status.reshape(fwd.shape[:-1]), err2.reshape(fwd.shape[:-1])

    def fb_pair(self, prev, nxt, levels, win, warp_mode, flow_scale=1.0, alpha=0.01, beta=0.5):
        """(fwd_total, bwd_total, status, err2): the level-0 compositions of oracle.flow_pair(prev, next) and
        oracle.flow_pair(next, prev) with exact window sums, and their check."""
        O = self.O
        fwd = O.flow_pair(prev, nxt, levels, win, warp_mode, O.SUMS_EXACT, flow_scale, want_cum=True)[1][0]
        bwd = O.flow_pair(nxt, prev, levels, win, warp_mode, O.SUMS_EXACT, flow_scale, want_cum=True)[1][0]
        return (fwd, bwd) + self.fb_check(fwd, bwd, flow_scale, alpha, beta)


@pytest.fixture(scope="session")
def tro(oracle):
    return TrackOracle(c_library("track_oracle"), oracle)


@pytest.fixture(scope="session")
def cro():
    return CornerOracle(c_library("corner_oracle"))


@pytest.fixture(scope="session")
def fbo(oracle):
    return FbOracle(c_library("fb_oracle"), oracle)


# ------------------------------------------------------------------------------------ comparison bars
# Each rule takes numpy arrays or torch tensors (compared where they are, so device tensors stay on the device).  The
# *_differ form returns '' when the two match and else what differs; the assert_* form fails with that message.
def _tensor(a, dtype=None):
    import torch

    if isinstance(a, torch.Tensor):
        return a
    a = np.ascontiguousarray(a, dtype)
    return torch.from_numpy(a if a.flags.writeable else a.copy())


def _pair(got, ref, dtype=None):
    g, r = _tensor(got, dtype), _tensor(ref, dtype)
    return g, r, "" if g.shape == r.shape else f"shapes differ: {tuple(g.shape)} vs {tuple(r.shape)}"


def _first(g, r, bad, what):
    i = tuple(bad.nonzero()[0].tolist())
    return f"{int(bad.sum())} of {bad.numel()} {what} differ, first at {list(i)}: got {g[i].item()!r} ref {r[i].item()!r}"


def _nan_positions(g, r):
    ng, nr = g.isnan(), r.isnan()
    if bool((ng != nr).any()):
        return ng, f"NaN positions differ at {int((ng != nr).sum())} values, first at {(ng != nr).nonzero()[0].tolist()}"
    return ng, ""


def bytes_differ(got, ref):
    """Equal shape, dtype and bytes: NaN payloads included."""
    g, r, e = _pair(got, ref)
    if e or g.dtype != r.dtype:
        return e or f"dtypes differ: {g.dtype} vs {r.dtype}"
    import torch

    bad = g.contiguous().view(torch.uint8) != r.contiguous().view(torch.uint8)
    return f"{int(bad.sum())} bytes differ" if bool(bad.any()) else ""


def bits_differ(got, ref):
    """float32: NaN at the same positions (any payload), every other value bit for bit (so 0.0 and -0.0 differ)."""
    g, r, e = _pair(got, ref, F32)
    if e:
        return e
    import torch

    ng, e = _nan_positions(g, r)
    if e:
        return e
    bad = (g.view(torch.int32) != r.view(torch.int32)) & ~ng
    return _first(g, r, bad, "values") if bool(bad.any()) else ""


def values_differ(got, ref):
    """NaN at the same positions, every other value equal as a number (so infinities of the same sign, and 0.0 == -0.0)."""
    g, r, e = _pair(got, ref)
    if e:
        return e
    ng, e = _nan_positions(g, r)
    if e:
        return e
    bad = (g != r) & ~ng
    return _first(g, r, bad, "values") if bool(bad.any()) else ""


def statuses_differ(got, ref):
    """Every status equal."""
    g, r, e = _pair(got, ref)
    if e:
        return e
    bad = g != r
    return _first(g, r, bad, "statuses") if bool(bad.any()) else ""


def assert_same_bytes(got, ref, what=""):
    assert not (e := bytes_differ(got, ref)), f"{what}: {e}"


def assert_same_bits(got, ref, what=""):
    assert not (e := bits_differ(got, ref)), f"{what}: {e}"


def assert_values_equal(got, ref, what=""):
    assert not (e := values_differ(got, ref)), f"{what}: {e}"


def assert_status_equal(got, ref, what=""):
    assert not (e := statuses_differ(got, ref)), f"{what}: {e}"


def assert_flow_within_tolerance(got: np.ndarray, ref: np.ndarray, what: str = "", ulps: bool = True):
    """The stated bar of the tolerance-mode solve, per level on identical inputs: non-finite values on exactly the same
    pixels, and |du|, |dv| <= TOL_ABS + TOL_REL * |ref| everywhere else."""
    fg, fr = np.isfinite(got), np.isfinite(ref)
    assert np.array_equal(fg, fr), f"{what}: finite masks differ at {np.argwhere(fg != fr)[:5]}"
    d = np.abs(got[fg].astype(np.float64) - ref[fg])
    lim = TOL_ABS + TOL_REL * np.abs(ref[fg])
    assert (d <= lim).all(), f"{what}: max abs diff {d.max():.3e} exceeds tolerance"
    # and in fact a few float ulps: exact integer determinant / numerators, one rounding each, 1-ulp reciprocal
    rel = d / np.maximum(np.abs(ref[fg]), 1e-30)
    big = np.abs(ref[fg]) > 1e-3
    if ulps and big.any():  # (not for sums like the cumulative flow, where terms cancel)
        assert rel[big].max() < 1e-6, f"{what}: relative error {rel[big].max():.3e}"


# ------------------------------------------------------------------------------------ the device and the shared context
def to_device(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def device_frames(imgs, pitch=None, stride=None, fill=0):
    """(n, h, w) uint8 -> (flat CUDA buffer, pitch, stride): image i at byte i * stride with row pitch `pitch` (default w,
    stride default pitch * h, 0 allowed), `fill` in every other byte.  The buffer ends with the last image's last pixel."""
    import torch

    n, h, w = imgs.shape
    pitch = pitch or w
    stride = pitch * h if stride is None else stride
    buf = np.full(stride * (n - 1) + pitch * (h - 1) + w, fill, np.uint8)
    np.lib.stride_tricks.as_strided(buf, (n, h, w), (stride, pitch, 1))[...] = imgs
    return torch.from_numpy(buf).cuda(), pitch, stride


@contextlib.contextmanager
def solve(ctx, mode):
    """The shared context in solve `mode` (OFB_SOLVE_*) for the block, and back in OFB_SOLVE_EXACT after it, also on
    failure.  Every test finds the context in the exact solve."""
    from cuda_optical_flow_2_b200 import SOLVE_EXACT

    assert ctx.solve == SOLVE_EXACT
    ctx.solve = mode
    try:
        yield ctx
    finally:
        ctx.solve = SOLVE_EXACT


@pytest.fixture
def fast_ctx(ctx):
    from cuda_optical_flow_2_b200 import SOLVE_FAST

    with solve(ctx, SOLVE_FAST):
        yield ctx


# ------------------------------------------------------------------------------------ worst-case image content
def _grid(w, h):
    return np.arange(w)[None, :], np.arange(h)[:, None]


def _u8(a, w, h):
    return np.ascontiguousarray(np.broadcast_to(a, (h, w)), dtype=np.uint8)


def flat(w, h, value):
    return np.full((h, w), value, np.uint8)


def binary_noise(w, h, seed):
    return (np.random.default_rng(seed).integers(0, 2, (h, w)) * 255).astype(np.uint8)


def uniform_noise(w, h, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w), dtype=np.uint8)


def checkerboard(w, h, cell):
    x, y = _grid(w, h)
    return _u8(255 * ((x // cell + y // cell) % 2), w, h)


def vertical_stripes(w, h, period):
    x, _ = _grid(w, h)
    return _u8(255 * ((x // (period // 2)) % 2), w, h)


def diagonal_stripes(w, h, period, anti=False):
    x, y = _grid(w, h)
    return _u8(255 * (((x - y if anti else x + y) // (period // 2)) % 2), w, h)


def impulses(w, h, seed):
    """Isolated 255 pixels on 0: one per 6x6 cell, at a seeded position inside the cell's upper-left 5x5."""
    rng = np.random.default_rng(seed)
    img = np.zeros((h, w), np.uint8)
    ys, xs = np.meshgrid(np.arange(0, h, 6), np.arange(0, w, 6), indexing="ij")
    ys, xs = ys + rng.integers(0, 5, ys.shape), xs + rng.integers(0, 5, xs.shape)
    keep = (ys < h) & (xs < w)
    img[ys[keep], xs[keep]] = 255
    return img


def step(w, h, at, axis):
    """0 before column (axis 1) or row (axis 0) `at`, 255 from there on."""
    x, y = _grid(w, h)
    return _u8(255 * ((x if axis == 1 else y) >= at), w, h)


def roll_x(img, s=1):
    return np.ascontiguousarray(np.roll(img, s, axis=1))


# name -> (w, h) -> (prev, next).  Periodic patterns move by one pixel; the noise pairs are independent frames (the
# largest |It|) or a shifted copy.
PAIRS = {
    "zeros": lambda w, h: (flat(w, h, 0), flat(w, h, 0)),
    "full": lambda w, h: (flat(w, h, 255), flat(w, h, 255)),
    "zero_to_full": lambda w, h: (flat(w, h, 0), flat(w, h, 255)),
    "full_to_zero": lambda w, h: (flat(w, h, 255), flat(w, h, 0)),
    "binary_noise": lambda w, h: (binary_noise(w, h, 11), binary_noise(w, h, 12)),
    "uniform_noise": lambda w, h: (uniform_noise(w, h, 21), np.ascontiguousarray(np.roll(uniform_noise(w, h, 21), (1, -1), (0, 1)))),
    "checker1": lambda w, h: (checkerboard(w, h, 1), roll_x(checkerboard(w, h, 1))),
    "checker2": lambda w, h: (checkerboard(w, h, 2), roll_x(checkerboard(w, h, 2))),
    "vstripes4": lambda w, h: (vertical_stripes(w, h, 4), roll_x(vertical_stripes(w, h, 4))),
    "diag4": lambda w, h: (diagonal_stripes(w, h, 4), roll_x(diagonal_stripes(w, h, 4))),
    "diag6": lambda w, h: (diagonal_stripes(w, h, 6), roll_x(diagonal_stripes(w, h, 6))),
    "diag8": lambda w, h: (diagonal_stripes(w, h, 8), roll_x(diagonal_stripes(w, h, 8))),
    "adiag4": lambda w, h: (diagonal_stripes(w, h, 4, True), roll_x(diagonal_stripes(w, h, 4, True))),
    "adiag6": lambda w, h: (diagonal_stripes(w, h, 6, True), roll_x(diagonal_stripes(w, h, 6, True))),
    "adiag8": lambda w, h: (diagonal_stripes(w, h, 8, True), roll_x(diagonal_stripes(w, h, 8, True))),
    "impulses": lambda w, h: (impulses(w, h, 31), np.ascontiguousarray(np.roll(impulses(w, h, 31), (1, 1), (0, 1)))),
    "step_x": lambda w, h: (step(w, h, w // 2, 1), step(w, h, w // 2 - 1, 1)),
    "step_y": lambda w, h: (step(w, h, h // 2, 0), step(w, h, h // 2 + 1, 0)),
}


def noise_pair(w, h, seed):
    """Uniform-noise frames: every byte of the warped frame enters some window sum with a nonzero weight."""
    rng = np.random.default_rng(seed)
    prev = rng.integers(0, 256, (h, w), dtype=np.uint8)
    nxt = np.ascontiguousarray(np.roll(prev, (1, -2), (0, 1)) ^ rng.integers(0, 16, (h, w), dtype=np.uint8))
    return prev, nxt


# ------------------------------------------------------------------------------------ corner content and the rule
def content(kind, w, h, seed=0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == "zeros":
        return np.zeros((h, w), np.uint8)
    if kind == "full":
        return np.full((h, w), 255, np.uint8)
    if kind == "checker":
        return (((xx + yy) & 1) * 255).astype(np.uint8)
    if kind == "stripes":  # vertical period-4 stripes: gy = 0 everywhere, det = 0
        return (((xx >> 1) & 1) * 255).astype(np.uint8)
    if kind == "noise":
        return rng.integers(0, 256, (h, w), dtype=np.uint8)
    if kind == "isotropic":  # a radial pattern: near-isotropic windows (disc close to 0)
        r = np.hypot(xx - w / 2 + 0.3, yy - h / 2 + 0.7)
        return (127.5 + 127.5 * np.cos(r * 0.9)).astype(np.uint8)
    if kind == "textured":
        from oracle import oracle as O

        return O.make_frame(w, h, 0.0, 0.0, 4, 1000 + seed)
    if kind == "natural":  # smooth blobs plus a little noise
        f = np.zeros((h, w))
        for _ in range(12):
            cx, cy, s, a = rng.uniform(0, w), rng.uniform(0, h), rng.uniform(2, 9), rng.uniform(-90, 90)
            f += a * np.exp(-((xx - cx) ** 2 + (yy - cy) ** 2) / (2 * s * s))
        return np.clip(128 + f + rng.normal(0, 3, (h, w)), 0, 255).astype(np.uint8)
    raise ValueError(kind)


def exact_sums(img, win):
    """A, D, B by scipy correlations in int64 (zero mode): Sobel fields, then the window sums."""
    from scipy.ndimage import correlate

    i = img.astype(np.int64)
    dx = np.array([[-1, 0, 1], [-2, 0, 2], [-1, 0, 1]], np.int64)
    gx = correlate(i, dx, mode="constant", cval=0)
    gy = correlate(i, dx.T, mode="constant", cval=0)
    box = np.ones((win, win), np.int64)
    return (correlate(gx * gx, box, mode="constant", cval=0), correlate(gy * gy, box, mode="constant", cval=0),
            correlate(gx * gy, box, mode="constant", cval=0))


def plain_greedy(score, win, max_corners, quality_level, min_distance, min_score):
    """The rule of include/ofb200.h, written the slow, obvious way."""
    h, w = score.shape
    m = win // 2 + 1
    if w < 2 * m + 1 or h < 2 * m + 1:
        return []
    inter = score[m:h - m, m:w - m]
    thr = max(F32(quality_level) * F32(inter.max()), F32(min_score))
    cands = []
    for y in range(m, h - m):
        for x in range(m, w - m):
            s = score[y, x]
            if not s > thr:
                continue
            ok = True
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    nx, ny = x + dx, y + dy
                    if (dx, dy) == (0, 0) or not (m <= nx <= w - 1 - m and m <= ny <= h - 1 - m):
                        continue
                    t = score[ny, nx]
                    if not (s > t or (s == t and y * w + x < ny * w + nx)):
                        ok = False
            if ok:
                cands.append((-float(s), y * w + x, x, y, s))
    cands.sort()
    md2 = float(min_distance) * float(min_distance)
    acc = []
    for _, _, x, y, s in cands:
        if len(acc) == max_corners:
            break
        if all(float((x - ax) ** 2 + (y - ay) ** 2) >= md2 for ax, ay, _ in acc):
            acc.append((x, y, s))
    return acc


# ------------------------------------------------------------------------------------ point sets
def border_points(w, h):
    """Every pixel of the four borders (corners included), as integer (x, y)."""
    xs = np.arange(w)
    ys = np.arange(1, h - 1)
    pts = [np.stack([xs, np.zeros_like(xs)], 1), np.stack([xs, np.full_like(xs, h - 1)], 1),
           np.stack([np.zeros_like(ys), ys], 1), np.stack([np.full_like(ys, w - 1), ys], 1)]
    return np.concatenate(pts).astype(F32)


def random_points(w, h, m, seed, margin=2.0):
    """m sub-pixel points over [-margin, w-1+margin] x [-margin, h-1+margin] (some start outside), the first ones replaced
    by the corners, exact last row / column, a NaN, an inf, a point 1/256 px past the last column and half-to-even ties
    of x * 256 / 2^k at levels 0..3."""
    rng = np.random.default_rng(seed)
    pts = np.stack([rng.uniform(-margin, w - 1 + margin, m), rng.uniform(-margin, h - 1 + margin, m)], 1).astype(F32)
    special = [(0, 0), (w - 1, h - 1), (w - 1, 0), (0, h - 1), (np.nan, 3), (4, np.inf), (w - 1 + 1 / 256, 2),
               (10.5 / 256, 2.5 / 256 + 3), (16.5 / 128, 9 + 0.5 / 128), (7.5 / 64 + 5, 3.5 / 64 + 1), (1.5 / 32 + 2, 0.5 / 32 + 4)]
    k = min(m, len(special))
    pts[:k] = np.array(special[:k], F32)
    return pts


# ------------------------------------------------------------------------------------ models
def np_fb_check(fwd, bwd, s, alpha=0.01, beta=0.5):
    """The forward-backward check of include/ofb200.h on one (h, w, 2) pair, float32 throughout (numpy rounds every
    operation on its own)."""
    s, alpha, beta = F32(s), F32(alpha), F32(beta)
    h, w = fwd.shape[:2]
    u, v = fwd[..., 0], fwd[..., 1]
    ii, jj = np.meshgrid(np.arange(h, dtype=np.int64), np.arange(w, dtype=np.int64), indexing="ij")
    with np.errstate(all="ignore"):
        fin = np.isfinite(u) & np.isfinite(v)
        du, dv = s * u, s * v
        ranged = fin & (np.abs(du) < F32(32768)) & (np.abs(dv) < F32(32768))
        X = jj * 256 + np.where(ranged, np.rint(du * F32(256)), F32(0)).astype(np.int64)
        Y = ii * 256 + np.where(ranged, np.rint(dv * F32(256)), F32(0)).astype(np.int64)
        inside = ranged & (X >= 0) & (X <= (w - 1) * 256) & (Y >= 0) & (Y <= (h - 1) * 256)
        X, Y = np.where(inside, X, 0), np.where(inside, Y, 0)
        x0, y0, wx, wy = X >> 8, Y >> 8, X & 255, Y & 255
        x1, y1 = np.where(wx > 0, x0 + 1, x0), np.where(wy > 0, y0 + 1, y0)
        b00, b01, b10, b11 = bwd[y0, x0], bwd[y0, x1], bwd[y1, x0], bwd[y1, x1]
        bfin = np.isfinite(b00).all(-1) & np.isfinite(b01).all(-1) & np.isfinite(b10).all(-1) & np.isfinite(b11).all(-1)
        fx = (wx.astype(F32) * F32(1 / 256))[..., None]
        fy = (wy.astype(F32) * F32(1 / 256))[..., None]
        top = b00 + fx * (b01 - b00)
        bot = b10 + fx * (b11 - b10)
        b = top + fy * (bot - top)
        bu, bv = b[..., 0], b[..., 1]
        eu, ev = s * (u + bu), s * (v + bv)
        e2 = eu * eu + ev * ev
        sbu, sbv = s * bu, s * bv
        mag2 = (du * du + dv * dv) + (sbu * sbu + sbv * sbv)
        cons = np.isfinite(e2) & (e2 <= alpha * mag2 + beta)
    ok = inside & bfin
    status = np.full((h, w), FB_OUTSIDE, np.uint8)
    status[~fin] = FB_FWD_NONFINITE
    status[inside & ~bfin] = FB_BWD_NONFINITE
    status[ok & cons] = FB_CONSISTENT
    status[ok & ~cons] = FB_INCONSISTENT
    err2 = np.where(ok, e2, F32(np.nan)).astype(F32)
    return status, err2


def u_of(c, s):
    """The displacement in px the oracle takes from a coarser vector component c at flow_scale s: (2 c) s in float32."""
    with np.errstate(over="ignore", invalid="ignore"):
        return (np.float32(2) * np.asarray(c, np.float32)) * np.float32(s)


def c_for(u_target, s):
    """A float32 coarser component whose displacement u_of(c, s) is exactly u_target where one exists within a few ulps
    of u_target / 2s, else the nearest float32 to u_target / 2s."""
    u_target = np.asarray(u_target, np.float32)
    c0 = np.asarray(u_target.astype(np.float64) / (2.0 * float(np.float32(s))), np.float32)
    best = c0.copy()
    hit = u_of(c0, s) == u_target
    lo, hi = c0.copy(), c0.copy()
    for _ in range(6):
        lo, hi = np.nextafter(lo, np.float32(-np.inf)), np.nextafter(hi, np.float32(np.inf))
        for cand in (lo, hi):
            take = ~hit & (u_of(cand, s) == u_target)
            best = np.where(take, cand, best)
            hit |= take
    return best


def oracle_warp(oracle, nxt, cum, mode, s):
    h, w = nxt.shape
    return oracle.warp(nxt, w, h, 0, 2, [np.zeros((h, w, 2), np.float32), cum], mode, np.float32(s))


def cta_rows(out_y0g, out_y1g, win):
    """Global rows [yw0, ylim) whose 2x2 blocks some CTA of a strip launch gathers: the first CTA stages from its first
    output row minus R + 1, lowered to an even global row; the last needs rows up to its last output row plus R + 1.
    (Every CTA in between covers a sub-range of this one, and the rule below is the same in each, so the union does not
    depend on the split.)"""
    r = win // 2
    yw0 = out_y0g - r - 1
    yw0 -= yw0 & 1
    return yw0, out_y1g + r + 1


def requested_rows(cum, w, h, mode, out_y0g, out_y1g, win, s=1.0):
    """The rows lk_warp_block_general (csrc/lk_level.cuh) asks for, over every 2x2 block a strip launch gathers:
    (mask of image rows (h,), mask of coarser rows (h >> 1,)).

    Per block at even global (xe, ye), inside the image and before the CTA's ylim, with coarser vector
    cf = cum[min(ye >> 1, ch - 1), min(xe >> 1, cw - 1)] (that coarser row is requested):
      bilinear: U, V = rint(cf * 512 s); if both are in range (|.| < 2^23) and any target of the block is inside the image,
                the three tap rows ye + (V >> 8) + 0..2, clamped to the image (the third also when its weight is 0);
      nearest:  per pixel the truncated target row int(y + v) of a target inside the image;
      both:     the pixel's own row for a pixel inside the image and before ylim whose target is skipped."""
    ch, cw = h >> 1, w >> 1
    yw0, ylim = cta_rows(out_y0g, out_y1g, win)
    ye = np.arange(max(yw0, 0), min(ylim, h), 2)
    xe = np.arange(0, w, 2)
    img = np.zeros(h, bool)
    crow = np.zeros(ch, bool)
    if ye.size == 0:
        return img, crow
    cy = np.minimum(ye >> 1, ch - 1)
    cx = np.minimum(xe >> 1, cw - 1)
    crow[cy] = True
    cf = cum[cy[:, None], cx[None, :]]  # (blocks rows, block columns, 2)
    YE, XE = np.broadcast_arrays(ye[:, None], xe[None, :])
    with np.errstate(invalid="ignore", over="ignore"):
        if mode == 2:
            s512 = np.float32(512.0) * np.float32(s)
            fu, fv = (cf[..., 0] * s512).astype(np.float32), (cf[..., 1] * s512).astype(np.float32)
            ranged = (np.abs(fu) < 8388608.0) & (np.abs(fv) < 8388608.0)
            U = np.where(ranged, np.rint(fu), 0).astype(np.int64)
            V = np.where(ranged, np.rint(fv), 0).astype(np.int64)
            anyt = np.zeros(YE.shape, bool)
            done = {}
            for r in range(2):
                for c in range(2):
                    inimg = (XE + c < w) & (YE + r < h) & (YE + r < ylim)
                    X, Y = ((XE + c) << 8) + U, ((YE + r) << 8) + V
                    d = ranged & inimg & (X >= 0) & (X <= (w - 1) << 8) & (Y >= 0) & (Y <= (h - 1) << 8)
                    done[r, c] = (inimg, d)
                    anyt |= d
            for k in range(3):
                img[np.clip(YE + (V >> 8) + k, 0, h - 1)[anyt]] = True
            for r in range(2):
                for c in range(2):
                    inimg, d = done[r, c]
                    img[(YE + r)[inimg & ~d]] = True
        else:
            s2 = np.float32(2.0) * np.float32(s)
            u, v = (cf[..., 0] * s2).astype(np.float32), (cf[..., 1] * s2).astype(np.float32)
            for r in range(2):
                for c in range(2):
                    inimg = (XE + c < w) & (YE + r < h) & (YE + r < ylim)
                    fx = ((XE + c).astype(np.float32) + u).astype(np.float32)
                    fy = ((YE + r).astype(np.float32) + v).astype(np.float32)
                    inr = (fx > -2147483648.0) & (fx < 2147483648.0) & (fy > -2147483648.0) & (fy < 2147483648.0)
                    nx = np.where(inr, np.trunc(fx), -1).astype(np.int64)
                    ny = np.where(inr, np.trunc(fy), -1).astype(np.int64)
                    d = inimg & inr & (nx >= 0) & (nx < w) & (ny >= 0) & (ny < h)
                    img[ny[d]] = True
                    img[(YE + r)[inimg & ~d]] = True
    return img, crow


def reach_flag(req, y_off, h_local, cum_y_off, cum_h_local):
    """The strip kernel's reach flag as the rule predicts it: a requested row outside the rows held."""
    img, crow = req
    held = np.zeros(img.size, bool)
    held[y_off:y_off + h_local] = True
    cheld = np.zeros(crow.size, bool)
    cheld[cum_y_off:cum_y_off + cum_h_local] = True
    return bool((img & ~held).any() or (crow & ~cheld).any())


@pytest.fixture
def rows(monkeypatch):
    """set(n): force n rows per CTA on every following launch (OFB_LK_ROWS, read by csrc/lk_win.cu on every launch);
    set(None): the cost model's own split."""

    def set_rows(n):
        if n is None:
            monkeypatch.delenv("OFB_LK_ROWS", raising=False)
        else:
            monkeypatch.setenv("OFB_LK_ROWS", str(n))

    set_rows(None)
    return set_rows


# ------------------------------------------------------------------------------------ checked pairs on row strips
FB_UNCHECKED = 5


def held_rows(y0, y1, h, fb_reach):
    """Rows of the level-0 backward total a strip's check holds: its own rows [y0, y1) and fb_reach more either side."""
    return max(0, y0 - fb_reach), min(h, y1 + fb_reach + 1)


def tap_rows_outside(fwd, y0, h, b0, b1, s):
    """For own rows fwd ((rows, w, 2), global rows y0 ..) of a frame h rows high: which pixels read backward taps at all
    (their whole-frame status is CONSISTENT, INCONSISTENT or BWD_NONFINITE) and which of those have a tap of non-zero
    weight outside rows [b0, b1)."""
    s = F32(s)
    rows, w = fwd.shape[:2]
    u, v = fwd[..., 0], fwd[..., 1]
    ii, jj = np.meshgrid(np.arange(y0, y0 + rows, dtype=np.int64), np.arange(w, dtype=np.int64), indexing="ij")
    with np.errstate(all="ignore"):
        fin = np.isfinite(u) & np.isfinite(v)
        du, dv = s * u, s * v
        ranged = fin & (np.abs(du) < F32(32768)) & (np.abs(dv) < F32(32768))
        X = jj * 256 + np.where(ranged, np.rint(du * F32(256)), F32(0)).astype(np.int64)
        Y = ii * 256 + np.where(ranged, np.rint(dv * F32(256)), F32(0)).astype(np.int64)
    reads = ranged & (X >= 0) & (X <= (w - 1) * 256) & (Y >= 0) & (Y <= (h - 1) * 256)
    ty0 = Y >> 8
    ty1 = np.where(Y & 255, ty0 + 1, ty0)
    return reads, reads & ((ty0 < b0) | (ty1 >= b1))


def assert_equals_whole(ranks, whole, want_err2, what):
    """Checks the flags (bit 2 allowed) and every rank's outputs of a checked pair (dist.NativeStrips made with fb_reach)
    against its rows of the whole-frame result `whole` (Context.flow_pairs_fb_device), with the pixels whose taps leave
    the held rows -- predicted from the whole-frame forward total -- UNCHECKED and err2 NaN."""
    import torch

    fwd, bwd, st, e2 = whole
    for ns in ranks:
        ns.check(allow_unchecked=True)
        y0, y1 = ns.own_rows(0)
        b0, b1 = held_rows(y0, y1, ns.h, ns.fb_reach)
        _, out = tap_rows_outside(fwd[0, y0:y1].cpu().numpy(), y0, ns.h, b0, b1, ns.flow_scale)
        out = torch.from_numpy(out).to(st.device)
        gf, gb, gs, ge = ns.own_fb()
        assert_same_bits(gf, fwd[0, y0:y1], f"{what} rank {ns.rank}: forward total")
        assert_same_bits(gb, bwd[0, y0:y1], f"{what} rank {ns.rank}: backward total")
        ref_st = torch.where(out, torch.full_like(st[0, y0:y1], FB_UNCHECKED), st[0, y0:y1])
        assert bool((gs == ref_st).all()), f"{what} rank {ns.rank}: status ({int((gs != ref_st).sum())} differ)"
        if want_err2:
            assert_same_bits(ge, torch.where(out, torch.full_like(ge, float("nan")), e2[0, y0:y1]), f"{what} rank {ns.rank}: err2")


# ------------------------------------------------------------------------------------ the frame stream
_STREAM_SHIFTS = [(0.0, 0.0), (1.5, -0.5), (2.25, 0.75), (0.5, 2.0), (-1.0, 1.25), (3.0, -1.5)]


def bgr_sequence(oracle, w, h, seed=61):
    return [oracle.make_bgr_frame(w, h, dx, dy, 8, seed) for dx, dy in _STREAM_SHIFTS]


def pyramid_launches(levels):
    return levels // 2  # two pyramid steps per launch where two are left: ceil((levels - 1) / 2)
