"""Warped levels on crafted coarser flow, and batches up to the grid limit of 65535 pairs.

The other warped-level tests pass in coarser flow that the library computed itself.  Callers can pass that flow
directly (`ofb_lk_level_device`'s cum_in, the drop-in `ofb_calc_opt_flow_host_u8c3`'s optFlowPyramid[k > level]), and
the flow values decide which of the bilinear gather's four code paths a 2x2 block takes (csrc/lk_level.cuh): the
straight-line gather from the staged window (lk_gather_smem), the image-border gather (lk_gather_border), the
nearest-sample gather (lk_gather_nearest) and the general path on global memory (lk_warp_block_general).  The fields
below are built to reach each path's edges: targets exactly on and one 1/256 step past the last column and row, 1/256-px
rounding ties, negative fractional offsets, blocks whose taps leave the staged window, non-finite and out-of-range
components (one component alone too), and nearest-mode truncations of j + u in (-1, 0) and at |x| >= 2^31.

CPU tests (no mark) restate the warp rule of include/ofb200.h / oracle/lk_oracle.c in numpy and check it against the
oracle byte for byte on every field, and check that the fields really reach what they claim.  GPU tests run one warped
level on each field and compare it with the oracle bit for bit, run the drop-in entry point on a crafted residual
pyramid, and run batches of 32767 to 65535 pairs.
"""
import functools

import numpy as np
import pytest

from support import assert_flow_within_tolerance, assert_values_equal, c_for, noise_pair, oracle_warp, solve, u_of

FLOW_SCALES = [1.0, 8.0 / 15.0, 3.0]
WINDOWS = [3, 9, 11, 19]
SHAPES = [(64, 48), (67, 45), (250, 161), (300, 130)]  # (67, 45): odd coarser width; 250 and 300: several column strips
FLT_MAX = np.float32(np.finfo(np.float32).max)
BELOW_32768 = np.nextafter(np.float32(32768), np.float32(0))


# ------------------------------------------------------------------------------------ helpers
def _coarse_index(w, h):
    """Per pixel of a level, the coarser pixel its vector comes from (indices clamped for odd sizes)."""
    cw, ch = w >> 1, h >> 1
    ti = np.minimum(np.arange(h) >> 1, ch - 1)[:, None]
    tj = np.minimum(np.arange(w) >> 1, cw - 1)[None, :]
    return np.broadcast_to(ti, (h, w)), np.broadcast_to(tj, (h, w))


def pixel_flow(cum, w, h, mode, s):
    """(u, v) in px per pixel of the warped level, as orc_cum_flow and the flow_scale multiply compute them."""
    if mode == 0:  # as written: the vector of coarser pixel (0, 0) for every pixel
        cu, cv = np.full((h, w), cum[0, 0, 0], np.float32), np.full((h, w), cum[0, 0, 1], np.float32)
    else:
        ti, tj = _coarse_index(w, h)
        cu, cv = cum[ti, tj, 0], cum[ti, tj, 1]
    with np.errstate(over="ignore", invalid="ignore"):
        u, v = np.float32(0) + np.float32(2) * cu, np.float32(0) + np.float32(2) * cv
        if np.float32(s) != np.float32(1):
            u, v = u * np.float32(s), v * np.float32(s)
    return u.astype(np.float32), v.astype(np.float32)


def bilinear_targets(u, v, w, h, range_test=True):
    """8.8 fixed-point targets X, Y and the mask of warped (not skipped) pixels."""
    jj, ii = np.meshgrid(np.arange(w), np.arange(h))
    with np.errstate(invalid="ignore"):
        ranged = (np.abs(u) < 32768) & (np.abs(v) < 32768) if range_test else np.ones(u.shape, bool)
        U = np.where(ranged, np.rint(u * np.float32(256)), 0).astype(np.int64)
        V = np.where(ranged, np.rint(v * np.float32(256)), 0).astype(np.int64)
    X, Y = jj * 256 + U, ii * 256 + V
    ok = ranged & (X >= 0) & (X <= (w - 1) * 256) & (Y >= 0) & (Y <= (h - 1) * 256)
    return X, Y, ok, ranged


def nearest_targets(u, v, w, h):
    """float add j + u, truncation toward zero; the mask of pixels whose target is inside the image and int range."""
    jj, ii = np.meshgrid(np.arange(w, dtype=np.float32), np.arange(h, dtype=np.float32))
    with np.errstate(invalid="ignore", over="ignore"):
        fx, fy = (jj + u).astype(np.float32), (ii + v).astype(np.float32)
        inr = (fx > -2147483648.0) & (fx < 2147483648.0) & (fy > -2147483648.0) & (fy < 2147483648.0)
        nx = np.where(inr, np.trunc(fx), -1).astype(np.int64)
        ny = np.where(inr, np.trunc(fy), -1).astype(np.int64)
    ok = inr & (nx >= 0) & (nx < w) & (ny >= 0) & (ny < h)
    return fx, fy, nx, ny, ok


def warp_model(nxt, cum, mode, s, nan_to_zero=False):
    """numpy restatement of orc_warp_u8 at a warped level (level 0 of 2, pyramid [zeros, cum]).  With nan_to_zero the
    bilinear rule converts a NaN component to 0 before anything else (what the staged-window gather did without its
    range test)."""
    h, w = nxt.shape
    u, v = pixel_flow(cum, w, h, mode, s)
    out = nxt.copy()
    n = nxt.astype(np.int64)
    if mode == 2:
        if nan_to_zero:
            u, v = np.where(np.isnan(u), np.float32(0), u), np.where(np.isnan(v), np.float32(0), v)
        X, Y, ok, _ = bilinear_targets(u, v, w, h)
        X, Y = np.where(ok, X, 0), np.where(ok, Y, 0)
        x0, y0, wx, wy = X >> 8, Y >> 8, X & 255, Y & 255
        x1, y1 = np.minimum(x0 + 1, w - 1), np.minimum(y0 + 1, h - 1)
        top = (256 - wx) * n[y0, x0] + wx * n[y0, x1]
        bot = (256 - wx) * n[y1, x0] + wx * n[y1, x1]
        val = ((256 - wy) * top + wy * bot + 32768) >> 16
        out[ok] = val[ok].astype(np.uint8)
    else:
        _, _, nx, ny, ok = nearest_targets(u, v, w, h)
        out[ok] = nxt[ny[ok], nx[ok]]
    return out


# ------------------------------------------------------------------------------------ window geometry (lk_level.cuh)
def tile_width(win):
    """Output columns per tile (LkCfg<WIN>::TWO)."""
    r = win // 2
    return min((128 - 2 * r) // 8, 16) * 8


def anchor_columns(w, win):
    """Coarser column of each column strip's anchor block: the tile's first block column (XB >> 1) + 32, clamped."""
    r, cw = win // 2, w >> 1
    sh = 0 if r & 1 else 1
    cols = []
    for x0 in range(0, w, tile_width(win)):
        c = ((x0 - r - 1 - sh) >> 1) + 32
        cols.append(c if 0 <= c < cw else cw - 1)
    return cols


def anchor_rows(h, win):
    """Coarser rows the anchors of a whole-height CTA come from: chunk starts (yw0 = -R-1, every 16 rows), and the
    clamped last row for the first chunk."""
    r, ch = win // 2, h >> 1
    rows = {ch - 1}
    for y in range(-r - 1, h, 16):
        if 0 <= (y >> 1) < ch:
            rows.add(y >> 1)
    return sorted(rows)


# ------------------------------------------------------------------------------------ crafted fields
# Each returns the coarser flow (h>>1, w>>1, 2) float32 of one pair of a level of w x h; displacements are u_of(c, s).
def field_smooth(w, h, s, rng):
    """A few pixels, smooth: every interior block is served from the staged window."""
    cw, ch = w >> 1, h >> 1
    y, x = np.mgrid[0:ch, 0:cw].astype(np.float64)
    ph = rng.uniform(0, 2 * np.pi, 4)
    u = 1.5 * np.sin(x / 7.0 + ph[0]) + 1.0 * np.cos(y / 5.0 + ph[1])
    v = 1.25 * np.cos(x / 6.0 + ph[2]) - 1.0 * np.sin(y / 9.0 + ph[3])
    return np.stack([c_for(u, s), c_for(v, s)], axis=-1)


def field_ties(w, h, s, rng):
    """u*256 and v*256 at k + 1/2: round half to even, odd and even k, both signs."""
    cw, ch = w >> 1, h >> 1
    k = rng.integers(-1400, 1400, (ch, cw, 2))
    return c_for((k + 0.5) / 256.0, s)


def field_negative_fractions(w, h, s, rng):
    """Negative fractional offsets: floor through >> 8, weights U & 255."""
    cw, ch = w >> 1, h >> 1
    frac = rng.integers(1, 256, (ch, cw, 2)) / 256.0
    whole = rng.integers(0, 4, (ch, cw, 2))
    return c_for(-(whole + frac), s)


def _block_pixels(w, h, rng):
    """Per coarser pixel, one of the level's pixels that take their vector from it, drawn at random: either pixel of
    its 2x2 block, or the last column / row of an odd size, which uses the clamped coarser index."""
    cw, ch = w >> 1, h >> 1
    j = 2 * np.arange(cw)[None, :] + rng.integers(0, 2, (ch, cw))
    i = 2 * np.arange(ch)[:, None] + rng.integers(0, 2, (ch, cw))
    if w & 1:
        j[:, -1] = w - 3 + rng.integers(0, 3, ch)
    if h & 1:
        i[-1, :] = h - 3 + rng.integers(0, 3, cw)
    return i, j


def field_edges(w, h, s, rng):
    """Targets exactly at X = 0, (w-1)*256, (w-1)*256 + 1 and -1 (and the same for Y) from either pixel of a block,
    including the pixels of an odd last column or row, which use the clamped coarser index."""
    cw, ch = w >> 1, h >> 1
    i, j = _block_pixels(w, h, rng)
    kind = rng.integers(0, 3, (ch, cw))  # 0: X edge, 1: Y edge, 2: both
    tx = np.array([0, (w - 1) * 256, (w - 1) * 256 + 1, -1])[rng.integers(0, 4, (ch, cw))]
    ty = np.array([0, (h - 1) * 256, (h - 1) * 256 + 1, -1])[rng.integers(0, 4, (ch, cw))]
    U = np.where(kind != 1, tx - 256 * j, rng.integers(-600, 600, (ch, cw)))
    V = np.where(kind != 0, ty - 256 * i, rng.integers(-600, 600, (ch, cw)))
    return np.stack([c_for(U / 256.0, s), c_for(V / 256.0, s)], axis=-1)


def field_escape_random(w, h, s, rng):
    """Per coarser pixel, flow of 8..40 px in either direction: blocks leave their anchor's window."""
    cw, ch = w >> 1, h >> 1
    mag = rng.uniform(8, 40, (ch, cw, 2)) * rng.choice([-1.0, 1.0], (ch, cw, 2))
    return c_for(mag, s)


def field_escape_checker(w, h, s, rng):
    """A checkerboard of two motions 20 px apart (4 x 4 coarser pixels per cell)."""
    cw, ch = w >> 1, h >> 1
    y, x = np.mgrid[0:ch, 0:cw]
    a, b = np.array([10.25, 4.125]), np.array([-9.75, -5.875])
    sel = ((x // 4 + y // 4) % 2).astype(bool)[..., None]
    return c_for(np.where(sel, a, b), s)


def special_values(s):
    """(u, v) coarser vectors that are non-finite, out of range or at the edge of the range test."""
    nan, inf = np.float32(np.nan), np.float32(np.inf)
    cf = lambda u: np.float32(c_for(u, s))  # noqa: E731
    return [
        (nan, nan), (inf, nan), (-inf, nan), (nan, -inf), (inf, cf(1.5)), (-inf, cf(-2.25)), (cf(0.75), inf),
        (np.float32(1.3), nan), (nan, np.float32(-0.7)), (cf(-3.5), nan), (nan, cf(2.0)),  # one NaN component
        (cf(BELOW_32768), cf(0.5)), (cf(-BELOW_32768), cf(-0.25)), (cf(32768), cf(1.0)), (cf(0.5), cf(-32768)),
        (cf(1e9), np.float32(0)), (np.float32(0), cf(-1e9)), (FLT_MAX, np.float32(1)), (-FLT_MAX, -FLT_MAX),
        (np.float32(1e-40), np.float32(-1e-45)), (np.float32(-0.0), np.float32(-0.0)), (np.float32(-0.0), cf(1.25)),
    ]


def field_nonfinite(w, h, s, rng):
    """Smooth flow with special vectors on interior blocks, on the image border and on the anchor blocks of every
    column strip (at the windows tested)."""
    out = field_smooth(w, h, s, rng)
    cw, ch = w >> 1, h >> 1
    vals = special_values(s)
    ring = [(0, j) for j in range(cw)] + [(ch - 1, j) for j in range(cw)] + [(i, 0) for i in range(ch)] + \
        [(i, cw - 1) for i in range(ch)]
    anchors = sorted({(i, j) for win in WINDOWS for j in anchor_columns(w, win) for i in anchor_rows(h, win)})
    inner = [(int(i), int(j)) for i, j in zip(rng.integers(2, ch - 2, 3 * len(vals)), rng.integers(2, cw - 2, 3 * len(vals)))]
    for group in (inner, [ring[k] for k in rng.permutation(len(ring))[: 2 * len(vals)]], anchors):
        off = int(rng.integers(0, len(vals)))
        for idx, (i, j) in enumerate(group):
            out[i, j] = vals[(idx + off) % len(vals)]
    return out


def field_nearest_edges(w, h, s, rng):
    """Nearest-sample targets j + u in (-1, 0) (truncated to column 0), at exactly -1, just below w, exactly w, and
    beyond int range; the same for rows."""
    cw, ch = w >> 1, h >> 1
    i, j = _block_pixels(w, h, rng)

    def targets(n):
        k = rng.integers(0, 7, (ch, cw))
        choices = np.stack([-rng.integers(1, 1024, (ch, cw)) / 1024.0, np.full((ch, cw), -1.0),
                            np.full((ch, cw), n - 1.0 / 1024.0), np.full((ch, cw), float(n)), np.full((ch, cw), 3.0e9),
                            np.full((ch, cw), -3.0e9), rng.uniform(0, n - 1, (ch, cw))])
        return np.take_along_axis(choices, k[None], 0)[0].astype(np.float32)

    fx, fy = targets(w), targets(h)
    return np.stack([c_for(fx - j.astype(np.float32), s), c_for(fy - i.astype(np.float32), s)], axis=-1)


FIELDS = {
    "smooth": field_smooth,
    "ties": field_ties,
    "negative_fractions": field_negative_fractions,
    "edges": field_edges,
    "escape_random": field_escape_random,
    "escape_checker": field_escape_checker,
    "nonfinite": field_nonfinite,
    "nearest_edges": field_nearest_edges,
}


@functools.lru_cache(maxsize=None)
def _field(name, w, h, s, seed):
    rng = np.random.default_rng([seed, w, h, sorted(FIELDS).index(name)])
    return np.ascontiguousarray(FIELDS[name](w, h, s, rng), np.float32)


def make_field(name, w, h, s, seed=0):
    return _field(name, w, h, float(s), seed).copy()


def expected_cum_out(cum, flow):
    h, w = flow.shape[:2]
    ti, tj = _coarse_index(w, h)
    with np.errstate(over="ignore", invalid="ignore"):
        return (np.float32(2) * cum[ti, tj] + flow).astype(np.float32)


# ------------------------------------------------------------------------------------ CPU: the model and the fields
@pytest.mark.parametrize("s", FLOW_SCALES)
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("name", sorted(FIELDS))
def test_warp_model_equals_oracle(oracle, name, mode, s):
    """The numpy restatement of the warp rule equals orc_warp_u8 byte for byte on every crafted field: this pins the
    oracle on values the reference goldens never contained."""
    for w, h in SHAPES:
        _, nxt = noise_pair(w, h, 5)
        cum = make_field(name, w, h, s)
        assert np.array_equal(warp_model(nxt, cum, mode, s), oracle_warp(oracle, nxt, cum, mode, s)), f"{name} {w}x{h}"


@pytest.mark.parametrize("s", FLOW_SCALES)
def test_fields_reach_their_edges(s):
    """The GPU tests see what they claim: targets exactly at 0, Xmax, Xmax + 1 and -1 on both axes (also from the
    clamped last column / row of odd sizes), ties of both parities and signs, range-skipped targets, one-NaN-component
    vectors, and blocks whose taps leave the staged window of their anchor."""
    for w, h in SHAPES:
        xmax, ymax = (w - 1) * 256, (h - 1) * 256
        u, v = pixel_flow(make_field("edges", w, h, s), w, h, 2, s)
        X, Y, _, _ = bilinear_targets(u, v, w, h)
        for what, T, top in (("X", X, xmax), ("Y", Y, ymax)):
            for t in (0, top, top + 1, -1):
                assert (T == t).sum() > 0, f"{w}x{h} s={s}: no target at {what} = {t}"
        if w & 1:
            assert np.isin(X[:, -1], [0, xmax, xmax + 1, -1]).any(), f"{w}x{h}: last (clamped) column never at an edge"
        if h & 1:
            assert np.isin(Y[-1, :], [0, ymax, ymax + 1, -1]).any(), f"{w}x{h}: last (clamped) row never at an edge"

        u, v = pixel_flow(make_field("ties", w, h, s), w, h, 2, s)
        for c in (u, v):
            t = c.astype(np.float64) * 256
            tie = t - np.floor(t) == 0.5
            k = np.floor(t)[tie]
            assert tie.mean() > 0.5, f"{w}x{h} s={s}: ties on {tie.mean():.2f} of the pixels"
            for par in (0, 1):
                for sign in (-1, 1):
                    assert ((k % 2 == par) & (np.sign(k + 0.5) == sign)).any(), f"{w}x{h} s={s}: tie class {par} {sign}"

        cum = make_field("nonfinite", w, h, s)
        u, v = pixel_flow(cum, w, h, 2, s)
        _, _, ok, ranged = bilinear_targets(u, v, w, h)
        finite = np.isfinite(u) & np.isfinite(v)
        assert (finite & ~ranged).sum() > 0, "no finite target skipped by the range test"
        assert (np.abs(u) == BELOW_32768).any() and (np.abs(u) == 32768).any(), f"s={s}: |u| at the range limit not hit"
        assert (np.isnan(u) ^ np.isnan(v)).sum() > 0, "no one-NaN-component vector"
        assert (np.isnan(cum[..., 0]) & ~np.isnan(cum[..., 1]) & np.isfinite(cum[..., 1])).any()
        assert (~np.isnan(cum[..., 0]) & np.isfinite(cum[..., 0]) & np.isnan(cum[..., 1])).any()
        for win in WINDOWS:  # special values on every column strip's anchor
            for j in anchor_columns(w, win):
                assert not np.isfinite(cum[:, j]).all() or (np.abs(u_of(cum[:, j], s)) >= 32768).any(), (w, win, j)

        for name in ("escape_random", "escape_checker"):
            for win in WINDOWS:
                assert escaping_blocks(make_field(name, w, h, s), w, h, win, s) > 0.1 * (w >> 1) * (h >> 1), (name, win)
        assert escaping_blocks(make_field("smooth", w, h, s), w, h, 9, s) == 0


def escaping_blocks(cum, w, h, win, s):
    """Blocks whose whole-pixel offset differs from the anchor's by more than the staged window's margin (8 columns;
    8 rows up to window 9, 6 above), with the anchor of the block's column strip taken at its 16-row chunk."""
    margin_y = 8 if win <= 9 else 6
    r = win // 2
    u, v = u_of(cum[..., 0], s), u_of(cum[..., 1], s)
    with np.errstate(invalid="ignore"):
        du, dv = np.floor(np.rint(u * 256) / 256), np.floor(np.rint(v * 256) / 256)
    ch, cw = cum.shape[:2]
    cols = anchor_columns(w, win)
    strip = np.minimum((2 * np.arange(cw)) // tile_width(win), len(cols) - 1)
    ac = np.array(cols)[strip]
    chunk_row = np.clip(((((2 * np.arange(ch)) + r + 1) // 16) * 16 - r - 1) >> 1, 0, ch - 1)
    escape = (np.abs(du - du[chunk_row[:, None], ac[None, :]]) > 7) | (np.abs(dv - dv[chunk_row[:, None], ac[None, :]]) > margin_y - 1)
    return int(escape.sum())


@pytest.mark.parametrize("win", [3, 19])
def test_one_wrong_byte_changes_the_flow(oracle, win):
    """On the noise frames, a single changed byte of the warped frame changes oracle.lk_level's flow -- at a corner, an
    edge and the interior -- so a bit-identity test sees one wrong byte."""
    for w, h in ((64, 48), (67, 45)):
        prev, nxt = noise_pair(w, h, 5)
        ref = oracle.lk_level(prev, nxt, win, oracle.SUMS_EXACT)
        for i, j in ((0, 0), (h - 1, w - 1), (0, w // 2), (h // 2, w // 3)):
            bad = nxt.copy()
            bad[i, j] ^= 1
            got = oracle.lk_level(prev, bad, win, oracle.SUMS_EXACT)
            assert not np.array_equal(got.view(np.uint32), ref.view(np.uint32)), f"{w}x{h} byte ({i}, {j})"


@pytest.mark.parametrize("s", FLOW_SCALES)
def test_nan_to_zero_rule_differs_from_the_oracle(oracle, s):
    """A gather that turns a NaN component into 0 (and so samples along the other component) instead of skipping the
    target differs from the oracle on the one-NaN-component vectors: the GPU test on this field fails on such a
    kernel."""
    for w, h in SHAPES:
        _, nxt = noise_pair(w, h, 5)
        cum = make_field("nonfinite", w, h, s)
        ref = oracle_warp(oracle, nxt, cum, 2, s)
        assert np.array_equal(warp_model(nxt, cum, 2, s), ref)
        wrong = warp_model(nxt, cum, 2, s, nan_to_zero=True)
        assert (wrong != ref).sum() > 0, f"{w}x{h}"
        u, v = pixel_flow(cum, w, h, 2, s)
        assert not ((wrong != ref) & ~(np.isnan(u) ^ np.isnan(v))).any(), "differences beyond the one-NaN targets"


def test_probe_example_from_the_rule():
    """The rule on one block: coarser vector (1.3, NaN) at bilinear warp keeps the unwarped pixel; the NaN-to-0 rule
    samples 2.6 px to the right instead."""
    w, h = 40, 24
    nxt = np.random.default_rng(0).integers(0, 256, (h, w), dtype=np.uint8)
    cum = np.zeros((h >> 1, w >> 1, 2), np.float32)
    cum[5, 7] = (1.3, np.nan)
    out, wrong = warp_model(nxt, cum, 2, 1.0), warp_model(nxt, cum, 2, 1.0, nan_to_zero=True)
    assert np.array_equal(out[10:12, 14:16], nxt[10:12, 14:16])
    U = int(np.rint(np.float32(1.3) * np.float32(512)))
    x0, wx = U >> 8, U & 255
    assert wrong[10, 14] == (((256 - wx) * int(nxt[10, 14 + x0]) + wx * int(nxt[10, 15 + x0])) * 256 + 32768) >> 16


# ------------------------------------------------------------------------------------ GPU: one warped level
def _run_level(ctx, oracle, fields, w, h, win, mode, s, want_cum, seed=0):
    """One warped level on a batch of pairs (one crafted field each) through lk_level_device; returns the device
    outputs and the oracle's (warped next -> lk_level) per pair."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    prevs, nexts, cums = [], [], []
    for k, name in enumerate(fields):
        prev, nxt = noise_pair(w, h, 100 + 7 * k + seed)
        prevs.append(prev)
        nexts.append(nxt)
        cums.append(make_field(name, w, h, s, seed + k))
    n = len(fields)
    cum_in = torch.from_numpy(np.stack(cums)).cuda()
    cum_out = torch.empty((n, h, w, 2), dtype=torch.float32, device="cuda") if want_cum else None
    flow = ctx.lk_level_device(planar_to_device(np.stack(prevs)), planar_to_device(np.stack(nexts)), w, win, warp_mode=mode,
                               flow_scale=float(np.float32(s)), cum_in=cum_in, cum_out=cum_out)
    torch.cuda.synchronize()
    flow = flow.cpu().numpy()
    cum_out = cum_out.cpu().numpy() if want_cum else None
    refs = [oracle.lk_level(prevs[k], oracle_warp(oracle, nexts[k], cums[k], mode, s), win, oracle.SUMS_EXACT) for k in range(n)]
    return flow, cum_out, refs, cums


BATCH_PARTNERS = ["nonfinite", "escape_checker", "edges"]


@pytest.mark.gpu
@pytest.mark.parametrize("s", FLOW_SCALES)
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("name", sorted(FIELDS))
def test_warped_level_on_crafted_flow(ctx, oracle, name, mode, s):
    """One warped level on each crafted field, bit-identical to the oracle's warp followed by its level; the cumulative
    output equals 2 cum[i>>1, j>>1] + flow.  Every shape runs at a different window (rotating with the field, so that
    every shape meets every window across the fields); two shapes run as batches of 3 pairs with different fields,
    which covers the pair stride of the coarser tile; the cumulative output alternates on and off."""
    idx = sorted(FIELDS).index(name)
    for k, (w, h) in enumerate(SHAPES):
        win = WINDOWS[(idx + k) % len(WINDOWS)]
        want_cum = (idx + k + mode) % 2 == 0
        fields = [name] if k % 2 == 0 else [BATCH_PARTNERS[(idx + k) % 3], name, BATCH_PARTNERS[(idx + k + 1) % 3]]
        flow, cum_out, refs, cums = _run_level(ctx, oracle, fields, w, h, win, mode, s, want_cum, seed=idx)
        for p in range(len(fields)):
            what = f"{fields[p]} (pair {p}) {w}x{h} win {win} mode {mode} s {s:.4f}"
            assert_values_equal(flow[p], refs[p], what)
            if want_cum:
                assert_values_equal(cum_out[p], expected_cum_out(cums[p], refs[p]), what + " cum_out")


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FIELDS))
def test_warped_level_on_crafted_flow_fast_solve(ctx, oracle, name):
    """The same fields once through the tolerance-mode kernels (separate instantiations of the same gather): within the
    stated bar of the oracle on the oracle's warped frame, non-finite values on the same pixels."""
    from cuda_optical_flow_2_b200 import SOLVE_FAST

    idx = sorted(FIELDS).index(name)
    with solve(ctx, SOLVE_FAST):
        for mode in (0, 1, 2):
            for k, (w, h) in enumerate(SHAPES[1:3]):
                win = WINDOWS[(idx + mode + 2 * k) % len(WINDOWS)]
                s = FLOW_SCALES[(idx + mode) % 3]
                fields = [name, BATCH_PARTNERS[(idx + mode) % 3]]
                flow, cum_out, refs, cums = _run_level(ctx, oracle, fields, w, h, win, mode, s, want_cum=k == 1, seed=idx)
                for p in range(len(fields)):
                    what = f"{fields[p]} {w}x{h} win {win} mode {mode}"
                    assert_flow_within_tolerance(flow[p], refs[p], what)
                    if k == 1:
                        assert_flow_within_tolerance(cum_out[p], expected_cum_out(cums[p], refs[p]), what + " cum_out", ulps=False)


@pytest.mark.gpu
@pytest.mark.parametrize("s", FLOW_SCALES)
def test_as_written_one_vector_per_pair(ctx, oracle, s):
    """Warp as written: the coarser vector at (0, 0) moves the whole frame.  A batch in which every pair has a different
    special value there -- the single vector is per pair."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    vals = special_values(s) + [(np.float32(c_for(-0.5, s)), np.float32(c_for(-0.25, s))),
                                (np.float32(c_for(3.75, s)), np.float32(c_for(-2.0, s)))]
    for w, h, win in ((64, 48, 9), (67, 45, 11)):
        prevs, nexts, cums = [], [], []
        for k, val in enumerate(vals):
            prev, nxt = noise_pair(w, h, 300 + k)
            cum = make_field("smooth", w, h, s, k)
            cum[0, 0] = val
            prevs.append(prev)
            nexts.append(nxt)
            cums.append(cum)
        cum_out = torch.empty((len(vals), h, w, 2), dtype=torch.float32, device="cuda")
        flow = ctx.lk_level_device(planar_to_device(np.stack(prevs)), planar_to_device(np.stack(nexts)), w, win, warp_mode=0,
                                   flow_scale=float(np.float32(s)), cum_in=torch.from_numpy(np.stack(cums)).cuda(), cum_out=cum_out)
        torch.cuda.synchronize()
        flow, cum_out = flow.cpu().numpy(), cum_out.cpu().numpy()
        for k in range(len(vals)):
            ref = oracle.lk_level(prevs[k], oracle_warp(oracle, nexts[k], cums[k], 0, s), win, oracle.SUMS_EXACT)
            assert_values_equal(flow[k], ref, f"pair {k} value {vals[k]} {w}x{h}")
            assert_values_equal(cum_out[k], expected_cum_out(cums[k], ref), f"pair {k} cum_out")


# ------------------------------------------------------------------------------------ GPU: the drop-in entry point
@pytest.mark.gpu
@pytest.mark.parametrize("at_origin", [False, True])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_drop_in_entry_on_crafted_residual_pyramid(ctx, oracle, mode, at_origin):
    """calc_opt_flow at level 0 with a crafted 3-level residual pyramid: +inf on level 2 and -inf on level 1 at the same
    position (their composition is NaN in one component only), one-NaN-component and out-of-range vectors, on top of
    escaping flow.  The composition of the caller's residuals (launch_compose_cum) and the warp equal the oracle's.
    at_origin puts the specials at coarser pixel (0, 0), the one vector the as-written warp uses."""
    w, h, levels, win = 132, 90, 3, 9
    prev, nxt = noise_pair(w, h, 77)
    rng = np.random.default_rng(9)
    flows = [np.zeros((h, w, 2), np.float32),
             (rng.uniform(-6, 6, (h >> 1, w >> 1, 2))).astype(np.float32),
             (rng.uniform(-3, 3, (h >> 2, w >> 2, 2))).astype(np.float32)]
    spots = [(0, 0)] if at_origin else [(3, 5), (0, 7), (h // 4 - 1, w // 4 - 1), (10, 0)]
    for n, (i, j) in enumerate(spots + ([] if at_origin else [(12, 20)])):
        flows[2][i, j, n % 2] = np.inf  # level 2 -> x4 at level 0, level 1 -> x2: inf - inf = NaN
        flows[1][2 * i, 2 * j, n % 2] = -np.inf
    if not at_origin:
        flows[1][7, 11] = (1.3, np.nan)
        flows[1][20, 30] = (np.nan, -0.7)
        flows[2][5, 9] = (20000.0, 0.5)  # x4: beyond 32768 px
        flows[1][30, 50] = (np.float32(BELOW_32768) / 2, 0.0)
        flows[2][15, 20] = (np.nan, np.nan)
    for s in (1.0, 8.0 / 15.0):
        got = [f.copy() for f in flows]
        ctx.calc_opt_flow(oracle.to_c3(prev), oracle.to_c3(nxt), w, h, got, 0, levels, win=win, warp_mode=mode,
                          flow_scale=float(np.float32(s)))
        warped = oracle.warp(nxt, w, h, 0, levels, flows, mode, np.float32(s))
        if mode == 2 and not at_origin:
            assert (warp_model_pyr_nan_mix(flows, w, h, s)).any(), "no one-NaN-component target"
        assert_values_equal(got[0], oracle.lk_level(prev, warped, win, oracle.SUMS_EXACT), f"mode {mode} s {s:.4f}")
        for k in (1, 2):
            assert np.array_equal(got[k].view(np.uint32), flows[k].view(np.uint32)), "coarser levels must stay untouched"


def warp_model_pyr_nan_mix(flows, w, h, s):
    """Pixels of level 0 whose composed displacement has exactly one NaN component."""
    ti1, tj1 = _coarse_index(w, h)
    ti2 = np.minimum(np.arange(h) >> 2, (h >> 2) - 1)[:, None]
    tj2 = np.minimum(np.arange(w) >> 2, (w >> 2) - 1)[None, :]
    with np.errstate(invalid="ignore", over="ignore"):
        c = np.float32(4) * flows[2][ti2, tj2] + np.float32(2) * flows[1][ti1, tj1]
    return np.isnan(c[..., 0]) ^ np.isnan(c[..., 1])


# ------------------------------------------------------------------------------------ GPU: batches at the grid limit
PERIOD = 7  # distinct pairs tiled through a batch: pair i is prototype i % 7, so pair or row-block mix-ups do not alias


def _prototypes(oracle, w, h):
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 4, 80 + i) for i in range(PERIOD)])
    nexts = np.stack([oracle.make_frame(w, h, 0.6 + 0.3 * i, 0.9 - 0.25 * i, 4, 80 + i) for i in range(PERIOD)])
    return prevs, nexts


def _tiled(imgs, n):
    from cuda_optical_flow_2_b200 import planar_to_device

    d = planar_to_device(imgs)
    return d.repeat((n + PERIOD - 1) // PERIOD, 1, 1)[:n].contiguous()


def _check_copies(t, n, what, chunk=8192):
    """Every pair of the (n, ...) tensor equals its prototype bit for bit, on the device; returns the prototypes taken from
    the last PERIOD pairs (the batch's tail) as numpy, in prototype order."""
    import torch

    v = t.view(n, -1).view(torch.int32)
    last = torch.arange(n - PERIOD, n, device=t.device)
    proto = torch.empty((PERIOD, v.shape[1]), dtype=torch.int32, device=t.device)
    proto[last % PERIOD] = v[last]
    for a in range(0, n, chunk):
        b = min(a + chunk, n)
        idx = torch.arange(a, b, device=t.device) % PERIOD
        same = (v[a:b] == proto[idx]).all(dim=1)
        if not bool(same.all()):
            first = a + int(torch.nonzero(~same)[0])
            raise AssertionError(f"{what}: pair {first} differs from prototype {first % PERIOD}")
    return proto.view(torch.float32).view((PERIOD,) + tuple(t.shape[1:])).cpu().numpy()


def _free():
    import torch

    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.mark.gpu
@pytest.mark.parametrize("levels", [2, 3])
@pytest.mark.parametrize("n", [32767, 32768])
def test_flow_pairs_device_around_the_per_frame_pyramid_split(ctx, oracle, n, levels):
    """n = 32767 builds both frames' pyramids in one launch (2n <= 65535), n = 32768 in one launch per frame: every copy
    equals its prototype, and the prototypes (from the tail) equal the oracle."""
    w, h, win = 40, 32, 9
    prevs, nexts = _prototypes(oracle, w, h)
    dp, dn = _tiled(prevs, n), _tiled(nexts, n)
    try:
        flows = ctx.flow_pairs_device(dp, dn, w, levels, win)
        for k in range(levels):
            got = _check_copies(flows[k], n, f"n {n} level {k}")
            for i in range(PERIOD):
                ref = oracle.flow_pair(prevs[i], nexts[i], levels, win, 2, oracle.SUMS_EXACT)
                assert_values_equal(got[i], ref[k], f"n {n} prototype {i} level {k}")
    finally:
        del dp, dn
        flows = None
        _free()


@pytest.mark.gpu
@pytest.mark.parametrize("n,w,h", [(65535, 24, 128), (64000, 16, 136)])
def test_tail_split_at_the_grid_limit(ctx, oracle, monkeypatch, n, w, h):
    """One column strip, at least 128 rows: the level-0 kernel cuts the batch's last wave of pairs into 4 row blocks
    each (csrc/lk_win.cu), and its grid z (pairs plus 3 per tail pair) must stay within 65535.  Every copy equals its
    prototype, the prototypes equal the oracle, and the result equals the launch with the tail switched off."""
    import torch

    levels, win = 2, 9
    prevs, nexts = _prototypes(oracle, w, h)
    dp, dn = _tiled(prevs, n), _tiled(nexts, n)
    try:
        flows = ctx.flow_pairs_device(dp, dn, w, levels, win)
        for k in range(levels):
            got = _check_copies(flows[k], n, f"level {k}")
            for i in range(PERIOD):
                ref = oracle.flow_pair(prevs[i], nexts[i], levels, win, 2, oracle.SUMS_EXACT)
                assert_values_equal(got[i], ref[k], f"prototype {i} level {k}")
        monkeypatch.setenv("OFB_LK_TAIL", "0")
        plain = ctx.flow_pairs_device(dp, dn, w, levels, win)
        torch.cuda.synchronize()
        for k in range(levels):
            assert torch.equal(flows[k].view(torch.int32), plain[k].view(torch.int32)), f"level {k}: tail on / off differ"
    finally:
        del dp, dn
        flows = plain = None
        _free()


@pytest.mark.gpu
def test_fb_entry_at_the_grid_limit(ctx, oracle):
    """flow_pairs_fb_device at 65535 pairs: the totals equal two flow_pairs_device calls bit for bit, the status equals
    fb_check_device on those totals, and the forward prototypes equal the oracle."""
    import torch

    n, w, h, levels, win = 65535, 24, 128, 2, 9
    prevs, nexts = _prototypes(oracle, w, h)
    dp, dn = _tiled(prevs, n), _tiled(nexts, n)
    try:
        fwd, bwd, status, _ = ctx.flow_pairs_fb_device(dp, dn, w, levels, win)
        tf = torch.empty_like(fwd)
        ctx.flow_pairs_device(dp, dn, w, levels, win, total_flow=tf)
        assert torch.equal(fwd.view(torch.int32), tf.view(torch.int32)), "forward totals differ"
        del tf
        tb = torch.empty_like(bwd)
        ctx.flow_pairs_device(dn, dp, w, levels, win, total_flow=tb)
        assert torch.equal(bwd.view(torch.int32), tb.view(torch.int32)), "backward totals differ"
        st, _ = ctx.fb_check_device(fwd, tb)
        assert torch.equal(status, st), "status differs from fb_check_device on the totals"
        del tb, st
        got = _check_copies(fwd, n, "forward total")
        for i in range(PERIOD):
            _, cums = oracle.flow_pair(prevs[i], nexts[i], levels, win, 2, oracle.SUMS_EXACT, 1.0, want_cum=True)
            assert_values_equal(got[i], cums[0], f"prototype {i} forward total")
    finally:
        del dp, dn
        fwd = bwd = status = None
        _free()


@pytest.mark.gpu
def test_65536_pairs_are_rejected(ctx):
    import torch

    from cuda_optical_flow_2_b200 import OfbError

    n, w, h = 65536, 16, 16
    img = torch.zeros((n, h, 64), dtype=torch.uint8, device="cuda")
    try:
        for levels in (1, 2):
            with pytest.raises(OfbError):
                ctx.flow_pairs_device(img, img, w, levels, 9)
        with pytest.raises(OfbError):
            ctx.lk_level_device(img, img, w, 9, cum_in=None)
        with pytest.raises(OfbError):
            ctx.flow_pairs_fb_device(img, img, w, 2, 9)
        # and the context still works
        one = ctx.flow_pairs_device(img[:1], img[:1], w, 2, 9)
        torch.cuda.synchronize()
        assert one[0].shape == (1, h, w, 2)
    finally:
        del img
        _free()
