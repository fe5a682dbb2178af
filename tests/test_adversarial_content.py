"""Parity on worst-case image content.

The other parity tests draw their frames from oracle.make_frame (smooth value noise).  The kernels' correctness rests on
value-range claims that smooth content never comes near:
  * prev and warped next share one 32-bit word per pixel, and the 3x3 stencils' partial sums stay below 2^16
    (csrc/lk_level.cuh, lk_v_row: Ix / Iy as two int16 halves, It by dp2a);
  * the five window sums are int32 running sums with wrap-around updates: |sum| <= WIN^2 * 1020 * 3825 < 2^31 for
    WIN <= 19;
  * the pyramid's packed [1 2 1] sums stay below 2^12 (an all-255 image reaches 4080);
  * the hand-written reciprocal lk_rcp is nvcc's for 0 or an integer determinant of magnitude 1 .. 2^62;
  * the tolerance-mode solve (SOLVE_FAST) stays within 1e-4 px + 1e-5 |ref| of the reference's double-precision solve
    with non-finite values on the same pixels -- also where |SIxIy| > 94,906,265, so that the reference's b*b rounds
    and its determinant of an exactly one-dimensional window is the rounding residue instead of 0.
The generators of support.PAIRS reach those ranges: flat 0 / 255 frames, binary and uniform noise, 1- and 2-px checkerboards,
vertical stripes of period 4 (|Ix| = 1020 at every pixel), diagonal and anti-diagonal stripes of periods 4, 6 and 8
(|SIxIy| beyond 2^26.5 at windows 17 and 19 for periods 6 and 8), single-pixel impulses, half-frame 0 -> 255 steps and
the pair 0 -> 255 (|It| = 3825 everywhere).

CPU tests (no mark) check on the oracle's exact integer sums that the inputs really reach those ranges and stay inside
int32, and check a numpy model of the tolerance-mode solve against the oracle.  GPU tests compare the kernels with the
oracle on the same content: bit for bit in EXACT mode and in the pyramid, within the stated bar in FAST mode.
"""
from fractions import Fraction

import numpy as np
import pytest

from support import (PAIRS, TOL_ABS, TOL_REL, assert_flow_within_tolerance, assert_values_equal, binary_noise, checkerboard,
                     device_frames, diagonal_stripes, fast_ctx, flat, roll_x, solve, to_device)  # noqa: F401 (fast_ctx is a fixture)

WINDOWS = [3, 5, 7, 9, 11, 13, 15, 17, 19]
SXY_EXACT_MAX = 94906265  # largest |b| with b*b < 2^53: beyond it the reference's b*b rounds in double


# ------------------------------------------------------------------------------------ content generators (PAIRS: support.py)
# single frames for the pyramid
FRAMES = {
    "full": lambda w, h: flat(w, h, 255),
    "binary_noise": lambda w, h: binary_noise(w, h, 41),
    "checker1": lambda w, h: checkerboard(w, h, 1),
}


# ------------------------------------------------------------------------------------ model of the tolerance-mode solve
def _fma(x: float, y: float, z: float) -> float:
    """x*y + z rounded once to double (Fraction arithmetic is exact; int / int true division rounds correctly)."""
    return float(Fraction(x) * Fraction(y) + Fraction(z))


def _exact_solve_one(a: int, b: int, d: int, tx: int, ty: int):
    """The reference's double-precision sequence (g_inv_matrix_float as nvcc contracts it, oracle orc_solve_one)."""
    bb = float(b) * float(b)
    det = float(a * d - int(bb))  # fma(a, d, -(b*b)): a*d is exact inside the fma, b*b is an integer-valued double
    if det == 0.0:
        return np.nan, np.nan
    pre = 1.0 / det
    ap, bp, dp = a * pre, b * pre, d * pre
    return np.float32(_fma(bp, ty, -(dp * tx))), np.float32(_fma(bp, tx, -(ap * ty)))


def fast_solve_model(sums, fallback: bool = True) -> np.ndarray:
    """lk_solve4_fast in numpy: int64 determinant and numerators, each rounded once to float32, times the float32
    reciprocal of the determinant (an IEEE division here; the kernel's rcp.approx is within an ulp of it).  With
    `fallback`, pixels with |SIxIy| > SXY_EXACT_MAX take the reference's double-precision sequence instead, as the
    kernel does."""
    a, d, b, tx, ty = (np.asarray(s, np.int64) for s in sums)
    fd = (a * d - b * b).astype(np.float32)
    fu = (b * ty - d * tx).astype(np.float32)
    fv = (b * tx - a * ty).astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        r = np.float32(1.0) / fd
        flow = np.stack([fu * r, fv * r], axis=-1)
    if fallback:
        for i, j in np.argwhere(np.abs(b) > SXY_EXACT_MAX):
            flow[i, j] = _exact_solve_one(int(a[i, j]), int(b[i, j]), int(d[i, j]), int(tx[i, j]), int(ty[i, j]))
    return flow


def count_beyond(got: np.ndarray, ref: np.ndarray) -> int:
    """Pixels outside the tolerance-mode bar: finite in one and not the other, or |d| > TOL_ABS + TOL_REL |ref|."""
    fg, fr = np.isfinite(got), np.isfinite(ref)
    with np.errstate(invalid="ignore"):
        far = fg & fr & (np.abs(got.astype(np.float64) - ref) > TOL_ABS + TOL_REL * np.abs(ref))
    return int(((fg != fr) | far).any(axis=-1).sum())


# ------------------------------------------------------------------------------------ CPU: ranges and the solve model
CPU_W, CPU_H = 96, 64


@pytest.mark.parametrize("name", sorted(PAIRS))
def test_window_sums_fit_int32(oracle, name):
    """The kernel keeps the five window sums as int32 running sums: every generator, every window."""
    prev, nxt = PAIRS[name](CPU_W, CPU_H)
    for win in WINDOWS:
        for q, s in zip(("Sxx", "Syy", "Sxy", "Sxt", "Syt"), oracle.lk_level_sums(prev, nxt, win)):
            assert np.abs(s).max() < 2 ** 31, f"{name} win {win}: {q} reaches {np.abs(s).max()}"


def test_generators_reach_the_claimed_ranges(oracle):
    """The content stays adversarial: if a generator quietly became tame, the GPU tests would prove nothing."""
    prev, nxt = PAIRS["vstripes4"](CPU_W, CPU_H)
    assert np.abs(oracle.conv(prev, oracle.DX))[1:-1, 1:-1].min() == 1020  # |Ix| = 1020 at every interior pixel
    assert oracle.lk_level_sums(prev, nxt, 19)[0].max() == 361 * 1020 ** 2
    for name in ("zero_to_full", "full_to_zero"):
        prev, nxt = PAIRS[name](CPU_W, CPU_H)
        it = oracle.conv(nxt, oracle.DT) - oracle.conv(prev, oracle.DT)
        assert np.abs(it).max() == 3825, name
    # |SIxIy| beyond 94,906,265 (b*b inexact in double) for diagonal stripes of period 6 at windows 17 and 19 and of
    # period 8 at 19; period 4 stays below it
    big = {(name, win): np.abs(oracle.lk_level_sums(*PAIRS[name](CPU_W, CPU_H), win)[2]).max()
           for name in ("diag4", "diag6", "diag8", "adiag4", "adiag6", "adiag8") for win in (15, 17, 19)}
    for anti in ("", "a"):
        assert big[(anti + "diag6", 17)] > SXY_EXACT_MAX and big[(anti + "diag6", 19)] > SXY_EXACT_MAX
        assert big[(anti + "diag8", 19)] > SXY_EXACT_MAX
        assert max(big[(anti + "diag4", win)] for win in (15, 17, 19)) <= SXY_EXACT_MAX
        assert max(big[(anti + p, 15)] for p in ("diag4", "diag6", "diag8")) <= SXY_EXACT_MAX


@pytest.mark.parametrize("name", sorted(PAIRS))
def test_fast_solve_model_within_tolerance_of_exact_oracle(oracle, name):
    """The tolerance-mode solve, modelled in numpy from the oracle's exact sums, meets its bar on every generator and
    window: the same non-finite pixels as the double-precision solve, |du|, |dv| <= 1e-4 + 1e-5 |ref| elsewhere."""
    prev, nxt = PAIRS[name](CPU_W, CPU_H)
    for win in WINDOWS:
        ref = oracle.lk_level(prev, nxt, win, oracle.SUMS_EXACT)
        model = fast_solve_model(oracle.lk_level_sums(prev, nxt, win))
        assert np.array_equal(np.isfinite(model), np.isfinite(ref)), f"{name} win {win}: finite masks differ"
        assert count_beyond(model, ref) == 0, f"{name} win {win}"


@pytest.mark.parametrize("period,counts", [(4, {9: 0, 13: 0, 15: 0, 17: 0, 19: 0}),
                                           (6, {9: 0, 13: 0, 15: 0, 17: 2392, 19: 2230}),
                                           (8, {19: 3344})])
def test_integer_solve_alone_breaks_on_diagonal_stripes(oracle, period, counts):
    """Why the tolerance-mode solve falls back to the double-precision sequence where |SIxIy| > 94,906,265: without
    that, the integer determinant of these exactly one-dimensional windows is 0 and the solve gives inf / NaN where the
    reference's determinant is the rounding residue of b*b and its flow is finite.  Counts of such pixels on a 96x64
    pair (diagonal stripes, next = prev moved 1 px in x); none remain with the fallback."""
    prev = diagonal_stripes(CPU_W, CPU_H, period)
    nxt = roll_x(prev)
    for win, n in counts.items():
        ref = oracle.lk_level(prev, nxt, win, oracle.SUMS_EXACT)
        sums = oracle.lk_level_sums(prev, nxt, win)
        raw = fast_solve_model(sums, fallback=False)
        lost = int((np.isfinite(ref) & ~np.isfinite(raw)).any(axis=-1).sum())
        assert lost == n, f"period {period} win {win}: {lost} pixels finite in the reference, not in the integer solve"
        assert count_beyond(raw, ref) == n, f"period {period} win {win}: other pixels beyond the tolerance"
        assert count_beyond(fast_solve_model(sums), ref) == 0, f"period {period} win {win} with the fallback"


# ------------------------------------------------------------------------------------ GPU
GPU_W, GPU_H = 203, 117  # more than one tile in both directions, odd width


def _coarsest(c, prev, nxt, win):
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w = prev.shape[1]
    flow = c.lk_level_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, win, cum_in=None)
    torch.cuda.synchronize()
    return flow.cpu().numpy()[0]


@pytest.mark.gpu
@pytest.mark.parametrize("win", WINDOWS)
@pytest.mark.parametrize("name", sorted(PAIRS))
def test_coarsest_level_identical_to_exact_oracle(ctx, oracle, name, win):
    """Bit for bit, including the diagonal-stripe windows whose double-precision determinant is a rounding residue
    (lk_rcp away from the determinants smooth content produces)."""
    prev, nxt = PAIRS[name](GPU_W, GPU_H)
    assert_values_equal(_coarsest(ctx, prev, nxt, win), oracle.lk_level(prev, nxt, win, oracle.SUMS_EXACT), f"{name} win {win}")


@pytest.mark.gpu
@pytest.mark.parametrize("win", WINDOWS)
@pytest.mark.parametrize("name", sorted(PAIRS))
def test_coarsest_level_fast_solve_within_tolerance(fast_ctx, oracle, name, win):
    prev, nxt = PAIRS[name](GPU_W, GPU_H)
    ref = oracle.lk_level(prev, nxt, win, oracle.SUMS_EXACT)
    assert_flow_within_tolerance(_coarsest(fast_ctx, prev, nxt, win), ref, f"{name} win {win}")


WARPED = ["binary_noise", "checker1", "diag6", "step_x", "zero_to_full"]


@pytest.mark.gpu
@pytest.mark.parametrize("want_total", [False, True])
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("w,h", [(256, 160), (262, 150)])
@pytest.mark.parametrize("win", [9, 19])
@pytest.mark.parametrize("name", WARPED)
def test_warped_levels_identical_to_oracle(ctx, oracle, name, win, w, h, mode, want_total):
    """Three levels through the batch entry point, every warp mode: residual flow of every level and the cumulative
    flow bit-identical to the oracle.  Adversarial content makes the coarser flow huge or non-finite in places, which
    sends blocks down the general gather path.  262x150 has odd coarser widths."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    levels = 3
    prev, nxt = PAIRS[name](w, h)
    total = torch.empty((1, h, w, 2), dtype=torch.float32, device="cuda") if want_total else None
    flows = ctx.flow_pairs_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, levels, win, warp_mode=mode,
                                  total_flow=total)
    torch.cuda.synchronize()
    ref, cums = oracle.flow_pair(prev, nxt, levels, win, mode, oracle.SUMS_EXACT, 1.0, want_cum=True)
    for k in range(levels - 1, -1, -1):
        assert_values_equal(flows[k][0].cpu().numpy(), ref[k], f"{name} win {win} level {k} mode {mode}")
    if want_total:
        assert_values_equal(total[0].cpu().numpy(), cums[0], f"{name} win {win} total flow")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("name,win", [("diag6", 17), ("diag6", 19), ("diag8", 19), ("adiag6", 17), ("adiag6", 19),
                                      ("adiag8", 19)])
def test_fast_solve_every_level_on_diagonal_stripes(ctx, oracle, name, win, mode):
    """The tolerance-mode kernel per level on the EXACT pipeline's inputs (pyramid level + coarser cumulative flow), on
    content whose |SIxIy| passes 94,906,265: residual and cumulative flow within the bar, same non-finite pixels."""
    import torch

    from cuda_optical_flow_2_b200 import SOLVE_FAST, planar_to_device

    w, h, levels = 256, 160, 3
    prev, nxt = PAIRS[name](w, h)
    assert np.abs(oracle.lk_level_sums(prev, nxt, win)[2]).max() > SXY_EXACT_MAX
    ref, cums = oracle.flow_pair(prev, nxt, levels, win, mode, oracle.SUMS_EXACT, 1.0, want_cum=True)
    pp, pn = oracle.gauss_pyramid(prev, levels), oracle.gauss_pyramid(nxt, levels)
    with solve(ctx, SOLVE_FAST):
        for k in range(levels - 1, -1, -1):
            cum_in = None if k == levels - 1 else torch.from_numpy(cums[k + 1][None].copy()).cuda()
            cum_out = torch.empty((1, h >> k, w >> k, 2), dtype=torch.float32, device="cuda")
            flow = ctx.lk_level_device(planar_to_device(pp[k][None]), planar_to_device(pn[k][None]), w >> k, win,
                                       cum_in=cum_in, warp_mode=mode, cum_out=cum_out)
            torch.cuda.synchronize()
            assert_flow_within_tolerance(flow.cpu().numpy()[0], ref[k], f"{name} mode {mode} level {k}")
            assert_flow_within_tolerance(cum_out.cpu().numpy()[0], cums[k], f"{name} mode {mode} level {k} cumulative",
                                         ulps=False)


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(101, 77), (2000, 70), (36, 300), (640, 480)])
@pytest.mark.parametrize("name", sorted(FRAMES))
def test_pyramid_byte_exact(ctx, oracle, name, w, h):
    """One and two pyramid steps on the content that drives the packed [1 2 1] sums to their top (4080 on all-255)."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    imgs = np.stack([FRAMES[name](w, h), 255 - FRAMES[name](w, h)])
    d = ctx.pyr_down_device(planar_to_device(imgs), w)
    d1, d2 = ctx.pyr_down2_device(planar_to_device(imgs), w)
    torch.cuda.synchronize()
    for i in range(len(imgs)):
        r1 = oracle.pyr_down(imgs[i])
        assert np.array_equal(d.cpu().numpy()[i, :, : w >> 1], r1), f"image {i}"
        assert np.array_equal(d1.cpu().numpy()[i, :, : w >> 1], r1), f"image {i} two steps, level +1"
        assert np.array_equal(d2.cpu().numpy()[i, :, : w >> 2], oracle.pyr_down(r1)), f"image {i} two steps, level +2"


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_mixed_batch_pairs_stay_apart(ctx, oracle, mode):
    """A batch mixing smooth and extreme pairs: every pair equals its single-pair run (extreme content must not leak into
    a neighbour's tiles) and, with the exact solve, the oracle."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, levels, win = 256, 160, 3, 19
    smooth = (oracle.make_frame(w, h, 0, 0, 8, 77), oracle.make_frame(w, h, 1.5, -0.75, 8, 77))
    pairs = [smooth, PAIRS["diag6"](w, h), smooth, PAIRS["zero_to_full"](w, h), PAIRS["binary_noise"](w, h),
             PAIRS["checker1"](w, h)]
    prevs, nexts = np.stack([p for p, _ in pairs]), np.stack([q for _, q in pairs])
    with solve(ctx, mode):
        batch = ctx.flow_pairs_device(planar_to_device(prevs), planar_to_device(nexts), w, levels, win)
        singles = [ctx.flow_pairs_device(planar_to_device(prevs[i:i + 1]), planar_to_device(nexts[i:i + 1]), w, levels, win)
                   for i in range(len(pairs))]
        torch.cuda.synchronize()
    for i in range(len(pairs)):
        ref = oracle.flow_pair(prevs[i], nexts[i], levels, win, 2, oracle.SUMS_EXACT) if mode == 0 else None
        for k in range(levels):
            got = batch[k][i].cpu().numpy()
            assert np.array_equal(got.view(np.uint32), singles[i][k][0].cpu().numpy().view(np.uint32)), f"pair {i} level {k}"
            if ref is not None:
                assert_values_equal(got, ref[k], f"pair {i} level {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(262, 150), (256, 160)])
def test_padding_bytes_are_never_read(ctx, oracle, w, h):
    """Device frames whose rows are padded only to a 16-byte pitch (w + 16 where w is already a multiple of 16), and a
    batch whose images lie further apart than pitch * h, with every padding byte 0xFF: results equal the zero-padded
    64-byte-pitch layout and the oracle."""
    import ctypes as C

    import torch

    from cuda_optical_flow_2_b200 import OfbParams, planar_to_device
    from cuda_optical_flow_2_b200.api import align_up
    from cuda_optical_flow_2_b200._lib import check

    levels, win, mode = 3, 9, 2
    pitch = align_up(w, 16) if w % 16 else w + 16
    pairs = [PAIRS["binary_noise"](w, h), PAIRS["diag6"](w, h)]
    prevs, nexts = np.stack([p for p, _ in pairs]), np.stack([q for _, q in pairs])
    n = len(pairs)
    plain = ctx.flow_pairs_device(planar_to_device(prevs), planar_to_device(nexts), w, levels, win, warp_mode=mode)
    plain = [f.cpu().numpy() for f in plain]

    # pitch align_up(w, 16) through the Python entry points (image stride = pitch * h)
    pad = ((0, 0), (0, 0), (0, pitch - w))
    dp, dn = to_device(np.pad(prevs, pad, constant_values=0xFF)), to_device(np.pad(nexts, pad, constant_values=0xFF))
    flows = ctx.flow_pairs_device(dp, dn, w, levels, win, warp_mode=mode)
    top = ctx.lk_level_device(dp, dn, w, win, cum_in=None)
    half = ctx.pyr_down_device(dp, w)
    torch.cuda.synchronize()
    for i in range(n):
        ref = oracle.flow_pair(prevs[i], nexts[i], levels, win, mode, oracle.SUMS_EXACT)
        for k in range(levels):
            assert np.array_equal(flows[k][i].cpu().numpy().view(np.uint32), plain[k][i].view(np.uint32)), f"pair {i} level {k}"
            assert_values_equal(flows[k][i].cpu().numpy(), ref[k], f"pair {i} level {k}")
        assert_values_equal(top[i].cpu().numpy(), oracle.lk_level(prevs[i], nexts[i], win, oracle.SUMS_EXACT), f"pair {i} one level")
        assert np.array_equal(half[i].cpu().numpy()[:, : w >> 1], oracle.pyr_down(prevs[i])), f"pair {i} pyramid"

    # image stride larger than pitch * h, through the C ABI itself
    stride = pitch * (h + 3) + 16
    bp, bn = device_frames(prevs, pitch, stride, 0xFF)[0], device_frames(nexts, pitch, stride, 0xFF)[0]
    out = [torch.empty((n, h >> k, w >> k, 2), dtype=torch.float32, device="cuda") for k in range(levels)]
    total = torch.empty((n, h, w, 2), dtype=torch.float32, device="cuda")
    p = OfbParams(w, h, levels, win, mode, 1.0, n)
    ptrs = (C.c_void_p * levels)(*[f.data_ptr() for f in out])
    check(ctx._lib.ofb_flow_pairs_device(ctx._h, C.byref(p), bp.data_ptr(), bn.data_ptr(), pitch, stride, ptrs,
                                         total.data_ptr(), None))
    torch.cuda.synchronize()
    for i in range(n):
        ref, cums = oracle.flow_pair(prevs[i], nexts[i], levels, win, mode, oracle.SUMS_EXACT, 1.0, want_cum=True)
        for k in range(levels):
            assert np.array_equal(out[k][i].cpu().numpy().view(np.uint32), plain[k][i].view(np.uint32)), f"stride: pair {i} level {k}"
            assert_values_equal(out[k][i].cpu().numpy(), ref[k], f"stride: pair {i} level {k}")
        assert_values_equal(total[i].cpu().numpy(), cums[0], f"stride: pair {i} total flow")
