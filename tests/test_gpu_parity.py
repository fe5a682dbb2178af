"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same inputs.

Bars (SURVEY.md section 8c):
  * pyramid levels: byte-exact;
  * flow against the oracle with EXACT window sums: bit-for-bit equal (the kernel does the same
    integer arithmetic and the same double-precision solve), non-finite pixels in the same places;
  * flow against the oracle with the reference's fp32-sequential window sums: equal wherever every
    window sum stays below 2^24 (the fp32 sums are then exact), otherwise max |du|,|dv| <= TOL_ABS
    + TOL_REL*|ref| on pixels where both are finite.
"""
import numpy as np
import pytest

from support import TOL_ABS, TOL_REL, assert_flow_within_tolerance, assert_values_equal, fast_ctx, solve  # noqa: F401

pytestmark = pytest.mark.gpu


def assert_flow_close(got: np.ndarray, ref: np.ndarray, what: str = ""):
    both = np.isfinite(got) & np.isfinite(ref)
    # where the reference's own fp32 rounding made one side non-finite the other may be huge: require
    # agreement of the masks except on (near-)singular pixels, which the caller avoids via textured input
    assert (np.isfinite(got) == np.isfinite(ref)).mean() > 0.9999, what
    d = np.abs(got[both] - ref[both])
    lim = TOL_ABS + TOL_REL * np.abs(ref[both])
    assert (d <= lim).all(), f"{what}: max abs diff {d.max():.3e} exceeds tolerance"


def frames(oracle, w, h, dx=1.0, dy=0.5, cell=4, seed=1234):
    return oracle.make_frame(w, h, 0.0, 0.0, cell, seed), oracle.make_frame(w, h, dx, dy, cell, seed)


# ------------------------------------------------------------------------------------ pyramid
@pytest.mark.parametrize("w,h", [(640, 480), (1920, 1080), (101, 77), (64, 34), (258, 130)])
def test_pyr_down_device_byte_exact(ctx, oracle, w, h):
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    imgs = np.stack([oracle.make_frame(w, h, 0, 0, 4, 100 + i) for i in range(3)])
    d = ctx.pyr_down_device(planar_to_device(imgs), w)
    torch.cuda.synchronize()
    got = d.cpu().numpy()[:, :, : w >> 1]
    for i in range(3):
        assert np.array_equal(got[i], oracle.pyr_down(imgs[i])), f"image {i}"


@pytest.mark.parametrize("w,h", [(640, 480), (1920, 1080), (101, 77), (64, 34), (258, 130), (2000, 70), (36, 300), (4, 4)])
def test_pyr_down2_device_byte_exact(ctx, oracle, w, h):
    """Two pyramid steps in one launch (level +2 formed from the level +1 bytes still in registers) = two oracle steps."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    imgs = np.stack([oracle.make_frame(w, h, 0, 0, 4, 200 + i) for i in range(3)])
    d1, d2 = ctx.pyr_down2_device(planar_to_device(imgs), w)
    torch.cuda.synchronize()
    g1, g2 = d1.cpu().numpy()[:, :, : w >> 1], d2.cpu().numpy()[:, :, : w >> 2]
    for i in range(3):
        r1 = oracle.pyr_down(imgs[i])
        assert np.array_equal(g1[i], r1), f"image {i} level +1"
        assert np.array_equal(g2[i], oracle.pyr_down(r1)), f"image {i} level +2"


@pytest.mark.parametrize("rows", [1, 3, 37])
def test_pyr_down_single_image_many_row_groups(ctx, oracle, rows):
    """One small image: the launcher shortens the row groups (down to 2 rows per thread) to fill the GPU."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h = 520, 4 * rows + 2
    img = oracle.make_frame(w, h, 0, 0, 4, 300 + rows)[None]
    d = ctx.pyr_down_device(planar_to_device(img), w)
    d1, d2 = ctx.pyr_down2_device(planar_to_device(img), w)
    torch.cuda.synchronize()
    r1 = oracle.pyr_down(img[0])
    assert np.array_equal(d.cpu().numpy()[0, :, : w >> 1], r1)
    assert np.array_equal(d1.cpu().numpy()[0, :, : w >> 1], r1)
    assert np.array_equal(d2.cpu().numpy()[0, :, : w >> 2], oracle.pyr_down(r1))


# ------------------------------------------------------------------------------------ single level
@pytest.mark.parametrize("w,h,win", [(640, 480, 5), (640, 480, 9), (320, 240, 19), (203, 117, 15), (64, 64, 3),
                                     (131, 59, 7), (250, 40, 11), (96, 200, 13), (128, 128, 17), (1920, 1080, 9)])
def test_lk_level_coarsest_identical_to_exact_oracle(ctx, oracle, w, h, win):
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    prev, nxt = frames(oracle, w, h)
    flow = ctx.lk_level_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, win, cum_in=None)
    torch.cuda.synchronize()
    got = flow.cpu().numpy()[0]
    ref = oracle.lk_level(prev, nxt, win, oracle.SUMS_EXACT)
    assert_values_equal(got, ref, f"{w}x{h} win {win}")


@pytest.mark.parametrize("w,h,win,cell", [(640, 480, 5, 8), (640, 480, 9, 8), (640, 480, 19, 2), (320, 240, 15, 4)])
def test_lk_level_vs_reference_fp32_sums(ctx, oracle, w, h, win, cell):
    """Against the reference's own rounding (fp32 sequential window sums)."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    prev, nxt = frames(oracle, w, h, cell=cell)
    flow = ctx.lk_level_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, win, cum_in=None)
    torch.cuda.synchronize()
    got = flow.cpu().numpy()[0]
    ref = oracle.lk_level(prev, nxt, win, oracle.SUMS_F32_SEQUENTIAL)
    sums = oracle.lk_level_sums(prev, nxt, win)
    if max(np.abs(s).max() for s in sums) < 2 ** 24:
        assert_values_equal(got, ref, "sums < 2^24: fp32 sums are exact")
    else:
        assert_flow_close(got, ref, "sums >= 2^24")


def test_flat_image_nonfinite_mask(ctx, oracle):
    """det == 0 windows: the reference writes inf/NaN (no threshold, OptFlowGpu.cu:1835); so do we."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h = 160, 96
    prev, nxt = frames(oracle, w, h)
    prev[20:70, 30:120] = 77
    nxt[20:70, 30:120] = 77
    flow = ctx.lk_level_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, 9)
    torch.cuda.synchronize()
    got = flow.cpu().numpy()[0]
    ref = oracle.lk_level(prev, nxt, 9, oracle.SUMS_EXACT)
    assert (~np.isfinite(ref)).sum() > 100
    assert_values_equal(got, ref)


# ------------------------------------------------------------------------------------ multi level
@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("w,h,levels,win", [(640, 480, 4, 9), (322, 246, 3, 5), (1920, 1080, 3, 9)])
def test_flow_pairs_device_identical_to_oracle(ctx, oracle, mode, w, h, levels, win):
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    n = 2
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 8, 500 + i) for i in range(n)])
    nexts = np.stack([oracle.make_frame(w, h, 2.5 + i, -1.25, 8, 500 + i) for i in range(n)])
    total = torch.empty((n, h, w, 2), dtype=torch.float32, device="cuda")
    flows = ctx.flow_pairs_device(planar_to_device(prevs), planar_to_device(nexts), w, levels, win, warp_mode=mode,
                                  total_flow=total)
    torch.cuda.synchronize()
    for i in range(n):
        ref, cums = oracle.flow_pair(prevs[i], nexts[i], levels, win, mode, oracle.SUMS_EXACT, 1.0, want_cum=True)
        for k in range(levels - 1, -1, -1):
            assert_values_equal(flows[k][i].cpu().numpy(), ref[k], f"pair {i} level {k} mode {mode}")
        assert_values_equal(total[i].cpu().numpy(), cums[0], f"pair {i} total flow")


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("win", [3, 7, 11, 13, 15, 17, 19])
@pytest.mark.parametrize("w,h,want_total", [(256, 160, False), (256, 160, True), (262, 150, False)])
def test_every_window_on_warped_levels_identical_to_oracle(ctx, oracle, mode, win, w, h, want_total):
    """The window sizes the other multi-level tests leave out, three levels, every warp mode: even sizes without the total
    flow (level 0 composes the coarser cumulative flow on the fly), with it (level 0 writes it), and a size whose coarser
    widths are odd (no tensor map for the coarser flow, clamped coarse indices)."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    levels = 3
    prev = oracle.make_frame(w, h, 0, 0, 6, 900 + win)
    nxt = oracle.make_frame(w, h, 1.75, -2.5, 6, 900 + win)
    total = torch.empty((1, h, w, 2), dtype=torch.float32, device="cuda") if want_total else None
    flows = ctx.flow_pairs_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, levels, win, warp_mode=mode,
                                  total_flow=total)
    torch.cuda.synchronize()
    ref, cums = oracle.flow_pair(prev, nxt, levels, win, mode, oracle.SUMS_EXACT, 1.0, want_cum=True)
    for k in range(levels - 1, -1, -1):
        assert_values_equal(flows[k][0].cpu().numpy(), ref[k], f"win {win} level {k} mode {mode}")
    if want_total:
        assert_values_equal(total[0].cpu().numpy(), cums[0], f"win {win} total flow")


@pytest.mark.parametrize("case", ["far_shift", "split_motion", "coarse_outliers"])
def test_staged_window_and_fallbacks_identical_to_oracle(ctx, oracle, case):
    """The warped levels gather from a window of `next` staged around the tile, displaced by the local coarser
    flow.  far_shift: a global motion far larger than the window margin (the window follows it); split_motion:
    two halves moving apart, so blocks near the seam leave the window and take the general path; coarse_outliers:
    large flat areas whose unthresholded solve gives inf / NaN / huge flow on the coarser levels."""
    import torch

    from cuda_optical_flow_2_b200 import WARP_BILINEAR, planar_to_device

    w, h, levels, win = 640, 480, 3, 9
    prev = oracle.make_frame(w, h, 0, 0, 8, 4242)
    if case == "far_shift":
        nxt = oracle.make_frame(w, h, 41.5, -27.25, 8, 4242)
    elif case == "split_motion":
        a, b = oracle.make_frame(w, h, 13.0, 9.5, 8, 4242), oracle.make_frame(w, h, -14.5, -11.0, 8, 4242)
        nxt = np.where(np.arange(w)[None, :] < w // 2, a, b).astype(np.uint8)
    else:
        prev = prev.copy()
        prev[100:300, 50:400] = 128  # flat: det == 0 there
        prev[350:, 500:] = 0
        nxt = np.roll(prev, (2, 3), axis=(0, 1))
    total = torch.empty((1, h, w, 2), dtype=torch.float32, device="cuda")
    flows = ctx.flow_pairs_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, levels, win,
                                  warp_mode=WARP_BILINEAR, total_flow=total)
    torch.cuda.synchronize()
    ref, cums = oracle.flow_pair(prev, nxt, levels, win, oracle.WARP_BILINEAR, oracle.SUMS_EXACT, 1.0, want_cum=True)
    for k in range(levels - 1, -1, -1):
        assert_values_equal(flows[k][0].cpu().numpy(), ref[k], f"{case} level {k}")
    assert_values_equal(total[0].cpu().numpy(), cums[0], f"{case} total flow")


def test_flow_scale(ctx, oracle):
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, levels, win = 320, 240, 3, 9
    prev, nxt = frames(oracle, w, h, 3.0, 1.0, 8)
    flows = ctx.flow_pairs_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, levels, win, warp_mode=2,
                                  flow_scale=8.0 / 15.0)
    torch.cuda.synchronize()
    ref = oracle.flow_pair(prev, nxt, levels, win, 2, oracle.SUMS_EXACT, np.float32(8.0 / 15.0))
    for k in range(levels):
        assert_values_equal(flows[k][0].cpu().numpy(), ref[k], f"level {k}")


# ------------------------------------------------------------------------------------ host wrappers
def test_gauss_pyramid_host_c3(ctx, oracle):
    w, h, levels = 640, 480, 4
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)  # channels differ: each is processed independently
    pyr = [img.copy()] + [np.zeros((h >> k, w >> k, 3), np.uint8) for k in range(1, levels)]
    ctx.gauss_pyramid(pyr, w, h, levels)
    for c in range(3):
        ref = oracle.gauss_pyramid(np.ascontiguousarray(img[:, :, c]), levels)
        for k in range(levels):
            assert np.array_equal(pyr[k][:, :, c], ref[k]), f"channel {c} level {k}"


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_calc_opt_flow_host_loop(ctx, oracle, mode):
    """The main.cu:256-262 loop through the drop-in per-level entry point."""
    w, h, levels, win = 320, 240, 3, 9
    prev, nxt = frames(oracle, w, h, 2.0, 1.0, 8)
    pp = oracle.gauss_pyramid(prev, levels)
    pn = oracle.gauss_pyramid(nxt, levels)
    flows = [np.zeros((h >> k, w >> k, 2), np.float32) for k in range(levels)]
    for k in range(levels - 1, -1, -1):
        ctx.calc_opt_flow(oracle.to_c3(pp[k]), oracle.to_c3(pn[k]), w >> k, h >> k, flows, k, levels, win=win,
                          warp_mode=mode)
    ref = oracle.flow_pair(prev, nxt, levels, win, mode, oracle.SUMS_EXACT)
    for k in range(levels):
        assert_values_equal(flows[k], ref[k], f"level {k} mode {mode}")


def test_stage_functions_host(ctx, oracle):
    w, h, win = 200, 120, 7
    prev, nxt = frames(oracle, w, h)
    c3 = oracle.to_c3(prev)
    ix = ctx.conv_3ch_1ch_tiled_uchar_float(c3, w, h, oracle.DX, 3, 3)
    iy = ctx.conv_3ch_1ch_tiled_uchar_float(c3, w, h, oracle.DY, 3, 3)
    it1 = ctx.conv_3ch_1ch_tiled_uchar_float(c3, w, h, oracle.DT, 3, 3)
    it2 = ctx.conv_3ch_1ch_tiled_uchar_float(oracle.to_c3(nxt), w, h, oracle.DT, 3, 3)
    assert np.array_equal(ix, oracle.conv(prev, oracle.DX))
    assert np.array_equal(iy, oracle.conv(prev, oracle.DY))
    assert np.array_equal(it1, oracle.conv(prev, oracle.DT))
    it = it2 - it1
    rng = np.random.default_rng(1)
    fa = (rng.standard_normal((h, w)) * 1000).astype(np.float32)  # non-integer floats: fp32 order must match too
    fb = (rng.standard_normal((h, w)) * 1000).astype(np.float32)
    assert np.array_equal(ctx.srm_1ch_float(fa, fb, w, h, win, win), oracle.srm_f32(fa, fb, win, win))
    sums = [ctx.srm_1ch_float(a, b, w, h, win, win) for a, b in ((ix, ix), (iy, iy), (ix, iy), (ix, it), (iy, it))]
    for s, (a, b) in zip(sums, ((ix, ix), (iy, iy), (ix, iy), (ix, it), (iy, it))):
        assert np.array_equal(s, oracle.srm_f32(a, b, win, win))
    flows = [np.zeros((h, w, 2), np.float32)]
    ctx.inverse_matrix_float(*sums, flows, 0, w, h)
    assert_values_equal(flows[0], oracle.solve_f32(*sums))
    # 5x5 mask with zeros, through the generic path
    m5 = np.arange(25, dtype=np.float32).reshape(5, 5) - 12
    assert np.array_equal(ctx.conv_3ch_1ch_tiled_uchar_float(c3, w, h, m5, 5, 5), oracle.conv(prev, m5))


def test_flow_pairs_host(ctx, oracle):
    w, h, levels, win = 256, 192, 3, 9
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 8, 900 + i) for i in range(3)])
    nexts = np.stack([oracle.make_frame(w, h, 1.5, 2.0 - i, 8, 900 + i) for i in range(3)])
    got1 = ctx.flow_pairs_host(prevs, nexts, levels, win)
    got3 = ctx.flow_pairs_host(np.stack([oracle.to_c3(p) for p in prevs]), np.stack([oracle.to_c3(p) for p in nexts]),
                               levels, win)
    for i in range(3):
        ref = oracle.flow_pair(prevs[i], nexts[i], levels, win, 2, oracle.SUMS_EXACT)
        for k in range(levels):
            assert_values_equal(got1[k][i], ref[k], f"planar pair {i} level {k}")
            assert_values_equal(got3[k][i], ref[k], f"c3 pair {i} level {k}")


# ------------------------------------------------------------------------------------ BASELINE.json configurations
def test_config0_640x480_one_level_win5(ctx, oracle):
    """configs[0]: single 640x480 pair, 1 level, 5x5 window (the case the reference CPU path runs)."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    prev, nxt = frames(oracle, 640, 480, 0.6, -0.4, 8)
    flows = ctx.flow_pairs_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), 640, 1, 5)
    torch.cuda.synchronize()
    assert_values_equal(flows[0][0].cpu().numpy(), oracle.lk_level(prev, nxt, 5, oracle.SUMS_EXACT), "config 0")
    assert_flow_close(flows[0][0].cpu().numpy(), oracle.lk_level(prev, nxt, 5, oracle.SUMS_F32_SEQUENTIAL), "config 0 vs fp32")


def test_config2_4k_four_levels_win15(ctx, oracle):
    """configs[2]: 3840x2160 pair, 4-level pyramid, 15x15 window."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, levels, win = 3840, 2160, 4, 15
    prev, nxt = frames(oracle, w, h, 5.0, -3.0, 16)
    flows = ctx.flow_pairs_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, levels, win)
    torch.cuda.synchronize()
    ref = oracle.flow_pair(prev, nxt, levels, win, 2, oracle.SUMS_EXACT)
    for k in range(levels):
        assert_values_equal(flows[k][0].cpu().numpy(), ref[k], f"4K level {k}")


def test_config3_batch_equals_single_pairs(ctx, oracle):
    """configs[3] property at a reduced count: every pair of a 1080p batch equals the same pair run alone
    (pairs share nothing), and the batch does not depend on the batch size."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, levels, win, n = 1920, 1080, 3, 9, 6
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 8, 40 + i) for i in range(n)])
    nexts = np.stack([oracle.make_frame(w, h, 1.0 + i, 0.5 * i, 8, 40 + i) for i in range(n)])
    dp, dn = planar_to_device(prevs), planar_to_device(nexts)
    batch = [f.clone() for f in ctx.flow_pairs_device(dp, dn, w, levels, win)]
    for i in (0, 3, 5):
        single = ctx.flow_pairs_device(dp[i:i + 1].contiguous(), dn[i:i + 1].contiguous(), w, levels, win)
        torch.cuda.synchronize()
        for k in range(levels):
            a, b = batch[k][i].cpu().numpy(), single[k][0].cpu().numpy()
            assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)])
    ref = oracle.flow_pair(prevs[5], nexts[5], levels, win, 2, oracle.SUMS_EXACT)
    for k in range(levels):
        assert_values_equal(batch[k][5].cpu().numpy(), ref[k], f"batch pair 5 level {k}")


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_big_batch_short_ctas_at_the_tail(ctx, oracle, mode, monkeypatch):
    """A batch of many pairs ends with a wave of short CTAs (csrc/lk_win.cu: the last pairs are cut into 4 row blocks so
    that the launch drains faster).  Small frames, 800 pairs: every copy of a pair -- in the full-height part and in the
    tail -- is bit-identical, equals the oracle, and equals the launch with the tail switched off."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, levels, win, distinct, n = 248, 136, 2, 9, 4, 800
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 4, 70 + i) for i in range(distinct)])
    nexts = np.stack([oracle.make_frame(w, h, 0.7 + i, 1.0 - i, 4, 70 + i) for i in range(distinct)])
    dp = planar_to_device(prevs).repeat(n // distinct, 1, 1)
    dn = planar_to_device(nexts).repeat(n // distinct, 1, 1)
    flows = [f.clone() for f in ctx.flow_pairs_device(dp, dn, w, levels, win, warp_mode=mode)]
    monkeypatch.setenv("OFB_LK_TAIL", "0")
    plain = ctx.flow_pairs_device(dp, dn, w, levels, win, warp_mode=mode)
    torch.cuda.synchronize()
    for k in range(levels):
        f = flows[k].view(torch.int32).view(n // distinct, distinct, -1)
        assert bool((f == f[0:1]).all()), f"level {k}: copies of the same pair differ inside one batch"
        assert bool((flows[k].view(torch.int32) == plain[k].view(torch.int32)).all()), f"level {k}: tail on / off differ"
    for i in range(distinct):
        ref = oracle.flow_pair(prevs[i], nexts[i], levels, win, mode, oracle.SUMS_EXACT)
        for k in range(levels):
            assert_values_equal(flows[k][n - distinct + i].cpu().numpy(), ref[k], f"pair {i} (tail copy), level {k}")


@pytest.mark.parametrize("mode", [0, 1])
def test_config3_one_ranks_share_of_the_full_batch(ctx, oracle, mode):
    """configs[3] at the size one of eight B200 gets (512 of the 4096 pairs of 1080p, the bench's per-launch class): the
    batch is 4 distinct pairs tiled, and every copy must be bit-identical to the first one of its kind in every level --
    a property that does not need the oracle at full size -- while pair 1 is checked against the oracle itself (exact
    solve) or against the tolerance (fast solve)."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, levels, win, distinct, n = 1920, 1080, 3, 9, 4, 512
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 8, 60 + i) for i in range(distinct)])
    nexts = np.stack([oracle.make_frame(w, h, 0.5 + i, 1.5 - i, 8, 60 + i) for i in range(distinct)])
    dp = planar_to_device(prevs).repeat(n // distinct, 1, 1)
    dn = planar_to_device(nexts).repeat(n // distinct, 1, 1)
    with solve(ctx, mode):
        flows = ctx.flow_pairs_device(dp, dn, w, levels, win)
        torch.cuda.synchronize()
    for k in range(levels):
        f = flows[k].view(torch.int32).view(n // distinct, distinct, -1)
        assert bool((f == f[0:1]).all()), f"level {k}: copies of the same pair differ inside one batch"
    ref = oracle.flow_pair(prevs[1], nexts[1], levels, win, 2, oracle.SUMS_EXACT)
    if mode == 0:
        for k in range(levels):
            assert_values_equal(flows[k][n - distinct + 1].cpu().numpy(), ref[k], f"last copy of pair 1, level {k}")
    else:
        got = flows[levels - 1][n - distinct + 1].cpu().numpy()
        fin = np.isfinite(ref[levels - 1])
        assert np.array_equal(np.isfinite(got), fin)
        d = np.abs(got[fin] - ref[levels - 1][fin])
        assert (d <= TOL_ABS + TOL_REL * np.abs(ref[levels - 1][fin])).all()


def test_config4_8k_whole_frame_vs_oracle(ctx, oracle):
    """configs[4] frame (7680x4320, 4 levels, window 9) on one GPU against the oracle; the row-strip
    split of the same frame is checked against this whole-frame result in tests/test_dist.py."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, levels, win = 7680, 4320, 4, 9
    prev, nxt = frames(oracle, w, h, 6.0, 4.0, 16)
    flows = ctx.flow_pairs_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, levels, win)
    torch.cuda.synchronize()
    ref = oracle.flow_pair(prev, nxt, levels, win, 2, oracle.SUMS_EXACT)
    for k in range(levels):
        assert_values_equal(flows[k][0].cpu().numpy(), ref[k], f"8K level {k}")


@pytest.mark.parametrize("w,h,levels,win", [(17, 9, 1, 3), (40, 33, 2, 5), (129, 65, 3, 9), (2, 2, 1, 3), (121, 240, 1, 19)])
def test_small_and_ragged_sizes(ctx, oracle, w, h, levels, win):
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    prev, nxt = frames(oracle, w, h, 0.7, 0.3, 4)
    flows = ctx.flow_pairs_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, levels, win)
    torch.cuda.synchronize()
    ref = oracle.flow_pair(prev, nxt, levels, win, 2, oracle.SUMS_EXACT)
    for k in range(levels):
        assert_values_equal(flows[k][0].cpu().numpy(), ref[k], f"{w}x{h} level {k}")


def test_bad_arguments_are_rejected(ctx):
    import torch

    from cuda_optical_flow_2_b200 import OfbError

    img = torch.zeros((1, 64, 64), dtype=torch.uint8, device="cuda")
    with pytest.raises(OfbError):
        ctx.flow_pairs_device(img, img, 64, 3, 8)  # even window
    with pytest.raises(OfbError):
        ctx.flow_pairs_device(img, img, 64, 7, 9)  # too many levels for 64x64
    with pytest.raises(OfbError):
        ctx.flow_pairs_device(img, img, 64, 2, 21)  # window too large
    bad = torch.zeros((1, 64, 72), dtype=torch.uint8, device="cuda")
    with pytest.raises(OfbError):
        ctx.flow_pairs_device(bad, bad, 64, 1, 9)  # pitch not a multiple of 16


# ------------------------------------------------------------------------------------ tolerance-mode solve (OFB_SOLVE_FAST)
@pytest.mark.parametrize("w,h,win", [(640, 480, 5), (640, 480, 9), (320, 240, 19), (203, 117, 15), (64, 64, 3),
                                     (131, 59, 7), (250, 40, 11), (96, 200, 13), (128, 128, 17), (1920, 1080, 9)])
def test_fast_solve_coarsest_level_within_tolerance(fast_ctx, oracle, w, h, win):
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    prev, nxt = frames(oracle, w, h)
    flow = fast_ctx.lk_level_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, win, cum_in=None)
    torch.cuda.synchronize()
    ref = oracle.lk_level(prev, nxt, win, oracle.SUMS_EXACT)
    assert_flow_within_tolerance(flow.cpu().numpy()[0], ref, f"{w}x{h} win {win}")


def test_fast_solve_flat_areas_same_nonfinite_pixels(fast_ctx, oracle):
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h = 160, 96
    prev, nxt = frames(oracle, w, h)
    prev[20:70, 30:120] = 77
    nxt[20:70, 30:120] = 77
    flow = fast_ctx.lk_level_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, 9)
    torch.cuda.synchronize()
    ref = oracle.lk_level(prev, nxt, 9, oracle.SUMS_EXACT)
    assert (~np.isfinite(ref)).sum() > 100
    assert_flow_within_tolerance(flow.cpu().numpy()[0], ref)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("w,h,levels,win", [(640, 480, 4, 9), (322, 246, 3, 5), (1920, 1080, 3, 9), (400, 300, 3, 15), (256, 160, 3, 3),
                                            (256, 160, 3, 7), (262, 150, 3, 11), (256, 160, 3, 13), (256, 160, 3, 17), (262, 150, 3, 19)])
def test_fast_solve_every_level_on_identical_inputs(ctx, oracle, mode, w, h, levels, win):
    """Per level, on the EXACT pipeline's inputs (pyramid level + coarser cumulative flow): the tolerance-mode
    kernel against the oracle's residual flow and cumulative flow of that level."""
    import torch

    from cuda_optical_flow_2_b200 import SOLVE_FAST, planar_to_device

    prev = oracle.make_frame(w, h, 0, 0, 8, 777)
    nxt = oracle.make_frame(w, h, 3.25, -1.75, 8, 777)
    ref, cums = oracle.flow_pair(prev, nxt, levels, win, mode, oracle.SUMS_EXACT, 1.0, want_cum=True)
    pp, pn = oracle.gauss_pyramid(prev, levels), oracle.gauss_pyramid(nxt, levels)
    with solve(ctx, SOLVE_FAST):
        for k in range(levels - 1, -1, -1):
            cum_in = None if k == levels - 1 else torch.from_numpy(cums[k + 1][None].copy()).cuda()
            cum_out = torch.empty((1, h >> k, w >> k, 2), dtype=torch.float32, device="cuda")
            flow = ctx.lk_level_device(planar_to_device(pp[k][None]), planar_to_device(pn[k][None]), w >> k, win,
                                       cum_in=cum_in, warp_mode=mode, cum_out=cum_out)
            torch.cuda.synchronize()
            assert_flow_within_tolerance(flow.cpu().numpy()[0], ref[k], f"mode {mode} level {k}")
            assert_flow_within_tolerance(cum_out.cpu().numpy()[0], cums[k], f"mode {mode} level {k} cumulative", ulps=False)


def test_fast_solve_whole_pipeline_close_to_exact(fast_ctx, oracle):
    """Through all levels the two modes can part at warped levels (a last-ulp difference of the coarser flow can flip
    its rounding to 1/256 px and so one bilinear weight); report and bound that: almost everywhere inside the
    per-level tolerance, and never by more than a few hundredths of a pixel."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, levels, win = 1920, 1080, 3, 9
    prev = oracle.make_frame(w, h, 0, 0, 8, 31)
    nxt = oracle.make_frame(w, h, 2.5, -1.25, 8, 31)
    total = torch.empty((1, h, w, 2), dtype=torch.float32, device="cuda")
    fast_ctx.flow_pairs_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, levels, win, total_flow=total)
    torch.cuda.synchronize()
    _, cums = oracle.flow_pair(prev, nxt, levels, win, 2, oracle.SUMS_EXACT, 1.0, want_cum=True)
    got, ref = total.cpu().numpy()[0], cums[0]
    assert np.array_equal(np.isfinite(got), np.isfinite(ref))
    fin = np.isfinite(ref)
    d = np.abs(got[fin] - ref[fin])
    lim = TOL_ABS + TOL_REL * np.abs(ref[fin])
    assert (d > lim).mean() < 1e-3, f"{(d > lim).mean():.2e} of the total-flow values beyond the per-level tolerance"
    well = np.abs(ref[fin]) < 100.0  # ill-conditioned windows amplify any input change without bound
    assert d[well].max() < 0.25, f"max |d| {d[well].max():.3e}"


@pytest.mark.parametrize("w,h", [(322, 246), (129, 65), (64, 48)])
def test_flow_pairs_host_c3_layout_any_width(ctx, oracle, w, h):
    """The 3-channel upload path (channel 0 -> planar): widths that are and are not multiples of 4 (vector / scalar
    de-interleave), and the total-flow-only variant of the host call."""
    levels, win = 2, 5
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 4, 300 + i) for i in range(2)])
    nexts = np.stack([oracle.make_frame(w, h, 0.75, -0.5 * i, 4, 300 + i) for i in range(2)])
    got = ctx.flow_pairs_host(np.stack([oracle.to_c3(p) for p in prevs]), np.stack([oracle.to_c3(p) for p in nexts]), levels, win)
    total = ctx.total_flow_pairs_host(prevs, nexts, levels, win)
    for i in range(2):
        ref, cums = oracle.flow_pair(prevs[i], nexts[i], levels, win, 2, oracle.SUMS_EXACT, 1.0, want_cum=True)
        for k in range(levels):
            assert_values_equal(got[k][i], ref[k], f"{w}x{h} pair {i} level {k}")
        assert_values_equal(total[i], cums[0], f"{w}x{h} pair {i} total flow")


@pytest.mark.parametrize("threads,n,w,h", [(1, 5, 130, 66), (4, 20, 322, 246), (3, 26, 64, 48)])
def test_flow_pairs_host_c3_host_threads(ctx, oracle, threads, n, w, h):
    """3-channel host images with channel 0 extracted by host threads into pinned staging buffers (ofb_ctx_set_host_threads):
    identical to the planar call, channels 1 and 2 are never looked at, and the staging buffers of a lane are reused
    across many sub-batches."""
    levels, win = 2, 5
    rng = np.random.default_rng(n)
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 4, 500 + i) for i in range(n)])
    nexts = np.stack([oracle.make_frame(w, h, 0.5, -0.25 * (i % 3), 4, 500 + i) for i in range(n)])
    p3 = rng.integers(0, 256, size=(n, h, w, 3), dtype=np.uint8)
    n3 = rng.integers(0, 256, size=(n, h, w, 3), dtype=np.uint8)
    p3[..., 0], n3[..., 0] = prevs, nexts
    ref = ctx.flow_pairs_host(prevs, nexts, levels, win)
    assert ctx.host_threads == 0
    dev = ctx.flow_pairs_host(p3, n3, levels, win)
    ctx.host_threads = threads
    try:
        assert ctx.host_threads == threads
        for rep in range(2):  # (second call: pool and staging buffers already exist)
            got = ctx.flow_pairs_host(p3, n3, levels, win)
            for k in range(levels):
                assert np.array_equal(got[k].view(np.uint32), ref[k].view(np.uint32)), f"level {k} rep {rep}"
                assert np.array_equal(dev[k].view(np.uint32), ref[k].view(np.uint32)), f"level {k} device extraction"
    finally:
        ctx.host_threads = 0
