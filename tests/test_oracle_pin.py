"""Pins the CPU oracle (oracle/lk_oracle.c) to the reference itself.  Runs without a GPU.

Two sources of truth, neither written by us:
  * tests/golden/ref_gpu_b200.npz -- outputs of the UNMODIFIED reference's GPU functions
    (gpu::conv_3ch_1ch_tiled_uchar_float, gpu::srm_1ch_float, gpu::inverse_matrix_float,
    gpu::gauss_pyramid, gpu::calc_opt_flow) run on a B200 at launch-valid sizes by
    oracle/make_golden.py (inputs are seeded synthetic frames, so only outputs are stored);
  * oracle/_ref/libofref.so -- the reference's CPU-side functions compiled from /root/reference
    (cpu::gauss_pyramid, cpu::shift_back_pyramid, utils::arr_sub_float), when it has been built.
The reference ships no tests or golden vectors of its own (SURVEY.md section 4).
"""
import os

import numpy as np
import pytest

from oracle.make_golden import DERIVATIVES, MULTI, SINGLE, WINDOWS, load
from support import assert_values_equal

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_gpu_b200.npz")


@pytest.fixture(scope="module")
def gold():
    return load(GOLDEN)


def test_golden_file_decodes(gold):
    """The stored form of oracle/make_golden.py gives back float32 arrays of the reference's shapes, and what it stores
    beside them is near zero: a decoding mistake shows here instead of as an oracle mismatch further down."""
    for name, w, h, *_ in SINGLE:
        for k in DERIVATIVES:
            assert gold[f"{name}_{k}"].dtype == np.float32 and gold[f"{name}_{k}"].shape == (h, w)
        for win in WINDOWS:
            assert gold[f"{name}_sums_w{win}"].dtype == np.float32 and gold[f"{name}_sums_w{win}"].shape == (5, h, w)
            assert gold[f"{name}_flow_w{win}"].dtype == np.float32 and gold[f"{name}_flow_w{win}"].shape == (h, w, 2)
        assert gold[f"{name}_entry_flow"].dtype == np.float32 and gold[f"{name}_entry_flow"].shape == (h, w, 2)
    name, w, h, levels, *_ = MULTI
    for k in range(levels):
        assert gold[f"{name}_loop_flow_l{k}"].dtype == np.float32 and gold[f"{name}_loop_flow_l{k}"].shape == (h >> k, w >> k, 2)
    for k in range(1, levels):
        assert gold[f"{name}_pyr_prev_l{k}"].dtype == np.uint8 and gold[f"{name}_pyr_prev_l{k}"].shape == (h >> k, w >> k)
    with np.load(GOLDEN) as z:
        for key in z.keys():
            if key.endswith("_xor_solve"):  # a double-precision solve rounds like the reference's almost everywhere
                assert (z[key] == 0).mean() > 0.99, key
            elif key.endswith("_minus_exact") and np.abs(gold[key[:-len("_minus_exact")]]).max() < 2 ** 24:
                assert not z[key].any(), key  # fp32 accumulation is exact below 2^24
    # the decoder's window sums against a direct sum over every 5x5 window (case a stays below 2^24 at window 5)
    ix, iy = gold["a_ix"].astype(np.int64), gold["a_iy"].astype(np.int64)
    it = (gold["a_it2"] - gold["a_it1"]).astype(np.int64)
    for k, p in enumerate((ix * ix, iy * iy, ix * iy, ix * it, iy * it)):
        direct = np.lib.stride_tricks.sliding_window_view(np.pad(p, 2), (5, 5)).sum(axis=(-2, -1))
        assert np.array_equal(direct, gold["a_sums_w5"][k]), f"sum {k}"


@pytest.mark.parametrize("case", SINGLE, ids=[c[0] for c in SINGLE])
def test_derivatives_match_reference_gpu(oracle, gold, case):
    name, w, h, dx, dy, cell, seed = case
    prev = oracle.make_frame(w, h, 0, 0, cell, seed)
    nxt = oracle.make_frame(w, h, dx, dy, cell, seed)
    assert np.array_equal(oracle.conv(prev, oracle.DX), gold[f"{name}_ix"])
    assert np.array_equal(oracle.conv(prev, oracle.DY), gold[f"{name}_iy"])
    assert np.array_equal(oracle.conv(prev, oracle.DT), gold[f"{name}_it1"])
    assert np.array_equal(oracle.conv(nxt, oracle.DT), gold[f"{name}_it2"])


@pytest.mark.parametrize("win", WINDOWS)
@pytest.mark.parametrize("case", SINGLE, ids=[c[0] for c in SINGLE])
def test_window_sums_solve_and_level_match_reference_gpu(oracle, gold, case, win):
    name, w, h, dx, dy, cell, seed = case
    prev = oracle.make_frame(w, h, 0, 0, cell, seed)
    nxt = oracle.make_frame(w, h, dx, dy, cell, seed)
    ix, iy = gold[f"{name}_ix"], gold[f"{name}_iy"]
    it = gold[f"{name}_it2"] - gold[f"{name}_it1"]
    ref_sums = gold[f"{name}_sums_w{win}"]
    pairs = ((ix, ix), (iy, iy), (ix, iy), (ix, it), (iy, it))
    for k, (a, b) in enumerate(pairs):
        assert np.array_equal(oracle.srm_f32(a, b, win, win), ref_sums[k]), f"sum {k}"
        # the exact integer sums equal the fp32 ones whenever those stayed below 2^24
        if np.abs(ref_sums[k]).max() < 2 ** 24:
            assert np.array_equal(oracle.srm_exact(a, b, win, win), ref_sums[k].astype(np.int64))
    ref_flow = gold[f"{name}_flow_w{win}"]
    assert_values_equal(oracle.solve_f32(*ref_sums), ref_flow)
    assert_values_equal(oracle.lk_level(prev, nxt, win, oracle.SUMS_F32_SEQUENTIAL), ref_flow)
    exact = oracle.lk_level(prev, nxt, win, oracle.SUMS_EXACT)
    if np.abs(ref_sums).max() < 2 ** 24:
        assert_values_equal(exact, ref_flow)
    else:  # fp32 rounding of the reference's sums: stated tolerance of the parity tests
        both = np.isfinite(exact) & np.isfinite(ref_flow)
        assert np.abs(exact[both] - ref_flow[both]).max() <= 1e-4


@pytest.mark.parametrize("case", SINGLE, ids=[c[0] for c in SINGLE])
def test_entry_point_single_level(oracle, gold, case):
    """gpu::calc_opt_flow with level == maxLevel-1 (no warp), window 19."""
    name, w, h, dx, dy, cell, seed = case
    prev = oracle.make_frame(w, h, 0, 0, cell, seed)
    nxt = oracle.make_frame(w, h, dx, dy, cell, seed)
    assert_values_equal(oracle.lk_level(prev, nxt, 19, oracle.SUMS_F32_SEQUENTIAL), gold[f"{name}_entry_flow"])


def test_pyramid_and_coarse_to_fine_loop_match_reference_gpu(oracle, gold):
    name, w, h, levels, dx, dy, cell, seed = MULTI
    prev = oracle.make_frame(w, h, 0, 0, cell, seed)
    nxt = oracle.make_frame(w, h, dx, dy, cell, seed)
    pp, pn = oracle.gauss_pyramid(prev, levels), oracle.gauss_pyramid(nxt, levels)
    for k in range(1, levels):
        assert np.array_equal(pp[k], gold[f"{name}_pyr_prev_l{k}"])
        assert np.array_equal(pn[k], gold[f"{name}_pyr_next_l{k}"])
    flows = oracle.flow_pair(prev, nxt, levels, 19, oracle.WARP_AS_WRITTEN, oracle.SUMS_F32_SEQUENTIAL)
    for k in range(levels - 1, -1, -1):
        ref = gold[f"{name}_loop_flow_l{k}"]
        wk, hk = w >> k, h >> k
        # Pixels the reference's warp skipped hold uninitialised heap beyond the first third of its
        # 3-channel buffer (OptFlowCPU.cpp:247); their influence reaches win/2 + 1 pixels.  The
        # global shift is the flow of pixel (0,0) of every coarser level (OptFlowCPU.cpp:260-261).
        u = sum(np.float32(1 << (m - k)) * gold[f"{name}_loop_flow_l{m}"][0, 0, 0] for m in range(levels - 1, k, -1))
        v = sum(np.float32(1 << (m - k)) * gold[f"{name}_loop_flow_l{m}"][0, 0, 1] for m in range(levels - 1, k, -1))
        jj, ii = np.meshgrid(np.arange(wk), np.arange(hk))
        nx = np.trunc(jj + np.float32(u)).astype(int) if k < levels - 1 else jj
        ny = np.trunc(ii + np.float32(v)).astype(int) if k < levels - 1 else ii
        skipped = (nx < 0) | (nx >= wk) | (ny < 0) | (ny >= hk)
        reach = 19 // 2 + 1
        tainted = np.zeros_like(skipped)
        ys, xs = np.nonzero(skipped)
        for y, x in zip(ys, xs):
            tainted[max(0, y - reach):y + reach + 1, max(0, x - reach):x + reach + 1] = True
        clean = ~tainted
        assert clean.mean() > 0.8
        eq = (flows[k] == ref) | (np.isnan(flows[k]) & np.isnan(ref))
        assert eq[clean].all(), f"level {k}: {(~eq[clean]).sum()} clean pixels differ"


# ------------------------------------------------------------------ compiled reference, CPU side
needs_ref = pytest.mark.skipif(not os.path.exists(os.path.join(os.path.dirname(__file__), "..", "oracle", "_ref",
                                                               "libofref.so")),
                               reason="oracle/_ref/libofref.so not built (needs /root/reference)")


@needs_ref
@pytest.mark.parametrize("w,h,levels", [(640, 480, 4), (320, 200, 3), (96, 64, 2)])
def test_pyramid_matches_reference_cpu(oracle, w, h, levels):
    img = oracle.make_frame(w, h, 0, 0, 4, 7)
    ref = oracle.ref_cpu_gauss_pyramid_c3(oracle.to_c3(img), levels)
    mine = oracle.gauss_pyramid(img, levels)
    for k in range(levels):
        for c in range(3):
            assert np.array_equal(ref[k][:, :, c], mine[k])


@needs_ref
def test_arr_sub_matches_reference(oracle):
    rng = np.random.default_rng(0)
    a = rng.standard_normal(1000).astype(np.float32)
    b = rng.standard_normal(1000).astype(np.float32)
    assert np.array_equal(oracle.ref_arr_sub(a, b), a - b)


@needs_ref
@pytest.mark.parametrize("level,shift", [(1, (0.9, -0.4)), (0, (-1.3, 0.6)), (0, (0.2, 0.2))])
def test_warp_as_written_matches_reference_cpu(oracle, level, shift):
    """cpu::shift_back_pyramid as written: a global shift by the flow of pixel (0,0)."""
    W0, H0, levels = 96, 64, 3
    rng = np.random.default_rng(3)
    flows = [rng.standard_normal((H0 >> k, W0 >> k, 2)).astype(np.float32) for k in range(levels)]
    for k in range(levels):
        flows[k][0, 0] = shift
    w, h = W0 >> level, H0 >> level
    img = oracle.make_frame(w, h, 0, 0, 4, 11)
    ref = oracle.ref_cpu_shift_back_c3(oracle.to_c3(img), level, levels, flows, prefill=0xAB)
    mine = oracle.warp(img, W0, H0, level, levels, flows, oracle.WARP_AS_WRITTEN)
    # where the reference wrote a pixel all three channels carry it; where it skipped, bytes beyond the
    # first w*h of the interleaved buffer keep the prefill (its memcpy copies only w*h bytes)
    u = sum(np.float32(1 << (k - level)) * np.float32(shift[0]) for k in range(levels - 1, level, -1))
    v = sum(np.float32(1 << (k - level)) * np.float32(shift[1]) for k in range(levels - 1, level, -1))
    jj, ii = np.meshgrid(np.arange(w), np.arange(h))
    nx, ny = np.trunc(jj + np.float32(u)).astype(int), np.trunc(ii + np.float32(v)).astype(int)
    written = (nx >= 0) & (nx < w) & (ny >= 0) & (ny < h)
    assert written.mean() > 0.8
    assert np.array_equal(ref[:, :, 0][written], mine[written])
    assert np.array_equal(ref[:, :, 1][written], mine[written])
    flat = ref.reshape(-1)
    skipped_bytes = np.repeat(~written.reshape(-1), 3)
    beyond = np.arange(flat.size) >= w * h
    assert (flat[skipped_bytes & beyond] == 0xAB).all()
    assert np.array_equal(mine[~written], img[~written])  # the oracle keeps the unwarped pixel


def test_warp_nearest_uses_per_pixel_flow(oracle):
    """NEAREST differs from AS_WRITTEN exactly by indexing the coarser flow at (i>>off, j>>off)."""
    W0, H0, levels = 64, 48, 2
    img = oracle.make_frame(W0, H0, 0, 0, 4, 5)
    f1 = np.zeros((H0 >> 1, W0 >> 1, 2), np.float32)
    f1[:, :, 0] = 1.0  # u = 2 px at level 0 everywhere
    f1[0, 0] = (0.0, 0.0)  # ... except the pixel AS_WRITTEN looks at
    flows = [np.zeros((H0, W0, 2), np.float32), f1]
    near = oracle.warp(img, W0, H0, 0, levels, flows, oracle.WARP_NEAREST)
    asw = oracle.warp(img, W0, H0, 0, levels, flows, oracle.WARP_AS_WRITTEN)
    assert np.array_equal(asw, img)
    assert np.array_equal(near[:, 2:W0 - 2], img[:, 4:W0])
    bil = oracle.warp(img, W0, H0, 0, levels, flows, oracle.WARP_BILINEAR)
    assert np.array_equal(bil[:, 2:W0 - 2], img[:, 4:W0])  # integer shift: bilinear == nearest


def test_bilinear_half_pixel(oracle):
    W0, H0 = 32, 16
    img = oracle.make_frame(W0, H0, 0, 0, 4, 9)
    f1 = np.full((H0 >> 1, W0 >> 1, 2), 0.0, np.float32)
    f1[:, :, 0] = 0.25  # u = 0.5 px
    out = oracle.warp(img, W0, H0, 0, 2, [np.zeros((H0, W0, 2), np.float32), f1], oracle.WARP_BILINEAR)
    exp = ((img[:, :-1].astype(int) * 128 + img[:, 1:].astype(int) * 128) * 256 + 32768) >> 16
    assert np.array_equal(out[:, :-1], exp.astype(np.uint8))
    assert np.array_equal(out[:, -1], img[:, -1])  # x + 0.5 > w-1: skipped, keeps the pixel


def test_cumulative_flow_is_the_main_cu_composition(oracle):
    w, h, levels = 64, 32, 3
    prev = oracle.make_frame(w, h, 0, 0, 4, 1)
    nxt = oracle.make_frame(w, h, 1.0, 0.0, 4, 1)
    flows, cums = oracle.flow_pair(prev, nxt, levels, 5, oracle.WARP_BILINEAR, oracle.SUMS_EXACT, 1.0, want_cum=True)
    i, j = 13, 37
    u = np.float32(0)
    for k in range(levels - 1, -1, -1):  # main.cu:136-147
        u = np.float32(u + np.float32(1 << k) * flows[k][i >> k, j >> k, 0])
    assert cums[0][i, j, 0] == u
    assert np.array_equal(np.nan_to_num(cums[levels - 1]), np.nan_to_num(flows[levels - 1] + 0.0))
