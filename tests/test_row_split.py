"""The fused level kernel at every row-block split.

A launch cuts each frame into row blocks of `rows_per_block` rows (csrc/lk_win.cu: a cost model of shape, batch size and
SM count), and every CTA derives its geometry from that number: its first staged row (lowered to an even global row), its
chunks, its last needed row `ylim`, the parity of the composing kernel's coarser tile, the anchor of its first chunk and
its ring slots.  The result must not depend on the split.  The other tests only reach the splits the cost model picks for
their shapes on one B200; these force others through the developer overrides the launcher reads on every launch:

  OFB_LK_ROWS        rows per CTA (clamped to the launch's rows);
  OFB_LK_TAIL        0 = no batch tail, n = the last wave of pairs cut into 2^n row blocks each;
  OFB_LK_TAIL_WAVES  the length of that tail in tenths of a wave.

A. one level (coarsest and warped, every window and warp mode, with and without cum_out) at rows per CTA from 1 to the
   frame height, on an even shape, an odd one without a tensor map for the coarser flow, and one whose last row block
   is a single row; exact solve bit-identical to the oracle, fast solve bit-identical to its own default split.
B. whole pipelines (3 levels: level 0 composing, writing the total flow, odd sizes) on smooth, far-moving, split-motion
   and adversarial content.
C. the batch tail at every shift and tail length, with tail rows that are not a multiple of the 16-row chunk.
D. row strips through ofb_lk_level_strip_device at windows of rows the strip schedule never produces: the contract
   "bit-identical unless the reach flag is raised", and the flag raised exactly when the general warp path's rule
   (restated here in numpy) asks for a row that is not held.
E. the peer-memory strip kernels (permuted row-block order, fused push counters) at other splits.
F. the pyramid's rows per thread (launch_pyr_roll) at each of its five values, and the strip pyramid step on minimal
   source rows.
"""
import numpy as np
import pytest

from support import (PAIRS, assert_flow_within_tolerance, assert_values_equal, bits_differ, c_for, noise_pair, oracle_warp,
                     reach_flag, requested_rows, rows, solve, values_differ)  # noqa: F401 (rows is a fixture)

WINDOWS = [3, 5, 7, 9, 11, 13, 15, 17, 19]
SHAPES_A = [(256, 160), (262, 150), (256, 161)]  # even; odd coarser width (no tensor map); 161 = 10 * 16 + 1 = 5 * 32 + 1


def rpb_values(win, h):
    """Rows per CTA to force: short blocks (below the window radius R), around R, 2R+1 and the 16-row chunk, the whole
    frame, and one more than it (the launcher clamps it to the frame)."""
    r = win // 2
    return sorted({1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, r, r + 1, 2 * r + 1, 2 * r + 2, 31, 32, 33, h - 1, h, h + 5})


def row_blocks(out_rows, rpb):
    """(first row, rows) of each row block of a launch, as lk_level_kernel derives them."""
    rpb = min(rpb, out_rows)
    return [(y, min(rpb, out_rows - y)) for y in range(0, out_rows, rpb)]


def test_rpb_values_reach_the_edges():
    """The forced splits include blocks shorter than the window radius and, on the odd shape, a last block of one row
    after a full one."""
    for win in WINDOWS:
        r = win // 2
        vals = rpb_values(win, 161)
        assert any(v < r for v in vals) or r <= 1
        assert any(row_blocks(161, v)[-1][1] == 1 and len(row_blocks(161, v)) > 1 for v in vals)
        assert row_blocks(161, 161 + 5) == [(0, 161)]
    assert {len(row_blocks(150, v)) for v in rpb_values(9, 150)} >= {1, 2, 5, 10, 150}


# --------------------------------------------------------------------------------------- D: the reach rule in numpy
def window_rows(out_y0g, out_y1g, win, h):
    """Rows of prev and next the window sums of the output rows read: the caller must hold these (ofb200.h)."""
    r = win // 2
    return max(out_y0g - r - 1, 0), min(out_y1g + r + 1, h)


STRIP_SHAPES = [(200, 91), (202, 91)]  # coarser width 100 (tensor map) and 101 (copied tile); odd height: clamped coarse row
STRIP_WINDOWS = [(0, 1), (0, 2), (0, 17), (37, 38), (40, 42), (37, 54), (90, 91), (89, 91), (74, 91)]  # global [y0, y1)


def strip_field(w, h, seed):
    """Coarser flow for the strip tests: vertical displacements up to +-7 px at 1/256-px rounding ties (both parities, both
    signs) and on whole rows, so that tap rows land on and one past every candidate bound; a few vectors skipped (NaN, out
    of range) so that unwarped rows are requested; horizontal flow small."""
    rng = np.random.default_rng([seed, w, h])
    cw, ch = w >> 1, h >> 1
    kind = rng.integers(0, 8, (ch, cw))
    k = rng.integers(-1800, 1800, (ch, cw))
    v = np.where(kind < 4, (k + 0.5) / 256.0, np.where(kind < 6, np.round(k / 256.0), k / 256.0))
    u = rng.integers(-600, 600, (ch, cw)) / 256.0
    cum = np.stack([c_for(u, 1.0), c_for(v, 1.0)], axis=-1).astype(np.float32)
    skip = rng.integers(0, 40, (ch, cw))
    cum[skip == 0, 1] = np.nan
    cum[skip == 1, 0] = np.float32(1e6)
    return np.ascontiguousarray(cum)


def strip_holdings(cum, w, h, mode, out_y0g, out_y1g, win):
    """(name, y_off, h_local, cum_y_off, cum_h_local) to run: the tight rows (what the window sums and the warp need),
    one row fewer at either end where that row is a warp request outside the output rows, one more above (the other
    parity of y_off), and the tight image rows with one coarser row short at either end."""
    req = requested_rows(cum, w, h, mode, out_y0g, out_y1g, win)
    img, crow = req
    wlo, whi = window_rows(out_y0g, out_y1g, win, h)
    rows = np.flatnonzero(img)
    lo, hi = min(wlo, int(rows.min())), max(whi, int(rows.max()) + 1)
    crows = np.flatnonzero(crow)
    clo, chi = int(crows.min()), int(crows.max()) + 1
    out = [("tight", lo, hi - lo, clo, chi - clo)]
    if img[lo] and lo < out_y0g:  # (a strip always holds its own output rows)
        out.append(("top-1", lo + 1, hi - lo - 1, clo, chi - clo))
    if img[hi - 1] and hi > out_y1g:
        out.append(("bottom-1", lo, hi - lo - 1, clo, chi - clo))
    if lo > 0:
        out.append(("above+1", lo - 1, hi - lo + 1, clo, chi - clo))
    if chi - clo > 1:
        out.append(("coarse top-1", lo, hi - lo, clo + 1, chi - clo - 1))
        out.append(("coarse bottom-1", lo, hi - lo, clo, chi - clo - 1))
    return out, req


@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("w,h", STRIP_SHAPES)
def test_strip_fields_fall_on_both_sides_of_the_reach_rule(mode, w, h):
    """Every strip case runs tight rows and one more above (rule: no flag) and rows one short (rule: flag); at many bounds
    the warp reaches beyond the rows the window sums need, so that the tight bound is a warp request; the field has
    1/256-px rounding ties."""
    cum = strip_field(w, h, 0)
    sides, far = set(), 0
    for win in (5, 11):
        for y0, y1 in STRIP_WINDOWS:
            hold, req = strip_holdings(cum, w, h, mode, y0, y1, win)
            for name, y_off, h_local, cy0, chl in hold:
                flag = reach_flag(req, y_off, h_local, cy0, chl)
                assert flag == (name not in ("tight", "above+1")), (win, y0, y1, name)
                sides.add(flag)
            wlo, whi = window_rows(y0, y1, win, h)
            rows = np.flatnonzero(req[0])
            far += int(rows.min() < wlo) + int(rows.max() >= whi)
    assert sides == {False, True}
    assert far > 10, "the warp should reach beyond the window rows at many bounds"
    # ties really occur: V * 512 at k + 1/2 for some blocks
    fv = cum[..., 1] * np.float32(512)
    with np.errstate(invalid="ignore"):
        ties_at_bound = int((np.abs(fv - np.floor(fv) - 0.5) == 0).sum())
    assert ties_at_bound > 100


def test_reach_rule_details():
    """The rule on hand-made vectors: the weight-0 third tap row is requested; a skipped target requests its own row;
    nearest truncation toward zero; rows at or past ylim are not requested."""
    w, h, win = 8, 40, 3
    cum = np.zeros((h >> 1, w >> 1, 2), np.float32)
    # block row 10..11: V = 2 * 256 exactly (cum.y = 1): bilinear taps 12, 13, 14 (14 has weight 0)
    cum[5, :, 1] = 1.0
    img, crow = requested_rows(cum, w, h, 2, 10, 12, win)
    assert img[12] and img[13] and img[14] and not img[15]
    # nearest mode: targets 10 + 2 = 12 and 11 + 2 = 13 only
    img1, _ = requested_rows(cum, w, h, 1, 10, 12, win)
    assert img1[12] and img1[13] and not img1[14]
    # NaN vectors: every pixel skipped, its own row requested, no taps -- blocks 8 .. 12, row 14 is the CTA's ylim
    cum[..., 1] = np.nan
    img, _ = requested_rows(cum, w, h, 2, 10, 12, win)
    assert np.flatnonzero(img).tolist() == [8, 9, 10, 11, 12, 13]
    # nearest: fy = 11 - 0.5 truncates to 10; fy = 10 - 0.5 -> 9
    cum[5, :, 1] = -0.25
    img1, _ = requested_rows(cum, w, h, 1, 10, 12, win)
    assert img1[9] and img1[10] and not img1[11]
    # window [20, 21), R = 1: blocks from row 18 (20 - 2 = 18, even) to ylim 23: block row 22 requests row 22 only
    cum[:] = 0
    img, crow = requested_rows(cum, w, h, 2, 20, 21, win)
    assert np.flatnonzero(crow).tolist() == [9, 10, 11]
    cum[11, :, 1] = 4.0  # block row 22: V = 8 rows down; row 23 is past ylim
    img, _ = requested_rows(cum, w, h, 2, 20, 21, win)
    assert img[30] and img[31] and img[32] and not img[23]
    img1, _ = requested_rows(cum, w, h, 1, 20, 21, win)
    assert img1[30] and not img1[31]


# --------------------------------------------------------------------------------------- F: pyramid rows per thread
def pyr_roll_rpt(sw, sh, n_images, sm_count):
    """Rows per thread launch_pyr_roll (csrc/pyramid.cu) picks for n_images frames of sw x sh."""
    dw, dh = sw >> 1, sh >> 1
    warps_x = ((dw + 7) // 8 + 30) // 31
    wpb = min(warps_x, 4)
    gx = (warps_x + wpb - 1) // wpb
    want = (sm_count if sm_count > 0 else 148) * 32
    rpt = 32
    while rpt > 2 and gx * wpb * ((dh + rpt - 1) // rpt) * n_images < want:
        rpt >>= 1
    return rpt


def batch_sizes_for_each_rpt(sw, sh, sm_count):
    """The smallest batch size at which launch_pyr_roll picks each of 2, 4, 8, 16 and 32 rows per thread."""
    out = {}
    for n in range(1, 65536):
        out.setdefault(pyr_roll_rpt(sw, sh, n, sm_count), n)
        if len(out) == 5:
            break
    return out


PYR_SHAPES = [(520, 75), (520, 76), (130, 150)]  # dh = 37 (odd), 38 (even, not a multiple of 4), 75 (odd)


@pytest.mark.parametrize("sm_count", [148, 132, 160])
@pytest.mark.parametrize("sw,sh", PYR_SHAPES)
def test_pyramid_batch_sizes_reach_every_rows_per_thread(sw, sh, sm_count):
    sizes = batch_sizes_for_each_rpt(sw, sh, sm_count)
    assert sorted(sizes) == [2, 4, 8, 16, 32]
    assert sizes[2] == 1 and max(sizes.values()) <= 4096
    for rpt, n in sizes.items():
        assert pyr_roll_rpt(sw, sh, n, sm_count) == rpt
        dh = sh >> 1
        assert rpt == 2 or dh % rpt != 0


# =================================================================================================== GPU
# --------------------------------------------------------------------------------------- A
@pytest.mark.gpu
@pytest.mark.parametrize("w,h", SHAPES_A)
@pytest.mark.parametrize("win", WINDOWS)
def test_one_level_at_every_rows_per_cta(ctx, oracle, rows, win, w, h):
    """The coarsest level and the warped level in all three warp modes (on the oracle's cumulative flow of the coarser
    level), each with and without cum_out, at every forced rows per CTA.  Exact solve: bit-identical to the oracle; fast
    solve: every pair bit-identical to the cost model's split and, there, within the tolerance bar of the oracle.  At rows
    per CTA up to 5 a batch of three distinct pairs, so that row blocks and pairs interleave in the grid."""
    import torch

    from cuda_optical_flow_2_b200 import SOLVE_EXACT, SOLVE_FAST, planar_to_device

    npair = 3
    prevs = [oracle.make_frame(w, h, 0, 0, 6, 3000 + 31 * win + i) for i in range(npair)]
    nexts = [oracle.make_frame(w, h, 1.75 - i, -2.5 + 0.75 * i, 6, 3000 + 31 * win + i) for i in range(npair)]
    dp, dn = planar_to_device(np.stack(prevs)), planar_to_device(np.stack(nexts))
    # level 0 of a 2-level pyramid; coarser flow and references from the oracle
    coarse = {}
    refs = {None: [oracle.lk_level(prevs[i], nexts[i], win, oracle.SUMS_EXACT) for i in range(npair)]}
    cum_ref = {None: refs[None]}
    for mode in (0, 1, 2):
        fl = [oracle.flow_pair(prevs[i], nexts[i], 2, win, mode, oracle.SUMS_EXACT, 1.0, want_cum=True) for i in range(npair)]
        coarse[mode] = torch.from_numpy(np.stack([f[1][1] for f in fl])).cuda()
        refs[mode] = [f[0][0] for f in fl]
        cum_ref[mode] = [f[1][0] for f in fl]
    dev = {m: torch.from_numpy(np.stack(refs[m])).cuda() for m in refs}
    dev_cum = {m: torch.from_numpy(np.stack(cum_ref[m])).cuda() for m in cum_ref}

    def run(mode, want_cum, n):
        cum_in = None if mode is None else coarse[mode][:n].contiguous()
        cum_out = torch.empty((n, h, w, 2), dtype=torch.float32, device="cuda") if want_cum else None
        flow = ctx.lk_level_device(dp[:n].contiguous(), dn[:n].contiguous(), w, win, warp_mode=2 if mode is None else mode,
                                   cum_in=cum_in, cum_out=cum_out)
        return flow, cum_out

    cases = [(m, c) for m in (None, 0, 1, 2) for c in (False, True)]
    for sm in (SOLVE_EXACT, SOLVE_FAST):
        with solve(ctx, sm):
            rows(None)
            base = {}
            for mode, want_cum in cases:
                base[mode, want_cum] = run(mode, want_cum, npair)
                if sm == SOLVE_FAST:
                    torch.cuda.synchronize()
                    for i in range(npair):
                        got = base[mode, want_cum][0][i].cpu().numpy()
                        assert_flow_within_tolerance(got, refs[mode][i], f"fast solve, mode {mode}, pair {i}, default split")
            for rpb in rpb_values(win, h):
                rows(rpb)
                for mode, want_cum in cases:
                    n = npair if rpb <= 5 else 1
                    flow, cum_out = run(mode, want_cum, n)
                    what = f"rows per CTA {rpb}, mode {mode}, cum_out {want_cum}, solve {sm}"
                    if sm == SOLVE_EXACT:
                        assert not (e := values_differ(flow, dev[mode][:n])), f"{what}: flow: {e}"
                        if want_cum:
                            assert not (e := values_differ(cum_out, dev_cum[mode][:n])), f"{what}: cum_out: {e}"
                    else:
                        e = bits_differ(flow, base[mode, want_cum][0][:n])
                        assert not e, f"{what}: flow against the default split: {e}"
                        if want_cum:
                            assert not (e := bits_differ(cum_out, base[mode, want_cum][1][:n])), f"{what}: cum_out: {e}"


# --------------------------------------------------------------------------------------- B
def _content(oracle, name, w, h):
    if name == "smooth":
        return oracle.make_frame(w, h, 0, 0, 6, 515), oracle.make_frame(w, h, 2.25, -1.5, 6, 515)
    if name == "far_shift":
        return oracle.make_frame(w, h, 0, 0, 8, 4242), oracle.make_frame(w, h, 41.5, -27.25, 8, 4242)
    if name == "split_motion":
        a, b = oracle.make_frame(w, h, 13.0, 9.5, 8, 4242), oracle.make_frame(w, h, -14.5, -11.0, 8, 4242)
        return oracle.make_frame(w, h, 0, 0, 8, 4242), np.where(np.arange(w)[None, :] < w // 2, a, b).astype(np.uint8)
    return PAIRS[name](w, h)


PIPE_RPB = [1, 2, 3, 5, 8, 9, 16, 17, 33]


@pytest.mark.gpu
@pytest.mark.parametrize("win", [5, 9, 15])
@pytest.mark.parametrize("content", ["smooth", "far_shift", "split_motion", "binary_noise", "diag6"])
@pytest.mark.parametrize("w,h,want_total", [(256, 160, False), (256, 160, True), (262, 150, False)])
def test_pipeline_at_every_rows_per_cta(ctx, oracle, rows, w, h, want_total, content, win):
    """flow_pairs_device, 3 levels, every warp mode, the forced rows per CTA applying to every level: 256x160 without the
    total flow (level 0 composes the coarser cumulative flow on the fly), with it, and 262x150 (odd coarser sizes).  Exact:
    every level and the total flow bit-identical to the oracle; fast: bit-identical to the cost model's split."""
    import torch

    from cuda_optical_flow_2_b200 import SOLVE_EXACT, SOLVE_FAST, planar_to_device

    levels = 3
    prev, nxt = _content(oracle, content, w, h)
    dp, dn = planar_to_device(prev[None]), planar_to_device(nxt[None])
    for mode in (0, 1, 2):
        ref, cums = oracle.flow_pair(prev, nxt, levels, win, mode, oracle.SUMS_EXACT, 1.0, want_cum=True)
        dref = [torch.from_numpy(r[None]).cuda() for r in ref]
        dtot = torch.from_numpy(cums[0][None]).cuda()

        def run():
            total = torch.empty((1, h, w, 2), dtype=torch.float32, device="cuda") if want_total else None
            return ctx.flow_pairs_device(dp, dn, w, levels, win, warp_mode=mode, total_flow=total), total

        for sm in (SOLVE_EXACT, SOLVE_FAST):
            with solve(ctx, sm):
                rows(None)
                base, base_total = run()
                for rpb in PIPE_RPB:
                    rows(rpb)
                    flows, total = run()
                    what = f"mode {mode}, rows per CTA {rpb}, solve {sm}"
                    for k in range(levels):
                        e = values_differ(flows[k], dref[k]) if sm == SOLVE_EXACT else bits_differ(flows[k], base[k])
                        assert not e, f"{what}, level {k}: {e}"
                    if want_total:
                        e = values_differ(total, dtot) if sm == SOLVE_EXACT else bits_differ(total, base_total)
                        assert not e, f"{what}, total flow: {e}"
                rows(None)


# --------------------------------------------------------------------------------------- C
def lk_min_blocks(win, lk_min_blocks=4):
    """LkCfg<WIN>::MIN_BLOCKS (csrc/lk_level.cuh): CTAs per SM that shared memory allows (with the ring in shared memory),
    at most LK_MIN_BLOCKS."""
    r, sub, ch, tile_w, ntw, ctw, nt, cpw = win // 2, 8, 16, 160, 176, 68, 128, 132
    up = lambda v: (v + 127) // 128 * 128  # noqa: E731
    nbr, margin_y = ch // 2, 8 if win <= 9 else 6
    tile_p = up(ch * tile_w)
    tile_q = max(tile_p, up((ch + 2 * margin_y + 2) * ntw))
    off_cum = 128 + tile_p + tile_q
    off_w = off_cum + nbr * ctw * 8 + up((nbr // 2 + 1) * (ctw // 2 + 2) * 8)
    off_ring = off_w + ch * 2 * 66 * 4 + 5 * sub * cpw * 4
    fit = (227 * 1024) // (off_ring + win * nt * 8 + 1024)
    return max(1, min(fit, lk_min_blocks))


def tail_split(w, out_rows, n_pairs, win, sm_count, shift, waves, nby=1):
    """(first tail pair, tail rows) of the batch tail launch_one (csrc/lk_win.cu) sets up for a whole-frame level, or None
    when the tail stays off."""
    two = min((128 - 2 * (win // 2)) // 8, 16) * 8
    strips = (w + two - 1) // two
    slots = (sm_count if sm_count > 0 else 148) * lk_min_blocks(win)
    tail_pairs = ((slots + strips - 1) // strips * waves + 9) // 10
    if 0 < shift <= 4:
        tail_pairs = min(tail_pairs, (65535 - n_pairs) // ((1 << shift) - 1))
    if (0 < shift <= 4 and nby == 1 and out_rows >= (2 * 16 << shift) and tail_pairs > 0 and n_pairs * strips >= 4 * slots
            and tail_pairs < n_pairs):
        return n_pairs - tail_pairs, (out_rows + (1 << shift) - 1) >> shift
    return None


TAIL_W, TAIL_H, TAIL_WIN, TAIL_DISTINCT = 120, 532, 9, 4  # one column strip at window 9 (LkCfg<9>::TWO = 120)


def tail_batch_size(sm_count):
    """Pairs enough for the tail (n * strips >= 4 * SMs * MIN_BLOCKS), a whole number of prototypes."""
    need = 4 * sm_count * lk_min_blocks(TAIL_WIN)
    return -(-need // TAIL_DISTINCT) * TAIL_DISTINCT


@pytest.mark.parametrize("sm_count", [148, 132, 160])
def test_tail_batch_engages_the_tail_on_every_level(sm_count):
    """With one row block per level, the tail test's batch switches the tail on at level 0 (532 rows, composing) for every
    shift 1-4 with tail rows 266, 133, 67 and 34 (none a multiple of 16), at level 1 (266 rows) for shifts 1-3 and at level
    2 (133 rows) for shifts 1-2; and not with more than one row block."""
    assert lk_min_blocks(9) == 4 and lk_min_blocks(19) >= 1
    n = tail_batch_size(sm_count)
    for waves in (1, 10, 30):
        rows0 = [tail_split(TAIL_W, TAIL_H, n, TAIL_WIN, sm_count, s, waves)[1] for s in (1, 2, 3, 4)]
        assert rows0 == [266, 133, 67, 34] and all(r % 16 for r in rows0)
        for k, shifts in ((1, (1, 2, 3)), (2, (1, 2))):
            for s in (1, 2, 3, 4):
                on = tail_split(TAIL_W >> k, TAIL_H >> k, n, TAIL_WIN, sm_count, s, waves) is not None
                assert on == (s in shifts), (k, s, waves)
        assert tail_split(TAIL_W, TAIL_H, n, TAIL_WIN, sm_count, 2, waves, nby=4) is None
        assert tail_split(TAIL_W, TAIL_H, n, TAIL_WIN, sm_count, 0, waves) is None


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1])
def test_batch_tail_at_every_shift_and_length(ctx, oracle, monkeypatch, mode):
    """A batch big enough that the launcher cuts its last pairs into 2^shift short row blocks, on a frame of one column
    strip whose 532 rows are not a multiple of 16, 3 levels, bilinear warp, no total flow (level 0 composes).  Every level
    is forced to one row block (the tail needs that), so that the tail engages at level 0 for every shift (tail rows 266,
    133, 67 and 34), at level 1 for shifts 1-3 and at level 2 for shifts 1-2 -- asserted from the restated switch with this
    GPU's SM count.  Every OFB_LK_TAIL in 1..4 and tail length 1, 10 and 30 tenths of a wave: bit-identical to the launch
    without a tail; exact solve: every copy of every prototype equals the oracle."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    w, h, win, distinct, levels = TAIL_W, TAIL_H, TAIL_WIN, TAIL_DISTINCT, 3
    n = tail_batch_size(ctx.sm_count)
    for shift in (1, 2, 3, 4):
        assert tail_split(w, h, n, win, ctx.sm_count, shift, 1) is not None, f"the tail would stay off at shift {shift}"
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 6, 880 + i) for i in range(distinct)])
    nexts = np.stack([oracle.make_frame(w, h, 1.25 - i, 0.5 + 0.75 * i, 6, 880 + i) for i in range(distinct)])
    dp = planar_to_device(prevs).repeat(n // distinct, 1, 1)
    dn = planar_to_device(nexts).repeat(n // distinct, 1, 1)
    with solve(ctx, mode):
        monkeypatch.setenv("OFB_LK_ROWS", str(h))  # clamped to each level's rows: one row block per level
        monkeypatch.setenv("OFB_LK_TAIL", "0")
        plain = [f.clone() for f in ctx.flow_pairs_device(dp, dn, w, levels, win)]
        refs = None
        if mode == 0:
            refs = []
            per = [oracle.flow_pair(prevs[i], nexts[i], levels, win, 2, oracle.SUMS_EXACT) for i in range(distinct)]
            for k in range(levels):
                refs.append(torch.from_numpy(np.stack([p[k] for p in per])).cuda())
            for k in range(levels):
                e = values_differ(plain[k].view(n // distinct, distinct, h >> k, w >> k, 2),
                                  refs[k].expand(n // distinct, -1, -1, -1, -1))
                assert not e, f"no tail, level {k}: {e}"
        for shift in (1, 2, 3, 4):
            for waves in (1, 10, 30):
                monkeypatch.setenv("OFB_LK_TAIL", str(shift))
                monkeypatch.setenv("OFB_LK_TAIL_WAVES", str(waves))
                flows = ctx.flow_pairs_device(dp, dn, w, levels, win)
                for k in range(levels):
                    e = bits_differ(flows[k], plain[k])
                    assert not e, f"tail {shift}, waves {waves}, level {k}: against no tail: {e}"
                    if refs is not None:  # every copy, those of the tail included
                        e = values_differ(flows[k].view(n // distinct, distinct, h >> k, w >> k, 2),
                                          refs[k].expand(n // distinct, -1, -1, -1, -1))
                        assert not e, f"tail {shift}, waves {waves}, level {k}: against the oracle: {e}"
                del flows


# --------------------------------------------------------------------------------------- D
@pytest.mark.gpu
@pytest.mark.parametrize("win", [5, 11])
@pytest.mark.parametrize("mode", [1, 2])
@pytest.mark.parametrize("w,h", STRIP_SHAPES)
def test_strip_windows_bit_identical_unless_flagged(ctx, oracle, rows, w, h, mode, win):
    """ofb_lk_level_strip_device on rows cut from whole frames: output windows of 1, 2 and 17 rows at the top, in the
    interior (odd and even first rows) and at the bottom; held rows exactly what the window sums and the warp need, one
    fewer at either end, one more above (y_off of the other parity); coarser rows tight and one short; 1, 3, 16 and the
    default rows per CTA.  The flag is raised exactly when the rule (requested_rows) asks for a row not held, and when it
    is not raised, flow and cum_out rows equal lk_level_device on the whole frame bit for bit.  Rows outside what a call
    holds are filled with other bytes and other flow, so that a read of them shows; rows outside the output window must
    stay untouched."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    prev, nxt = noise_pair(w, h, 77 + w)
    cum = strip_field(w, h, 1)
    rows(None)
    P, N = planar_to_device(prev[None]), planar_to_device(nxt[None])
    cum_d = torch.from_numpy(cum[None]).cuda()
    whole_cum = torch.empty((1, h, w, 2), dtype=torch.float32, device="cuda")
    whole = ctx.lk_level_device(P, N, w, win, warp_mode=mode, cum_in=cum_d, cum_out=whole_cum)
    torch.cuda.synchronize()
    ref = oracle.lk_level(prev, oracle_warp(oracle, nxt, cum, mode, 1.0), win, oracle.SUMS_EXACT)
    assert_values_equal(whole[0].cpu().numpy(), ref, "whole frame")
    # garbage copies: other bytes / other flow everywhere a call does not hold
    Pg, Ng = planar_to_device((255 - prev)[None])[0], planar_to_device(np.roll(nxt, 7, 1)[None])[0]
    cum_g = torch.from_numpy(np.ascontiguousarray(cum[::-1] * np.float32(-1.5) + np.float32(3.25))).cuda()
    sentinel = float("-1.25e30")
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    counts = {False: 0, True: 0}
    for y0, y1 in STRIP_WINDOWS:
        hold, req = strip_holdings(cum, w, h, mode, y0, y1, win)
        for name, y_off, h_local, cy0, chl in hold:
            expect = reach_flag(req, y_off, h_local, cy0, chl)
            pb, nb, cb = Pg.clone(), Ng.clone(), cum_g.clone()
            pb[y_off:y_off + h_local] = P[0, y_off:y_off + h_local]
            nb[y_off:y_off + h_local] = N[0, y_off:y_off + h_local]
            cb[cy0:cy0 + chl] = cum_d[0, cy0:cy0 + chl]
            for rpb in (None, 1, 3, 16):
                rows(rpb)
                for want_cum in (False, True):
                    flow = torch.full((h_local, w, 2), sentinel, dtype=torch.float32, device="cuda")
                    cout = torch.full((h_local, w, 2), sentinel, dtype=torch.float32, device="cuda") if want_cum else None
                    flag.zero_()
                    ctx.lk_level_strip_device(pb[y_off:y_off + h_local], nb[y_off:y_off + h_local], w, y_off, h, y0 - y_off,
                                              y1 - y_off, win, mode, 1.0, cb[cy0:cy0 + chl], cy0, flow, cum_out=cout,
                                              overflow_flag=flag)
                    what = f"rows [{y0},{y1}) held {name} [{y_off},{y_off + h_local}) coarse [{cy0},{cy0 + chl}), " \
                           f"rows per CTA {rpb}, cum_out {want_cum}"
                    got = int(flag.item())
                    assert got in (0, 1), f"{what}: flag {got}"
                    assert bool(got) == expect, f"{what}: flag {got}, the rule says {int(expect)}"
                    counts[expect] += 1
                    lo, hi = y0 - y_off, y1 - y_off
                    for t, ref in ((flow, whole), (cout, whole_cum)):
                        if t is None:
                            continue
                        assert bool((t[:lo] == sentinel).all() and (t[hi:] == sentinel).all()), f"{what}: wrote outside its rows"
                        if not expect:
                            assert not (e := bits_differ(t[lo:hi], ref[0, y0:y1])), f"{what}: {e}"
    assert counts[False] > 0 and counts[True] > 0


# --------------------------------------------------------------------------------------- E
@pytest.mark.gpu
@pytest.mark.parametrize("rpb", [1, 3, 16])
@pytest.mark.parametrize("world", [2, 3])
def test_peer_memory_strips_at_other_splits(ctx, oracle, rows, world, rpb):
    """Row strips with the halo exchange fused into the level kernels (peer-memory transport, ranks in this process), with
    the forced rows per CTA: many row blocks, the pushing blocks scheduled first (permuted order) and the push counters
    sized from the split.  Two pairs back to back, every level and the total flow bit-identical to the whole frame, and no
    flag (neither a timed-out neighbour nor a reach overflow)."""
    import torch

    from cuda_optical_flow_2_b200 import WARP_BILINEAR, planar_to_device
    from cuda_optical_flow_2_b200.dist import NativeStrips

    W, H, levels, win = 320, 240, 3, 9
    dev = torch.device("cuda", 0)
    ranks = [NativeStrips(ctx, W, H, levels, win, world, rk, dev, WARP_BILINEAR, 1.0, 16, transport="local")
             for rk in range(world)]
    try:
        NativeStrips.connect_local(ranks)
        for trial, (dx, dy) in enumerate([(2.25, -1.5), (-1.0, 3.25)]):
            prev = oracle.make_frame(W, H, 0, 0, 8, 610 + trial)
            nxt = oracle.make_frame(W, H, dx, dy, 8, 610 + trial)
            dp, dn = planar_to_device(prev[None]), planar_to_device(nxt[None])
            rows(None)
            total = torch.empty((1, H, W, 2), dtype=torch.float32, device=dev)
            whole = ctx.flow_pairs_device(dp, dn, W, levels, win, warp_mode=WARP_BILINEAR, total_flow=total)
            torch.cuda.synchronize()
            rows(rpb)
            inputs = []
            for ns in ranks:
                y0, y1 = ns.own_rows(0)
                inputs.append((dp[0, y0:y1], dn[0, y0:y1]))
            NativeStrips.run_local_sequenced(ranks, inputs, torch.cuda.current_stream().cuda_stream)
            for ns in ranks:
                ns.check()
            for ns in ranks:
                for k in range(levels):
                    y0, y1 = ns.own_rows(k)
                    assert not (e := bits_differ(ns.own_flow(k), whole[k][0, y0:y1])), f"pair {trial} rank {ns.rank} level {k}: {e}"
                y0, y1 = ns.own_rows(0)
                assert not (e := bits_differ(ns.own_flow(0, total=True), total[0, y0:y1])), f"pair {trial} rank {ns.rank} total: {e}"
    finally:
        torch.cuda.synchronize()
        for ns in ranks:
            ns.close()


@pytest.mark.gpu
def test_checked_peer_memory_strips_at_three_rows_per_cta(ctx, oracle, rows):
    """A checked pair (both directions and the forward-backward check) on three ranks at 3 rows per CTA: every output
    bit-identical to the whole-frame ofb_flow_pairs_fb_device rows, no flag."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device
    from cuda_optical_flow_2_b200.dist import NativeStrips

    W, H, levels, win, world = 320, 240, 3, 9, 3
    dev = torch.device("cuda", 0)
    ranks = [NativeStrips(ctx, W, H, levels, win, world, rk, dev, 2, 1.0, 16, transport="local", fb_reach=16)
             for rk in range(world)]
    try:
        NativeStrips.connect_local(ranks)
        prev = oracle.make_frame(W, H, 0, 0, 8, 640)
        nxt = oracle.make_frame(W, H, 1.5, -0.75, 8, 640)
        dp, dn = planar_to_device(prev[None]), planar_to_device(nxt[None])
        fwd, bwd, st, e2 = ctx.flow_pairs_fb_device(dp, dn, W, levels, win, want_err2=True)
        torch.cuda.synchronize()
        rows(3)
        inputs = [(dp[0, ns.own_rows(0)[0]:ns.own_rows(0)[1]], dn[0, ns.own_rows(0)[0]:ns.own_rows(0)[1]]) for ns in ranks]
        NativeStrips.run_local_sequenced_fb(ranks, inputs, want_err2=True, stream=torch.cuda.current_stream().cuda_stream)
        for ns in ranks:
            ns.check()
            y0, y1 = ns.own_rows(0)
            gf, gb, gs, ge = ns.own_fb()
            assert not (e := bits_differ(gf, fwd[0, y0:y1])), f"rank {ns.rank} forward total: {e}"
            assert not (e := bits_differ(gb, bwd[0, y0:y1])), f"rank {ns.rank} backward total: {e}"
            assert torch.equal(gs, st[0, y0:y1]), f"rank {ns.rank} status"
            assert not (e := bits_differ(ge, e2[0, y0:y1])), f"rank {ns.rank} err2: {e}"
    finally:
        torch.cuda.synchronize()
        for ns in ranks:
            ns.close()


# --------------------------------------------------------------------------------------- F
@pytest.mark.gpu
@pytest.mark.parametrize("sw,sh", PYR_SHAPES)
def test_pyramid_at_every_rows_per_thread(ctx, oracle, sw, sh):
    """One and two pyramid steps of batches sized so that launch_pyr_roll picks each of 2, 4, 8, 16 and 32 rows per
    thread (restated above), byte-exact against the oracle for every image.  The two-step entry passes the context's SM
    count to launch_pyr_roll; the one-step entry goes through launch_pyr_down, which passes none (launch_pyr_roll then
    assumes 148 SMs), so each is sized with the count its launcher uses."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    distinct = 3
    imgs = np.stack([oracle.make_frame(sw, sh, 0, 0, 3, 950 + i) for i in range(distinct)])
    r1 = np.stack([oracle.pyr_down(im) for im in imgs])
    r2 = np.stack([oracle.pyr_down(im) for im in r1])
    d1r, d2r = torch.from_numpy(r1).cuda(), torch.from_numpy(r2).cuda()
    src = planar_to_device(imgs)
    for steps, sm_count in ((1, 0), (2, ctx.sm_count)):
        sizes = batch_sizes_for_each_rpt(sw, sh, sm_count)
        assert sorted(sizes) == [2, 4, 8, 16, 32]
        for rpt, n in sorted(sizes.items()):
            batch = src.repeat(-(-n // distinct), 1, 1)[:n].contiguous()
            idx = torch.arange(n, device="cuda") % distinct
            what = f"{rpt} rows per thread ({n} images), {steps} step(s)"
            if steps == 1:
                assert torch.equal(ctx.pyr_down_device(batch, sw)[:, :, :sw >> 1], d1r[idx]), what
            else:
                a, b = ctx.pyr_down2_device(batch, sw)
                assert torch.equal(a[:, :, :sw >> 1], d1r[idx]), f"{what}: level +1"
                assert torch.equal(b[:, :, :sw >> 2], d2r[idx]), f"{what}: level +2"


@pytest.mark.gpu
@pytest.mark.parametrize("sw,sh", [(520, 75), (130, 150), (66, 33)])
def test_pyramid_strip_on_minimal_source_rows(ctx, oracle, sw, sh):
    """ofb_pyr_down_strip_device with exactly source rows 2y0-1 .. 2y1-1 held (odd src_y_off except at the top), single
    destination rows at the top, in the interior and at the bottom, and longer runs; the rows around the held ones hold
    other bytes, so that a read past them shows.  Byte-exact against the oracle."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    img = oracle.make_frame(sw, sh, 0, 0, 3, 970 + sw)
    ref = oracle.pyr_down(img)
    dh, dw = sh >> 1, sw >> 1
    full = planar_to_device(img[None])[0]
    junk = planar_to_device((img ^ 0x5A)[None])[0]
    cases = [(0, 1), (1, 2), (dh // 2, dh // 2 + 1), (dh - 1, dh), (0, dh), (3, dh - 2), (dh - 5, dh)]
    for y0, y1 in cases:
        s0, s1 = max(2 * y0 - 1, 0), 2 * (y1 - 1) + 2
        buf = junk.clone()
        buf[s0:s1] = full[s0:s1]
        dst = torch.full((y1 - y0, full.shape[1]), 0xEE, dtype=torch.uint8, device="cuda")
        ctx.pyr_down_strip_device(buf[s0:s1], sw, s0, dst, y0, y1)
        torch.cuda.synchronize()
        assert np.array_equal(dst[:, :dw].cpu().numpy(), ref[y0:y1]), f"rows [{y0},{y1}) from source [{s0},{s1})"
