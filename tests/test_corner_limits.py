"""Shi-Tomasi corners at their limits: the launch grids' stride loops, raster indices near 2^31, the selection's chunk
boundaries, ties across the kernels' seams, the threshold, caller buffers and streams, workspace reuse and the slot limit.

Everything is compared with the C restatement tests/corner_oracle.c bit for bit (maps, corners, scores, counts and the NaN
tail).  Where a whole-frame restatement would be too large (the 2^31-pixel frame), the reference is built from crops of the
frame and a sparse restatement of the candidate rule, which is itself checked against `plain_greedy` on the CPU.

CPU tests (no mark): the score on content that drives its double arithmetic past 2^53, the launcher's choice of the
selection grid restated in Python, the sparse reference, and the planning arithmetic of the slot limit.
GPU tests: every other item; each output is allocated with guard bands that must survive every call.
"""
import decimal
import math

import numpy as np
import pytest

from support import F32, assert_same_bits, content, cro, device_frames, exact_sums, plain_greedy  # noqa: F401 (cro is a fixture)

WINS = list(range(3, 20, 2))
FLT_MAX = float(np.finfo(F32).max)
G = 64  # guard elements before and after every output buffer


def f32_next(x, toward):
    return float(np.nextafter(F32(x), F32(toward)))


# ------------------------------------------------------------------------------------ launch arithmetic, restated
def score_grid(w, h):
    """corner_score_kernel: 32 x 32 tiles, grid.y capped at 65535, tiles stepped by grid.y."""
    tiles_y = (h - 1) // 32 + 1
    return (w - 1) // 32 + 1, min(tiles_y, 65535), tiles_y


def cand_grid(iw, ih):
    """corner_cand_kernel: 32 x 8 threads over the interior, grid.y capped at 65535, rows stepped by 8 grid.y."""
    return (iw + 31) // 32, min((ih + 7) // 8, 65535)


def plan(w, h, n, win):
    """plan_corners: interior margin and size, candidate slots per image (ceil(iw/2) ceil(ih/2)) and in all."""
    m = win // 2 + 1
    iw, ih = max(w - 2 * m, 0), max(h - 2 * m, 0)
    cap = ((iw + 1) // 2) * ((ih + 1) // 2) if iw and ih else 0
    return m, iw, ih, cap, cap * n


def select_grid(md, iw, ih):
    """launch_detect_corners' selection grid: cell side c, grid size gw x gh, and reach, the largest |dx| looked up."""
    md2 = float(md) * float(md)
    c = int(min(math.floor(float(md) / math.sqrt(2.0)), float(1 << 30)))
    c = max(c, 1)
    while c > 1 and 2.0 * (c - 1) * (c - 1) >= md2:
        c -= 1
    gw, gh = (iw + c - 1) // c, (ih + c - 1) // c
    reach = int(min(math.ceil(float(md)), float(max(iw, ih))))
    return c, gw, gh, reach


# ------------------------------------------------------------------------------------ content
def worst(kind, w=64, h=64, seed=0):
    """Content whose exact sums push the score's int64 -> double conversions past 2^53."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == "checker3":  # 3x3 blocks: det > 2^53 at window 19
        return ((((xx // 3) + (yy // 3)) & 1) * 255).astype(np.uint8)
    if kind == "bnoise2":  # binary noise in 2x2 blocks: det > 2^53 at window 19
        b = rng.integers(0, 2, ((h + 1) // 2, (w + 1) // 2))
        return (np.kron(b, np.ones((2, 2), np.int64))[:h, :w] * 255).astype(np.uint8)
    if kind == "stripes_impulses":  # period-4 stripes with 1 % flipped pixels: disc > 2^53 with det != 0
        img = ((xx >> 1) & 1) * 255
        return np.where(rng.random((h, w)) < 0.01, 255 - img, img).astype(np.uint8)
    if kind == "impulses":
        return np.where(rng.random((h, w)) < 0.06, 255, 0).astype(np.uint8)
    if kind == "steps":  # 0 -> 255 steps: horizontal, vertical and diagonal edges and their crossings
        return (255 * ((xx >= 21) ^ (yy >= 37) ^ (xx + 2 * yy >= 90))).astype(np.uint8)
    raise ValueError(kind)


WORST = ["checker3", "bnoise2", "stripes_impulses", "impulses", "steps"]


# ------------------------------------------------------------------------------------ GPU helpers: guarded outputs
def _guarded(count, dtype, fill):
    import torch

    buf = torch.full((G + count + G,), fill, dtype=dtype, device="cuda")
    return buf, buf[G:G + count]


def _guards_intact(buf, fill):
    return bool((buf[:G] == fill).all()) and bool((buf[-G:] == fill).all())


def _map_g(ctx, dev, pitch, stride, w, h, n, win, stream=None):
    import torch

    from cuda_optical_flow_2_b200 import _lib

    buf, out = _guarded(n * h * w, torch.float32, float("nan"))
    _lib.check(_lib.load().ofb_min_eig_map_device(ctx._h, dev.data_ptr(), pitch, stride, w, h, n, win, out.data_ptr(), stream))
    torch.cuda.synchronize()
    assert bool(torch.isnan(buf[:G]).all()) and bool(torch.isnan(buf[-G:]).all()), "map guard overwritten"
    return out.view(n, h, w)


SENT = -7.25


def _detect_g(ctx, dev, pitch, stride, w, h, n, win, mc, ql=0.01, md=10.0, ms=0.0, with_scores=True, stream=None):
    """ofb_detect_corners_device into guarded outputs; the guards are checked before anything is returned."""
    import torch

    from cuda_optical_flow_2_b200 import _lib

    cb, corners = _guarded(n * mc * 2, torch.float32, SENT)
    sb, scores = _guarded(n * mc, torch.float32, SENT)
    kb, counts = _guarded(n, torch.int32, -7)
    _lib.check(_lib.load().ofb_detect_corners_device(ctx._h, dev.data_ptr(), pitch, stride, w, h, n, win, mc, ql, md, ms,
                                                     corners.data_ptr(), scores.data_ptr() if with_scores else None,
                                                     counts.data_ptr(), stream))
    torch.cuda.synchronize()
    assert _guards_intact(cb, SENT) and _guards_intact(kb, -7), "corner / count guard overwritten"
    if with_scores:
        assert _guards_intact(sb, SENT), "score guard overwritten"
    else:
        assert bool((sb == SENT).all()), "scores written although NULL was passed"
    return (corners.view(n, mc, 2).cpu().numpy(), scores.view(n, mc).cpu().numpy() if with_scores else None,
            counts.cpu().numpy())


def _assert_detect(cro, imgs, got, win, mc, ql=0.01, md=10.0, ms=0.0, refs=None):
    corners, scores, counts = got
    for i, img in enumerate(imgs):
        rc, rs, rn = refs[i] if refs is not None else cro.detect(img, win, mc, quality_level=ql, min_distance=md,
                                                                 min_score=ms)
        assert counts[i] == rn, (i, counts[i], rn)
        assert_same_bits(corners[i], rc, f"image {i} corners")
        if scores is not None:
            assert_same_bits(scores[i], rs, f"image {i} scores")
    return counts


# ==================================================================================== 1. worst-case content
@pytest.mark.parametrize("win", WINS)
@pytest.mark.parametrize("kind", WORST)
def test_worst_case_score_within_one_ulp(cro, kind, win):
    """The restatement stays within one float ulp of a 50-digit evaluation of l1 / win^2 where det and disc pass 2^53."""
    img = worst(kind, seed=win)
    h, w = img.shape
    got = cro.score(img, win)
    A, D, B = exact_sums(img, win)
    assert (A + D).max() < 2 ** 31  # the kernel forms S = A + D in int32
    decimal.getcontext().prec = 50
    n2 = decimal.Decimal(win * win)
    for y in range(h):
        for x in range(w):
            a, d, b = int(A[y, x]), int(D[y, x]), int(B[y, x])
            g = float(got[y, x])
            if a * d - b * b == 0:
                assert g == 0.0, (x, y, g)
                continue
            lam = (decimal.Decimal(a + d) - decimal.Decimal((a - d) ** 2 + 4 * b * b).sqrt()) / 2 / n2
            ref = float(lam)
            assert abs(g - ref) <= float(np.spacing(F32(ref))), (x, y, g, ref)


def test_worst_case_content_reaches_past_2_53():
    """The content of the test above is what it claims: det > 2^53 on thousands of pixels (3x3 checkerboard, 2x2 binary
    noise), disc > 2^53 with det != 0 (stripes with impulses), and S = A + D far inside int32 (measured 3.8e8 at most;
    the bound 2 * 361 * 1020^2 = 7.5e8 holds for any content)."""
    assert 2 * 19 * 19 * 1020 ** 2 < 2 ** 31
    seen = {}
    for kind in WORST:
        for win in WINS:
            A, D, B = exact_sums(worst(kind, seed=win), win)
            det, disc = A * D - B * B, (A - D) ** 2 + 4 * B * B
            assert (A + D).max() < 2 ** 31 and disc.min() >= 0
            seen[kind, win] = (int((det > 2 ** 53).sum()), int(((disc > 2 ** 53) & (det != 0)).sum()))
    assert seen["checker3", 19][0] > 2000 and seen["bnoise2", 19][0] > 2000
    assert seen["stripes_impulses", 19][1] > 2000


@pytest.mark.gpu
@pytest.mark.parametrize("win", WINS)
def test_worst_case_content_kernel(ctx, cro, win):
    imgs = np.stack([worst(k, seed=win) for k in WORST])
    n, h, w = imgs.shape
    dev, pitch, stride = device_frames(imgs)
    got = _map_g(ctx, dev, pitch, stride, w, h, n, win).cpu().numpy()
    for i, k in enumerate(WORST):
        assert_same_bits(got[i], cro.score(imgs[i], win), f"{k} map")
    for kw in (dict(ql=0.0, md=0.0), dict(ql=0.01, md=3.0)):
        _assert_detect(cro, imgs, _detect_g(ctx, dev, pitch, stride, w, h, n, win, 200, **kw), win, 200, **kw)


# ==================================================================================== 2. tall frames
TALL_W, TALL_H = 40, 2_100_037
TALL19_W, TALL19_H = 24, 524_280 + 2 * 10 + 517


def test_tall_frames_step_every_grid_stride_loop():
    """From the launch arithmetic: the 40 x 2,100,037 frame makes the score kernel's tile loop and the candidate kernel's
    row loop take more than one step, and so does the window-19 frame for the candidate kernel."""
    _, gy, tiles = score_grid(TALL_W, TALL_H)
    assert gy == 65535 and tiles > gy
    _, iw, ih, _, _ = plan(TALL_W, TALL_H, 1, 3)
    assert cand_grid(iw, ih)[1] == 65535 and ih > 8 * 65535
    _, iw, ih, _, _ = plan(TALL19_W, TALL19_H, 1, 19)
    assert TALL19_W >= 24 and cand_grid(iw, ih)[1] == 65535 and ih > 8 * 65535
    # the 1-wide and 1-tall extremes of the frame limit: 2^26 tiles, and ty * 32 would pass 2^31 after the last tile
    w1, gy1, tiles1 = score_grid(1, 2 ** 31 - 1)
    assert (w1, gy1, tiles1) == (1, 65535, 2 ** 26) and (tiles1 + gy1 - 1) * 32 >= 2 ** 31
    assert score_grid(2 ** 31 - 1, 1)[0] == 2 ** 26


_tall_cache = {}


def _tall(cro, kind, w, h, win, seed):
    """The frame, its restated map and the restated detections (md 0 and 3, max_corners 2^20), computed once."""
    key = (kind, w, h, win, seed)
    if key not in _tall_cache:
        img = np.random.default_rng(seed).integers(0, 256, (h, w), dtype=np.uint8) if kind == "noise" else \
            np.tile(worst("bnoise2", w, 4096, seed), (h // 4096 + 1, 1))[:h]
        smap = cro.score(img, win)
        sel = {md: cro.select(smap, win, 1 << 20, quality_level=0.0, min_distance=md) for md in (0.0, 3.0)}
        _tall_cache[key] = img, smap, sel
    return _tall_cache[key]


@pytest.mark.gpu
@pytest.mark.parametrize("n,win", [(1, 3), (2, 3), (1, 19)])
def test_tall_frames(ctx, cro, n, win):
    """The whole map and the detections (2^20 corners reached) on frames taller than the grids' caps."""
    w, h = (TALL_W, TALL_H) if win == 3 else (TALL19_W, TALL19_H)
    frames = [_tall(cro, k, w, h, win, s) for k, s in (("noise", 1), ("bnoise2", 2))[:n]]
    imgs = np.stack([f[0] for f in frames])
    dev, pitch, stride = device_frames(imgs)
    got = _map_g(ctx, dev, pitch, stride, w, h, n, win).cpu().numpy()
    for i in range(n):
        assert_same_bits(got[i], frames[i][1], f"image {i} map")
    del got
    for md in (0.0, 3.0):
        counts = _assert_detect(cro, imgs, _detect_g(ctx, dev, pitch, stride, w, h, n, win, 1 << 20, ql=0.0, md=md), win,
                                1 << 20, ql=0.0, md=md, refs=[f[2][md] for f in frames])
        if win == 3:
            assert (counts == 1 << 20).all()


@pytest.mark.gpu
@pytest.mark.parametrize("w,h", [(1, 2 ** 31 - 1), (2 ** 31 - 1, 1)])
def test_one_pixel_wide_and_tall_frames(ctx, w, h):
    """The largest 1-wide and 1-tall frames: the Sobel fields have no cross-derivative, so every score is 0; every pixel
    is written (the map starts NaN), nothing past it, and detection finds nothing.  Before the tile loop compared tile
    indices instead of ty * 32 < h, the 1-wide frame wrapped past 2^31 and wrote before the map; a frame this wide made
    the host's (w + 31) / 32 overflow."""
    import torch

    img = torch.full((w * h,), 255, dtype=torch.uint8, device="cuda")
    img[::7] = 0
    out = _map_g(ctx, img, w, w * h, w, h, 1, 3)
    assert int(torch.count_nonzero(out)) == 0 and not bool(torch.isnan(out).any())
    del out
    corners, scores, counts = _detect_g(ctx, img, w, w * h, w, h, 1, 3, 5, ql=0.0, md=0.0)
    assert counts[0] == 0 and np.isnan(corners).all() and np.isnan(scores).all()


# ==================================================================================== 3. the largest frame
def sparse_candidates(pieces, W, H, win, ql, ms):
    """The candidate rule of include/ofb200.h on a W x H map that is 0 outside `pieces` [(x0, y0, scores)] (pieces at least
    2 px apart): threshold over the interior, strict key-order local maximum among interior 8-neighbours.  Returns keys
    (-score, raster index, x, y, score) in key order."""
    m = win // 2 + 1
    mx = F32(0)
    for x0, y0, s in pieces:
        hh, ww = s.shape
        ys, xs = slice(max(m - y0, 0), max(min(H - m - y0, hh), 0)), slice(max(m - x0, 0), max(min(W - m - x0, ww), 0))
        if s[ys, xs].size:
            mx = max(mx, s[ys, xs].max())
    thr = max(F32(ql) * mx, F32(ms))
    out = []
    for x0, y0, s in pieces:
        hh, ww = s.shape
        p = np.zeros((hh + 2, ww + 2), F32)  # one pixel of the zero frame around the piece
        p[1:-1, 1:-1] = s
        yy, xx = np.mgrid[y0:y0 + hh, x0:x0 + ww]
        inter = (xx >= m) & (xx <= W - 1 - m) & (yy >= m) & (yy <= H - 1 - m)
        ok = inter & (s > thr)
        for dy in (-1, 0, 1):
            for dx in (-1, 0, 1):
                if dx == dy == 0:
                    continue
                q = p[1 + dy:1 + dy + hh, 1 + dx:1 + dx + ww]
                nin = (xx + dx >= m) & (xx + dx <= W - 1 - m) & (yy + dy >= m) & (yy + dy <= H - 1 - m)
                earlier = dy < 0 or (dy == 0 and dx < 0)
                ok &= ~nin | ((s > q) if earlier else (s >= q))
        for y, x in zip(*np.nonzero(ok)):
            gy_, gx_ = int(y0 + y), int(x0 + x)
            out.append((-float(s[y, x]), gy_ * W + gx_, gx_, gy_, s[y, x]))
    out.sort()
    return out


def greedy(cands, max_corners, md):
    md2 = float(md) * float(md)
    acc = []
    for _, _, x, y, s in cands:
        if len(acc) == max_corners:
            break
        if all(float((x - ax) ** 2 + (y - ay) ** 2) >= md2 for ax, ay, _ in acc):
            acc.append((x, y, s))
    return acc


def crop_layout(W, H, k, seed):
    """k crop origins (48 x 48 crops) spread over a W x H frame, with crops in the last rows and columns."""
    rng = np.random.default_rng(seed)
    pos = {(W - 48, H - 48), (W - 48, 0), (0, H - 48), (W // 2, H - 48), (W - 48, H // 2), (0, 0)}
    while len(pos) < k:
        x, y = int(rng.integers(0, (W - 48) // 64)) * 64, int(rng.integers(0, (H - 48) // 64)) * 64
        pos.add((x, y))
    return sorted(pos)


def crop_content(seed):
    """A 48 x 48 crop: natural content with a zero border of 3 px, so that its scores are 0 on its edge and it can sit
    anywhere in a zero frame (at window 3 a score reaches 2 px past the content)."""
    c = np.zeros((48, 48), np.uint8)
    c[3:45, 3:45] = content("natural", 42, 42, seed) if seed % 2 else content("noise", 42, 42, seed)
    return c


@pytest.mark.parametrize("md,mc", [(0.0, 10_000), (3.0, 10_000), (10.0, 37)])
def test_sparse_reference_equals_plain_greedy(cro, md, mc):
    """The sparse reference of the largest-frame test equals plain_greedy and the restatement on a whole small frame."""
    W, H, win = 400, 300, 3
    frame = np.zeros((H, W), np.uint8)
    pieces = []
    for i, (x0, y0) in enumerate(crop_layout(W, H, 9, 4)):
        frame[y0:y0 + 48, x0:x0 + 48] = crop_content(i)
        pieces.append((x0, y0, cro.score(frame[y0:y0 + 48, x0:x0 + 48], win)))
    smap = cro.score(frame, win)
    for x0, y0, s in pieces:
        assert_same_bits(smap[y0:y0 + 48, x0:x0 + 48], s, "crop map")
    acc = greedy(sparse_candidates(pieces, W, H, win, 0.01, 0.0), mc, md)
    assert acc == plain_greedy(smap, win, mc, 0.01, md, 0.0)
    c, s, n = cro.select(smap, win, mc, quality_level=0.01, min_distance=md)
    assert n == len(acc) and np.array_equal(c[:n], np.array([(x, y) for x, y, _ in acc], F32))


@pytest.mark.gpu
def test_largest_frame(cro):
    """65535 x 32768 = 2^31 - 32768 pixels (the map's last raster index is within 2^16 of 2^31), zeros except 40 crops of
    content, some in the last rows and columns (candidate raster indices above 2^30, columns above 65400).  The map equals
    the restatement of each crop and is 0 elsewhere; the detections equal the sparse reference.  Device memory measured on
    one NVIDIA B200 (1000 W power limit): 10.1 GiB for the frame and the map, 33.6 GiB for the frame and the detection
    workspace (map, keys in and out, cell grid and sort storage: 15.8 bytes per pixel).  The only case of this size."""
    from cuda_optical_flow_2_b200 import Context

    W, H, win = 65535, 32768, 3
    assert W * H == 2 ** 31 - 32768
    with Context(0) as ctx:  # its own workspace, measured here and freed at the end
        _largest_frame(ctx, cro, W, H, win)


def _largest_frame(ctx, cro, W, H, win):
    import torch

    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info()[0]
    img = torch.zeros((H, W), dtype=torch.uint8, device="cuda")
    pieces = []
    for i, (x0, y0) in enumerate(crop_layout(W, H, 40, 11)):
        c = crop_content(i)
        img[y0:y0 + 48, x0:x0 + 48] = torch.from_numpy(c).cuda()
        pieces.append((x0, y0, cro.score(c, win)))
    dev = img.view(-1)
    smap = _map_g(ctx, dev, W, W * H, W, H, 1, win)[0]
    peak_map = free0 - torch.cuda.mem_get_info()[0]
    for x0, y0, s in pieces:
        assert_same_bits(smap[y0:y0 + 48, x0:x0 + 48].cpu().numpy(), s, f"crop ({x0}, {y0})")
        smap[y0:y0 + 48, x0:x0 + 48] = 0
    assert int(torch.count_nonzero(smap)) == 0  # 0 (and no NaN) outside the crops
    del smap
    torch.cuda.empty_cache()
    peak = 0
    for md, mc in ((0.0, 20_000), (3.0, 20_000), (12.0, 701)):
        cands = sparse_candidates(pieces, W, H, win, 0.01, 0.0)
        assert max(k[1] for k in cands) > 2 ** 30 and max(k[2] for k in cands) > 65400
        acc = greedy(cands, mc, md)
        corners, scores, counts = _detect_g(ctx, dev, W, W * H, W, H, 1, win, mc, ql=0.01, md=md)
        peak = max(peak, free0 - torch.cuda.mem_get_info()[0])
        ref_c = np.full((mc, 2), np.nan, F32)
        ref_s = np.full(mc, np.nan, F32)
        if acc:
            ref_c[:len(acc)] = [(x, y) for x, y, _ in acc]
            ref_s[:len(acc)] = [s for _, _, s in acc]
        assert counts[0] == len(acc), (md, counts[0], len(acc))
        assert_same_bits(corners[0], ref_c, f"md {md} corners")
        assert_same_bits(scores[0], ref_s, f"md {md} scores")
    print(f"largest frame ({torch.cuda.get_device_name()}): frame + map {peak_map / 2 ** 30:.1f} GiB, frame + detection "
          f"workspace {peak / 2 ** 30:.1f} GiB")


# ==================================================================================== 4. chunk boundaries of the selection
def lattice(nx, ny, sx, sy, win, bright, jitter=None):
    """An nx x ny lattice of isolated impulses with spacing (sx, sy) >= win + 3, each its own single candidate; bright(i, j)
    sets the impulse's brightness, so its score, so its order."""
    m = win // 2 + 1
    off = m + win
    w, h = off * 2 + sx * (nx - 1) + 1, off * 2 + sy * (ny - 1) + 1
    img = np.zeros((h, w), np.uint8)
    for j in range(ny):
        for i in range(nx):
            img[off + j * sy, off + i * sx] = bright(i, j)
    return img


def checker_bright(i, j):
    """A checkerboard colouring of the lattice: bright (200) impulses, then dim (100) ones, in key order.  With
    min_distance just above the spacing every dim impulse conflicts only with bright ones, which all come first: at 1024
    candidates chunk 0 holds exactly the bright ones, so every conflict of a later chunk is found in the grid."""
    return 200 if (i + j) % 2 == 0 else 100


LATTICES = {511: (73, 7), 512: (32, 16), 513: (27, 19), 1024: (32, 32), 1025: (41, 25), 1537: (53, 29)}


@pytest.mark.parametrize("count", sorted(LATTICES))
@pytest.mark.parametrize("win", [3, 5, 9])
def test_lattice_candidate_counts(cro, count, win):
    """Each impulse of the lattice is exactly one candidate: the candidate counts straddle the 512-key chunks."""
    nx, ny = LATTICES[count]
    s = win + 3
    img = lattice(nx, ny, s, s, win, checker_bright)
    _, _, n = cro.detect(img, win, 1 << 20, quality_level=0.0, min_distance=0.0)
    assert n == count


MD_SWEEP = [1.0, f32_next(1, 2), 2.0, f32_next(2, 3), float(F32(math.sqrt(5))), f32_next(math.sqrt(5), 0),
            f32_next(math.sqrt(5), 3), 5.0, f32_next(5, 0), 7.5, 31.9, 500.0, 1e6, FLT_MAX]


def test_selection_grid_restated():
    """For every min_distance used here and at shapes up to the frame limit: a cell never holds two accepted corners
    (2 (c-1)^2 < md^2), the grid covers the interior, the looked-up cells cover every |dx|, |dy| that can conflict, and
    the grid arithmetic stays inside int."""
    mds = sorted(set(MD_SWEEP + [0.0, 1.5, 2.5, 3.0, 6.5, 8.5, 10.0, f32_next(10, 11), 12.0, 12.5, 4.9, 5.1, 7.1, 6.9]))
    for md in mds:
        md2 = md * md
        if md2 <= 1.0:
            continue  # no suppression
        for W, H in ((40, 30), (3840, 2160), (65535, 32768), (40, 2_100_037), (5, (2 ** 31 - 1) // 5), (429_496_729, 5)):
            _, iw, ih, cap, _ = plan(W, H, 1, 3)
            if not cap:
                continue
            c, gw, gh, reach = select_grid(md, iw, ih)
            assert c >= 1 and 2 * (c - 1) ** 2 < md2
            assert gw * c >= iw and gh * c >= ih and iw + c - 1 < 2 ** 31 and gw * gh <= iw * ih
            far = min(math.ceil(md) - 1, max(iw, ih) - 1)  # the largest integer |dx| with dx^2 < md^2, inside the interior
            assert far * far < md2 and reach >= far
            for gx in sorted({0, 1, c - 1, c, iw // 2, iw - 1}):
                if not 0 <= gx < iw:
                    continue
                cx0, cx1 = max(0, gx - reach) // c, min(gw - 1, (gx + reach) // c)
                assert cx0 <= max(0, gx - far) // c and cx1 >= min(iw - 1, gx + far) // c
                assert gx + reach < 2 ** 31


@pytest.mark.gpu
@pytest.mark.parametrize("count", sorted(LATTICES))
def test_chunk_boundaries(ctx, cro, count):
    """Lattices of 511 .. 1537 candidates at windows 3 and 9: max_corners running out at count - 1, 512, 1024 and in the
    middle of a chunk; min_distance just above the spacing (each dim impulse's conflicts are bright ones, which fill the
    earlier chunks: the grid lookup), at the spacing, and the sweep."""
    nx, ny = LATTICES[count]
    for win in (3, 9):
        s = win + 3
        img = lattice(nx, ny, s, s, win, checker_bright)[None]
        h, w = img.shape[1:]
        dev, pitch, stride = device_frames(img)
        mcs = sorted({count - 1, 512, 1024, 300, count + 3, 1 << 20} - {0})
        for md in [f32_next(s, s + 1), float(s), 0.0] + MD_SWEEP:
            for mc in (mcs if md in (f32_next(s, s + 1), 0.0) else [count + 3]):
                _assert_detect(cro, img, _detect_g(ctx, dev, pitch, stride, w, h, 1, win, mc, ql=0.0, md=md), win, mc, ql=0.0,
                               md=md)


@pytest.mark.gpu
def test_exact_distance_lattice(ctx, cro):
    """Impulses on a 6 x 8 lattice: horizontal neighbours 6 apart, vertical 8, diagonal exactly 10 (6-8-10).  md 10 keeps
    the diagonal pairs, nextafter(10, 11) separates them; 1537 candidates, three chunks."""
    img = lattice(53, 29, 6, 8, 3, lambda i, j: 60 + (i * 7 + j * 13) % 190)[None]
    h, w = img.shape[1:]
    dev, pitch, stride = device_frames(img)
    got = {}
    for md in (6.0, f32_next(6, 7), 8.0, f32_next(8, 9), 10.0, f32_next(10, 11), f32_next(10, 0)):
        got[md] = _assert_detect(cro, img, _detect_g(ctx, dev, pitch, stride, w, h, 1, 3, 2000, ql=0.0, md=md), 3, 2000, ql=0.0,
                                 md=md)[0]
    assert got[10.0] > got[f32_next(10, 11)] and got[6.0] > got[f32_next(6, 7)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["noise", "natural"])
def test_min_distance_sweep_4k(ctx, cro, kind):
    w, h, win = 3840, 2160, 3
    img = content(kind, w, h, 21)[None] if kind == "noise" else \
        np.tile(content("natural", 480, 270, 21), (8, 8))[None]
    dev, pitch, stride = device_frames(img)
    smap = cro.score(img[0], win)
    for md in [0.0] + MD_SWEEP:
        ref = cro.select(smap, win, 1 << 20, quality_level=0.0, min_distance=md)
        _assert_detect(cro, img, _detect_g(ctx, dev, pitch, stride, w, h, 1, win, 1 << 20, ql=0.0, md=md), win, 1 << 20,
                       ql=0.0, md=md, refs=[ref])


# ==================================================================================== 5. ties across seams
def mirrored(w, h, ax, ay, seed):
    """Random content mirrored about every column boundary ax + 32 k and row boundary ay + 32 k: equal scores on the two
    pixels next to each axis (away from the frame edge)."""
    t = np.random.default_rng(seed).integers(0, 256, (32, 32), dtype=np.uint8)
    q = np.block([[t, t[:, ::-1]], [t[::-1], t[::-1, ::-1]]])  # period 64, symmetric about 0 and 32 (mod 64)
    reps = np.tile(q, (h // 64 + 3, w // 64 + 3))
    return np.ascontiguousarray(reps[64 - ay % 64:64 - ay % 64 + h, 64 - ax % 64:64 - ax % 64 + w])


@pytest.mark.gpu
@pytest.mark.parametrize("win", [3, 9, 19])
def test_ties_across_seams(ctx, cro, win):
    """Mirror axes on the score kernel's 32-column and 32-row tile seams, on the candidate kernel's warp seam (interior
    column x - m a multiple of 32) and its 8-row block seam; periodic content (a 7 x 5 tile) with md just above and below
    the periods."""
    m = win // 2 + 1
    w, h = 203, 157
    imgs = np.stack([mirrored(w, h, 0, 0, 1), mirrored(w, h, m, m, 2), mirrored(w, h, m, m + 8, 3),
                     np.tile(np.random.default_rng(4).integers(0, 256, (5, 7), dtype=np.uint8), (h // 5 + 1, w // 7 + 1))[:h, :w]])
    s0 = cro.score(imgs[0], win)
    x = 64 + 32
    assert (s0[40:110, x - 1] == s0[40:110, x]).all() and (s0[x - 1, 40:110] == s0[x, 40:110]).all()
    s1 = cro.score(imgs[1], win)
    assert (s1[40:110, m + 63] == s1[40:110, m + 64]).all()
    dev, pitch, stride = device_frames(imgs)
    got = _map_g(ctx, dev, pitch, stride, w, h, len(imgs), win).cpu().numpy()
    for i in range(len(imgs)):
        assert_same_bits(got[i], cro.score(imgs[i], win), f"image {i} map")
    for md in (0.0, 2.5, 4.9, 5.0, f32_next(5, 6), 6.9, 7.0, f32_next(7, 8)):
        _assert_detect(cro, imgs, _detect_g(ctx, dev, pitch, stride, w, h, len(imgs), win, 3000, ql=0.0, md=md), win, 3000,
                       ql=0.0, md=md)


# ==================================================================================== 6. the threshold
def bright_frame(w, h, seed):
    """Near-white content (245..254): against the zero padding outside the frame the image's largest scores are in the
    border band, while the interior sees only the weak texture."""
    return (245 + np.random.default_rng(seed).integers(0, 10, (h, w))).astype(np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("win", [3, 9])
def test_threshold(ctx, cro, win):
    w, h = 120, 90
    m = win // 2 + 1
    img = bright_frame(w, h, win)
    smap = cro.score(img, win)
    inter = smap[m:h - m, m:w - m]
    assert smap.max() > 4 * inter.max() > 0  # over the whole frame, quality_level 0.5 would leave nothing
    dev, pitch, stride = device_frames(img[None])
    n = _assert_detect(cro, img[None], _detect_g(ctx, dev, pitch, stride, w, h, 1, win, 5000, ql=0.5, md=0.0), win, 5000,
                       ql=0.5, md=0.0)[0]
    assert n > 0
    # min_score at a candidate's exact score (excluded) and one ulp below (included)
    _, rs, rn = cro.detect(img, win, 5000, quality_level=0.0, min_distance=0.0)
    s = F32(rs[rn // 3])
    counts = []
    for ms in (float(s), f32_next(s, 0)):
        counts.append(_assert_detect(cro, img[None], _detect_g(ctx, dev, pitch, stride, w, h, 1, win, 5000, ql=0.0, md=0.0,
                                                               ms=ms), win, 5000, ql=0.0, md=0.0, ms=ms)[0])
    assert counts[1] > counts[0]
    # quality_level * max equal to a candidate's score
    mx = F32(inter.max())
    hit = None
    for c in rs[1:rn]:
        ql = F32(c) / mx
        for q in (ql, np.nextafter(ql, F32(0)), np.nextafter(ql, F32(1))):
            if q <= 1 and F32(q) * mx == F32(c):
                hit = float(q)
                break
        if hit is not None:
            break
    assert hit is not None
    n_eq = _assert_detect(cro, img[None], _detect_g(ctx, dev, pitch, stride, w, h, 1, win, 5000, ql=hit, md=0.0), win, 5000,
                          ql=hit, md=0.0)[0]
    assert 0 < n_eq < rn


# ==================================================================================== 7. caller buffers and streams
@pytest.mark.gpu
@pytest.mark.parametrize("mc", [1, 7, 513])
def test_caller_buffers(ctx, cro, mc):
    """Guarded outputs with odd max_corners (per-image slices at 8- but not 16-byte offsets), scores NULL, pitch = w with
    odd w, an odd image stride that is not a multiple of the pitch, and stride 0 with one image."""
    w, h, win = 67, 45, 5
    imgs = np.stack([content(k, w, h, i) for i, k in enumerate(["natural", "noise", "textured"])])
    for pitch, stride in ((w, w * h), (w, w * h + 13), (80, 80 * h + 7)):
        dev, pitch, stride = device_frames(imgs, pitch, stride, 0xFF)
        assert_same_bits(_map_g(ctx, dev, pitch, stride, w, h, 3, win).cpu().numpy(),
                         np.stack([cro.score(i, win) for i in imgs]), f"map, pitch {pitch} stride {stride}")
        for sc in (True, False):
            _assert_detect(cro, imgs, _detect_g(ctx, dev, pitch, stride, w, h, 3, win, mc, ql=0.0, md=3.0, with_scores=sc),
                           win, mc, ql=0.0, md=3.0)
    dev, pitch, _ = device_frames(imgs[:1], w)
    assert_same_bits(_map_g(ctx, dev, pitch, 0, w, h, 1, win).cpu().numpy()[0], cro.score(imgs[0], win), "stride 0")
    _assert_detect(cro, imgs[:1], _detect_g(ctx, dev, pitch, 0, w, h, 1, win, mc, ql=0.0, md=3.0), win, mc, ql=0.0, md=3.0)


@pytest.mark.gpu
def test_stream_with_work_queued_ahead(ctx, cro):
    """The frames are written on a side stream behind a long spin kernel; detection on that stream must see them."""
    import torch

    w, h, win, n, mc = 256, 192, 7, 3, 400
    imgs = np.stack([content("natural", w, h, 30 + i) for i in range(n)])
    src = torch.from_numpy(imgs).cuda()
    dev = torch.zeros_like(src)
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(50_000_000)
        dev.copy_(src)
        got = _detect_g(ctx, dev, w, w * h, w, h, n, win, mc, ql=0.0, md=4.0, stream=side.cuda_stream)
        smap = _map_g(ctx, dev, w, w * h, w, h, n, win, stream=side.cuda_stream).cpu().numpy()
    _assert_detect(cro, imgs, got, win, mc, ql=0.0, md=4.0)
    for i in range(n):
        assert_same_bits(smap[i], cro.score(imgs[i], win), f"image {i} map")


@pytest.mark.gpu
def test_refusals_leave_guards_untouched(ctx):
    """Every refusal of test_corners' list, on guarded outputs: nothing launched, no output or guard written."""
    import torch

    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    w, h, n, mc = 64, 48, 2, 7
    img = torch.zeros((n, h, 64), dtype=torch.uint8, device="cuda")
    cb, corners = _guarded(n * mc * 2, torch.float32, 7.0)
    sb, scores = _guarded(n * mc, torch.float32, 7.0)
    kb, counts = _guarded(n, torch.int32, 7)
    mb, smap = _guarded(n * h * w, torch.float32, 7.0)
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
        torch.cuda.synchronize()
        for b, fill in ((cb, 7.0), (sb, 7.0), (kb, 7), (mb, 7.0)):
            assert bool((b == fill).all()), kw
    for kw, code in [(dict(nn=0), inv), (dict(nn=65536), inv), (dict(win=8), uns), (dict(im=None), inv), (dict(out=None), inv),
                     (dict(out=smap.data_ptr() + 2), inv), (dict(pitch=32), inv), (dict(ww=65536, hh=32768), inv)]:
        assert score_map(**kw) == code, (kw, lib.ofb_last_error())
        torch.cuda.synchronize()
        assert bool((mb == 7.0).all()), kw
    assert ctx.launch_count == before


# ==================================================================================== 8. workspace reuse
def reuse_sequence():
    """A fixed sequence of about 30 calls: n 1 and 3, suppression on and off, growing and shrinking shapes, every window,
    map-only calls, a tracker call, and a reservation at a larger size followed by smaller calls."""
    rng = np.random.default_rng(2024)
    shapes = [(40, 30), (200, 150), (64, 300), (33, 17), (400, 260), (90, 70), (7, 7), (320, 33), (150, 220), (48, 48)]
    seq = []
    for i in range(30):
        w, h = shapes[i % len(shapes)]
        win = WINS[i % len(WINS)]
        n = 1 if i % 2 == 0 else 3
        md = (0.0, 3.0, 1.0, 7.5)[(i // 2) % 4]
        op = "map" if i % 5 == 4 else "detect"
        if i == 12:
            op = "track"
        if i == 20:
            op = "reserve"
        seq.append(dict(op=op, w=w, h=h, win=win, n=n, md=md, mc=int(rng.integers(1, 600)), ql=float(rng.choice([0.0, 0.01])),
                        seed=i))
    return seq


def _run_call(ctx, cro, oracle, call):
    import torch

    w, h, n, win = call["w"], call["h"], call["n"], call["win"]
    if call["op"] == "reserve":
        ctx.reserve_corners(1000, 800, 3, 19, 4000)
        return None
    if call["op"] == "track":
        from cuda_optical_flow_2_b200 import planar_to_device

        prev = np.stack([oracle.make_frame(160, 120, 0, 0, 4, call["seed"] + i) for i in range(n)])
        nxt = np.stack([oracle.make_frame(160, 120, 0.6, -0.3, 4, call["seed"] + i) for i in range(n)])
        p, q = planar_to_device(prev), planar_to_device(nxt)
        pts = torch.from_numpy(np.random.default_rng(call["seed"]).uniform(10, 110, (n, 64, 2)).astype(F32)).cuda()
        flow, st = ctx.track_points_device(p, q, 160, 2, 9, pts)
        torch.cuda.synchronize()
        return [flow.cpu().numpy(), st.cpu().numpy()]
    imgs = np.stack([content(("natural", "noise")[i % 2], w, h, call["seed"] * 10 + i) for i in range(n)])
    dev, pitch, stride = device_frames(imgs)
    if call["op"] == "map":
        got = _map_g(ctx, dev, pitch, stride, w, h, n, win).cpu().numpy()
        for i in range(n):
            assert_same_bits(got[i], cro.score(imgs[i], win), f"{call} map {i}")
        return [got]
    got = _detect_g(ctx, dev, pitch, stride, w, h, n, win, call["mc"], ql=call["ql"], md=call["md"])
    _assert_detect(cro, imgs, got, win, call["mc"], ql=call["ql"], md=call["md"])
    return list(got)


@pytest.mark.gpu
def test_workspace_reuse(cro, oracle):
    """One fresh context runs the sequence; every result equals the restatement and the same call on a fresh context."""
    import torch

    from cuda_optical_flow_2_b200 import Context

    torch.cuda.synchronize()
    seq = reuse_sequence()
    assert {c["n"] for c in seq} == {1, 3} and {c["win"] for c in seq} == set(WINS)
    assert {c["op"] for c in seq} == {"map", "detect", "track", "reserve"}
    with Context(0) as a:
        for call in seq:
            got = _run_call(a, cro, oracle, call)
            if got is None:
                continue
            with Context(0) as b:
                ref = _run_call(b, cro, oracle, call)
            for g, r in zip(got, ref):
                assert np.array_equal(np.asarray(g).view(np.uint8), np.asarray(r).view(np.uint8)), call


# ==================================================================================== 9. refusals at the slot limit
def test_slot_limit_planning():
    """65535 images of 370 x 370 at window 3 hold 65535 * 183^2 >= 2^31 candidate slots and are refused.  2^31 - 1 is prime,
    so the largest total a shape can reach below the limit is 2^31 - 2: 34881 images of 376 x 666 (iw 372, ih 662,
    186 * 331 slots each), which passes; one row more per image passes the limit."""
    assert plan(370, 370, 65535, 3)[4] >= 2 ** 31
    assert all((2 ** 31 - 1) % p for p in range(2, 46341))
    m, iw, ih, cap, total = plan(376, 666, 34881, 3)
    assert (iw, ih, cap) == (372, 662, 186 * 331) and total == 2 ** 31 - 2
    assert plan(376, 668, 34881, 3)[4] >= 2 ** 31
    assert 376 * 666 < 2 ** 31 and 34881 <= 65535


@pytest.mark.gpu
def test_slot_limit_refusal(ctx):
    """The refusal comes from the planning arithmetic alone: the frames and outputs passed are far too small for the shape,
    and nothing may touch them."""
    import torch

    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    n, w, h, mc = 65535, 370, 370, 3
    img = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    cb, corners = _guarded(64, torch.float32, SENT)
    sb, scores = _guarded(64, torch.float32, SENT)
    kb, counts = _guarded(64, torch.int32, -7)
    torch.cuda.synchronize()
    before = ctx.launch_count
    rc = lib.ofb_detect_corners_device(ctx._h, img.data_ptr(), w, w * h, w, h, n, 3, mc, 0.01, 3.0, 0.0, corners.data_ptr(),
                                       scores.data_ptr(), counts.data_ptr(), None)
    assert rc == _lib.OFB_ERR_UNSUPPORTED
    assert f"{n} images of {w}x{h} hold {plan(w, h, n, 3)[4]} candidate slots".encode() in lib.ofb_last_error()
    assert lib.ofb_ctx_reserve_corners(ctx._h, w, h, n, 3, mc) == _lib.OFB_ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert ctx.launch_count == before
    assert bool((cb == SENT).all()) and bool((sb == SENT).all()) and bool((kb == -7).all())
