"""Row strips thinner than their halo (csrc/strips.cu, dist.NativeStrips).

When strips are thinner than the rows a rank holds around them, a rank's halo rows come from -- and its own rows go to --
ranks that are not adjacent.  That takes code paths the adjacent-only plans never reach: the level-0 image exchange to up
to 4 ranks (2 copy segments each), the copy and wait kernels that take over a cumulative-flow exchange the level kernel's
two push / wait slots cannot carry (mixed with the fused form on the other exchanges of the same pair), and a fused push
from every row block of a strip.  Plans whose exchanges fan out further than the runner carries are refused at create.

CPU: a plain restatement of the halo-row table (the image-buffer rows of ofb_strips_plan_query, the exchanges and their
send / receive lists, the end-of-pair handshake) against the library on every rank and level; a sweep of a few thousand
plans in which the library refuses exactly the plans the restatement finds over the limits; dist.StripPlan and the library
refusing the same plans for too few coarsest rows; every GPU case below in its intended class; the motion of every GPU
case inside `reach` by the warp rule (support.requested_rows), so that a flag is a failure.
GPU: ranks in this process on one device, phases interleaved on one stream (as test_dist.py): three pairs back to back per
plan bit-identical to the whole frame in both solve modes, both per-pixel warp modes and flow_scale 1 and 8/15, with the
launches per pair counted from the restated table (fused and separate exchanges, with and without the total flow); forced
row splits; checked pairs; CUDA graph replay; refusals on every rank; and, with 4 or 8 GPUs, the whole pair per process over
CUDA IPC.
"""
import ctypes as C
import itertools
import os

import pytest

from support import BIL, NEAR, S815, assert_equals_whole, assert_same_bits, reach_flag, requested_rows, rows, solve  # noqa: F401

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PEER_MAX_DST, PEER_MAX_SEG = 4, 8  # csrc/strips.cu: ranks one exchange sends to / receives from; copy segments per exchange
OFB_OK, OFB_ERR_INVALID, OFB_ERR_UNSUPPORTED = 0, 1, 3


# ------------------------------------------------------------------------------------------ the halo-row table, restated
class Table:
    """The schedule of ofb_strips_create / _create_fb (fb_reach None: a plain handle) written out for every rank.

    rows[k][rank] = (y0, y1, by0, by1, cy0, cy1, eb0, eb1) as ofb_strips_plan_query reports them; send[x][rank] /
    recv[x][rank] = [(peer, lo, hi)] per exchange x (0 = level-0 images, j = cumulative flow of level L-j, L-1+j its backward
    twin, 2L-1 the backward total rows the checks sample); sources[rank] / done_from[rank] = the ranks of the end-of-pair
    handshake."""

    def __init__(self, W, H, levels, win, world, reach, fb_reach=None):
        self.W, self.H, self.L, self.win, self.world, self.reach, self.fb_reach = W, H, levels, win, world, reach, fb_reach
        r, L = win // 2, levels
        halo = r + 2 + reach + 2
        hc = H >> (L - 1)
        bound = [rk * hc // world for rk in range(world)]
        self.rows = [[None] * world for _ in range(L)]
        for rk in range(world):
            for k in range(L - 1, -1, -1):  # coarse to fine: a level's buffer also holds what building the next one takes
                h = H >> k
                y0 = bound[rk] << (L - 1 - k)
                y1 = h if rk == world - 1 else bound[rk + 1] << (L - 1 - k)
                by0, by1 = max(0, y0 - halo), min(h, y1 + halo)
                cy0, cy1 = (max(0, (y0 - r - 2) >> 1), min(H >> (k + 1), ((y1 + r + 1) >> 1) + 1)) if k < L - 1 else (0, 0)
                eb0, eb1 = by0, by1
                if k < L - 1:
                    ceb0, ceb1 = self.rows[k + 1][rk][6:]
                    eb0, eb1 = min(by0, max(0, 2 * ceb0 - 1)), max(by1, min(h, 2 * (ceb1 - 1) + 2))
                self.rows[k][rk] = (y0, y1, by0, by1, cy0, cy1, eb0, eb1)
        self.nx = L if fb_reach is None else 2 * L
        self.send = [[[] for _ in range(world)] for _ in range(self.nx)]
        self.recv = [[[] for _ in range(world)] for _ in range(self.nx)]
        for x in range(self.nx):
            ex = [self.exchange_rows(x, rk) for rk in range(world)]
            for rk, peer in itertools.permutations(range(world), 2):
                (m0, m1, _, _), (_, _, pw0, pw1) = ex[rk], ex[peer]
                if max(m0, pw0) < min(m1, pw1):
                    self.send[x][rk].append((peer, max(m0, pw0), min(m1, pw1)))
                    self.recv[x][peer].append((rk, max(m0, pw0), min(m1, pw1)))
        for x in range(self.nx):
            for rk in range(world):
                self.recv[x][rk].sort()
        self.done_from = [sorted({p for x in range(self.nx) for p, _, _ in self.send[x][rk]}) for rk in range(world)]
        self.sources = [sorted({p for x in range(self.nx) for p, _, _ in self.recv[x][rk]}) for rk in range(world)]

    def fb_rows(self, rank):
        y0, y1 = self.rows[0][rank][:2]
        return max(0, y0 - self.fb_reach), min(self.H, y1 + self.fb_reach + 1)

    def exchange_rows(self, x, rank):
        """(own rows, window) of exchange x on `rank`: the rows it owns that others may need, and the rows its buffer holds."""
        L = self.L
        if x == 0:
            y0, y1, _, _, _, _, eb0, eb1 = self.rows[0][rank]
            return y0, y1, eb0, eb1
        if x == 2 * L - 1:
            return self.rows[0][rank][:2] + self.fb_rows(rank)
        j = x if x < L else x - (L - 1)
        return self.rows[L - j][rank][:2] + self.rows[L - 1 - j][rank][4:6]

    def fan_out(self, x):
        """Most ranks exchange x sends to or receives from on any rank."""
        return max(max(len(self.send[x][rk]), len(self.recv[x][rk])) for rk in range(self.world))

    def over_limit(self):
        """What the runner could not carry, or None."""
        for rk in range(self.world):
            for x in range(self.nx):
                if len(self.send[x][rk]) > PEER_MAX_DST or len(self.recv[x][rk]) > PEER_MAX_DST:
                    return f"exchange {x} on rank {rk}: {len(self.send[x][rk])} / {len(self.recv[x][rk])} ranks"
            if 2 * len(self.send[0][rk]) > PEER_MAX_SEG:
                return f"image exchange on rank {rk}: {2 * len(self.send[0][rk])} segments"
            if len(self.sources[rk]) > 2 * PEER_MAX_DST or len(self.done_from[rk]) > 2 * PEER_MAX_DST:
                return f"handshake of rank {rk}: {len(self.sources[rk])} / {len(self.done_from[rk])} ranks"
        return None

    def launches(self, fused=True, checked=False):
        """Kernel launches of one pair over all ranks: the image push and wait where the image exchange has peers, L-1
        pyramid steps, L level kernels per direction, per cumulative-flow exchange a copy kernel unless the fused slots (at
        most 2 targets) carried it and a wait kernel unless the level kernel waited itself (at most 2 sources); in a checked
        pair the check-row exchange (copy kernel unless level 0's slots carried it, always a wait kernel) and the check; the
        end-of-pair handshake."""
        L, n = self.L, 0
        cum = list(range(1, L)) + (list(range(L, 2 * L - 1)) if checked else [])
        for rk in range(self.world):
            n += bool(self.send[0][rk]) + bool(self.recv[0][rk]) + (L - 1) + L * (2 if checked else 1)
            for x in cum:
                s, r = len(self.send[x][rk]), len(self.recv[x][rk])
                n += (s > 0 and not (fused and s <= 2)) + (r > 0 and not (fused and r <= 2))
            if checked:
                s, r = len(self.send[2 * L - 1][rk]), len(self.recv[2 * L - 1][rk])
                n += (s > 0 and not (fused and s <= 2)) + (r > 0) + 1
            n += self.world > 1
        return n


def query(W, H, levels, win, world, rank, reach, level):
    """(rc, out8) of ofb_strips_plan_query."""
    from cuda_optical_flow_2_b200 import _lib

    out = (C.c_int * 8)()
    rc = _lib.load().ofb_strips_plan_query(W, H, levels, win, world, rank, reach, level, out)
    return rc, tuple(out)


# ------------------------------------------------------------------------------------------ the cases the GPU runs
# name -> (W, H, levels, win, world, reach, class).  Class ("image", n): the image exchange fans out to n ranks and every
# cumulative-flow exchange to at most 2 (the kernels' own slots); ("cum", n, ranks): some cumulative-flow exchange fans out
# to n, and the ranks on which one exceeds 2 (copy and wait kernels) are `ranks`.
CASES = {
    "image3-320x240x3-4": (320, 240, 3, 9, 4, 16, ("image", 3)),
    "image3-1920x1080x5-4": (1920, 1080, 5, 9, 4, 16, ("image", 3)),
    "image4-320x240x3-5": (320, 240, 3, 9, 5, 16, ("image", 4)),
    "image4-321x243x3-5": (321, 243, 3, 9, 5, 16, ("image", 4)),
    "image4-1920x1080x4w9-8": (1920, 1080, 4, 9, 8, 16, ("image", 4)),
    "image4-1920x1080x4w15-8": (1920, 1080, 4, 15, 8, 16, ("image", 4)),
    "image4-1920x1080x3-12": (1920, 1080, 3, 9, 12, 16, ("image", 4)),
    "image4-1920x1080x3-16": (1920, 1080, 3, 9, 16, 16, ("image", 4)),
    "cum3-320x52x3-5": (320, 52, 3, 9, 5, 16, ("cum", 3, [1, 3])),
    "cum3-333x52x3-5-reach2": (333, 52, 3, 9, 5, 2, ("cum", 3, [1, 3])),
    "cum4-320x48x3-5-reach0": (320, 48, 3, 9, 5, 0, ("cum", 4, [2])),
    "cum4-320x40x4w3-5-reach0": (320, 40, 4, 3, 5, 0, ("cum", 4, [1, 2, 3])),
}
# checked handles: name -> (W, H, levels, win, world, reach, fb_reach, {exchange: fan-out})
FB_CASES = {
    "checked-320x52x3-5": (320, 52, 3, 9, 5, 16, 16, {0: 4, 1: 3, 3: 3, 5: 4}),
    "checked-640x480x3-8": (640, 480, 3, 9, 8, 16, 100, {0: 4, 1: 2, 3: 2, 5: 4}),
}
# plans over the limits: (W, H, levels, win, world, reach, fb_reach)
REFUSED = {
    "1920x1080x5-8": (1920, 1080, 5, 9, 8, 16, None),
    "320x240x3-8": (320, 240, 3, 9, 8, 16, None),
    "checked-640x480x3-8-fb200": (640, 480, 3, 9, 8, 16, 200),
}
# per pair (dx, dy) of next against prev: small vertical motion where reach is small
MOTION = {16: [(2.25, -1.5), (-3.0, 0.75), (0.5, 2.0)], 2: [(2.25, -0.5), (-3.0, 0.25), (0.5, 0.75)],
          0: [(2.25, -0.25), (-3.0, 0.125), (0.5, 0.25)]}
# (solve, warp mode, flow_scale) per case: every case exact and fast bilinear and exact nearest, some at flow_scale 8/15
VARIANTS = [(name, v) for name in CASES for v in [("exact", BIL, 1.0), ("fast", BIL, 1.0), ("exact", NEAR, 1.0)]] + \
    [(name, ("exact", BIL, S815)) for name in ("image4-320x240x3-5", "cum3-320x52x3-5", "cum4-320x48x3-5-reach0")]


def frames(oracle, W, H, seed, dx, dy):
    return oracle.make_frame(W, H, 0, 0, 8, seed), oracle.make_frame(W, H, dx, dy, 8, seed)


# ------------------------------------------------------------------------------------------------------------------ CPU
def test_restated_table_matches_plan_query():
    """Every rank and level of plans that are accepted, plain and thin: own rows, kernel rows, coarser rows and the image
    buffer rows (with what building the coarser levels' halo rows locally takes) equal ofb_strips_plan_query."""
    n = 0
    for W, H, levels, win, world, reach, _ in list(CASES.values()) + [(640, 480, 3, 9, 2, 16, 0), (1001, 777, 3, 19, 3, 2, 0),
                                                                      (64, 24, 1, 3, 4, 0, 0), (333, 97, 5, 5, 3, 0, 0)]:
        t = Table(W, H, levels, win, world, reach)
        assert t.over_limit() is None
        for rk in range(world):
            for k in range(levels):
                rc, out = query(W, H, levels, win, world, rk, reach, k)
                assert rc == OFB_OK and out == t.rows[k][rk], (W, H, levels, win, world, rk, k, out, t.rows[k][rk])
                n += 1
    assert n > 300


def sweep_plans():
    """A few thousand plans: odd and even widths, H 24..700, 1-5 levels, windows 3 / 5 / 9 / 19, 1-16 ranks, reach 0 / 2 / 16."""
    heights = [24, 25, 31, 40, 48, 52, 64, 97, 120, 161, 240, 243, 361, 480, 511, 700]
    for i, (H, levels, win, world, reach) in enumerate(itertools.product(heights, range(1, 6), (3, 5, 9, 19), range(1, 17),
                                                                          (0, 2, 16))):
        if i % 3 == 0:  # every third combination: about 4,000 plans
            yield (37, 320, 333, 64, 7)[i % 5], H, levels, win, world, reach


def test_refusal_sweep_matches_restated_limits():
    """ofb_strips_plan_query refuses exactly the plans whose restated table fans out past what the runner carries
    (OFB_ERR_UNSUPPORTED, on every rank alike: the first and the last are asked), and too few coarsest rows or columns
    with OFB_ERR_INVALID; accepted plans report the restated rows.  The peers of every exchange are a run of ranks around
    the rank (the library scans outward from it).  Plans at the limit are accepted, and every plan on more than 5 ranks
    whose coarsest strips are all 1 or all 2 rows is refused (on 5 ranks or fewer no rank has more than 4 others)."""
    from cuda_optical_flow_2_b200 import _lib

    verdicts = {OFB_OK: 0, OFB_ERR_INVALID: 0, OFB_ERR_UNSUPPORTED: 0}
    at_limit = one_row = 0
    for W, H, levels, win, world, reach in sweep_plans():
        what = (W, H, levels, win, world, reach)
        rc0, _ = query(W, H, levels, win, world, 0, reach, 0)
        rc1, out = query(W, H, levels, win, world, world - 1, reach, levels - 1)
        assert rc0 == rc1, what
        verdicts[rc0] += 1
        hc = H >> (levels - 1)
        if hc < world or (W >> (levels - 1)) < 1:
            assert rc0 == OFB_ERR_INVALID, what
            continue
        t = Table(W, H, levels, win, world, reach)
        over = t.over_limit()
        assert rc0 == (OFB_OK if over is None else OFB_ERR_UNSUPPORTED), f"{what}: restated {over}"
        if over is not None:
            assert "limit of" in _lib.load().ofb_last_error().decode(), what
        else:
            assert out == t.rows[levels - 1][world - 1], what
            at_limit += max(t.fan_out(x) for x in range(t.nx)) == PEER_MAX_DST
        if hc in (world, 2 * world) and world > 5:
            one_row += 1
            assert over is not None, what
        for x in range(t.nx):
            for rk in range(world):
                peers = sorted({p for p, _, _ in t.send[x][rk] + t.recv[x][rk]} | {rk})
                assert peers == list(range(peers[0], peers[-1] + 1)), (what, x, rk, peers)
    assert sum(verdicts.values()) > 3000 and min(verdicts.values()) > 300, verdicts
    assert at_limit > 100 and one_row > 10


def test_strip_plan_refuses_what_the_library_refuses():
    """dist.StripPlan raises for exactly the plans whose coarsest level has fewer rows than strips, as the library does
    (levels >= 4 at window 3 and reach 0 included, where the old rule let 3 coarsest rows on 4 ranks through)."""
    from cuda_optical_flow_2_b200.dist import StripPlan

    n = 0
    for W, H, levels, win, world, reach in list(sweep_plans()) + [(64, 24, 4, 3, 4, 0), (64, 40, 5, 3, 3, 0), (640, 48, 4, 3, 7, 0)]:
        if (W >> (levels - 1)) < 1:
            continue
        rc, _ = query(W, H, levels, win, world, 0, reach, 0)
        try:
            plan = StripPlan(W, H, levels, win, world, reach)
        except ValueError:
            plan = None
        assert (plan is None) == (rc == OFB_ERR_INVALID), (W, H, levels, win, world, reach, rc)
        if plan is None:
            n += 1
        else:
            plan.validate()
    assert n > 300


@pytest.mark.parametrize("name", sorted(CASES))
def test_case_class(name):
    W, H, levels, win, world, reach, cls = CASES[name]
    t = Table(W, H, levels, win, world, reach)
    assert t.over_limit() is None
    cum = range(1, levels)
    if cls[0] == "image":
        assert t.fan_out(0) == cls[1] and all(t.fan_out(x) <= 2 for x in cum)
    else:
        assert max(t.fan_out(x) for x in cum) == cls[1]
        assert [rk for rk in range(world) if any(max(len(t.send[x][rk]), len(t.recv[x][rk])) > 2 for x in cum)] == cls[2]
    # a thin plan: some rank exchanges rows with a rank that is not adjacent
    assert any(abs(p - rk) > 1 for x in range(t.nx) for rk in range(world) for p, _, _ in t.send[x][rk])


@pytest.mark.parametrize("name", sorted(FB_CASES))
def test_checked_case_class(name):
    W, H, levels, win, world, reach, fb_reach, fans = FB_CASES[name]
    t = Table(W, H, levels, win, world, reach, fb_reach)
    assert t.over_limit() is None and {x: t.fan_out(x) for x in fans} == fans


@pytest.mark.parametrize("name", sorted(REFUSED))
def test_refused_case_class(name):
    """Over the limit, while rank 0's own exchanges fit."""
    W, H, levels, win, world, reach, fb_reach = REFUSED[name]
    t = Table(W, H, levels, win, world, reach, fb_reach)
    assert t.over_limit() is not None
    assert all(len(t.send[x][0]) <= PEER_MAX_DST and len(t.recv[x][0]) <= PEER_MAX_DST for x in range(t.nx))


@pytest.mark.parametrize("name", sorted(CASES))
def test_case_motion_stays_inside_reach(oracle, name):
    """The warp rule (support.requested_rows) on the oracle's cumulative flow of every pair, warp mode and flow_scale the
    GPU runs on this case asks for no row a rank does not hold: on the GPU a reach flag is a failure."""
    W, H, levels, win, world, reach, _ = CASES[name]
    t = Table(W, H, levels, win, world, reach)
    modes = {(m, s) for n, (_, m, s) in VARIANTS if n == name}
    for trial, (dx, dy) in enumerate(MOTION[reach]):
        prev, nxt = frames(oracle, W, H, 500 + trial, dx, dy)
        for mode, s in sorted(modes):
            _, cums = oracle.flow_pair(prev, nxt, levels, win, mode, oracle.SUMS_EXACT, s, want_cum=True)
            for rk in range(world):
                for k in range(levels - 1):
                    y0, y1, _, _, cy0, cy1, eb0, eb1 = t.rows[k][rk]
                    req = requested_rows(cums[k + 1], W >> k, H >> k, mode, y0, y1, win, s)
                    assert not reach_flag(req, eb0, eb1 - eb0, cy0, cy1 - cy0), (trial, mode, s, rk, k)


# ------------------------------------------------------------------------------------------------------------------ GPU
def make_ranks(ctx, W, H, levels, win, world, reach, mode=BIL, flow_scale=1.0, fb_reach=None):
    import torch

    from cuda_optical_flow_2_b200.dist import NativeStrips

    dev = torch.device("cuda", 0)
    ranks = []
    try:
        for rk in range(world):
            ranks.append(NativeStrips(ctx, W, H, levels, win, world, rk, dev, mode, flow_scale, reach, transport="local",
                                      fb_reach=fb_reach))
        NativeStrips.connect_local(ranks)
    except BaseException:
        close(ranks)
        raise
    return ranks


def close(ranks):
    import torch

    torch.cuda.synchronize()
    for ns in ranks:
        ns.close()


def device_pair(oracle, W, H, seed, dx, dy):
    from cuda_optical_flow_2_b200 import planar_to_device

    prev, nxt = frames(oracle, W, H, seed, dx, dy)
    return planar_to_device(prev[None]), planar_to_device(nxt[None])


def own_inputs(ranks, dp, dn):
    return [(dp[0, y0:y1], dn[0, y0:y1]) for y0, y1 in (ns.own_rows(0) for ns in ranks)]


def run_plain(ctx, ranks, inputs):
    """One plain pair, phase by phase on the current stream; returns its launches."""
    import torch

    from cuda_optical_flow_2_b200.dist import NativeStrips

    n0 = ctx.launch_count
    NativeStrips.run_local_sequenced(ranks, inputs, torch.cuda.current_stream().cuda_stream)
    return ctx.launch_count - n0


def assert_plain_equals_whole(ranks, whole, total, what, with_total=True):
    """No flag, and every rank's residual flow of every level (and the total flow) equal to its rows of the whole frame."""
    for ns in ranks:
        ns.check()
        for k in range(len(whole)):
            y0, y1 = ns.own_rows(k)
            assert_same_bits(ns.own_flow(k), whole[k][0, y0:y1], f"{what} rank {ns.rank} level {k}")
        if with_total:
            y0, y1 = ns.own_rows(0)
            assert_same_bits(ns.own_flow(0, total=True), total[0, y0:y1], f"{what} rank {ns.rank} total flow")


def whole_frame(ctx, dp, dn, W, levels, win, mode, flow_scale):
    import torch

    total = torch.empty((1, dp.shape[1], W, 2), dtype=torch.float32, device=dp.device)
    whole = ctx.flow_pairs_device(dp, dn, W, levels, win, warp_mode=mode, flow_scale=flow_scale, total_flow=total)
    torch.cuda.synchronize()
    return whole, total


@pytest.mark.gpu
@pytest.mark.parametrize("name,variant", VARIANTS, ids=[f"{n}-{v[0]}-{'bil' if v[1] == BIL else 'near'}-{v[2]:.3f}"
                                                         for n, v in VARIANTS])
def test_thin_strips_equal_whole_frame(ctx, oracle, name, variant):
    """Three pairs back to back (epochs, the done handshake) on every rank, each bit-identical to the whole frame at every
    level and in the total flow, with the launches of each pair what the restated table counts; then the last pair again
    with the separate copy / wait kernels (set_fused(False): same bits, the count of that form) and without the total flow
    (set_total(False): same residual flows, same count)."""
    from cuda_optical_flow_2_b200 import SOLVE_EXACT, SOLVE_FAST

    W, H, levels, win, world, reach, _ = CASES[name]
    kind, mode, s = variant
    t = Table(W, H, levels, win, world, reach)
    with solve(ctx, SOLVE_FAST if kind == "fast" else SOLVE_EXACT):
        ranks = make_ranks(ctx, W, H, levels, win, world, reach, mode, s)
        try:
            for trial, (dx, dy) in enumerate(MOTION[reach]):
                dp, dn = device_pair(oracle, W, H, 500 + trial, dx, dy)
                whole, total = whole_frame(ctx, dp, dn, W, levels, win, mode, s)
                n = run_plain(ctx, ranks, own_inputs(ranks, dp, dn))
                assert n == t.launches(), f"pair {trial}: {n} launches, the table counts {t.launches()}"
                assert_plain_equals_whole(ranks, whole, total, f"pair {trial}")
            for ns in ranks:
                ns.set_fused(False)
            n = run_plain(ctx, ranks, own_inputs(ranks, dp, dn))
            assert n == t.launches(fused=False), f"separate kernels: {n} launches, the table counts {t.launches(fused=False)}"
            assert_plain_equals_whole(ranks, whole, total, "separate kernels")
            for ns in ranks:
                ns.set_fused(True)
                ns.set_total(False)
            n = run_plain(ctx, ranks, own_inputs(ranks, dp, dn))
            assert n == t.launches(), f"without the total flow: {n} launches"
            assert_plain_equals_whole(ranks, whole, total, "without the total flow", with_total=False)
        finally:
            close(ranks)


@pytest.mark.gpu
@pytest.mark.parametrize("rpb", [1, 2, 3])
@pytest.mark.parametrize("name", ["cum3-320x52x3-5", "image4-320x240x3-5"])
def test_thin_strips_at_forced_row_splits(ctx, oracle, rows, name, rpb):
    """1, 2 and 3 rows per CTA: the rows a neighbour needs span every row block of a thin strip, so every CTA pushes
    (the fused push counter expects blocks x column strips of them).  Bit-identical, no flag, the table's launch count."""
    W, H, levels, win, world, reach, _ = CASES[name]
    t = Table(W, H, levels, win, world, reach)
    dp, dn = device_pair(oracle, W, H, 500, *MOTION[reach][0])
    whole, total = whole_frame(ctx, dp, dn, W, levels, win, BIL, 1.0)
    ranks = make_ranks(ctx, W, H, levels, win, world, reach)
    try:
        rows(rpb)
        n = run_plain(ctx, ranks, own_inputs(ranks, dp, dn))
        assert n == t.launches()
        assert_plain_equals_whole(ranks, whole, total, f"{rpb} rows per CTA")
    finally:
        close(ranks)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("name", sorted(FB_CASES))
def test_thin_checked_pairs_equal_whole_frame(ctx, oracle, name, fused):
    """Checked pairs whose check rows come from up to 4 ranks and whose backward cumulative flow fans out to 3: two pairs
    back to back, every output as the whole-frame ofb_flow_pairs_fb_device (assert_equals_whole), launches as counted."""
    import torch

    from cuda_optical_flow_2_b200.dist import NativeStrips

    W, H, levels, win, world, reach, fb_reach, _ = FB_CASES[name]
    t = Table(W, H, levels, win, world, reach, fb_reach)
    ranks = make_ranks(ctx, W, H, levels, win, world, reach, fb_reach=fb_reach)
    try:
        for ns in ranks:
            ns.set_fused(fused)
        for trial, (dx, dy) in enumerate(MOTION[reach][:2]):
            dp, dn = device_pair(oracle, W, H, 520 + trial, dx, dy)
            whole = ctx.flow_pairs_fb_device(dp, dn, W, levels, win, want_err2=True)
            torch.cuda.synchronize()
            n0 = ctx.launch_count
            NativeStrips.run_local_sequenced_fb(ranks, own_inputs(ranks, dp, dn), want_err2=True,
                                                stream=torch.cuda.current_stream().cuda_stream)
            n = ctx.launch_count - n0
            assert n == t.launches(fused, checked=True), f"pair {trial}: {n} launches, the table counts {t.launches(fused, True)}"
            assert_equals_whole(ranks, whole, True, f"pair {trial}")
    finally:
        close(ranks)


@pytest.mark.gpu
@pytest.mark.parametrize("checked", [False, True])
def test_thin_pair_replays_as_cuda_graph(ctx, oracle, checked):
    """A thin pair (image exchange to 4 ranks, copy and wait kernels for the cumulative flow of ranks 1 and 3; checked:
    check rows from 4 ranks too) captured as one CUDA graph, phase by phase; two replays on new frames written in place,
    each bit-identical to the whole frame."""
    import torch

    from cuda_optical_flow_2_b200.dist import NativeStrips

    W, H, levels, win, world, reach = 320, 52, 3, 9, 5, 16
    fb_reach = 16 if checked else None
    ranks = make_ranks(ctx, W, H, levels, win, world, reach, fb_reach=fb_reach)
    side = torch.cuda.Stream()
    try:
        ins = [ns.input_rows() for ns in ranks]

        def load(seed, dx, dy):
            dp, dn = device_pair(oracle, W, H, seed, dx, dy)
            for ns, (pin, nin) in zip(ranks, ins):
                y0, y1 = ns.own_rows(0)
                pin[:, :W].copy_(dp[0, y0:y1, :W])
                nin[:, :W].copy_(dn[0, y0:y1, :W])
            if checked:
                whole = ctx.flow_pairs_fb_device(dp, dn, W, levels, win, want_err2=True)
            else:
                whole = whole_frame(ctx, dp, dn, W, levels, win, BIL, 1.0)
            torch.cuda.synchronize()
            return whole

        def pair(stream):
            if checked:
                NativeStrips.run_local_sequenced_fb(ranks, ins, want_err2=True, stream=stream)
            else:
                NativeStrips.run_local_sequenced(ranks, ins, stream)

        load(530, 1.0, 1.0)
        pair(side.cuda_stream)  # warm-up pair, eager
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
            pair(torch.cuda.current_stream().cuda_stream)
        for trial, (dx, dy) in enumerate(MOTION[reach][:2]):
            whole = load(540 + trial, dx, dy)
            with torch.cuda.stream(side):
                g.replay()
            torch.cuda.synchronize()
            if checked:
                assert_equals_whole(ranks, whole, True, f"replay {trial}")
            else:
                assert_plain_equals_whole(ranks, *whole, f"replay {trial}")
    finally:
        close(ranks)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(REFUSED))
def test_over_limit_plans_refused_on_every_rank(ctx, name):
    """ofb_strips_create / _create_fb refuse a plan over the limits with OFB_ERR_UNSUPPORTED on EVERY rank -- rank 0,
    whose own exchanges fit, included -- naming the limit, and launch nothing.  No pair is ever enqueued here: a handle
    that a create returns is destroyed unconnected before the assertions."""
    import torch

    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    W, H, levels, win, world, reach, fb_reach = REFUSED[name]
    torch.cuda.synchronize()
    n0 = ctx.launch_count
    got = []
    for rk in range(world):
        h = C.c_void_p()
        if fb_reach is None:
            rc = lib.ofb_strips_create(ctx._h, W, H, levels, win, BIL, C.c_float(1.0), world, rk, reach, C.byref(h))
        else:
            rc = lib.ofb_strips_create_fb(ctx._h, W, H, levels, win, BIL, C.c_float(1.0), world, rk, reach, fb_reach, C.byref(h))
        msg = lib.ofb_last_error().decode() if rc else ""
        if h.value:
            lib.ofb_strips_destroy(h)
        got.append((rk, rc, msg))
    assert all(rc == OFB_ERR_UNSUPPORTED for _, rc, _ in got), got
    assert all("limit of 4" in msg and "fewer ranks" in msg for _, _, msg in got), got[0]
    torch.cuda.synchronize()
    assert ctx.launch_count == n0


@pytest.mark.gpu
@pytest.mark.parametrize("levels,world", [(5, 4), (4, 8)])
def test_thin_strips_across_processes(levels, world):
    """One process per GPU over CUDA IPC, each rank enqueuing its whole pair at once (scripts/run_strips.py under torchrun):
    1920x1080, window 9, image fan-out 3 on 4 ranks (5 levels) and 4 on 8 ranks (4 levels), with real cross-GPU waits; bit
    for bit the whole frame.  Skipped with fewer GPUs."""
    import json
    import socket
    import subprocess
    import sys

    import torch

    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "scripts", "run_strips.py"), "--w", "1920", "--h", "1080", "--levels",
           str(levels), "--win", "9", "--reps", "4", "--check"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    rec = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert rec["n_gpus"] == world and rec["bit_identical_to_whole_frame"] is True
