"""The forward-backward check on host batches (ofb_flow_pairs_fb_host) and on the frame stream
(ofb_stream_push_bgr_host_fb).

Both run the device-side body of ofb_flow_pairs_fb_device, so every output must be bit-identical to that call on the same
frames: for host batches the planar frames uploaded with planar_to_device, for the stream its preprocessed frames (the
oracle's grayscale, and with the bilateral filter that gray image through Context.bilateral_planar_device).  The status is
also checked against the C restatement of the check (tests/fb_oracle.c, compiled here into a temporary directory) on the
returned totals.  The refactored upload of ofb_flow_pairs_host / _ex is checked for unchanged bytes and an unchanged
number of launches, counted from the sub-batch plan.
"""
import contextlib
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from support import ASW, BIL, NEAR, S815, assert_same_bytes, bgr_sequence, fbo, pyramid_launches, solve  # noqa: F401 (fbo: a fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------ launches counted from the plan
def n_sub_batches(n, lanes=3):
    """Sub-batches of the host pipeline (csrc/ofb_api.cu host_pipeline, default lanes)."""
    sub = min(max(n // (8 * lanes), 1), 8)
    return -(-n // sub)


def host_launches(n, levels, channels, host_threads, fb):
    """Kernel launches of one batched host call: per sub-batch the device-side channel extraction (3-channel input without
    host threads), the pyramid build, the level loop (twice with the check) and the check."""
    per = (2 if channels == 3 and host_threads == 0 else 0) + pyramid_launches(levels) + levels * (2 if fb else 1) + (1 if fb else 0)
    return n_sub_batches(n) * per


def test_launch_plan_arithmetic():
    assert [n_sub_batches(n) for n in (1, 7, 24, 48, 53, 100, 192, 203)] == [1, 7, 24, 24, 27, 25, 24, 26]
    assert [pyramid_launches(L) for L in (1, 2, 3, 4, 5)] == [0, 1, 1, 2, 2]


def test_null_context_and_stream_are_rejected():
    from cuda_optical_flow_2_b200 import _lib

    lib = _lib.load()
    p = _lib.OfbParams(64, 64, 2, 9, BIL, 1.0, 1)
    assert lib.ofb_flow_pairs_fb_host(None, C.byref(p), None, None, 1, 0.01, 0.5, None, None, None, None) == _lib.OFB_ERR_INVALID
    assert b"NULL" in lib.ofb_last_error()
    assert lib.ofb_stream_push_bgr_host_fb(None, None, 0.01, 0.5, None, None, None, None, None, None) == _lib.OFB_ERR_INVALID
    assert b"NULL" in lib.ofb_last_error()


# ------------------------------------------------------------------------------------ GPU helpers
class Pinned:
    """Pinned host copies of numpy arrays (ofb_host_alloc), freed by the fixture."""

    def __init__(self):
        from cuda_optical_flow_2_b200 import _lib

        self._lib, self.lib, self.ptrs = _lib, _lib.load(), []

    def copy(self, a):
        p = C.c_void_p()
        self._lib.check(self.lib.ofb_host_alloc(C.byref(p), max(a.nbytes, 1)))
        self.ptrs.append(p)
        out = np.frombuffer((C.c_uint8 * a.nbytes).from_address(p.value), dtype=a.dtype).reshape(a.shape)
        out[...] = a
        return out

    def free(self):
        for p in self.ptrs:
            self.lib.ofb_host_free(p)
        self.ptrs = []


@pytest.fixture
def pinned():
    pin = Pinned()
    yield pin
    pin.free()


@contextlib.contextmanager
def settings(ctx, kind, host_threads=0):
    """The shared context in the "exact" or "fast" solve and with `host_threads` host threads, both restored afterwards."""
    from cuda_optical_flow_2_b200 import SOLVE_EXACT, SOLVE_FAST

    with solve(ctx, SOLVE_FAST if kind == "fast" else SOLVE_EXACT):
        ctx.host_threads = host_threads
        try:
            yield ctx
        finally:
            ctx.host_threads = 0


def gray_pairs(oracle, w, h, n, seed):
    prevs = np.stack([oracle.make_frame(w, h, 0, 0, 4, seed + i) for i in range(n)])
    nexts = np.stack([oracle.make_frame(w, h, 1.25 + 0.5 * (i % 5), -0.75 + 0.25 * (i % 3), 4, seed + i) for i in range(n)])
    return prevs, nexts


def with_channels(gray, rng):
    """(n, h, w) gray -> (n, h, w, 3) with channel 0 the gray image and other noise in channels 1 and 2 (never read)."""
    c3 = rng.integers(0, 256, size=gray.shape + (3,), dtype=np.uint8)
    c3[..., 0] = gray
    return c3


# ------------------------------------------------------------------------------------ GPU: host batches
HOST_CASES = [
    # channels, host threads, pinned, n, w, h, levels, win, warp, solve, want_bwd, want_err2, flow_scale
    (1, 0, False, 1, 96, 64, 3, 9, BIL, "exact", True, True, 1.0),  # one sub-batch
    (1, 0, True, 7, 96, 64, 4, 3, NEAR, "fast", True, False, 1.0),  # seven sub-batches of one pair over three lanes
    (3, 0, False, 53, 96, 64, 2, 19, ASW, "exact", False, True, 1.0),  # sub-batches of two, a ragged last one
    (3, 4, True, 53, 97, 61, 3, 9, BIL, "fast", True, True, S815),  # odd sizes, host extraction
    (3, 4, False, 7, 96, 64, 1, 9, BIL, "exact", True, True, 1.0),  # one level: the total is the residual flow
    (1, 0, True, 203, 64, 48, 2, 5, NEAR, "exact", False, False, 1.0),  # sub-batches of eight, ragged
    (1, 0, False, 7, 133, 71, 4, 19, BIL, "exact", True, True, S815),
    (1, 0, True, 3, 1920, 1080, 3, 9, BIL, "fast", True, False, 1.0),
    (3, 4, True, 2, 1920, 1080, 4, 19, ASW, "exact", False, True, 1.0),
]


def _host_id(c):
    return f"c{c[0]}-t{c[1]}-{'pinned' if c[2] else 'pageable'}-n{c[3]}-{c[4]}x{c[5]}-L{c[6]}-w{c[7]}-m{c[8]}-{c[9]}" \
           f"{'-bwd' if c[10] else ''}{'-err2' if c[11] else ''}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", HOST_CASES, ids=[_host_id(c) for c in HOST_CASES])
def test_fb_host_equals_fb_device(ctx, oracle, fbo, pinned, case):
    from cuda_optical_flow_2_b200 import planar_to_device

    channels, threads, pin, n, w, h, levels, win, mode, kind, want_bwd, want_err2, s = case
    prevs, nexts = gray_pairs(oracle, w, h, n, seed=40 + n)
    rng = np.random.default_rng(n)
    hp, hn = (prevs, nexts) if channels == 1 else (with_channels(prevs, rng), with_channels(nexts, rng))
    if pin:
        hp, hn = pinned.copy(hp), pinned.copy(hn)
    with settings(ctx, kind, threads):
        before = ctx.launch_count
        fwd, bwd, st, e2 = ctx.flow_pairs_fb_host(hp, hn, levels, win, warp_mode=mode, flow_scale=s, want_bwd=want_bwd,
                                                  want_err2=want_err2)
        launches = ctx.launch_count - before
        ref = ctx.flow_pairs_fb_device(planar_to_device(prevs), planar_to_device(nexts), w, levels, win, warp_mode=mode,
                                       flow_scale=s, want_err2=True)
    rf, rb, rst, re2 = (t.cpu().numpy() for t in ref)
    assert launches == host_launches(n, levels, channels, threads, fb=True)
    assert_same_bytes(fwd, rf, "forward total")
    assert_same_bytes(st, rst, "status")
    assert (bwd is not None) == want_bwd and (e2 is not None) == want_err2
    if want_bwd:
        assert_same_bytes(bwd, rb, "backward total")
        ost, oe2 = fbo.fb_check(fwd, bwd, s)
        assert_same_bytes(st, ost, "status against orc_fb_check")
        if want_err2:
            assert_same_bytes(e2, oe2, "err2 against orc_fb_check")
    if want_err2:
        assert_same_bytes(e2, re2, "err2")


EX_CASES = [(1, 0, 53, 96, 64, 3), (3, 0, 7, 160, 120, 4), (3, 4, 24, 97, 61, 2), (1, 0, 1, 96, 64, 1), (3, 4, 3, 64, 48, 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("channels,threads,n,w,h,levels", EX_CASES)
def test_host_ex_bytes_and_launches_unchanged(ctx, oracle, channels, threads, n, w, h, levels):
    """ofb_flow_pairs_host / _ex after the upload moved into the shared pipeline: the same bytes as
    ofb_flow_pairs_device on the same frames, and the launches the sub-batch plan predicts."""
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    win = 9
    prevs, nexts = gray_pairs(oracle, w, h, n, seed=700 + n)
    rng = np.random.default_rng(n + 1)
    hp, hn = (prevs, nexts) if channels == 1 else (with_channels(prevs, rng), with_channels(nexts, rng))
    with settings(ctx, "exact", threads):
        c0 = ctx.launch_count
        total = ctx.total_flow_pairs_host(hp, hn, levels, win)
        c1 = ctx.launch_count
        flows = ctx.flow_pairs_host(hp, hn, levels, win)
        c2 = ctx.launch_count
        ref_total = torch.empty((n, h, w, 2), dtype=torch.float32, device="cuda")
        ref = ctx.flow_pairs_device(planar_to_device(prevs), planar_to_device(nexts), w, levels, win, total_flow=ref_total)
    expect = host_launches(n, levels, channels, threads, fb=False)
    assert (c1 - c0, c2 - c1) == (expect, expect)
    for k in range(levels):
        assert_same_bytes(flows[k], ref[k].cpu().numpy(), f"level {k}")
    # (one level: the host call downloads the residual flow as the total, the kernel has nothing to compose)
    assert_same_bytes(total, (ref_total if levels > 1 else ref[0]).cpu().numpy(), "total flow")


@pytest.mark.gpu
def test_fb_host_profile_records(ctx, oracle):
    from cuda_optical_flow_2_b200 import PROFILE_FB_CHECK

    n = 7
    prevs, nexts = gray_pairs(oracle, 96, 64, n, seed=3)
    ctx.profile_enable(True)
    try:
        ctx.flow_pairs_fb_host(prevs, nexts, 3, 9)
        ms, recs = ctx.profile_read(PROFILE_FB_CHECK)
    finally:
        ctx.profile_enable(False)
    assert recs == n_sub_batches(n) and ms > 0


@pytest.mark.gpu
def test_fb_host_bad_arguments_enqueue_nothing(ctx):
    from cuda_optical_flow_2_b200 import OfbError, _lib

    lib = _lib.load()
    n, w, h = 2, 64, 48
    frames = np.zeros((n, h, w), np.uint8)
    fwd = np.zeros((n, h, w, 2), np.float32)
    st = np.zeros((n, h, w), np.uint8)
    u8, f32 = lambda a: a.ctypes.data_as(_lib.u8p), lambda a: a.ctypes.data_as(_lib.f32p)

    def call(status=st, scale=1.0, alpha=0.01, channels=1, fw=fwd):
        p = _lib.OfbParams(w, h, 2, 9, BIL, scale, n)
        return lib.ofb_flow_pairs_fb_host(ctx._h, C.byref(p), u8(frames), u8(frames), channels, alpha, 0.5,
                                          f32(fw) if fw is not None else None, None,
                                          u8(status) if status is not None else None, None)

    before = ctx.launch_count
    inv = _lib.OFB_ERR_INVALID
    assert call(status=None) == inv
    assert call(fw=None) == inv
    assert call(scale=0.0) == inv and b"flow_scale" in lib.ofb_last_error()
    assert call(scale=-1.0) == inv
    assert call(alpha=-0.01) == inv and b"alpha" in lib.ofb_last_error()
    assert call(channels=2) == inv
    assert ctx.launch_count == before
    with pytest.raises(OfbError, match="beta"):
        ctx.flow_pairs_fb_host(frames, frames, 2, 9, beta=-1.0)
    assert ctx.launch_count == before
    assert call() == _lib.OFB_OK


# ------------------------------------------------------------------------------------ GPU: the frame stream
def preprocessed(ctx, oracle, frame, bil):
    """The stream's level 0 of a frame as a (1, h, pitch) device tensor: the oracle's grayscale, then optionally the
    bilateral filter on the device."""
    from cuda_optical_flow_2_b200 import planar_to_device

    h, w, _ = frame.shape
    g = planar_to_device(np.ascontiguousarray(oracle.grayscale_c3(frame)[:, :, 0])[None])
    return ctx.bilateral_planar_device(g[0], w, bil, 2.0, 10.0)[None] if bil else g


STREAM_CASES = [
    # w, h, levels, win, warp, bilateral window, solve, flow_scale
    (96, 64, 1, 9, BIL, 0, "exact", 1.0),
    (101, 67, 2, 5, NEAR, 5, "fast", 1.0),
    (133, 71, 3, 9, BIL, 0, "fast", S815),
    (160, 120, 4, 19, ASW, 5, "exact", 1.0),
    (203, 117, 3, 9, BIL, 5, "exact", S815),
]


@pytest.mark.gpu
@pytest.mark.parametrize("w,h,levels,win,mode,bil,kind,s", STREAM_CASES)
def test_stream_fb_equals_fb_device(ctx, oracle, fbo, w, h, levels, win, mode, bil, kind, s):
    """Every push after the first against ofb_flow_pairs_fb_device on the previous and current preprocessed frames, and
    the forward outputs against a second stream's plain push."""
    frames = bgr_sequence(oracle, w, h)
    with settings(ctx, kind):
        fb = ctx.open_stream(w, h, levels, win, warp_mode=mode, flow_scale=s, bil_win=bil)
        plain = ctx.open_stream(w, h, levels, win, warp_mode=mode, flow_scale=s, bil_win=bil)
        try:
            assert fb.push_fb(frames[0]) is None and plain.push(frames[0]) is None
            prev = preprocessed(ctx, oracle, frames[0], bil)
            for t in range(1, len(frames)):
                got = fb.push_fb(frames[t], want_levels=True, want_bwd=True, want_err2=True)
                flows, total = plain.push(frames[t], want_total=True)
                cur = preprocessed(ctx, oracle, frames[t], bil)
                rf, rb, rst, re2 = (x[0].cpu().numpy() for x in ctx.flow_pairs_fb_device(prev, cur, w, levels, win, warp_mode=mode,
                                                                                         flow_scale=s, want_err2=True))
                assert_same_bytes(got["fwd_total"], rf, f"push {t} forward total")
                assert_same_bytes(got["bwd_total"], rb, f"push {t} backward total")
                assert_same_bytes(got["status"], rst, f"push {t} status")
                assert_same_bytes(got["err2"], re2, f"push {t} err2")
                assert_same_bytes(got["status"], fbo.fb_check(got["fwd_total"], got["bwd_total"], s)[0], f"push {t} orc_fb_check")
                assert_same_bytes(got["fwd_total"], total, f"push {t} forward total against push")
                for k in range(levels):
                    assert_same_bytes(got["levels"][k], flows[k], f"push {t} level {k} against push")
                prev = cur
        finally:
            fb.close()
            plain.close()


@pytest.mark.gpu
def test_stream_mixed_pushes(ctx, oracle):
    """push and push_fb alternating on one stream give what two separate streams give; the plain push launches what its
    plan says."""
    w, h, levels, win, bil = 150, 98, 3, 9, 5
    frames = bgr_sequence(oracle, w, h, seed=9) + bgr_sequence(oracle, w, h, seed=10)[1:3]
    mixed, only_plain, only_fb = (ctx.open_stream(w, h, levels, win, bil_win=bil) for _ in range(3))
    try:
        for t, f in enumerate(frames):
            a = only_plain.push(f, want_total=True)
            b = only_fb.push_fb(f, want_levels=True, want_bwd=True, want_err2=True)
            if t % 2:
                c0 = ctx.launch_count
                m = mixed.push(f, want_total=True)
                # grayscale, bilateral filter (range table + filter), pyramid, levels
                assert ctx.launch_count - c0 == 1 + 2 + pyramid_launches(levels) + levels
                if a is None:
                    assert m is None
                    continue
                for k in range(levels):
                    assert_same_bytes(m[0][k], a[0][k], f"frame {t} level {k}")
                assert_same_bytes(m[1], a[1], f"frame {t} total")
            else:
                m = mixed.push_fb(f, want_levels=True, want_bwd=True, want_err2=True)
                if b is None:
                    assert m is None
                    continue
                for key in ("fwd_total", "bwd_total", "status", "err2"):
                    assert_same_bytes(m[key], b[key], f"frame {t} {key}")
                for k in range(levels):
                    assert_same_bytes(m["levels"][k], b["levels"][k], f"frame {t} level {k}")
    finally:
        for s in (mixed, only_plain, only_fb):
            s.close()


@pytest.mark.gpu
def test_stream_first_push_writes_nothing_and_rejected_calls_keep_the_sequence(ctx, oracle):
    from cuda_optical_flow_2_b200 import OfbError, _lib

    lib = _lib.load()
    w, h, levels = 96, 64, 2
    frames = bgr_sequence(oracle, w, h)
    st = ctx.open_stream(w, h, levels, 9)
    unscaled = ctx.open_stream(w, h, levels, 9, flow_scale=0.0)
    try:
        with pytest.raises(OfbError, match="alpha"):
            st.push_fb(frames[0], alpha=-1.0)
        with pytest.raises(OfbError, match="flow_scale"):
            unscaled.push_fb(frames[0])
        fwd = np.full((h, w, 2), 7.0, np.float32)
        bwd, err2 = fwd.copy(), np.full((h, w), 7.0, np.float32)
        status = np.full((h, w), 0xAB, np.uint8)
        lv = [np.full((h >> k, w >> k, 2), 7.0, np.float32) for k in range(levels)]
        ptrs = (_lib.f32p * levels)(*[a.ctypes.data_as(_lib.f32p) for a in lv])
        f32, u8 = lambda a: a.ctypes.data_as(_lib.f32p), lambda a: a.ctypes.data_as(_lib.u8p)
        assert lib.ofb_stream_push_bgr_host_fb(st._h, u8(frames[0]), 0.01, 0.5, ptrs, f32(fwd), None, None, None,
                                               None) == _lib.OFB_ERR_INVALID  # NULL status: rejected
        has = C.c_int(5)
        assert lib.ofb_stream_push_bgr_host_fb(st._h, u8(frames[0]), 0.01, 0.5, ptrs, f32(fwd), f32(bwd), u8(status), f32(err2),
                                               C.byref(has)) == _lib.OFB_OK
        assert has.value == 0  # the rejected calls did not advance the sequence: this was its first frame
        assert (fwd == 7.0).all() and (bwd == 7.0).all() and (err2 == 7.0).all() and (status == 0xAB).all()
        assert all((a == 7.0).all() for a in lv)
        assert st.push_fb(frames[1]) is not None
    finally:
        st.close()
        unscaled.close()


SERIAL_SCRIPT = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
from cuda_optical_flow_2_b200 import Context
d = np.load(sys.argv[2])
frames, (w, h, levels, win, bil) = d["frames"], d["cfg"].tolist()
out = {}
with Context(0) as ctx:
    st = ctx.open_stream(w, h, levels, win, bil_win=bil)
    for t, f in enumerate(frames):
        r = st.push_fb(f, want_levels=True, want_bwd=True, want_err2=True)
        assert (r is None) == (t == 0)
        if r is not None:
            for key in ("fwd_total", "bwd_total", "status", "err2"):
                out[f"{key}_{t}"] = r[key]
            for k, a in enumerate(r["levels"]):
                out[f"level{k}_{t}"] = a
    st.close()
np.savez(sys.argv[3], **out)
"""


@pytest.mark.gpu
def test_stream_serial_override_gives_the_same_bytes(oracle, tmp_path):
    """OFB_FB_SERIAL=1 runs the backward level loop after the forward one on the context stream instead of beside it on
    the stream's second CUDA stream: byte-identical results.  In subprocesses: the library reads the override once."""
    w, h, levels, win, bil = 203, 117, 3, 9, 5
    inp = tmp_path / "in.npz"
    np.savez(inp, frames=np.stack(bgr_sequence(oracle, w, h, seed=23)), cfg=np.array([w, h, levels, win, bil]))
    res = {}
    for serial in (False, True):
        env = {k: v for k, v in os.environ.items() if k != "OFB_FB_SERIAL"}
        if serial:
            env["OFB_FB_SERIAL"] = "1"
        out = tmp_path / f"out_{int(serial)}.npz"
        r = subprocess.run([sys.executable, "-c", SERIAL_SCRIPT, ROOT, str(inp), str(out)], env=env, capture_output=True,
                           text=True, timeout=600)
        assert r.returncode == 0, r.stderr
        res[serial] = np.load(out)
    assert sorted(res[False].files) == sorted(res[True].files) and len(res[False].files) == 5 * (4 + levels)
    for key in res[False].files:
        assert_same_bytes(res[True][key], res[False][key], key)
