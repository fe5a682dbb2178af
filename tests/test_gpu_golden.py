"""The CUDA path against the reference-GPU golden vectors DIRECTLY (tests/golden/ref_gpu_b200.npz: outputs of the
unmodified reference's GPU functions on a B200, oracle/make_golden.py), without the oracle in between: single levels
at windows 5/9/15/19, the gpu::calc_opt_flow entry point (window 19), the pyramid, and the 3-level main.cu loop at the
reference's real defaults (window 19, warp as written) through the drop-in per-level entry point.

Bars: bit-identical wherever the reference's fp32 window sums are exact (every sum below 2^24); otherwise
|du|, |dv| <= 1e-4 px + 1e-5 |ref| (the reference rounds its sums, the CUDA path keeps them exact).  The loop compares the
pixels the reference's uninitialised `shifted` buffer does not taint (same mask as tests/test_oracle_pin.py)."""
import os

import numpy as np
import pytest

from oracle.make_golden import MULTI, SINGLE, WINDOWS, load
from support import TOL_ABS, TOL_REL, assert_values_equal

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "ref_gpu_b200.npz")


@pytest.fixture(scope="module")
def gold():
    return load(GOLDEN)


def compare(got, ref, exact, what, mask=None):
    if mask is None:
        mask = np.ones(ref.shape[:2], bool)
    g, r = got[mask], ref[mask]
    if exact:
        assert_values_equal(g, r, what)
        return
    both = np.isfinite(g) & np.isfinite(r)
    assert (np.isfinite(g) == np.isfinite(r)).mean() > 0.9999, what
    d = np.abs(g[both] - r[both])
    assert (d <= TOL_ABS + TOL_REL * np.abs(r[both])).all(), f"{what}: max |d| {d.max():.3e}"


@pytest.mark.parametrize("win", WINDOWS)
@pytest.mark.parametrize("case", SINGLE, ids=[c[0] for c in SINGLE])
def test_single_level_against_reference_gpu_golden(ctx, oracle, gold, case, win):
    import torch

    from cuda_optical_flow_2_b200 import planar_to_device

    name, w, h, dx, dy, cell, seed = case
    prev = oracle.make_frame(w, h, 0, 0, cell, seed)
    nxt = oracle.make_frame(w, h, dx, dy, cell, seed)
    flow = ctx.lk_level_device(planar_to_device(prev[None]), planar_to_device(nxt[None]), w, win, cum_in=None)
    torch.cuda.synchronize()
    exact = np.abs(gold[f"{name}_sums_w{win}"]).max() < 2 ** 24
    compare(flow.cpu().numpy()[0], gold[f"{name}_flow_w{win}"], exact, f"case {name} window {win}")


@pytest.mark.parametrize("case", SINGLE, ids=[c[0] for c in SINGLE])
def test_entry_point_against_reference_gpu_golden(ctx, oracle, gold, case):
    """gpu::calc_opt_flow(prev, next, w, h, pyr, level = maxLevel - 1, maxLevel) through the drop-in host entry point with
    its defaults (window 19)."""
    name, w, h, dx, dy, cell, seed = case
    prev = oracle.make_frame(w, h, 0, 0, cell, seed)
    nxt = oracle.make_frame(w, h, dx, dy, cell, seed)
    flows = [np.zeros((h, w, 2), np.float32)]
    ctx.calc_opt_flow(oracle.to_c3(prev), oracle.to_c3(nxt), w, h, flows, 0, 1)
    exact = np.abs(gold[f"{name}_sums_w19"]).max() < 2 ** 24
    compare(flows[0], gold[f"{name}_entry_flow"], exact, f"case {name} entry point")


def test_pyramid_and_main_loop_against_reference_gpu_golden(ctx, oracle, gold):
    """main.cu:250-262 at the reference's defaults: gpu::gauss_pyramid, then gpu::calc_opt_flow per level with window 19
    and the warp as written."""
    name, w, h, levels, dx, dy, cell, seed = MULTI
    prev = oracle.make_frame(w, h, 0, 0, cell, seed)
    nxt = oracle.make_frame(w, h, dx, dy, cell, seed)
    pp = [oracle.to_c3(prev)] + [np.zeros((h >> k, w >> k, 3), np.uint8) for k in range(1, levels)]
    pn = [oracle.to_c3(nxt)] + [np.zeros((h >> k, w >> k, 3), np.uint8) for k in range(1, levels)]
    ctx.gauss_pyramid(pp, w, h, levels)
    ctx.gauss_pyramid(pn, w, h, levels)
    for k in range(1, levels):
        assert np.array_equal(pp[k][:, :, 0], gold[f"{name}_pyr_prev_l{k}"]), f"prev pyramid level {k}"
        assert np.array_equal(pn[k][:, :, 0], gold[f"{name}_pyr_next_l{k}"]), f"next pyramid level {k}"
    flows = [np.zeros((h >> k, w >> k, 2), np.float32) for k in range(levels)]
    for k in range(levels - 1, -1, -1):
        ctx.calc_opt_flow(pp[k], pn[k], w >> k, h >> k, flows, k, levels)  # defaults: window 19, as written
    for k in range(levels - 1, -1, -1):
        ref = gold[f"{name}_loop_flow_l{k}"]
        wk, hk = w >> k, h >> k
        # pixels the reference's warp skipped hold uninitialised heap (OptFlowCPU.cpp:247); their influence reaches
        # win/2 + 1 pixels.  The global shift is the flow of pixel (0,0) of every coarser level (OptFlowCPU.cpp:260-261).
        u = sum(np.float32(1 << (m - k)) * gold[f"{name}_loop_flow_l{m}"][0, 0, 0] for m in range(levels - 1, k, -1))
        v = sum(np.float32(1 << (m - k)) * gold[f"{name}_loop_flow_l{m}"][0, 0, 1] for m in range(levels - 1, k, -1))
        jj, ii = np.meshgrid(np.arange(wk), np.arange(hk))
        nx = np.trunc(jj + np.float32(u)).astype(int) if k < levels - 1 else jj
        ny = np.trunc(ii + np.float32(v)).astype(int) if k < levels - 1 else ii
        skipped = (nx < 0) | (nx >= wk) | (ny < 0) | (ny >= hk)
        reach = 19 // 2 + 1
        tainted = np.zeros_like(skipped)
        for y, x in zip(*np.nonzero(skipped)):
            tainted[max(0, y - reach):y + reach + 1, max(0, x - reach):x + reach + 1] = True
        assert (~tainted).mean() > 0.8
        compare(flows[k], ref, False, f"main loop level {k}", mask=~tainted)


def _read_flo(path):
    with open(path, "rb") as f:
        tag = np.frombuffer(f.read(4), np.float32)[0]
        w, h = np.frombuffer(f.read(8), np.int32)
        assert tag == np.float32(202021.25)
        return np.frombuffer(f.read(), np.float32).reshape(h, w, 2)


@pytest.mark.parametrize("warp,win", [(2, 9), (0, 19)])
def test_cpp_driver_runs_the_drop_in_header(oracle, tmp_path, warp, win):
    """The C++ host driver (csrc/driver_main.cpp, the role of main.cu) is EXECUTED: it drives the frame loop through the
    `namespace gpu` wrappers of include/OptFlowGpuB200.hpp (gauss_pyramid, calc_opt_flow per level, pyramid swap), composes
    the total flow and writes it as .flo files, which must equal the oracle's composition for the same frames bit for bit."""
    import subprocess

    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "cuda_optical_flow_2_b200", "ofb_driver")
    assert os.path.exists(exe), "the driver binary is built by `make -C cuda_optical_flow_2_b200/csrc` / __graft_entry__.build()"
    w, h, levels, frames, step = 320, 240, 3, 2, 1.5
    prefix = str(tmp_path / "flow")
    r = subprocess.run([exe, "--w", str(w), "--h", str(h), "--levels", str(levels), "--frames", str(frames), "--win", str(win),
                        "--warp", str(warp), "--step", str(step), "--flo", prefix, "--arrows", "20"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("median composed flow") == frames
    for f in range(1, frames + 1):
        prev = oracle.make_frame(w, h, np.float32(step * (f - 1)), np.float32(0.5 * step * (f - 1)), 8, 1234)
        nxt = oracle.make_frame(w, h, np.float32(step * f), np.float32(0.5 * step * f), 8, 1234)
        _, cums = oracle.flow_pair(prev, nxt, levels, win, warp, oracle.SUMS_EXACT, 1.0, want_cum=True)
        got = _read_flo(f"{prefix}_{f:04d}.flo")
        ref = cums[0]
        same = (got == ref) | (np.isnan(got) & np.isnan(ref))
        assert same.all(), f"frame {f}: {(~same).sum()} of {same.size} values differ"
