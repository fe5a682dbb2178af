"""Generate tests/golden/ref_gpu_b200.npz by running the UNMODIFIED reference's GPU functions on a B200.

TEST INFRASTRUCTURE ONLY.  Run on a B200 with oracle/_ref/libofref.so built (`make -C oracle ref`):

    python oracle/make_golden.py <out.npz>

then copy the file to tests/golden/.  Inputs are the seeded synthetic frames of orc_make_frame, so
only the reference's OUTPUTS are stored.  Sizes are launch-valid for the reference's swapped
<<<block, grid>>> launches (SURVEY.md Q6): width and height multiples of 32 with
(w/32)*(h/32) <= 1024, at every level that is used.

The file keeps every output bit for bit in a compact form (as plain float32 arrays they take 2.8 MB):
derivatives as int16 (they are integers), window sums as their difference from the exact integer window
sums of those derivatives (zero wherever the reference's fp32 accumulation stayed exact), and single-level
flows as the XOR of their bits with a double-precision solve of those sums (zero wherever both round
alike).  Tests read it through load(), which returns the reference's arrays under their original names.
"""
from __future__ import annotations

import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import oracle as O  # noqa: E402

# (name, w, h, dx, dy, cell, seed)
SINGLE = [("a", 64, 64, 1.0, 0.5, 4, 1234), ("b", 96, 64, -0.75, 1.25, 8, 77), ("c", 128, 96, 2.0, -1.0, 2, 4242)]
WINDOWS = [5, 9, 15, 19]
MULTI = ("m", 256, 128, 3, 3.0, 1.5, 8, 99)  # name, w, h, levels, dx, dy, cell, seed


def main(out_path: str) -> None:
    g = {}
    for name, w, h, dx, dy, cell, seed in SINGLE:
        prev = O.make_frame(w, h, 0, 0, cell, seed)
        nxt = O.make_frame(w, h, dx, dy, cell, seed)
        pc3, nc3 = O.to_c3(prev), O.to_c3(nxt)
        ix = O.ref_gpu_conv(pc3, O.DX)
        iy = O.ref_gpu_conv(pc3, O.DY)
        it1 = O.ref_gpu_conv(pc3, O.DT)
        it2 = O.ref_gpu_conv(nc3, O.DT)
        it = O.ref_arr_sub(it2, it1)
        g[f"{name}_ix"], g[f"{name}_iy"], g[f"{name}_it1"], g[f"{name}_it2"] = ix, iy, it1, it2
        for win in WINDOWS:
            sums = [O.ref_gpu_srm(a, b, win, win) for a, b in ((ix, ix), (iy, iy), (ix, iy), (ix, it), (iy, it))]
            g[f"{name}_sums_w{win}"] = np.stack(sums)
            inv = O.ref_gpu_inverse(*sums)
            g[f"{name}_flow_w{win}"] = O.ref_gpu_lk_level_win(pc3, nc3, win)
            # the composed level is the same call sequence: store it once
            assert np.array_equal(inv.view(np.uint32), g[f"{name}_flow_w{win}"].view(np.uint32))
        # the entry point itself, single level (window hard-coded 19, OptFlowGpu.cu:1944-1945)
        flow = np.full((h, w, 2), -7.0, np.float32)
        pyr = (O._f32p * 1)(flow.ctypes.data_as(O._f32p))
        O.ref().ref_gpu_calc_opt_flow(pc3.ctypes.data_as(O._u8p), nc3.ctypes.data_as(O._u8p), w, h, pyr, 0, 1)
        g[f"{name}_entry_flow"] = flow
    # pyramid + the main.cu:256-262 loop through gpu::calc_opt_flow (warp as written, window 19)
    name, w, h, levels, dx, dy, cell, seed = MULTI
    prev = O.make_frame(w, h, 0, 0, cell, seed)
    nxt = O.make_frame(w, h, dx, dy, cell, seed)
    pp = O.ref_gpu_gauss_pyramid_c3(O.to_c3(prev), levels)
    pn = O.ref_gpu_gauss_pyramid_c3(O.to_c3(nxt), levels)
    for k in range(1, levels):
        g[f"{name}_pyr_prev_l{k}"] = pp[k][:, :, 0].copy()
        g[f"{name}_pyr_next_l{k}"] = pn[k][:, :, 0].copy()
        assert np.array_equal(pp[k][:, :, 0], pp[k][:, :, 1]) and np.array_equal(pp[k][:, :, 0], pp[k][:, :, 2])
    flows = [np.full((h >> k, w >> k, 2), -7.0, np.float32) for k in range(levels)]
    fptr = (O._f32p * levels)(*[f.ctypes.data_as(O._f32p) for f in flows])
    for k in range(levels - 1, -1, -1):
        O.ref().ref_gpu_calc_opt_flow(pp[k].ctypes.data_as(O._u8p), pn[k].ctypes.data_as(O._u8p), w >> k, h >> k, fptr, k,
                                      levels)
    for k in range(levels):
        g[f"{name}_loop_flow_l{k}"] = flows[k]
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    np.savez_compressed(out_path, **pack(g))
    print(f"wrote {out_path}: {len(g)} arrays, {sum(v.nbytes for v in g.values())} bytes raw")


# ------------------------------------------------------------------ storage form (see the module docstring)
DERIVATIVES = ("ix", "iy", "it1", "it2")
ENTRY_WIN = 19  # the window gpu::calc_opt_flow hard-codes


def _exact_sums(d: dict, win: int) -> np.ndarray:
    """The five window sums (xx, yy, xy, xt, yt) of int64 derivatives, exact, zero outside the image."""
    ix, iy, it = d["ix"], d["iy"], d["it2"] - d["it1"]
    h, w = ix.shape
    r = win // 2
    out = []
    for a in (ix * ix, iy * iy, ix * iy, ix * it, iy * it):
        c = np.zeros((h + 2 * r + 1, w + 2 * r + 1), np.int64)
        c[1 + r:1 + r + h, 1 + r:1 + r + w] = a
        c = c.cumsum(0).cumsum(1)
        out.append(c[win:, win:] - c[:h, win:] - c[win:, :w] + c[:h, :w])
    return np.stack(out)


def _solve_bits(sums: np.ndarray) -> np.ndarray:
    """uint32 bits of the 2x2 solve of float32 sums in double precision (a predictor: it need not match exactly)."""
    a, d, b, xt, yt = sums.astype(np.float64)
    with np.errstate(all="ignore"):
        p = 1.0 / (a * d - b * b)
        flow = np.stack([b * p * yt - d * p * xt, b * p * xt - a * p * yt], axis=-1).astype(np.float32)
    return flow.view(np.uint32)


def unpack(z) -> dict:
    """Stored form (a mapping of arrays) -> the reference's arrays under their original names."""
    g = {}
    for name, *_ in SINGLE:
        d = {k: z[f"{name}_{k}"].astype(np.int64) for k in DERIVATIVES}
        g.update({f"{name}_{k}": v.astype(np.float32) for k, v in d.items()})
        for win in WINDOWS:
            sums = (_exact_sums(d, win) + z[f"{name}_sums_w{win}_minus_exact"]).astype(np.float32)
            g[f"{name}_sums_w{win}"] = sums
            g[f"{name}_flow_w{win}"] = (z[f"{name}_flow_w{win}_xor_solve"] ^ _solve_bits(sums)).view(np.float32)
        g[f"{name}_entry_flow"] = (z[f"{name}_entry_flow_xor_solve"] ^ _solve_bits(g[f"{name}_sums_w{ENTRY_WIN}"])).view(np.float32)
    g.update({k: z[k] for k in z.keys() if k.startswith(MULTI[0] + "_")})
    return g


def pack(g: dict) -> dict:
    """The reference's arrays -> stored form; checks that unpack() gives every bit back."""
    z = {}
    for name, *_ in SINGLE:
        d = {k: g[f"{name}_{k}"].astype(np.int64) for k in DERIVATIVES}
        z.update({f"{name}_{k}": v.astype(np.int16) for k, v in d.items()})
        for win in WINDOWS:
            sums = g[f"{name}_sums_w{win}"]
            z[f"{name}_sums_w{win}_minus_exact"] = (sums.astype(np.int64) - _exact_sums(d, win)).astype(np.int32)
            z[f"{name}_flow_w{win}_xor_solve"] = g[f"{name}_flow_w{win}"].view(np.uint32) ^ _solve_bits(sums)
        z[f"{name}_entry_flow_xor_solve"] = g[f"{name}_entry_flow"].view(np.uint32) ^ _solve_bits(g[f"{name}_sums_w{ENTRY_WIN}"])
    z.update({k: v for k, v in g.items() if k.startswith(MULTI[0] + "_")})
    back = unpack(z)
    assert back.keys() == g.keys(), "stored form does not cover every array"
    for k, v in g.items():
        assert back[k].dtype == v.dtype and np.array_equal(back[k].view(np.uint8), v.view(np.uint8)), f"{k} does not round-trip"
    return z


def load(path: str) -> dict:
    with np.load(path) as z:
        return unpack(z)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "gpurun_out/ref_gpu_b200.npz")
