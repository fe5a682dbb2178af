"""Host-side mirror of the reference's `namespace gpu` interface for the pyramidal LK path.

Function names, argument order and meaning follow OptFlowGpu.cuh (reference): `gauss_pyramid` (:21),
`calc_opt_flow` (:33), `conv_3ch_1ch_tiled_uchar_float` (:17), `srm_1ch_float` (:25),
`inverse_matrix_float` (:31).  Host images are numpy u8 arrays in the reference layout
(h, w, 3 interleaved channels); flow is float32 (h, w, 2).  Everything computes on the GPU through
the C ABI in include/ofb200.h -- there is no CPU path here.

The device-resident entry points (`flow_pairs_device`, `flow_pairs_fb_device`, `fb_check_device`, `lk_level_device`,
`pyr_down_device`) take
torch CUDA tensors only as owners of device memory; torch does none of the arithmetic.  The forward-backward check also
runs on host batches (`flow_pairs_fb_host`) and on the frame stream (`FrameStream.push_fb`).  `track_points_device`
follows a list of sub-pixel points through the pyramids (the KLT tracker), and `detect_corners_device` finds points for it
to start from (Shi-Tomasi corners on the tracker's own texture measure).
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

from . import _lib as L
from ._lib import SOLVE_EXACT, SOLVE_FAST, WARP_AS_WRITTEN, WARP_BILINEAR, WARP_NEAREST, OfbError, OfbParams  # noqa: F401

REFERENCE_WINDOW = 19  # OptFlowGpu.cu:1944-1945


def _u8(a: np.ndarray) -> np.ndarray:
    if a.dtype != np.uint8 or not a.flags["C_CONTIGUOUS"]:
        raise TypeError("expected a C-contiguous uint8 array")
    return a


def _f32(a: np.ndarray) -> np.ndarray:
    if a.dtype != np.float32 or not a.flags["C_CONTIGUOUS"]:
        raise TypeError("expected a C-contiguous float32 array")
    return a


def _ptrs(arrs: Sequence[np.ndarray], t):
    return (t * len(arrs))(*[a.ctypes.data_as(t) for a in arrs])


def _optp(a: Optional[np.ndarray], t):
    return a.ctypes.data_as(t) if a is not None else None


def align_up(v: int, a: int) -> int:
    return (v + a - 1) // a * a


def _batch_shape(prev: np.ndarray, next: np.ndarray) -> tuple[int, int, int, int]:
    """(channels, n, h, w) of a host batch: (n, h, w) planar gray or (n, h, w, 3) reference layout."""
    if prev.ndim == 4:
        if prev.shape[3] != 3:
            raise ValueError("4-d input must be (n, h, w, 3)")
        channels, (n, h, w) = 3, prev.shape[:3]
    elif prev.ndim == 3:
        channels, (n, h, w) = 1, prev.shape
    else:
        raise ValueError("prev must be (n,h,w) or (n,h,w,3)")
    if next.shape != prev.shape:
        raise ValueError("prev and next differ in shape")
    return channels, n, h, w


class Context:
    """One per GPU (ofb_ctx): owns the device workspace reused across calls."""

    def __init__(self, device: int = 0):
        self._lib = L.load()
        h = C.c_void_p()
        L.check(self._lib.ofb_ctx_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.ofb_ctx_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def sm_count(self) -> int:
        v = C.c_int()
        L.check(self._lib.ofb_ctx_sm_count(self._h, C.byref(v)))
        return v.value

    @property
    def launch_count(self) -> int:
        v = C.c_ulonglong()
        L.check(self._lib.ofb_ctx_launch_count(self._h, C.byref(v)))
        return v.value

    @property
    def solve(self) -> int:
        """SOLVE_EXACT (default; the reference's double-precision operation order, bit-identical flow) or SOLVE_FAST
        (exact 64-bit integer determinant and numerators, one float reciprocal; |d| <= 1e-4 px + 1e-5 |ref| per level)."""
        v = C.c_int()
        L.check(self._lib.ofb_ctx_get_solve(self._h, C.byref(v)))
        return v.value

    @solve.setter
    def solve(self, mode: int) -> None:
        L.check(self._lib.ofb_ctx_set_solve(self._h, int(mode)))

    @property
    def host_threads(self) -> int:
        """Host threads that extract channel 0 of 3-channel host images in `flow_pairs_host` (0: the device does it
        after uploading all three channels)."""
        v = C.c_int(0)
        L.check(self._lib.ofb_ctx_get_host_threads(self._h, C.byref(v)))
        return v.value

    @host_threads.setter
    def host_threads(self, n: int) -> None:
        L.check(self._lib.ofb_ctx_set_host_threads(self._h, int(n)))

    def reserve_pairs(self, w: int, h: int, levels: int, win: int, n_pairs: int) -> None:
        """Size the context workspace for flow_pairs_device calls of this shape now (a later growth would invalidate
        CUDA graphs captured from earlier calls)."""
        p = OfbParams(w, h, levels, win, WARP_BILINEAR, 1.0, n_pairs)
        L.check(self._lib.ofb_ctx_reserve_pairs(self._h, C.byref(p)))

    def reserve_pairs_fb(self, w: int, h: int, levels: int, win: int, n_pairs: int) -> None:
        """As reserve_pairs, for flow_pairs_fb_device calls of this shape."""
        p = OfbParams(w, h, levels, win, WARP_BILINEAR, 1.0, n_pairs)
        L.check(self._lib.ofb_ctx_reserve_pairs_fb(self._h, C.byref(p)))

    def profile_enable(self, on: bool = True) -> None:
        """CUDA-event timing around each fused-LK launch (tag = level), the pyramid build, the forward-backward check and
        the point tracker's kernel and the corner detector's kernels."""
        L.check(self._lib.ofb_ctx_profile_enable(self._h, 1 if on else 0))

    def profile_read(self, tag: int) -> tuple[float, int]:
        """(summed milliseconds, number of records) for a tag: a pyramid level, PROFILE_PYRAMID, PROFILE_FB_CHECK,
        PROFILE_TRACK or PROFILE_CORNERS."""
        ms, n = C.c_double(), C.c_ulonglong()
        L.check(self._lib.ofb_ctx_profile_read(self._h, int(tag), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    # ---------------------------------------------------------------- reference-named host API
    def gauss_pyramid(self, pyramid: Sequence[np.ndarray], w: int, h: int, levels: int) -> None:
        """gpu::gauss_pyramid (OptFlowGpu.cu:1262): fills pyramid[1..levels-1] from pyramid[0] in place.
        pyramid[k] is a (h>>k, w>>k, 3) uint8 array."""
        for k in range(levels):
            if pyramid[k].shape != (h >> k, w >> k, 3):
                raise ValueError(f"pyramid[{k}] has shape {pyramid[k].shape}, expected {(h >> k, w >> k, 3)}")
        arrs = [_u8(p) for p in pyramid[:levels]]
        L.check(self._lib.ofb_gauss_pyramid_host_u8c3(self._h, _ptrs(arrs, L.u8p), w, h, levels))

    def calc_opt_flow(self, prev: np.ndarray, next: np.ndarray, w: int, h: int, optFlowPyramid: Sequence[np.ndarray],
                      level: int, maxLevel: int, win: int = REFERENCE_WINDOW, warp_mode: int = WARP_AS_WRITTEN,
                      flow_scale: float = 1.0) -> None:
        """gpu::calc_opt_flow (OptFlowGpu.cu:1909): one level; reads optFlowPyramid[k > level], writes
        optFlowPyramid[level] in place.  Defaults reproduce the reference (window 19, its warp as written)."""
        if prev.shape != (h, w, 3) or next.shape != (h, w, 3):
            raise ValueError("prev/next must be (h, w, 3) uint8")
        arrs = [_f32(f) for f in optFlowPyramid[:maxLevel]]
        for k in range(level, maxLevel):
            exp = (h >> (k - level), w >> (k - level), 2)
            if arrs[k].shape != exp:
                raise ValueError(f"optFlowPyramid[{k}] has shape {arrs[k].shape}, expected {exp}")
        ptrs = (L.f32p * maxLevel)(*[a.ctypes.data_as(L.f32p) for a in arrs])
        L.check(self._lib.ofb_calc_opt_flow_host_u8c3(self._h, _u8(prev).ctypes.data_as(L.u8p),
                                                      _u8(next).ctypes.data_as(L.u8p), w, h, ptrs, level, maxLevel, win,
                                                      warp_mode, C.c_float(flow_scale)))

    def conv_3ch_1ch_tiled_uchar_float(self, src: np.ndarray, w: int, h: int, mask: np.ndarray, mw: int, mh: int) -> np.ndarray:
        """gpu::conv_3ch_1ch_tiled_uchar_float (OptFlowGpu.cu:1100)."""
        if src.shape != (h, w, 3):
            raise ValueError("src must be (h, w, 3) uint8")
        mask = np.ascontiguousarray(mask, np.float32).reshape(-1)
        if mask.size != mw * mh:
            raise ValueError("mask size does not match mw*mh")
        dst = np.empty((h, w), np.float32)
        L.check(self._lib.ofb_conv_3ch_1ch_u8_f32_host(self._h, _u8(src).ctypes.data_as(L.u8p), w, h,
                                                       dst.ctypes.data_as(L.f32p), mask.ctypes.data_as(L.f32p), mw, mh))
        return dst

    def srm_1ch_float(self, arr1: np.ndarray, arr2: np.ndarray, w: int, h: int, ww: int, wh: int) -> np.ndarray:
        """gpu::srm_1ch_float (OptFlowGpu.cu:1597)."""
        if arr1.shape != (h, w) or arr2.shape != (h, w):
            raise ValueError("arr1/arr2 must be (h, w) float32")
        dst = np.empty((h, w), np.float32)
        L.check(self._lib.ofb_srm_1ch_f32_host(self._h, _f32(arr1).ctypes.data_as(L.f32p), _f32(arr2).ctypes.data_as(L.f32p),
                                               w, h, ww, wh, dst.ctypes.data_as(L.f32p)))
        return dst

    def inverse_matrix_float(self, sumIx2, sumIy2, sumIxIy, sumIxIt, sumIyIt, optFlowPyramid: Sequence[np.ndarray],
                             level: int, w: int, h: int) -> None:
        """gpu::inverse_matrix_float (OptFlowGpu.cu:1858): writes optFlowPyramid[level] in place."""
        sums = [_f32(s) for s in (sumIx2, sumIy2, sumIxIy, sumIxIt, sumIyIt)]
        for s in sums:
            if s.shape != (h, w):
                raise ValueError("sums must be (h, w) float32")
        arrs = [_f32(f) for f in optFlowPyramid[:level + 1]]
        if arrs[level].shape != (h, w, 2):
            raise ValueError("optFlowPyramid[level] must be (h, w, 2) float32")
        ptrs = (L.f32p * (level + 1))(*[a.ctypes.data_as(L.f32p) for a in arrs])
        L.check(self._lib.ofb_inverse_matrix_f32_host(self._h, *[s.ctypes.data_as(L.f32p) for s in sums], ptrs, level, w, h))

    # ---- debug derivative views: showTest (main.cu:19-92) without the windows ----
    def conv_3ch_1ch_tiled(self, src: np.ndarray, w: int, h: int, mask: np.ndarray, mw: int, mh: int) -> np.ndarray:
        """gpu::conv_3ch_1ch_tiled: (h, w, 3) u8 in, (h, w) u8 out."""
        mask = np.ascontiguousarray(mask, np.float32).reshape(-1)
        dst = np.empty((h, w), np.uint8)
        L.check(self._lib.ofb_conv_3ch_1ch_u8_u8_host(self._h, _u8(src).ctypes.data_as(L.u8p), w, h, dst.ctypes.data_as(L.u8p),
                                                      mask.ctypes.data_as(L.f32p), mw, mh))
        return dst

    def debug_view(self, prev_level: Optional[np.ndarray], cur_level: np.ndarray, w: int, h: int, level: int, which: int) -> np.ndarray:
        """One window of showTest: thresholded derivative of a pyramid level, upscaled by 2^level."""
        out = np.empty((h << level, w << level), np.uint8)
        pp = _u8(prev_level).ctypes.data_as(L.u8p) if prev_level is not None else None
        L.check(self._lib.ofb_debug_view_host_u8c3(self._h, pp, _u8(cur_level).ctypes.data_as(L.u8p), w, h, level, which,
                                                   out.ctypes.data_as(L.u8p)))
        return out

    # ---- flow composition and export: the headless part of visualizeFlowField (main.cu:114-174) ----
    def compose_flow(self, flow_pyramid: Sequence[np.ndarray], w: int, h: int, levels: int, level: int = 0) -> np.ndarray:
        """Total flow of `level` from the residual pyramid (composition rule main.cu:136-147)."""
        flows = [_f32(f) for f in flow_pyramid]
        out = np.empty((h >> level, w >> level, 2), np.float32)
        L.check(self._lib.ofb_compose_flow_host(self._h, _ptrs(flows, L.f32p), w, h, levels, level, out.ctypes.data_as(L.f32p)))
        return out

    def flow_arrows(self, flow_pyramid: Sequence[np.ndarray], w: int, h: int, levels: int, level: int, arrow_res: int) -> np.ndarray:
        """(n, 4) int32 array of (x0, y0, x1, y1): the arrows main.cu:125-171 draws."""
        flows = [_f32(f) for f in flow_pyramid]
        # one arrow per grid point at most: the grid step is (w >> level) // arrow_res in both directions (main.cu:125-133)
        step = max((w >> level) // max(arrow_res, 1), 1)
        cap = -(-(w >> level) // step) * -(-(h >> level) // step)
        buf = np.empty((cap, 4), np.int32)
        n = C.c_int(0)
        L.check(self._lib.ofb_flow_arrows_host(self._h, _ptrs(flows, L.f32p), w, h, levels, level, arrow_res,
                                               buf.ctypes.data_as(L.i32p), cap, C.byref(n)))
        if n.value > cap:  # (the C side reports the full count and truncates the list: ask again with room for all)
            cap = n.value
            buf = np.empty((cap, 4), np.int32)
            L.check(self._lib.ofb_flow_arrows_host(self._h, _ptrs(flows, L.f32p), w, h, levels, level, arrow_res,
                                                   buf.ctypes.data_as(L.i32p), cap, C.byref(n)))
        return buf[: min(n.value, cap)].copy()

    def grayscale_avg(self, src: np.ndarray, h: int, w: int) -> np.ndarray:
        """gpu::grayscale_avg(src, dest, h, w) (OptFlowGpu.cu:75; height before width like the reference)."""
        if src.shape != (h, w, 3):
            raise ValueError("src must be (h, w, 3) uint8")
        dst = np.empty_like(src)
        L.check(self._lib.ofb_grayscale_avg_host_u8c3(self._h, _u8(src).ctypes.data_as(L.u8p), dst.ctypes.data_as(L.u8p), h, w))
        return dst

    def bilinear_filter(self, src: np.ndarray, gray: np.ndarray, w: int, h: int, ww: int, wh: int, sigmaS: float,
                        sigmaB: float) -> np.ndarray:
        """gpu::bilinear_filter (OptFlowGpu.cu:2050): the bilateral pre-filter of main.cu:240."""
        if src.shape != (h, w, 3) or gray.shape != (h, w, 3):
            raise ValueError("src/gray must be (h, w, 3) uint8")
        dst = np.empty_like(src)
        L.check(self._lib.ofb_bilinear_filter_host_u8c3(self._h, _u8(src).ctypes.data_as(L.u8p), _u8(gray).ctypes.data_as(L.u8p),
                                                        dst.ctypes.data_as(L.u8p), w, h, ww, wh, float(sigmaS), float(sigmaB)))
        return dst

    def bilateral_planar_device(self, gray, w: int, ww: int, sigmaS: float, sigmaB: float, dst=None, stream: int = 0):
        """Bilateral filter of a planar (h, pitch) uint8 CUDA tensor (src == gray)."""
        import torch

        h, pitch = gray.shape
        if dst is None:
            dst = torch.zeros_like(gray)
        L.check(self._lib.ofb_bilateral_planar_device(self._h, gray.data_ptr(), pitch, w, h, ww, ww, float(sigmaS), float(sigmaB),
                                                      dst.data_ptr(), dst.stride(0), C.c_void_p(stream)))
        return dst

    def open_stream(self, w: int, h: int, levels: int, win: int, warp_mode: int = WARP_BILINEAR, flow_scale: float = 1.0,
                    bil_win: int = 0, bil_sigma_s: float = 2.0, bil_sigma_b: float = 10.0) -> "FrameStream":
        """Frame sequence in the role of main.cu:222-275 (defaults of main.cu:236-240 for the pre-filter)."""
        return FrameStream(self, w, h, levels, win, warp_mode, flow_scale, bil_win, bil_sigma_s, bil_sigma_b)

    # ---------------------------------------------------------------- whole-pair host API
    def flow_pairs_host(self, prev: np.ndarray, next: np.ndarray, levels: int, win: int,
                        warp_mode: int = WARP_BILINEAR, flow_scale: float = 1.0,
                        out: Optional[Sequence[np.ndarray]] = None) -> list[np.ndarray]:
        """The loop of main.cu:246-262 for a batch with host buffers.  prev/next: (n, h, w) gray or
        (n, h, w, 3) reference layout (a single pair may omit n).  Returns the residual flow of every
        level, level 0 first, each (n, h>>k, w>>k, 2)."""
        if prev.ndim == 4:
            if prev.shape[3] != 3:
                raise ValueError("4-d input must be (n, h, w, 3)")
            channels = 3
            n, h, w = prev.shape[0], prev.shape[1], prev.shape[2]
        elif prev.ndim == 3:
            channels = 1
            n, h, w = prev.shape
        elif prev.ndim == 2:
            channels = 1
            n, (h, w) = 1, prev.shape
        else:
            raise ValueError("prev must be (n,h,w), (h,w) or (n,h,w,3)")
        if next.shape != prev.shape:
            raise ValueError("prev and next differ in shape")
        p = OfbParams(w, h, levels, win, warp_mode, flow_scale, n)
        if out is None:
            out = [np.empty((n, h >> k, w >> k, 2), np.float32) for k in range(levels)]
        ptrs = (L.f32p * levels)(*[_f32(o).ctypes.data_as(L.f32p) for o in out])
        L.check(self._lib.ofb_flow_pairs_host(self._h, C.byref(p), _u8(prev).ctypes.data_as(L.u8p),
                                              _u8(next).ctypes.data_as(L.u8p), channels, ptrs))
        return list(out)

    def total_flow_pairs_host(self, prev: np.ndarray, next: np.ndarray, levels: int, win: int,
                              warp_mode: int = WARP_BILINEAR, flow_scale: float = 1.0,
                              out: Optional[np.ndarray] = None) -> np.ndarray:
        """As flow_pairs_host, but only the level-0 composition of main.cu:136-147 (the total flow, (n, h, w, 2))
        leaves the device: 8 bytes per pixel over PCIe instead of 10.5."""
        channels, n, h, w = _batch_shape(prev, next)
        p = OfbParams(w, h, levels, win, warp_mode, flow_scale, n)
        if out is None:
            out = np.empty((n, h, w, 2), np.float32)
        L.check(self._lib.ofb_flow_pairs_host_ex(self._h, C.byref(p), _u8(prev).ctypes.data_as(L.u8p),
                                                 _u8(next).ctypes.data_as(L.u8p), channels, None,
                                                 _f32(out).ctypes.data_as(L.f32p)))
        return out

    def flow_pairs_fb_host(self, prev: np.ndarray, next: np.ndarray, levels: int, win: int, warp_mode: int = WARP_BILINEAR,
                           flow_scale: float = 1.0, alpha: float = 0.01, beta: float = 0.5, want_bwd: bool = False,
                           want_err2: bool = False):
        """flow_pairs_fb_device for host batches: prev/next as in total_flow_pairs_host.  Returns numpy arrays
        (fwd_total (n, h, w, 2), bwd_total or None, status (n, h, w) uint8 FB_* codes, err2 (n, h, w) or None); the
        outputs not asked for are not downloaded."""
        channels, n, h, w = _batch_shape(prev, next)
        p = OfbParams(w, h, levels, win, warp_mode, flow_scale, n)
        fwd = np.empty((n, h, w, 2), np.float32)
        bwd = np.empty((n, h, w, 2), np.float32) if want_bwd else None
        status = np.empty((n, h, w), np.uint8)
        err2 = np.empty((n, h, w), np.float32) if want_err2 else None
        L.check(self._lib.ofb_flow_pairs_fb_host(self._h, C.byref(p), _u8(prev).ctypes.data_as(L.u8p),
                                                 _u8(next).ctypes.data_as(L.u8p), channels, C.c_float(alpha), C.c_float(beta),
                                                 fwd.ctypes.data_as(L.f32p), _optp(bwd, L.f32p), status.ctypes.data_as(L.u8p),
                                                 _optp(err2, L.f32p)))
        return fwd, bwd, status, err2

    # ---------------------------------------------------------------- device-resident API
    def flow_pairs_device(self, prev, next, w: int, levels: int, win: int, warp_mode: int = WARP_BILINEAR,
                          flow_scale: float = 1.0, flows=None, total_flow=None, stream: int = 0):
        """prev/next: torch.uint8 CUDA tensors (n, h, pitch) with pitch % 16 == 0 and pitch >= w.
        Returns the list of residual-flow tensors (n, h>>k, w>>k, 2); pass `flows` to reuse buffers."""
        import torch

        if prev.dtype != torch.uint8 or prev.dim() != 3 or not prev.is_contiguous() or prev.shape != next.shape:
            raise ValueError("prev/next must be contiguous uint8 (n, h, pitch) CUDA tensors of equal shape")
        n, h, pitch = prev.shape
        if flows is None:
            flows = [torch.empty((n, h >> k, w >> k, 2), dtype=torch.float32, device=prev.device) for k in range(levels)]
        p = OfbParams(w, h, levels, win, warp_mode, flow_scale, n)
        ptrs = (C.c_void_p * levels)(*[f.data_ptr() for f in flows])
        L.check(self._lib.ofb_flow_pairs_device(self._h, C.byref(p), prev.data_ptr(), next.data_ptr(), pitch, pitch * h,
                                                ptrs, total_flow.data_ptr() if total_flow is not None else None,
                                                C.c_void_p(stream)))
        return flows

    def fb_check_device(self, fwd, bwd, flow_scale: float = 1.0, alpha: float = 0.01, beta: float = 0.5, status=None,
                        err2=None, want_err2: bool = False, stream: int = 0):
        """Forward-backward consistency check of two total-flow fields: fwd / bwd are float32 (n, h, w, 2) CUDA tensors
        in flow units, flow_scale px per unit.  Returns (status (n, h, w) uint8 of FB_* codes, err2 (n, h, w) float32
        squared error in px^2 or None); passing `err2` implies want_err2."""
        import torch

        if fwd.dtype != torch.float32 or fwd.dim() != 4 or fwd.shape[3] != 2 or fwd.shape != bwd.shape or \
                not (fwd.is_contiguous() and bwd.is_contiguous()):
            raise ValueError("fwd/bwd must be contiguous float32 (n, h, w, 2) CUDA tensors of equal shape")
        n, h, w, _ = fwd.shape
        if status is None:
            status = torch.empty((n, h, w), dtype=torch.uint8, device=fwd.device)
        if err2 is None and want_err2:
            err2 = torch.empty((n, h, w), dtype=torch.float32, device=fwd.device)
        L.check(self._lib.ofb_fb_check_device(self._h, fwd.data_ptr(), bwd.data_ptr(), w, h, n, C.c_float(flow_scale),
                                              C.c_float(alpha), C.c_float(beta), status.data_ptr(),
                                              err2.data_ptr() if err2 is not None else None, C.c_void_p(stream)))
        return status, err2

    def flow_pairs_fb_device(self, prev, next, w: int, levels: int, win: int, warp_mode: int = WARP_BILINEAR,
                             flow_scale: float = 1.0, alpha: float = 0.01, beta: float = 0.5, want_err2: bool = False,
                             stream: int = 0):
        """Flow prev->next and next->prev from one pyramid build, and their forward-backward check.  prev/next as in
        flow_pairs_device.  Returns (fwd_total, bwd_total, status, err2 or None): the totals (n, h, w, 2) as
        flow_pairs_device's total_flow, status (n, h, w) uint8 FB_* codes."""
        import torch

        if prev.dtype != torch.uint8 or prev.dim() != 3 or not prev.is_contiguous() or prev.shape != next.shape:
            raise ValueError("prev/next must be contiguous uint8 (n, h, pitch) CUDA tensors of equal shape")
        n, h, pitch = prev.shape
        dev = prev.device
        fwd = torch.empty((n, h, w, 2), dtype=torch.float32, device=dev)
        bwd = torch.empty((n, h, w, 2), dtype=torch.float32, device=dev)
        status = torch.empty((n, h, w), dtype=torch.uint8, device=dev)
        err2 = torch.empty((n, h, w), dtype=torch.float32, device=dev) if want_err2 else None
        p = OfbParams(w, h, levels, win, warp_mode, flow_scale, n)
        L.check(self._lib.ofb_flow_pairs_fb_device(self._h, C.byref(p), prev.data_ptr(), next.data_ptr(), pitch, pitch * h,
                                                   C.c_float(alpha), C.c_float(beta), fwd.data_ptr(), bwd.data_ptr(),
                                                   status.data_ptr(), err2.data_ptr() if err2 is not None else None,
                                                   C.c_void_p(stream)))
        return fwd, bwd, status, err2

    def track_points_device(self, prev, next, w: int, levels: int, win: int, points, flow_scale: float = 1.0, iters: int = 30,
                            eps: float = 0.01, min_eig: float = 0.0, stream: int = 0):
        """Sparse pyramidal Lucas-Kanade (the KLT tracker): follow `points`, a float32 (n, m, 2) CUDA tensor of (x, y)
        level-0 positions (m points per pair), from prev to next through `levels` pyramid levels with up to `iters`
        Gauss-Newton iterations per level, stopping a level early once both components of an update are below `eps` px
        (the defaults are OpenCV's).  prev/next as in flow_pairs_device.  Returns (flow (n, m, 2) float32 in flow units --
        s * flow px with s = flow_scale --, status (n, m) uint8 PT_* codes).  min_eig > 0 marks points whose window's
        smaller structure-tensor eigenvalue, divided by win^2, is below it PT_LOW_TEXTURE (rule: include/ofb200.h); that
        value is the score of min_eig_map_device."""
        import torch

        if prev.dtype != torch.uint8 or prev.dim() != 3 or not prev.is_contiguous() or prev.shape != next.shape:
            raise ValueError("prev/next must be contiguous uint8 (n, h, pitch) CUDA tensors of equal shape")
        n, h, pitch = prev.shape
        if not (prev.is_cuda and next.device == prev.device):
            raise ValueError("prev/next must be CUDA tensors on one device")
        if points.dtype != torch.float32 or points.dim() != 3 or points.shape[0] != n or points.shape[2] != 2 or \
                not points.is_contiguous() or points.device != prev.device:
            raise ValueError("points must be a contiguous float32 (n, m, 2) CUDA tensor on prev's device, one row per pair")
        m = points.shape[1]
        flow = torch.empty((n, m, 2), dtype=torch.float32, device=prev.device)
        status = torch.empty((n, m), dtype=torch.uint8, device=prev.device)
        p = OfbParams(w, h, levels, win, WARP_BILINEAR, flow_scale, n)
        L.check(self._lib.ofb_track_points_device(self._h, C.byref(p), prev.data_ptr(), next.data_ptr(), pitch, pitch * h,
                                                  points.data_ptr(), m, int(iters), C.c_float(eps), C.c_float(min_eig),
                                                  flow.data_ptr(), status.data_ptr(), C.c_void_p(stream)))
        return flow, status

    @staticmethod
    def _corner_images(imgs, w: int):
        import torch

        if not isinstance(imgs, torch.Tensor) or imgs.dtype != torch.uint8 or imgs.dim() != 3 or not imgs.is_contiguous() \
                or not imgs.is_cuda:
            raise ValueError("imgs must be a contiguous uint8 (n, h, pitch) CUDA tensor")
        n, h, pitch = imgs.shape
        if not 1 <= w <= pitch:
            raise ValueError(f"w {w} outside 1..pitch {pitch}")
        return n, h, pitch

    def min_eig_map_device(self, imgs, w: int, win: int, stream: int = 0):
        """The Shi-Tomasi score of every pixel of the (n, h, pitch) uint8 images (the layout track_points_device takes):
        the smaller eigenvalue of the window's structure tensor of the tracker's Sobel fields, over win^2 -- the value the
        tracker compares with min_eig (rule: include/ofb200.h).  Returns (n, h, w) float32."""
        import torch

        n, h, pitch = self._corner_images(imgs, w)
        out = torch.empty((n, h, w), dtype=torch.float32, device=imgs.device)
        L.check(self._lib.ofb_min_eig_map_device(self._h, imgs.data_ptr(), pitch, pitch * h, w, h, n, win, out.data_ptr(),
                                                 C.c_void_p(stream)))
        return out

    def detect_corners_device(self, imgs, w: int, win: int, max_corners: int, quality_level: float = 0.01,
                              min_distance: float = 10.0, min_score: float = 0.0, stream: int = 0):
        """Shi-Tomasi corners (goodFeaturesToTrack) of each of the (n, h, pitch) uint8 images: interior strict local maxima
        of the score above max(quality_level * the image's largest score, min_score), strongest first, at least
        min_distance px apart, at most max_corners per image (rule: include/ofb200.h).  Returns (corners (n, max_corners, 2)
        float32 integer (x, y), scores (n, max_corners) float32, counts (n,) int32); the slots past an image's count are NaN,
        so `corners` can go straight to track_points_device as its points.  Nothing waits on the host."""
        import torch

        n, h, pitch = self._corner_images(imgs, w)
        dev = imgs.device
        corners = torch.empty((n, max_corners, 2), dtype=torch.float32, device=dev) if max_corners >= 1 else None
        scores = torch.empty((n, max_corners), dtype=torch.float32, device=dev) if max_corners >= 1 else None
        counts = torch.empty((n,), dtype=torch.int32, device=dev)
        L.check(self._lib.ofb_detect_corners_device(self._h, imgs.data_ptr(), pitch, pitch * h, w, h, n, win, int(max_corners),
                                                    C.c_float(quality_level), C.c_float(min_distance), C.c_float(min_score),
                                                    corners.data_ptr() if corners is not None else None,
                                                    scores.data_ptr() if scores is not None else None, counts.data_ptr(),
                                                    C.c_void_p(stream)))
        return corners, scores, counts

    def reserve_corners(self, w: int, h: int, n_images: int, win: int, max_corners: int) -> None:
        """Size the context workspace for detect_corners_device calls of this shape now (CUDA graph capture)."""
        L.check(self._lib.ofb_ctx_reserve_corners(self._h, w, h, n_images, win, max_corners))

    def pyr_down_device(self, src, sw: int, dst=None, stream: int = 0):
        """src: torch.uint8 (n, sh, pitch) -> dst (n, sh>>1, pitch_d)."""
        import torch

        n, sh, sp = src.shape
        dw, dh = sw >> 1, sh >> 1
        if dst is None:
            dst = torch.zeros((n, dh, align_up(dw, 64)), dtype=torch.uint8, device=src.device)
        dp = dst.shape[2]
        L.check(self._lib.ofb_pyr_down_device(self._h, src.data_ptr(), sp, sp * sh, sw, sh, dst.data_ptr(), dp, dp * dh, n,
                                              C.c_void_p(stream)))
        return dst

    def pyr_down2_device(self, src, sw: int, stream: int = 0):
        """Two pyramid steps in one launch: src (n, sh, pitch) -> (dst1 (n, sh>>1, pitch1), dst2 (n, sh>>2, pitch2))."""
        import torch

        n, sh, sp = src.shape
        d1 = torch.zeros((n, sh >> 1, align_up(sw >> 1, 64)), dtype=torch.uint8, device=src.device)
        d2 = torch.zeros((n, sh >> 2, align_up(sw >> 2, 64)), dtype=torch.uint8, device=src.device)
        L.check(self._lib.ofb_pyr_down2_device(self._h, src.data_ptr(), sp, sp * sh, sw, sh, d1.data_ptr(), d1.shape[2],
                                               d1.shape[2] * d1.shape[1], d2.data_ptr(), d2.shape[2], d2.shape[2] * d2.shape[1],
                                               n, C.c_void_p(stream)))
        return d1, d2

    def pyr_down_strip_device(self, src, sw: int, src_y_off: int, dst, dst_y0: int, dst_y1: int, stream: int = 0):
        """Row-strip pyramid step: src (rows, pitch) holds global rows from src_y_off; dst (dst_y1-dst_y0, pitch_d)."""
        L.check(self._lib.ofb_pyr_down_strip_device(self._h, src.data_ptr(), src.stride(0), sw, src.shape[0], src_y_off,
                                                    dst.data_ptr(), dst.stride(0), dst_y0, dst_y1, C.c_void_p(stream)))
        return dst

    def lk_level_device(self, prev, next, w: int, win: int, warp_mode: int = WARP_BILINEAR, flow_scale: float = 1.0,
                        cum_in=None, flow_out=None, cum_out=None, stream: int = 0):
        """One fused LK level on (n, h, pitch) uint8 tensors; cum_in is the (n, h>>1, w>>1, 2) cumulative
        flow of the coarser level or None for the coarsest level."""
        import torch

        n, h, pitch = prev.shape
        if flow_out is None:
            flow_out = torch.empty((n, h, w, 2), dtype=torch.float32, device=prev.device)
        L.check(self._lib.ofb_lk_level_device(self._h, prev.data_ptr(), next.data_ptr(), pitch, pitch * h, w, h, n, win,
                                              warp_mode, C.c_float(flow_scale),
                                              cum_in.data_ptr() if cum_in is not None else None, flow_out.data_ptr(),
                                              cum_out.data_ptr() if cum_out is not None else None, C.c_void_p(stream)))
        return flow_out

    def lk_level_strip_device(self, prev, next, w: int, y_off: int, h_global: int, out_y0: int, out_y1: int, win: int,
                              warp_mode: int, flow_scale: float, cum_in, cum_y_off: int, flow_out, cum_out=None,
                              overflow_flag=None, stream: int = 0):
        """Row-strip variant: prev/next are (h_local, pitch) uint8 holding global rows [y_off, y_off+h_local)."""
        h_local, pitch = prev.shape
        cum_h_local = cum_in.shape[0] if cum_in is not None else 0
        L.check(self._lib.ofb_lk_level_strip_device(
            self._h, prev.data_ptr(), next.data_ptr(), pitch, w, h_local, y_off, h_global, out_y0, out_y1, win, warp_mode,
            C.c_float(flow_scale), cum_in.data_ptr() if cum_in is not None else None, cum_y_off, cum_h_local,
            flow_out.data_ptr(), cum_out.data_ptr() if cum_out is not None else None,
            overflow_flag.data_ptr() if overflow_flag is not None else None, C.c_void_p(stream)))
        return flow_out


class FrameStream:
    """ofb_stream: push BGR frames one by one; every push after the first returns the flow against the
    previous frame, whose pyramid stays on the device."""

    def __init__(self, ctx: Context, w, h, levels, win, warp_mode, flow_scale, bil_win, bil_sigma_s, bil_sigma_b):
        self._ctx, self._lib = ctx, ctx._lib
        self.w, self.h, self.levels = w, h, levels
        p = OfbParams(w, h, levels, win, warp_mode, flow_scale, 1)
        hnd = C.c_void_p()
        L.check(self._lib.ofb_stream_create(ctx._h, C.byref(p), bil_win, float(bil_sigma_s), float(bil_sigma_b), C.byref(hnd)))
        self._h = hnd

    def push(self, frame_bgr: np.ndarray, want_total: bool = False):
        """Returns None for the first frame, else (flows, total) with flows[k] of shape (h>>k, w>>k, 2)."""
        if frame_bgr.shape != (self.h, self.w, 3):
            raise ValueError("frame must be (h, w, 3) uint8")
        flows = [np.empty((self.h >> k, self.w >> k, 2), np.float32) for k in range(self.levels)]
        total = np.empty((self.h, self.w, 2), np.float32) if want_total else None
        ptrs = (L.f32p * self.levels)(*[f.ctypes.data_as(L.f32p) for f in flows])
        has = C.c_int(0)
        L.check(self._lib.ofb_stream_push_bgr_host(self._h, _u8(frame_bgr).ctypes.data_as(L.u8p), ptrs,
                                                   total.ctypes.data_as(L.f32p) if want_total else None, C.byref(has)))
        return (flows, total) if has.value else None

    def push_fb(self, frame_bgr: np.ndarray, alpha: float = 0.01, beta: float = 0.5, want_levels: bool = False,
                want_bwd: bool = False, want_err2: bool = False):
        """push with the forward-backward check: returns None for the first frame, else a dict with `fwd_total` (h, w, 2),
        `status` (h, w) uint8 FB_* codes and, as asked, `levels` (the forward residual flows, level 0 first), `bwd_total`
        (h, w, 2) and `err2` (h, w).  Mixes freely with push on one stream."""
        if frame_bgr.shape != (self.h, self.w, 3):
            raise ValueError("frame must be (h, w, 3) uint8")
        out = {"fwd_total": np.empty((self.h, self.w, 2), np.float32), "status": np.empty((self.h, self.w), np.uint8)}
        if want_levels:
            out["levels"] = [np.empty((self.h >> k, self.w >> k, 2), np.float32) for k in range(self.levels)]
        if want_bwd:
            out["bwd_total"] = np.empty((self.h, self.w, 2), np.float32)
        if want_err2:
            out["err2"] = np.empty((self.h, self.w), np.float32)
        ptrs = _ptrs(out["levels"], L.f32p) if want_levels else None
        has = C.c_int(0)
        L.check(self._lib.ofb_stream_push_bgr_host_fb(self._h, _u8(frame_bgr).ctypes.data_as(L.u8p), C.c_float(alpha),
                                                      C.c_float(beta), ptrs, out["fwd_total"].ctypes.data_as(L.f32p),
                                                      _optp(out.get("bwd_total"), L.f32p), out["status"].ctypes.data_as(L.u8p),
                                                      _optp(out.get("err2"), L.f32p), C.byref(has)))
        return out if has.value else None

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ofb_stream_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def write_flo(path: str, flow: np.ndarray) -> None:
    """Middlebury .flo file of an (h, w, 2) float32 flow field."""
    f = _f32(flow)
    L.check(L.load().ofb_write_flo(os.fsencode(path), f.ctypes.data_as(L.f32p), f.shape[1], f.shape[0]))


def planar_to_device(imgs: np.ndarray, device="cuda:0"):
    """(n, h, w) uint8 numpy -> torch (n, h, pitch) with pitch = align_up(w, 64); padding is zero."""
    import torch

    n, h, w = imgs.shape
    pitch = align_up(w, 64)
    t = torch.zeros((n, h, pitch), dtype=torch.uint8, device=device)
    t[:, :, :w] = torch.from_numpy(np.ascontiguousarray(imgs)).to(device)
    return t
