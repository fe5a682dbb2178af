"""ctypes binding of libofb200.so (the C ABI in include/ofb200.h).

The shared library is built in-tree by `make -C cuda_optical_flow_2_b200/csrc` (or
`__graft_entry__.build()`).  There is no Python or CPU fallback: if the library is missing the
import of anything that computes raises, and on a machine without a B200 every compute entry
point returns OFB_ERR_CUDA, surfaced here as OfbError.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# OFB200_LIB lets a developer point at an experimental build of the same library
LIB_PATH = os.environ.get("OFB200_LIB") or os.path.join(_HERE, "libofb200.so")

OFB_OK, OFB_ERR_INVALID, OFB_ERR_CUDA, OFB_ERR_UNSUPPORTED, OFB_ERR_NOMEM = 0, 1, 2, 3, 4
WARP_AS_WRITTEN, WARP_NEAREST, WARP_BILINEAR = 0, 1, 2
SOLVE_EXACT, SOLVE_FAST = 0, 1
MAX_LEVELS, MAX_WINDOW = 8, 19
PROFILE_PYRAMID, PROFILE_FB_CHECK, PROFILE_TRACK, PROFILE_CORNERS = 100, 101, 102, 103
# per-pixel status of the forward-backward consistency check (ofb_fb_check_device)
FB_CONSISTENT, FB_INCONSISTENT, FB_OUTSIDE, FB_FWD_NONFINITE, FB_BWD_NONFINITE = 0, 1, 2, 3, 4
FB_UNCHECKED = 5  # row strips only: a tap the check needs lies outside the backward rows the rank holds
# per-point status of the sparse tracker (ofb_track_points_device)
PT_TRACKED, PT_NONFINITE, PT_LOW_TEXTURE, PT_OUTSIDE = 0, 1, 2, 3

u8p = C.POINTER(C.c_uint8)
f32p = C.POINTER(C.c_float)
i32p = C.POINTER(C.c_int)


class OfbParams(C.Structure):
    _fields_ = [("w", C.c_int), ("h", C.c_int), ("levels", C.c_int), ("win", C.c_int), ("warp_mode", C.c_int),
                ("flow_scale", C.c_float), ("n_pairs", C.c_int)]


class OfbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"ofb200 error {code}: {msg}")
        self.code = code


# every symbol include/ofb200.h declares: name -> (restype, argtypes)
_vp = C.c_void_p
_sz = C.c_size_t
SIGNATURES = {
    "ofb_last_error": (C.c_char_p, []),
    "ofb_version": (C.c_int, []),
    "ofb_ctx_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "ofb_ctx_destroy": (C.c_int, [_vp]),
    "ofb_ctx_device": (C.c_int, [_vp, i32p]),
    "ofb_ctx_sm_count": (C.c_int, [_vp, i32p]),
    "ofb_ctx_reserve_pairs": (C.c_int, [_vp, C.POINTER(OfbParams)]),
    "ofb_ctx_set_solve": (C.c_int, [_vp, C.c_int]),
    "ofb_ctx_get_solve": (C.c_int, [_vp, i32p]),
    "ofb_ctx_set_host_threads": (C.c_int, [_vp, C.c_int]),
    "ofb_ctx_get_host_threads": (C.c_int, [_vp, i32p]),
    "ofb_c3_extract_host": (C.c_int, [_vp, _vp, _sz, C.c_int]),
    "ofb_ctx_launch_count": (C.c_int, [_vp, C.POINTER(C.c_ulonglong)]),
    "ofb_ctx_profile_enable": (C.c_int, [_vp, C.c_int]),
    "ofb_ctx_profile_read": (C.c_int, [_vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_ulonglong)]),
    "ofb_flow_pairs_device": (C.c_int, [_vp, C.POINTER(OfbParams), _vp, _vp, _sz, _sz, C.POINTER(_vp), _vp, _vp]),
    "ofb_fb_check_device": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, _vp, _vp,
                                      _vp]),
    "ofb_flow_pairs_fb_device": (C.c_int, [_vp, C.POINTER(OfbParams), _vp, _vp, _sz, _sz, C.c_float, C.c_float, _vp, _vp, _vp,
                                           _vp, _vp]),
    "ofb_flow_pairs_fb_host": (C.c_int, [_vp, C.POINTER(OfbParams), u8p, u8p, C.c_int, C.c_float, C.c_float, f32p, f32p, u8p,
                                         f32p]),
    "ofb_stream_push_bgr_host_fb": (C.c_int, [_vp, u8p, C.c_float, C.c_float, C.POINTER(f32p), f32p, f32p, u8p, f32p, i32p]),
    "ofb_ctx_reserve_pairs_fb": (C.c_int, [_vp, C.POINTER(OfbParams)]),
    "ofb_track_points_device": (C.c_int, [_vp, C.POINTER(OfbParams), _vp, _vp, _sz, _sz, _vp, C.c_int, C.c_int, C.c_float,
                                          C.c_float, _vp, _vp, _vp]),
    "ofb_min_eig_map_device": (C.c_int, [_vp, _vp, _sz, _sz, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp]),
    "ofb_detect_corners_device": (C.c_int, [_vp, _vp, _sz, _sz, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                            C.c_float, C.c_float, _vp, _vp, _vp, _vp]),
    "ofb_ctx_reserve_corners": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "ofb_pyr_down_device": (C.c_int, [_vp, _vp, _sz, _sz, C.c_int, C.c_int, _vp, _sz, _sz, C.c_int, _vp]),
    "ofb_pyr_down2_device": (C.c_int, [_vp, _vp, _sz, _sz, C.c_int, C.c_int, _vp, _sz, _sz, _vp, _sz, _sz, C.c_int, _vp]),
    "ofb_pyr_down_strip_device": (C.c_int, [_vp, _vp, _sz, C.c_int, C.c_int, C.c_int, _vp, _sz, C.c_int, C.c_int, _vp]),
    "ofb_lk_level_device": (C.c_int, [_vp, _vp, _vp, _sz, _sz, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                      _vp, _vp, _vp, _vp]),
    "ofb_lk_level_strip_device": (C.c_int, [_vp, _vp, _vp, _sz, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.c_int, C.c_int, C.c_float, _vp, C.c_int, C.c_int, _vp, _vp, _vp, _vp]),
    "ofb_c3_to_planar_device": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp, _sz, _sz, _vp]),
    "ofb_gauss_pyramid_host_u8c3": (C.c_int, [_vp, C.POINTER(u8p), C.c_int, C.c_int, C.c_int]),
    "ofb_calc_opt_flow_host_u8c3": (C.c_int, [_vp, u8p, u8p, C.c_int, C.c_int, C.POINTER(f32p), C.c_int, C.c_int,
                                              C.c_int, C.c_int, C.c_float]),
    "ofb_conv_3ch_1ch_u8_f32_host": (C.c_int, [_vp, u8p, C.c_int, C.c_int, f32p, f32p, C.c_int, C.c_int]),
    "ofb_srm_1ch_f32_host": (C.c_int, [_vp, f32p, f32p, C.c_int, C.c_int, C.c_int, C.c_int, f32p]),
    "ofb_inverse_matrix_f32_host": (C.c_int, [_vp, f32p, f32p, f32p, f32p, f32p, C.POINTER(f32p), C.c_int, C.c_int,
                                              C.c_int]),
    "ofb_flow_pairs_host": (C.c_int, [_vp, C.POINTER(OfbParams), u8p, u8p, C.c_int, C.POINTER(f32p)]),
    "ofb_flow_pairs_host_ex": (C.c_int, [_vp, C.POINTER(OfbParams), u8p, u8p, C.c_int, C.POINTER(f32p), f32p]),
    "ofb_grayscale_avg_host_u8c3": (C.c_int, [_vp, u8p, u8p, C.c_int, C.c_int]),
    "ofb_bilinear_filter_host_u8c3": (C.c_int, [_vp, u8p, u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                                C.c_double]),
    "ofb_bilateral_planar_device": (C.c_int, [_vp, _vp, _sz, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                                              _vp, _sz, _vp]),
    "ofb_stream_create": (C.c_int, [_vp, C.POINTER(OfbParams), C.c_int, C.c_double, C.c_double, C.POINTER(_vp)]),
    "ofb_stream_push_bgr_host": (C.c_int, [_vp, u8p, C.POINTER(f32p), f32p, i32p]),
    "ofb_stream_destroy": (C.c_int, [_vp]),
    "ofb_strips_plan_query": (C.c_int, [C.c_int] * 8 + [i32p]),
    "ofb_strips_create": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int,
                                    C.POINTER(_vp)]),
    "ofb_strips_own_rows": (C.c_int, [_vp, C.c_int, i32p, i32p]),
    "ofb_strips_run_device": (C.c_int, [_vp, _vp, _vp, _sz, _vp]),
    "ofb_strips_run_phase_device": (C.c_int, [_vp, _vp, _vp, _sz, C.c_int, _vp]),
    "ofb_strips_result": (C.c_int, [_vp, C.c_int, C.POINTER(_vp), C.POINTER(_vp)]),
    "ofb_strips_check": (C.c_int, [_vp, _vp, i32p]),
    "ofb_strips_destroy": (C.c_int, [_vp]),
    "ofb_strips_input": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_sz)]),
    "ofb_strips_set_total": (C.c_int, [_vp, C.c_int]),
    "ofb_strips_set_fused": (C.c_int, [_vp, C.c_int]),
    "ofb_strips_peer_handle": (C.c_int, [_vp, _vp]),
    "ofb_strips_peer_connect": (C.c_int, [_vp, _vp]),
    "ofb_strips_peer_arena": (C.c_int, [_vp, C.POINTER(_vp)]),
    "ofb_strips_peer_connect_local": (C.c_int, [_vp, C.POINTER(_vp)]),
    "ofb_strips_create_fb": (C.c_int, [_vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.POINTER(_vp)]),
    "ofb_strips_run_fb_device": (C.c_int, [_vp, _vp, _vp, _sz, C.c_float, C.c_float, C.c_int, _vp]),
    "ofb_strips_run_fb_phase_device": (C.c_int, [_vp, _vp, _vp, _sz, C.c_float, C.c_float, C.c_int, C.c_int, _vp]),
    "ofb_strips_fb_result": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "ofb_conv_3ch_1ch_u8_u8_host": (C.c_int, [_vp, u8p, C.c_int, C.c_int, u8p, f32p, C.c_int, C.c_int]),
    "ofb_debug_view_host_u8c3": (C.c_int, [_vp, u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p]),
    "ofb_compose_flow_host": (C.c_int, [_vp, C.POINTER(f32p), C.c_int, C.c_int, C.c_int, C.c_int, f32p]),
    "ofb_flow_arrows_host": (C.c_int, [_vp, C.POINTER(f32p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, i32p, C.c_int, i32p]),
    "ofb_write_flo": (C.c_int, [C.c_char_p, f32p, C.c_int, C.c_int]),
    "ofb_host_alloc": (C.c_int, [C.POINTER(_vp), _sz]),
    "ofb_host_free": (C.c_int, [_vp]),
}

_lib = None


def load() -> C.CDLL:
    """Load libofb200.so and attach the prototypes.  Raises if the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `make -C cuda_optical_flow_2_b200/csrc` "
                              "(there is no fallback implementation)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int) -> None:
    if rc != OFB_OK:
        raise OfbError(rc, load().ofb_last_error().decode("utf-8", "replace"))
