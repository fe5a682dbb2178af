"""B200-native dense pyramidal Lucas-Kanade path (and a sparse point tracker on the same pyramids) behind the reference's `namespace gpu` interface.

The package holds only what that path needs: csrc/ (hand-written sm_100a kernels + the C ABI of
include/ofb200.h), api.py (host-side mirror of the reference's entry points) and dist.py (frame-batch
sharding and row-strip partitioning over torch.distributed).  There is no CPU implementation here.
"""
from ._lib import (FB_BWD_NONFINITE, FB_CONSISTENT, FB_FWD_NONFINITE, FB_INCONSISTENT, FB_OUTSIDE, FB_UNCHECKED, LIB_PATH, MAX_LEVELS,
                   MAX_WINDOW, PROFILE_FB_CHECK, PROFILE_PYRAMID, PROFILE_TRACK, PROFILE_CORNERS, PT_LOW_TEXTURE, PT_NONFINITE, PT_OUTSIDE,
                   PT_TRACKED, SOLVE_EXACT, SOLVE_FAST, WARP_AS_WRITTEN, WARP_BILINEAR,
                   WARP_NEAREST, OfbError, OfbParams)
from .api import REFERENCE_WINDOW, Context, align_up, planar_to_device, write_flo

__all__ = ["Context", "OfbError", "OfbParams", "WARP_AS_WRITTEN", "WARP_NEAREST", "WARP_BILINEAR", "SOLVE_EXACT", "SOLVE_FAST", "MAX_LEVELS",
           "MAX_WINDOW", "REFERENCE_WINDOW", "LIB_PATH", "align_up", "planar_to_device", "write_flo", "FB_CONSISTENT",
           "FB_INCONSISTENT", "FB_OUTSIDE", "FB_FWD_NONFINITE", "FB_BWD_NONFINITE", "FB_UNCHECKED", "PROFILE_PYRAMID", "PROFILE_FB_CHECK",
           "PROFILE_TRACK", "PROFILE_CORNERS", "PT_TRACKED", "PT_NONFINITE", "PT_LOW_TEXTURE", "PT_OUTSIDE"]
