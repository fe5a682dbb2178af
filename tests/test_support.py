"""The comparison bars of support.py reject what they claim to reject, and accept what they claim to accept, in their numpy
and torch forms (CPU tensors here; the same code runs on device tensors)."""
import numpy as np
import pytest

from support import (F32, assert_same_bits, assert_same_bytes, assert_status_equal, assert_values_equal, bits_differ,
                     bytes_differ, statuses_differ, values_differ)

BARS = {"bytes": (bytes_differ, assert_same_bytes), "bits": (bits_differ, assert_same_bits),
        "values": (values_differ, assert_values_equal), "statuses": (statuses_differ, assert_status_equal)}
FLOW = np.array([[1.0, -2.5, 0.0], [np.nan, np.inf, 7.0]], F32)


def nan_with_payload(payload):
    return np.array(0x7FC00000 | payload, np.uint32).view(F32)


def edited(a, *changes):
    a = a.copy()
    for at, v in changes:
        a[at] = v
    return a


# (bar, what, got, ref, the bar must reject)
CASES = [
    ("bits", "identical", FLOW.copy(), FLOW, False),
    ("bits", "-0.0 vs 0.0", edited(FLOW, ((0, 2), -0.0)), FLOW, True),
    ("bits", "NaN moved", edited(FLOW, ((1, 0), 5.0), ((1, 2), np.nan)), FLOW, True),
    ("bits", "one flipped low bit", edited(FLOW, ((0, 0), np.nextafter(F32(1), F32(2)))), FLOW, True),
    ("bits", "NaN payloads differ", edited(FLOW, ((1, 0), nan_with_payload(1))), FLOW, False),
    ("values", "identical", FLOW.copy(), FLOW, False),
    ("values", "-0.0 vs 0.0", edited(FLOW, ((0, 2), -0.0)), FLOW, False),
    ("values", "inf vs finite", edited(FLOW, ((1, 1), 3e38)), FLOW, True),
    ("values", "NaN moved", edited(FLOW, ((1, 0), 5.0), ((1, 2), np.nan)), FLOW, True),
    ("bytes", "identical", FLOW.copy(), FLOW, False),
    ("bytes", "NaN payloads differ", edited(FLOW, ((1, 0), nan_with_payload(1))), FLOW, True),
    ("statuses", "identical", np.array([0, 1, 2, 3, 4], np.uint8), np.array([0, 1, 2, 3, 4], np.uint8), False),
    ("statuses", "one status changed", np.array([0, 1, 2, 4, 4], np.uint8), np.array([0, 1, 2, 3, 4], np.uint8), True),
]


@pytest.mark.parametrize("form", ["numpy", "torch"])
@pytest.mark.parametrize("bar,what,got,ref,reject", CASES, ids=[f"{c[0]}-{c[1]}" for c in CASES])
def test_bar(bar, what, got, ref, reject, form):
    if form == "torch":
        import torch

        got, ref = torch.from_numpy(got), torch.from_numpy(ref)
    differ, assert_form = BARS[bar]
    assert bool(differ(got, ref)) == reject
    if reject:
        with pytest.raises(AssertionError):
            assert_form(got, ref, what)
    else:
        assert_form(got, ref, what)
