"""CPU: seeded fuzz of the oracles (oracle/warp_oracle.c, oracle/resize_oracle.py) against the live
cv2 build, over the shapes, types and geometries of tests/cv2_cases.py.

The golden files pin the oracles on fixed shapes; this file looks for corners nobody listed: cv2's
column block width, tiny frames, 1-pixel rows and columns, rounding ties, coordinates that saturate,
horizons inside the output.  A failure message carries the whole case (and its seed).
"""
import numpy as np
import pytest

from oracle import resize_oracle as ro
from oracle import warp_oracle as wo
from tests import cv2_cases as cc
from tests import util

cv2 = pytest.importorskip("cv2")

WARP_SEED, N_WARP = 20261020, 16000
RESIZE_SEED, N_RESIZE = 20261021, 6000


def cv2_warp(src, case):
    b = list(case["border"]) + [0.0] * (4 - case["channels"])
    out = cv2.warpPerspective(src, case["H"], case["dsize"], flags=case["flags"],
                              borderMode=cv2.BORDER_CONSTANT, borderValue=b)
    return out.reshape(case["dsize"][1], case["dsize"][0], case["channels"])


def test_warp_oracle_matches_cv2():
    deviating = 0
    for case in cc.warp_cases(WARP_SEED, N_WARP):
        src = cc.warp_src(case)
        ref = cv2_warp(src, case)
        out = wo.warp_perspective(src, case["H"], case["dsize"], flags=case["flags"],
                                  borderValue=case["border"])
        if cc.nearest_deviation_applies(case["dtype"], case["flags"], case["channels"]):
            bad = cc.unexplained_nearest_deviations(out, ref, src, case["H"], case["flags"], case["border"],
                                                    case["geom"] in cc.DEGENERATE)
            assert len(bad) == 0, "oracle != cv2 beyond the documented nearest deviation at %d px " \
                "(first (y, x) %s): %s" % (len(bad), bad[:4].tolist(), cc.describe(case))
            deviating += not util.bits_equal(out, ref)
        else:
            assert util.bits_equal(out, ref), "oracle != cv2 at %d px: %s" % (
                int(np.sum(out != ref)), cc.describe(case))
    # the deviation is real (the fuzz reaches it), so the test above asserts it rather than skips it
    assert deviating > 0


def test_warp_generator_reaches_its_corners():
    cases = cc.warp_cases(WARP_SEED, N_WARP)
    seen = {(c["dtype"], c["channels"], c["flags"]) for c in cases}
    assert len(seen) == 2 * 4 * 4
    assert {c["geom"] for c in cases} == set(cc.WARP_GEOMETRIES)
    assert any(c["src_hw"] == (1, 1) for c in cases) and any(c["src_hw"] == (2, 2) for c in cases)
    assert any(c["src_hw"][0] == 1 < c["src_hw"][1] for c in cases)
    assert any(c["src_hw"][1] == 1 < c["src_hw"][0] for c in cases)
    assert any(c["dsize"][1] < 16 and c["dsize"][0] > c["bw0"] for c in cases)  # several blocks a row
    assert any(c["dsize"][0] == c["bw0"] < 1024 // min(16, c["dsize"][1]) for c in cases)
    assert any(c["dsize"][0] % 4 for c in cases)
    assert any(not np.any(c["H"]) for c in cases)  # the zero matrix


def test_resize_oracle_matches_cv2():
    for case in cc.resize_cases(RESIZE_SEED, N_RESIZE):
        src = cc.resize_src(case)
        ref = cv2.resize(src, case["dsize"]).reshape(case["dsize"][1], case["dsize"][0], case["channels"])
        out = ro.resize(src, case["dsize"])
        assert util.bits_equal(out, ref), "oracle != cv2 at %d bytes: %s" % (
            int(np.sum(out != ref)), cc.describe(case))


def test_resize_generator_reaches_its_corners():
    cases = cc.resize_cases(RESIZE_SEED, N_RESIZE)
    assert {c["kind"] for c in cases} == set(cc.RESIZE_KINDS)
    half2 = [c for c in cases if c["channels"] == 2 and c["src_hw"] == (2 * c["dsize"][1], 2 * c["dsize"][0])]
    assert len(half2) >= 20
    for k in (2, 3, 4):
        assert any(c["src_hw"] == (k * c["dsize"][1], k * c["dsize"][0]) for c in cases)
        assert any(c["src_hw"][0] == k * c["dsize"][1] and c["src_hw"][1] != k * c["dsize"][0] for c in cases)
