"""Seeded INTER_AREA resize cases for tests/test_oracle_resize_area.py (CPU, against live cv2) and
tests/test_resize_area_gpu.py (GPU): shapes on every branch cv2.resize takes for INTER_AREA --
integer cells (2x, 3x, 4x in one or both axes, dst == src), general downscales (non-integer
factors, odd sources next to 2x, 1-pixel dst sizes) and the bilinear emulation (upscales, and one
axis up with the other down).  Case i draws from ``np.random.default_rng([seed, i])`` only, and
``describe`` gives a failure message that carries the whole case.
"""
import numpy as np

KINDS = ("arbitrary", "integer", "downscale", "odd_next_to_half", "upscale", "mixed", "one_pixel",
         "same_size")


def describe(case):
    return "; ".join("%s=%r" % kv for kv in case.items())


def area_case(seed, i, max_side=130, nv12=False):
    """One case: src (h, w), dsize (dst_w, dst_h), channels.  nv12: even source sizes (W % 4 == 2
    included) and 3 channels."""
    rng = np.random.default_rng([seed, i])
    kind = KINDS[i % len(KINDS)]

    def r(lo, hi):
        return int(rng.integers(lo, hi + 1))

    if kind == "arbitrary":
        sh, sw, dh, dw = r(1, max_side), r(1, max_side), r(1, max_side), r(1, max_side)
    elif kind == "integer":
        kx, ky = int(rng.choice([1, 2, 3, 4])), int(rng.choice([1, 2, 3, 4]))
        dh, dw = r(1, max_side // ky), r(1, max_side // kx)
        sh, sw = ky * dh, kx * dw
    elif kind == "downscale":
        dh, dw = r(1, max_side // 2), r(1, max_side // 2)
        sh, sw = r(dh, max_side), r(dw, max_side)
    elif kind == "odd_next_to_half":
        dh, dw = r(1, max_side // 2 - 1), r(1, max_side // 2 - 1)
        sh, sw = max(1, 2 * dh + r(-1, 1)), max(1, 2 * dw + int(rng.choice([-1, 1])))
    elif kind == "upscale":
        sh, sw = r(1, 40), r(1, 40)
        dh, dw = r(sh, 5 * sh + 8), r(sw, 5 * sw + 8)
    elif kind == "mixed":
        sh, sw = r(1, max_side), r(1, max_side)
        dh, dw = r(1, sh), r(sw + 1, 2 * max_side)
        if rng.random() < 0.5:
            sh, sw, dh, dw = sw, sh, dw, dh
    elif kind == "one_pixel":
        sh, sw, dh, dw = r(1, max_side), r(1, max_side), r(1, max_side), r(1, max_side)
        which = r(0, 3)
        if which == 0:
            sh = 1
        elif which == 1:
            sw = 1
        elif which == 2:
            dh = 1
        else:
            dw = 1
    else:  # same_size
        sh, sw = r(1, max_side), r(1, max_side)
        dh, dw = sh, sw
    ch = 3 if nv12 else r(1, 4)
    if nv12:
        # even sources; the integer cases keep their factor, W % 4 == 2 half of the time
        sh, sw = 2 * ((sh + 1) // 2), 2 * ((sw + 1) // 2)
        if kind == "integer":
            sh, sw = 2 * ky * dh, 2 * kx * dw
            dh, dw = 2 * dh, 2 * dw
        elif sw % 4 == 0 and rng.random() < 0.5:
            sw += 2
    return {"seed": seed, "index": i, "kind": kind, "nv12": nv12, "channels": ch, "src_hw": (sh, sw),
            "dsize": (dw, dh)}


def area_cases(seed, count, **kw):
    return [area_case(seed, i, **kw) for i in range(count)]


def area_src(case, n=None):
    """The case's source: uint8 (h, w, c) frames, or (h * 3 / 2, w) NV12 frames; n of them if n."""
    rng = np.random.default_rng([case["seed"], case["index"], 1])
    h, w = case["src_hw"]
    one = (h * 3 // 2, w) if case["nv12"] else (h, w, case["channels"])
    return rng.integers(0, 256, one if n is None else (n,) + one, dtype=np.uint8)
