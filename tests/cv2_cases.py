"""Seeded case generators for the live-cv2 parity tests (tests/test_oracle_cv2_fuzz.py on the CPU,
tests/test_cv2_parity_gpu.py on the GPU): cv2.warpPerspective and cv2.resize at the shapes, types
and geometries where a restatement of cv2 goes wrong.

Every case is a plain dict that ``describe`` turns into a message carrying everything needed to
reproduce it (shapes, dtype, channels, flags, border, the matrix written out with repr, the seed).
Case i of a generator draws from ``np.random.default_rng([seed, i])`` only, so a case can be
regenerated on its own.
"""
import numpy as np

from oracle import warp_oracle as wo

WARP_FLAGS = (0, 1, 16, 17)
WARP_GEOMETRIES = ("perspective", "horizon", "saturate", "minify", "magnify", "singular", "shift",
                   "edge")
DEGENERATE = ("singular", "horizon")
RESIZE_KINDS = ("arbitrary", "exact_both", "exact_one_axis", "odd_next_to_half", "upscale",
                "one_pixel")


def block_width(dst_w, dst_h):
    """cv2's column block of the warp: bw0 = min(1024 / min(16, dst_h), dst_w)."""
    return min(1024 // min(16, dst_h), dst_w)


def describe(case):
    return "; ".join("%s=%r" % (k, v.tolist() if isinstance(v, np.ndarray) and k != "H" else v)
                     for k, v in case.items())


# ---------------------------------------------------------------------------------------- warp

def _src_size(rng):
    k = int(rng.integers(0, 10))
    if k == 0:
        return 1, 1
    if k == 1:
        return 2, 2
    if k == 2:
        return 1, int(rng.integers(2, 131))  # 1 x N
    if k == 3:
        return int(rng.integers(2, 131)), 1  # N x 1
    if k == 4:
        return int(rng.integers(1, 9)), int(rng.integers(1, 9))
    return int(rng.integers(1, 131)), int(rng.integers(1, 131))


def _dst_size(rng):
    """(dst_w, dst_h) that move cv2's block width around: rows shorter than 16 (bw0 = 1024 / h),
    rows narrower than one block, rows of several blocks, and tiny frames."""
    k = int(rng.integers(0, 4))
    if k == 0:
        dh = int(rng.integers(1, 16))
        dw = int(rng.integers(1, min(2 * (1024 // dh) + 8, 1400)))
    elif k == 1:
        dh, dw = int(rng.integers(16, 81)), int(rng.integers(1, 64))
    elif k == 2:
        dh, dw = int(rng.integers(16, 81)), int(rng.integers(65, 201))
    else:
        dh, dw = int(rng.integers(1, 5)), int(rng.integers(1, 5))
    if dw % 4 == 0 and rng.random() < 0.5:
        dw += 1  # widths that are not a multiple of 4
    return dw, dh


def _quad_map(frm, to):
    """3x3 projective map taking the 4 points frm to the 4 points to (float64 DLT)."""
    A, b = [], []
    for (x, y), (u, v) in zip(frm, to):
        A.append([x, y, 1, 0, 0, 0, -u * x, -u * y])
        A.append([0, 0, 0, x, y, 1, -v * x, -v * y])
        b += [u, v]
    h = np.linalg.solve(np.array(A, np.float64), np.array(b, np.float64))
    return np.append(h, 1.0).reshape(3, 3)


def _dst_corners(dw, dh):
    return np.array([[0, 0], [dw - 1, 0], [dw - 1, dh - 1], [0, dh - 1]], np.float64)


def _src_corners(sw, sh):
    return np.array([[0, 0], [sw - 1, 0], [sw - 1, sh - 1], [0, sh - 1]], np.float64)


def _dst_to_src(geom, rng, sw, sh, dw, dh):
    """dst -> src map of one geometry class (all but "singular")."""
    dc = _dst_corners(max(dw, 2), max(dh, 2))
    sc = _src_corners(max(sw, 2), max(sh, 2))
    if geom == "perspective":
        span = np.array([max(sw, 2), max(sh, 2)], np.float64)
        return _quad_map(dc, sc + rng.normal(size=(4, 2)) * span * 0.25)
    if geom == "horizon":
        M = _quad_map(dc, sc + rng.normal(size=(4, 2)) * 2.0)
        M = M / M[2, 2]
        x0, y0 = rng.uniform(0, dw), rng.uniform(0, dh)  # w changes sign through (x0, y0)
        g, h = rng.normal(size=2) / max(dw, dh)
        M[2] = [g, h, -(g * x0 + h * y0)]
        return M
    if geom == "saturate":
        s = 10.0 ** rng.uniform(4, 12) * rng.choice([-1.0, 1.0])
        M = np.diag([s, s * rng.choice([-1.0, 1.0]), 1.0]) + rng.normal(size=(3, 3)) * [[s, s, s], [s, s, s], [0, 0, 0]] * 0.1
        if rng.random() < 0.3:
            M = np.diag([1.0, 1.0, 10.0 ** -rng.uniform(6, 14)])  # tiny w: huge coordinates
            M[:2, 2] = rng.normal(size=2)
        return M
    if geom in ("minify", "magnify"):
        k = rng.uniform(5, 100) if geom == "minify" else 1.0 / rng.uniform(5, 50)
        M = np.array([[k, rng.normal() * 0.1 * k, rng.uniform(-sw, sw)],
                      [rng.normal() * 0.1 * k, k, rng.uniform(-sh, sh)],
                      [rng.normal() * 1e-3 * k / max(sw, sh), rng.normal() * 1e-3 * k / max(sw, sh), 1.0]])
        return M
    if geom == "shift":
        k = int(rng.integers(0, 4))
        tx, ty = 0.0, 0.0
        if k == 1:
            tx, ty = [float(v) for v in rng.integers(-3, 4, 2)]
        elif k == 2:
            tx, ty = [float(v) + 0.5 for v in rng.integers(-3, 3, 2)]  # exact ties
        elif k == 3:
            tx, ty = float(rng.integers(-3, 3)) + 0.5, float(rng.integers(-3, 4))
        return np.array([[1.0, 0.0, tx], [0.0, 1.0, ty], [0.0, 0.0, 1.0]])
    if geom == "edge":
        # source coordinates that land within +-0.5 px of each frame edge
        if rng.random() < 0.5:
            e = rng.uniform(-0.6, 0.6, size=(4, 2))
            return _quad_map(dc + rng.uniform(-3, 3, size=(4, 2)), _src_corners(sw, sh).astype(np.float64) + e)
        ex, ey = rng.uniform(-0.5, 0.5, 2)
        ax = (sw - 1 + 2 * ex) / max(dw - 1, 1)
        ay = (sh - 1 + 2 * ey) / max(dh - 1, 1)
        return np.array([[ax, 0.0, -ex], [0.0, ay, -ey], [0.0, 0.0, 1.0]])
    raise ValueError(geom)


def _singular(rng, ipp):
    k = int(rng.integers(0, 4))
    if k == 0 or ipp:
        return np.zeros((3, 3))
    if k == 1:
        return np.outer(rng.normal(size=3), rng.normal(size=3))  # rank 1
    M = rng.normal(size=(3, 3))
    M[2] = M[0] * rng.normal() + M[1] * rng.normal()  # rank 2 ...
    if k == 3:
        M[2] += rng.normal(size=3) * 10.0 ** -rng.uniform(6, 13)  # ... or nearly so
    return M


def _border(rng, dtype, ch):
    if rng.random() < 0.4:
        return tuple([0.0] * ch)
    if dtype == "uint8":
        vals = [float(v) for v in rng.integers(0, 256, ch)]
        if rng.random() < 0.3:  # cv2 saturates and rounds the border half to even
            vals[int(rng.integers(0, ch))] = float(rng.choice([-7.0, 300.0, 12.5, 13.5]))
        return tuple(vals)
    return tuple(float(v) for v in np.round(rng.uniform(-50, 50, ch), 2))


def warp_case(seed, i, dtypes=("uint8", "float32")):
    rng = np.random.default_rng([seed, i])
    geom = WARP_GEOMETRIES[i % len(WARP_GEOMETRIES)]
    dtype = dtypes[int(rng.integers(0, len(dtypes)))]
    ch = int(rng.integers(1, 5))
    flags = WARP_FLAGS[int(rng.integers(0, 4))]
    sh, sw = _src_size(rng)
    dw, dh = _dst_size(rng)
    if geom == "singular":
        # passed as it is, with or without WARP_INVERSE_MAP.  Only the zero matrix for the formats
        # of the nearest deviation: cv2 4.13 does not return on some near-singular float maps there.
        H = _singular(rng, nearest_deviation_applies(dtype, flags, ch))
    else:
        try:
            M = _dst_to_src(geom, rng, sw, sh, dw, dh)
            H = M if flags & 16 else np.linalg.inv(M)
        except np.linalg.LinAlgError:  # degenerate draw: fall back to the identity
            H = np.eye(3)
    return {"seed": seed, "index": i, "geom": geom, "dtype": dtype, "channels": ch,
            "src_hw": (sh, sw), "dsize": (dw, dh), "bw0": block_width(dw, dh), "flags": flags,
            "border": _border(rng, dtype, ch), "H": H}


def warp_cases(seed, count, **kw):
    return [warp_case(seed, i, **kw) for i in range(count)]


def warp_src(case, n=None, src_hw=None):
    """Seeded source frame(s) of a case: (h, w, c), or (n, h, w, c) when n is given."""
    rng = np.random.default_rng([case["seed"], case["index"], 1])
    h, w = src_hw or case["src_hw"]
    shape = (h, w, case["channels"]) if n is None else (n, h, w, case["channels"])
    if case["dtype"] == "uint8":
        return rng.integers(0, 256, shape, dtype=np.uint8)
    return rng.uniform(-100, 100, shape).astype(np.float32)


def effective_map(H, flags):
    """dst -> src map cv2 uses: H itself with WARP_INVERSE_MAP, else cv2.invert(H)."""
    return np.asarray(H, np.float64) if flags & 16 else wo.invert3x3(H)


def nearest_deviation_applies(dtype, flags, ch):
    """The one documented deviation from cv2 4.13: float (float32, and so float16) INTER_NEAREST
    warps of 1 or 4 channels, where cv2's own result depends on how it dispatches the shape."""
    return dtype in ("float32", "float16") and (flags & 7) == 0 and ch in (1, 4)


def unexplained_nearest_deviations(out, ref, src, H, flags, border, degenerate=False):
    """Pixels where ``out`` differs from cv2's ``ref`` for none of the documented reasons (with
    ``degenerate`` -- a near-singular map, or one with a horizon -- cv2 may also hold the border
    value at any pixel the project samples):
    (a) cv2 holds the border value and the continuous source coordinate lies outside
        [0, W-1] x [0, H-1] by at most half a pixel;
    (b) a source coordinate is a half-pixel tie (to 1e-6 px) and cv2 holds one of the two source
        pixels next to it, rounding exact ties half up where the project rounds half to even;
    (c) the map sends the pixel to infinity, see below.
    out / ref (h, w, c) of src's dtype, src (H, W, c); returns the (y, x) of such pixels."""
    h, w, c = ref.shape
    bits = {1: np.uint8, 2: np.uint16, 4: np.uint32}[ref.dtype.itemsize]
    diff = np.any(out.reshape(h, w, c).view(bits) != ref.view(bits), axis=2)
    if not diff.any():
        return np.zeros((0, 2), np.int64)
    bv = np.array(border, np.float64).astype(ref.dtype)
    at_border = np.all(ref == bv[None, None, :c], axis=2)
    M = effective_map(H, flags)
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float64)
    with np.errstate(all="ignore"):
        W = M[2, 0] * xs + M[2, 1] * ys + M[2, 2]
        X = (M[0, 0] * xs + M[0, 1] * ys + M[0, 2]) / W
        Y = (M[1, 0] * xs + M[1, 1] * ys + M[1, 2]) / W
    sh, sw = src.shape[:2]
    eps = 1e-6
    near = (X >= -0.5 - eps) & (X <= sw - 0.5 + eps) & (Y >= -0.5 - eps) & (Y <= sh - 0.5 + eps)
    outside = (X < 0) | (X > sw - 1) | (Y < 0) | (Y > sh - 1)
    explained = at_border & near & outside
    with np.errstate(all="ignore"):
        tie = (np.abs(X - np.floor(X) - 0.5) < eps) | (np.abs(Y - np.floor(Y) - 0.5) < eps)

        def idx(v, s, e):
            return np.clip(np.nan_to_num(np.floor(v + 0.5 + e), nan=0.0), 0, s - 1).astype(np.int64)

        either = np.zeros_like(diff)
        for ex in (-eps, eps):
            for ey in (-eps, eps):
                either |= np.all(ref.view(bits) == src.view(bits)[idx(Y, sh, ey), idx(X, sw, ex)], axis=2)
    explained |= tie & near & ~outside & either
    # (c) the map sends the pixel to infinity (w == 0): cv2 holds the border value, the project
    #     follows cv2's remap convention (coordinate 0 when w == 0) and samples pixel (0, 0)
    with np.errstate(all="ignore"):
        far = ~(np.abs(X) < 1e6) | ~(np.abs(Y) < 1e6)
    origin = np.all(out.reshape(h, w, c).view(bits) == src.view(bits)[0, 0], axis=2)
    explained |= at_border & far & origin
    if degenerate:
        explained |= at_border
    return np.argwhere(diff & ~explained)


# -------------------------------------------------------------------------------------- resize

def resize_case(seed, i, max_side=130):
    rng = np.random.default_rng([seed, i])
    kind = RESIZE_KINDS[i % len(RESIZE_KINDS)]
    ch = int(rng.integers(1, 5))

    def r(lo, hi):
        return int(rng.integers(lo, hi + 1))

    if kind == "arbitrary":
        sh, sw, dh, dw = r(1, max_side), r(1, max_side), r(1, max_side), r(1, max_side)
    elif kind == "exact_both":
        k = int(rng.choice([2, 3, 4]))
        dh, dw = r(1, max_side // k), r(1, max_side // k)
        sh, sw = k * dh, k * dw
    elif kind == "exact_one_axis":
        k = int(rng.choice([2, 3, 4]))
        dh, dw = r(1, max_side // k), r(1, max_side)
        sh, sw = k * dh, r(1, max_side)
        if rng.random() < 0.5:
            sh, sw, dh, dw = sw, sh, dw, dh
    elif kind == "odd_next_to_half":
        dh, dw = r(1, max_side // 2 - 1), r(1, max_side // 2 - 1)
        sh = 2 * dh + int(rng.choice([-1, 0, 1]))
        sw = 2 * dw + int(rng.choice([-1, 1]))
        sh = max(sh, 1)
        if rng.random() < 0.5:
            sh, sw, dh, dw = sw, sh, dw, dh
    elif kind == "upscale":
        sh, sw = r(1, 40), r(1, 40)
        dh, dw = int(sh * rng.uniform(1.0, 6.0)) + 1, int(sw * rng.uniform(1.0, 6.0)) + 1
    else:  # one_pixel
        sh, sw, dh, dw = r(1, max_side), r(1, max_side), r(1, max_side), r(1, max_side)
        which = int(rng.integers(0, 4))
        if which == 0:
            sh = 1
        elif which == 1:
            sw = 1
        elif which == 2:
            dh = 1
        else:
            dw = 1
    return {"seed": seed, "index": i, "kind": kind, "channels": ch, "src_hw": (sh, sw),
            "dsize": (dw, dh)}


def resize_cases(seed, count, **kw):
    return [resize_case(seed, i, **kw) for i in range(count)]


def resize_src(case, n=None):
    rng = np.random.default_rng([case["seed"], case["index"], 1])
    h, w = case["src_hw"]
    shape = (h, w, case["channels"]) if n is None else (n, h, w, case["channels"])
    return rng.integers(0, 256, shape, dtype=np.uint8)
