"""oracle/resize_oracle.py -- TEST INFRASTRUCTURE ONLY.

numpy restatement of ``cv2.resize(img, (new_u, new_v))`` (default INTER_LINEAR, uint8) as the
reference calls it for the small-frame path (/root/reference/vis_homo.py:90, next to the warp at
:91 whose homography comes from ``Calib.scale(align_corners=False)``, bev/calib.py:142-198).

The arithmetic lives in OpenCV (third party, unpinned by the reference; this image resolves it to
opencv-python-headless 4.13.0.92); its published algorithm for 8-bit bilinear resize is:

* per dst column: fx = float((dx + 0.5) * scale_x - 0.5) with scale_x = 1 / (dst_w / src_w) in
  double; sx = floor(fx); fx -= sx; columns left of the image take (sx, fx) = (0, 0), columns at
  or right of the last pixel (src_w - 1, 0); weights short(rint((1 - fx) * 2048)),
  short(rint(fx * 2048)), computed in float.
* per dst row the same formula WITHOUT that clamp: the weights keep their fraction and the two
  row indices sy, sy + 1 are clipped into the image instead.
* horizontal pass in int: S = p[sx] * a0 + p[sx + 1] * a1; vertical pass
  ((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2.
* one exception: 2-channel frames downscaled by exactly 2 in both axes take the round-half-even
  mean of each 2x2 block (``half_mean_2x2``).

Pinned bit-for-bit against cv2 4.13.0.92 in the build container by oracle/gen_golden.py (all
shapes of tests/golden/resize_kat.json: the generator asserts equality before it stores cv2's
hashes) and on the fixtures by tests/test_oracle_resize.py.  Never imported by bev_b200/.
"""
import numpy as np

COEF_BITS = 11
COEF_SCALE = 1 << COEF_BITS


def axis_coefficients(ssize, dsize, clamp):
    """(index, w0, w1) per dst position along one axis; ``clamp`` = the x-axis border rule."""
    scale = 1.0 / (float(dsize) / float(ssize))
    d = np.arange(dsize, dtype=np.float64)
    f = ((d + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int32)
    f = (f - s.astype(np.float32)).astype(np.float32)
    if clamp:
        lo = s < 0
        f[lo] = 0
        s[lo] = 0
        hi = s >= ssize - 1
        f[hi] = 0
        s[hi] = ssize - 1
    w1 = np.rint(f * np.float32(COEF_SCALE)).astype(np.int32)
    w0 = np.rint((np.float32(1) - f) * np.float32(COEF_SCALE)).astype(np.int32)
    return s, w0, w1


def resize(img, dsize):
    """cv2.resize(img, dsize) for uint8 (H, W) or (H, W, C); dsize = (width, height)."""
    img = np.asarray(img)
    assert img.dtype == np.uint8
    squeeze = img.ndim == 2
    if squeeze:
        img = img[:, :, None]
    h, w, c = img.shape
    dw, dh = int(dsize[0]), int(dsize[1])
    if c == 2 and w == 2 * dw and h == 2 * dh:
        out = half_mean_2x2(img)
        return out[:, :, 0] if squeeze else out
    sx, a0, a1 = axis_coefficients(w, dw, True)
    sy, b0, b1 = axis_coefficients(h, dh, False)
    px = img.astype(np.int32)
    sx1 = np.minimum(sx + 1, w - 1)
    r0, r1 = np.clip(sy, 0, h - 1), np.clip(sy + 1, 0, h - 1)
    rows = px[:, sx] * a0[None, :, None] + px[:, sx1] * a1[None, :, None]
    s0, s1 = rows[r0], rows[r1]
    out = (((b0[:, None, None] * (s0 >> 4)) >> 16) + ((b1[:, None, None] * (s1 >> 4)) >> 16) + 2) >> 2
    out = out.astype(np.uint8)
    return out[:, :, 0] if squeeze else out


def half_mean_2x2(img):
    """cv2 sends an exact 2x downscale in both axes to INTER_AREA; for 2-channel uint8 frames that
    gives the mean of each 2x2 block rounded half to even.  (For 1, 3 and 4 channels it gives
    (a + b + c + d + 2) >> 2, which the bilinear formula above already equals.)"""
    p = img.astype(np.int32)
    s = p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2]
    q, r = s >> 2, s & 3
    return (q + ((r > 2) | ((r == 2) & ((q & 1) == 1)))).astype(np.uint8)


def touched_pixels(ssize, dsize):
    """Distinct source pixels any tap with a non-zero weight reads (for the roofline)."""
    w, h = ssize
    sx, a0, a1 = axis_coefficients(w, dsize[0], True)
    sy, b0, b1 = axis_coefficients(h, dsize[1], False)
    cols = np.zeros(w, bool)
    cols[sx[a0 != 0]] = True
    cols[np.minimum(sx + 1, w - 1)[a1 != 0]] = True
    rows = np.zeros(h, bool)
    rows[np.clip(sy, 0, h - 1)[b0 != 0]] = True
    rows[np.clip(sy + 1, 0, h - 1)[b1 != 0]] = True
    return int(cols.sum()) * int(rows.sum())
