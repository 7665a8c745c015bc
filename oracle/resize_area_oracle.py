"""oracle/resize_area_oracle.py -- TEST INFRASTRUCTURE ONLY.

numpy restatement of ``cv2.resize(img, dsize, interpolation=cv2.INTER_AREA)`` for uint8 frames
with 1 to 4 channels, as OpenCV 4.13 (opencv-python-headless 4.13.0.92) computes it.  With
scale = 1 / (dsize / ssize) in double per axis, cv2 takes one of three branches:

* ``fast``: both scales >= 1 and both within DBL_EPSILON of an integer (kx, ky).  The integer sum
  s of each kx x ky cell, then saturate_cast<uchar>(s * (1.f / (kx * ky))) in float (round half to
  even).  At kx = ky = 2 with 1, 3 or 4 channels cv2's SIMD row takes (s + 2) >> 2 instead, tail
  columns included; 2 channels keep the float rule.
* ``area``: both scales >= 1 otherwise.  Per axis a table of (dst, src, alpha) entries in double
  (``axis_table``, cv2's computeResizeAreaTab): an optional partial first cell, the full cells,
  an optional partial last cell, 1e-3 thresholds, cellWidth = min(scale, ssize - fsx1).  Per
  source row buf[dx] += S[sx] * alpha in table order, then sum = beta * buf for the first source
  row of a dst row and sum += beta * buf for the others, all float32 and unfused;
  saturate_cast<uchar> (round half to even) at the end.
* ``linear``: any axis upscales.  cv2's INTER_LINEAR fixed-point machinery with the area
  coefficients sx = floor(dx * scale), fx = float((dx + 1) - (sx + 1) / scale),
  fx = 0 if fx <= 0 else fx - floor(fx); the column clamp at the last pixel, the row clip, the
  11-bit weights and the vertical pass are resize_oracle.py's.

Pinned bit for bit against live cv2 by tests/test_oracle_resize_area.py (a seeded fuzz over all
three branches) and by the cv2 hashes of tests/golden/resize_area_hash.json.  Never imported by
bev_b200/.
"""
import math

import numpy as np

from . import nv12_oracle

COEF_SCALE = 2048
DBL_EPSILON = np.finfo(np.float64).eps
f32 = np.float32


def scales(ssize, dsize):
    """(scale_x, scale_y) as cv2 computes them; ssize / dsize = (width, height)."""
    return tuple(1.0 / (float(d) / float(s)) for s, d in zip(ssize, dsize))


def branch(ssize, dsize):
    """'fast', 'area' or 'linear': the branch cv2.resize takes for INTER_AREA."""
    sx, sy = scales(ssize, dsize)
    if sx >= 1 and sy >= 1:
        fast = all(abs(s - int(math.floor(s + 0.5))) < DBL_EPSILON for s in (sx, sy))
        return "fast" if fast else "area"
    return "linear"


def axis_table(ssize, dsize, scale):
    """computeResizeAreaTab: (dst index, src index, float32 alpha) arrays in cv2's table order."""
    di, si, al = [], [], []
    for d in range(dsize):
        fs1 = d * scale
        fs2 = fs1 + scale
        cw = min(scale, ssize - fs1)
        s1, s2 = math.ceil(fs1), math.floor(fs2)
        s2 = min(s2, ssize - 1)
        s1 = min(s1, s2)
        if s1 - fs1 > 1e-3:
            di.append(d), si.append(s1 - 1), al.append(f32((s1 - fs1) / cw))
        for s in range(s1, s2):
            di.append(d), si.append(s), al.append(f32(1.0 / cw))
        if fs2 - s2 > 1e-3:
            di.append(d), si.append(s2), al.append(f32(min(min(fs2 - s2, 1.0), cw) / cw))
    return np.array(di, np.int64), np.array(si, np.int64), np.array(al, f32)


def _padded(table, dsize):
    """The table as (dsize, n) src index / alpha arrays, entries in table order; unused slots
    have alpha 0 (adding S * 0 = +0 leaves a float32 sum unchanged)."""
    di, si, al = table
    counts = np.bincount(di, minlength=dsize)
    n = int(counts.max())
    idx = np.zeros((dsize, n), np.int64)
    alpha = np.zeros((dsize, n), f32)
    first = np.concatenate([[0], np.cumsum(counts)[:-1]])
    slot = np.arange(len(di)) - first[di]
    idx[di, slot] = si
    alpha[di, slot] = al
    # unused slots repeat the last source index so every gather stays inside the image
    for k in range(1, n):
        unused = k >= counts
        idx[unused, k] = idx[unused, k - 1]
    return idx, alpha


def _area(px, dsize):
    h, w, _ = px.shape
    dw, dh = dsize
    sx, sy = scales((w, h), dsize)
    xi, xa = _padded(axis_table(w, dw, sx), dw)
    yi, ya = _padded(axis_table(h, dh, sy), dh)
    p = px.astype(f32)
    buf = np.zeros((h, dw, px.shape[2]), f32)
    for k in range(xi.shape[1]):
        buf = buf + p[:, xi[:, k]] * xa[None, :, k, None]
    out = ya[:, 0, None, None] * buf[yi[:, 0]]
    for k in range(1, yi.shape[1]):
        out = out + ya[:, k, None, None] * buf[yi[:, k]]
    return np.clip(np.rint(out), 0, 255).astype(np.uint8)


def _fast(px, dsize):
    h, w, c = px.shape
    dw, dh = dsize
    kx, ky = w // dw, h // dh
    s = px.astype(np.int64).reshape(dh, ky, dw, kx, c).sum(axis=(1, 3))
    if kx == 2 and ky == 2 and c != 2:
        return ((s + 2) >> 2).astype(np.uint8)
    r = s.astype(f32) * (f32(1) / f32(kx * ky))
    return np.clip(np.rint(r), 0, 255).astype(np.uint8)


def linear_axis(ssize, dsize, scale, clamp):
    """(index, w0, w1) per dst position of cv2's bilinear emulation of INTER_AREA."""
    inv = float(dsize) / float(ssize)
    d = np.arange(dsize)
    s = np.floor(d * scale).astype(np.int64)
    f = ((d + 1) - (s + 1) * inv).astype(f32)
    f = np.where(f <= 0, f32(0), (f - np.floor(f)).astype(f32)).astype(f32)
    if clamp:
        hi = s >= ssize - 1
        f[hi] = 0
        s[hi] = ssize - 1
    w1 = np.rint(f * f32(COEF_SCALE)).astype(np.int64)
    w0 = np.rint((f32(1) - f) * f32(COEF_SCALE)).astype(np.int64)
    return s, w0, w1


def _linear(px, dsize):
    h, w, _ = px.shape
    dw, dh = dsize
    scx, scy = scales((w, h), dsize)
    sx, a0, a1 = linear_axis(w, dw, scx, True)
    sy, b0, b1 = linear_axis(h, dh, scy, False)
    p = px.astype(np.int64)
    rows = p[:, sx] * a0[None, :, None] + p[:, np.minimum(sx + 1, w - 1)] * a1[None, :, None]
    s0, s1 = rows[np.clip(sy, 0, h - 1)], rows[np.clip(sy + 1, 0, h - 1)]
    out = (((b0[:, None, None] * (s0 >> 4)) >> 16) + ((b1[:, None, None] * (s1 >> 4)) >> 16) + 2) >> 2
    return out.astype(np.uint8)


def resize(img, dsize):
    """cv2.resize(img, dsize, interpolation=cv2.INTER_AREA) for uint8 (H, W) or (H, W, C);
    dsize = (width, height)."""
    img = np.asarray(img)
    assert img.dtype == np.uint8
    squeeze = img.ndim == 2
    px = img[:, :, None] if squeeze else img
    dsize = (int(dsize[0]), int(dsize[1]))
    kind = branch((px.shape[1], px.shape[0]), dsize)
    out = {"fast": _fast, "area": _area, "linear": _linear}[kind](px, dsize)
    return out[:, :, 0] if squeeze else out


def resize_nv12(f, dsize):
    """cv2.resize(cv2.cvtColor(f, COLOR_YUV2BGR_NV12), dsize, interpolation=INTER_AREA) of one
    (H*3/2, W) NV12 frame."""
    return resize(nv12_oracle.nv12_to_bgr(f), dsize)


def _touched_axes(ssize, dsize):
    """Per axis, a bool mask of the source positions a tap with a non-zero weight reads."""
    masks = []
    scs = scales(ssize, dsize)
    kind = branch(ssize, dsize)
    for axis in range(2):
        n, dn, sc = int(ssize[axis]), int(dsize[axis]), scs[axis]
        m = np.zeros(n, bool)
        if kind == "fast":
            m[:dn * int(round(sc))] = True
        elif kind == "area":
            _, si, al = axis_table(n, dn, sc)
            m[si[al != 0]] = True
        else:
            s, w0, w1 = linear_axis(n, dn, sc, axis == 0)
            m[np.clip(s, 0, n - 1)[w0 != 0]] = True
            m[np.clip(s + 1, 0, n - 1)[w1 != 0]] = True
        masks.append(m)
    return masks


def touched_pixels(ssize, dsize):
    """Distinct source pixels the resize reads (for the benchmark's algorithmic bytes)."""
    cols, rows = _touched_axes(ssize, dsize)
    return int(cols.sum()) * int(rows.sum())


def touched_samples_nv12(ssize, dsize):
    """(luma, chroma): distinct luma pixels the resize reads and the distinct U,V pairs they use."""
    cols, rows = _touched_axes(ssize, dsize)
    luma = int(cols.sum()) * int(rows.sum())
    chroma = int(cols.reshape(-1, 2).any(1).sum()) * int(rows.reshape(-1, 2).any(1).sum())
    return luma, chroma
