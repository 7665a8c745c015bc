"""oracle/yuv420_oracle.py -- TEST INFRASTRUCTURE ONLY.

numpy restatement of ``cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)`` (cv2 4.13): BT.601 limited
range in 20-bit fixed point.  Luma is computed per pixel; the U and V of each 2x2 block come from
its top-left pixel alone (cv2 does not average the block).  The result is an (H * 3 / 2, W) uint8
array: H rows of Y, then the (H/2, W/2) U plane packed row-major into the next H/4 rows, then V the
same way.  NV12 holds the same Y rows followed by H/2 rows of interleaved U, V bytes.  Pinned
against live cv2 and against the cv2 hashes of tests/golden/yuv420_hash.json by
tests/test_oracle_yuv420.py.
"""
import numpy as np

COLOR_BGR2YUV_I420 = 128

# 20-bit fixed-point BT.601 limited-range coefficients of cv2's RGB -> YUV 4:2:0 conversion
_CRY, _CGY, _CBY = 269484, 528482, 102760
_CRU, _CGU, _CBU = -155188, -305135, 460324
_CRV, _CGV, _CBV = 460324, -385875, -74448
_HALF = 1 << 19


def _check(bgr):
    bgr = np.asarray(bgr)
    if bgr.dtype != np.uint8 or bgr.ndim != 3 or bgr.shape[2] != 3 or bgr.shape[0] % 2 or bgr.shape[1] % 2 \
            or bgr.size == 0:
        raise ValueError("BGR frame must be uint8 (H, W, 3) with H, W even, got %s %s" % (bgr.dtype, bgr.shape))
    return bgr


def _planes(bgr):
    """(Y (H, W), U (H/2, W/2), V (H/2, W/2)) uint8 planes of a BGR frame."""
    b, g, r = (bgr[..., c].astype(np.int64) for c in range(3))
    y = (_CRY * r + _CGY * g + _CBY * b + _HALF + (16 << 20)) >> 20
    tl = (slice(0, None, 2), slice(0, None, 2))  # the top-left pixel of every 2x2 block
    u = (_CRU * r[tl] + _CGU * g[tl] + _CBU * b[tl] + _HALF + (128 << 20)) >> 20
    v = (_CRV * r[tl] + _CGV * g[tl] + _CBV * b[tl] + _HALF + (128 << 20)) >> 20
    return tuple(np.clip(p, 0, 255).astype(np.uint8) for p in (y, u, v))


def bgr_to_i420(bgr):
    """(H, W, 3) BGR, H and W even -> (H * 3 / 2, W) I420, byte-identical to cv2."""
    bgr = _check(bgr)
    h, w = bgr.shape[:2]
    y, u, v = _planes(bgr)
    return np.concatenate([y.reshape(-1), u.reshape(-1), v.reshape(-1)]).reshape(h * 3 // 2, w)


def bgr_to_nv12(bgr):
    """(H, W, 3) BGR, H and W even -> (H * 3 / 2, W) NV12: the Y rows of bgr_to_i420, then H/2 rows
    of interleaved U, V."""
    bgr = _check(bgr)
    h, w = bgr.shape[:2]
    y, u, v = _planes(bgr)
    return np.concatenate([y, np.stack([u, v], -1).reshape(h // 2, w)])


def i420_to_nv12(f):
    """Relayout of an (H * 3 / 2, W) I420 frame as NV12 (same bytes, chroma interleaved)."""
    f = np.asarray(f)
    rows, w = f.shape
    h = rows // 3 * 2
    c = f[h:].reshape(-1)
    u, v = c[:c.size // 2], c[c.size // 2:]
    return np.concatenate([f[:h], np.stack([u, v], -1).reshape(h // 2, w)])


def convert(bgr, layout):
    """bgr_to_i420 or bgr_to_nv12 by name ("i420" / "nv12")."""
    return {"i420": bgr_to_i420, "nv12": bgr_to_nv12}[layout](bgr)


def all_triples_bgr(r0=0, rows=4096):
    """2x2-block rows r0 .. r0 + rows - 1 of an 8192 x 8192 BGR image in which the 2^24 (B, G, R)
    triples each fill one 2x2 block (so every triple is also a chroma sample): block k (row-major)
    holds the triple (k >> 16, (k >> 8) & 255, k & 255)."""
    k = np.arange(r0 * 4096, (r0 + rows) * 4096, dtype=np.int64).reshape(rows, 4096)
    px = np.stack([k >> 16, (k >> 8) & 255, k & 255], -1).astype(np.uint8)
    return np.repeat(np.repeat(px, 2, 0), 2, 1)


def touched(n, h, w, bgr_in=True):
    """Algorithmic bytes of a conversion of n frames of h x w: 3 bytes/pixel read (BGR) and 1.5
    bytes/pixel written (YUV 4:2:0)."""
    return n * h * w * (3 if bgr_in else 0) + n * h * w * 3 // 2
