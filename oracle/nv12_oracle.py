"""oracle/nv12_oracle.py -- TEST INFRASTRUCTURE ONLY.

numpy restatement of ``cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)`` (cv2 4.13): BT.601 limited range
in 20-bit fixed point, chroma replicated over each 2x2 luma block.  Pinned against live cv2 and
against the cv2 hashes of tests/golden/nv12_hash.json by tests/test_oracle_nv12.py.  A warp of an
NV12 frame is ``warp_oracle.warp_perspective(nv12_to_bgr(f), ...)``, which is what cv2 computes
when it is handed the converted frame.

Also the host-side coordinate map of the warp (the dst->src arithmetic of warp_oracle.c, in
unfused float64 numpy) for counting the luma and chroma samples a warp touches.
"""
import numpy as np

COLOR_YUV2BGR_NV12 = 91

# 20-bit fixed-point BT.601 limited-range coefficients (cv2 4.13)
_CY, _CVR, _CVG, _CUG, _CUB = 1220542, 1673527, -852492, -409993, 2116026
_HALF = 1 << 19


def seeded_nv12(seed, h, w):
    """Seeded uniform-noise NV12 frame: (h * 3 / 2, w) uint8, h and w even."""
    rng = np.random.default_rng(seed)
    return rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)


def all_triples_nv12():
    """One 4096 x 4096 NV12 frame holding each of the 2^24 (Y, U, V) triples once: chroma sample
    k (row-major) carries the pair (U, V) = divmod(k // 64, 256), and its 2x2 luma block the four
    Y values 4 * (k % 64) .. 4 * (k % 64) + 3."""
    k = np.arange(2048 * 2048, dtype=np.int64).reshape(2048, 2048)
    pair, j = k // 64, k % 64
    uv = np.stack([pair >> 8, pair & 255], -1).astype(np.uint8).reshape(2048, 4096)
    Y = np.empty((4096, 4096), np.uint8)
    for dy in range(2):
        for dx in range(2):
            Y[dy::2, dx::2] = 4 * j + 2 * dy + dx
    return np.concatenate([Y, uv])


def yuv_to_bgr(Y, U, V):
    """Per-sample conversion of broadcastable uint8 arrays -> (..., 3) uint8 BGR."""
    y = np.maximum(Y.astype(np.int64) - 16, 0) * _CY
    u = U.astype(np.int64) - 128
    v = V.astype(np.int64) - 128
    r = (y + _CVR * v + _HALF) >> 20
    g = (y + _CVG * v + _CUG * u + _HALF) >> 20
    b = (y + _CUB * u + _HALF) >> 20
    return np.clip(np.stack([b, g, r], -1), 0, 255).astype(np.uint8)


def nv12_to_bgr(f):
    """(H * 3 / 2, W) NV12 frame, H and W even -> (H, W, 3) BGR, byte-identical to cv2."""
    f = np.asarray(f)
    rows, w = f.shape
    h = rows * 2 // 3
    if f.dtype != np.uint8 or rows % 3 or rows == 0 or w % 2:
        raise ValueError("NV12 frame must be uint8 (H*3/2, W) with H, W even, got %s %s" % (f.dtype, f.shape))
    Y = f[:h]
    uv = f[h:].reshape(h // 2, w // 2, 2)
    U = np.repeat(np.repeat(uv[:, :, 0], 2, 0), 2, 1)
    V = np.repeat(np.repeat(uv[:, :, 1], 2, 0), 2, 1)
    return yuv_to_bgr(Y, U, V)


def _invert3x3(H):
    """cv2.invert's adjugate order (warp_oracle.invert3x3 without the compiled library)."""
    (a00, a01, a02), (a10, a11, a12), (a20, a21, a22) = np.asarray(H, np.float64).reshape(3, 3)
    d = a00 * (a11 * a22 - a12 * a21) - a01 * (a10 * a22 - a12 * a20) + a02 * (a10 * a21 - a11 * a20)
    if d == 0.0:
        return np.zeros((3, 3))
    d = 1.0 / d
    return np.array([[(a11 * a22 - a12 * a21) * d, (a02 * a21 - a01 * a22) * d, (a01 * a12 - a02 * a11) * d],
                     [(a12 * a20 - a10 * a22) * d, (a00 * a22 - a02 * a20) * d, (a02 * a10 - a00 * a12) * d],
                     [(a10 * a21 - a11 * a20) * d, (a01 * a20 - a00 * a21) * d, (a00 * a11 - a01 * a10) * d]])


def coord_map(dsize, M, flags=1):
    """Quantised source coordinates (X, Y) of every dst pixel, int arrays (dh, dw): 1/32 px for
    bilinear, whole pixels for nearest.  cv2's block-column split and evaluation order; numpy
    float64 operations are never fused, so this equals the device arithmetic."""
    dw, dh = int(dsize[0]), int(dsize[1])
    Mi = np.asarray(M, np.float64).reshape(3, 3) if flags & 16 else _invert3x3(M)
    bh0 = min(16, dh)
    bw0 = min(1024 // bh0, dw)
    x = np.arange(dw)
    xb = ((x // bw0) * bw0).astype(np.float64)[None, :]
    x1 = (x - (x // bw0) * bw0).astype(np.float64)[None, :]
    y = np.arange(dh, dtype=np.float64)[:, None]
    m = Mi.reshape(-1)
    X0 = m[0] * xb + m[1] * y + m[2]
    Y0 = m[3] * xb + m[4] * y + m[5]
    W0 = m[6] * xb + m[7] * y + m[8]
    w = W0 + m[6] * x1
    scale = 32.0 if (flags & 7) == 1 else 1.0
    with np.errstate(divide="ignore", invalid="ignore"):
        w = np.where(w != 0.0, scale / np.where(w != 0.0, w, 1.0), 0.0)
    X = np.clip((X0 + m[0] * x1) * w, -2147483648.0, 2147483647.0)
    Y = np.clip((Y0 + m[3] * x1) * w, -2147483648.0, 2147483647.0)
    return np.rint(X).astype(np.int64), np.rint(Y).astype(np.int64)


def touched_samples(ssize, dsize, M, flags=1):
    """(luma, chroma): distinct in-frame luma pixels the warp's taps reference (4 bilinear, 1
    nearest) and the distinct chroma samples (U,V pairs) those pixels use."""
    sw, sh = int(ssize[0]), int(ssize[1])
    X, Y = coord_map(dsize, M, flags)
    linear = (flags & 7) == 1
    sx = np.clip(X >> 5 if linear else X, -32768, 32767).reshape(-1)
    sy = np.clip(Y >> 5 if linear else Y, -32768, 32767).reshape(-1)
    nt = 2 if linear else 1
    luma = np.zeros((sh, sw), bool)
    for j in range(nt):
        for i in range(nt):
            u, v = sx + i, sy + j
            ok = (u >= 0) & (u < sw) & (v >= 0) & (v < sh)
            luma[v[ok], u[ok]] = True
    chroma = luma.reshape(sh // 2, 2, sw // 2, 2).any(axis=(1, 3))
    return int(luma.sum()), int(chroma.sum())
