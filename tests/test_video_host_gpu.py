"""GPU: the host-buffer warp of video frames (bevk_warp_perspective_video_host) for every pair of
BGR, I420 and NV12 frame formats, bit for bit against cv2's own chain cvtColor -> warpPerspective ->
cvtColor.  The device workspace is filled with frames of another seed before the checked calls, so
a luma or chroma row that the upload misses shows up as wrong bytes."""
import cv2
import numpy as np
import pytest
import torch

from bev_b200 import _native, homo
from oracle import yuv420_oracle as yo

pytestmark = pytest.mark.gpu

FORMATS = ("bgr", "i420", "nv12")
PAIRS = [(s, d) for s in FORMATS for d in FORMATS]
BV = (30, 60, 200)
HORIZON = np.array([[1.0, 0.2, -3.0], [0.1, 1.1, -2.0], [0.0, 0.03, -0.5]])  # w changes sign in the BEV


def frames(fmt, n, h, w, seed):
    rng = np.random.default_rng(seed)
    if fmt == "bgr":
        return rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    return rng.integers(0, 256, (n, h * 3 // 2, w), dtype=np.uint8)


def cv2_chain(f, sfmt, dfmt, M, dsize, flags, bv=0):
    """What a cv2 user computes for one frame: decode to BGR, warp, encode."""
    bgr = {"bgr": lambda: f, "i420": lambda: cv2.cvtColor(f, cv2.COLOR_YUV2BGR_I420),
           "nv12": lambda: cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)}[sfmt]()
    b = tuple(bv) if np.ndim(bv) else (bv, bv, bv)
    bev = cv2.warpPerspective(bgr, M, dsize, flags=flags, borderMode=cv2.BORDER_CONSTANT, borderValue=b)
    if dfmt == "bgr":
        return bev
    i420 = cv2.cvtColor(bev, cv2.COLOR_BGR2YUV_I420)
    return i420 if dfmt == "i420" else yo.i420_to_nv12(i420)


def quad_map(rng, ssize, dsize, rows):
    """A forward map that takes a random quadrilateral of source rows `rows` onto the whole BEV."""
    w, _ = ssize
    y0, y1 = rows
    src = np.array([[rng.uniform(0.1, 0.4) * w, y0 + rng.uniform(0, 3)],
                    [rng.uniform(0.6, 0.9) * w, y0 + rng.uniform(0, 3)],
                    [rng.uniform(0.8, 1.0) * w, y1 - rng.uniform(0, 3)],
                    [rng.uniform(0.0, 0.2) * w, y1 - rng.uniform(0, 3)]])
    dst = np.array([[0, 0], [dsize[0], 0], [dsize[0], dsize[1]], [0, dsize[1]]], np.float64)
    return cv2.getPerspectiveTransform(src.astype(np.float32), dst.astype(np.float32))


def poison(sfmt, dfmt, n, ssize, dsize, seed):
    """Run the same shapes through the shared device workspace with frames of another seed and a
    horizon-crossing map, which uploads whole frames."""
    assert _native.warp_host_rows(ssize, dsize, HORIZON, 16) == (0, ssize[1] - 1)
    _native.warp_perspective_video_host(frames(sfmt, n, ssize[1], ssize[0], seed + 1000), HORIZON, dsize, sfmt, dfmt,
                                        flags=16)


def check(out, f, sfmt, dfmt, Ms, idx, dsize, flags, bv, what):
    for i in range(len(f)):
        M = Ms[i if idx is None and len(Ms) > 1 else (0 if idx is None else idx[i])]
        ref = cv2_chain(f[i], sfmt, dfmt, M, dsize, flags, bv)
        assert out[i].shape == ref.shape and out[i].dtype == np.uint8, (what, out[i].shape, ref.shape)
        if not np.array_equal(out[i], ref):
            bad = np.argwhere(out[i] != ref)
            pytest.fail("%s: frame %d differs from cv2 at %d positions, first %s" % (what, i, len(bad), bad[0]))


@pytest.mark.parametrize("ssize,dsize", [((480, 270), (256, 192)), ((482, 272), (130, 98))], ids=["w4", "w2"])
@pytest.mark.parametrize("flags", [0, 1])
@pytest.mark.parametrize("sfmt,dfmt", PAIRS, ids=["%s-%s" % p for p in PAIRS])
def test_every_pair_vs_cv2(sfmt, dfmt, flags, ssize, dsize):
    """All nine pairs, nearest and bilinear, widths with w % 4 == 0 (word gathers) and == 2 (bytes);
    270 rows put the I420 V plane's first row in the middle of a row."""
    rng = np.random.default_rng([ssize[0], flags, FORMATS.index(sfmt), FORMATS.index(dfmt)])
    n = 5
    f = frames(sfmt, n, ssize[1], ssize[0], rng.integers(1 << 30))
    H = quad_map(rng, ssize, dsize, (40, ssize[1] - 30))
    poison(sfmt, dfmt, n, ssize, dsize, 1)
    out = homo.warp_perspective_video_host(f, H, dsize, sfmt, dfmt, flags=flags, borderValue=BV)
    check(out, f, sfmt, dfmt, H[None], None, dsize, flags, BV, "%s -> %s flags %d" % (sfmt, dfmt, flags))
    one = homo.warp_perspective_video_host(f[2], H, dsize, sfmt, dfmt, flags=flags, borderValue=BV)
    assert np.array_equal(one, out[2])  # an unbatched frame


@pytest.mark.parametrize("sfmt,dfmt", [("i420", "i420"), ("nv12", "bgr"), ("i420", "nv12"), ("bgr", "i420")])
@pytest.mark.parametrize("n", [41, 64])
def test_matrix_tables_and_chunks(sfmt, dfmt, n):
    """Per-frame matrices, a mat_index table with more runs than one launch takes (BEVK_MAX_GROUPS,
    16) in one upload chunk, and a horizon-crossing map; 41 frames are not a multiple of the chunk."""
    ssize, dsize = (480, 270), (128, 96)
    rng = np.random.default_rng([n, FORMATS.index(sfmt), FORMATS.index(dfmt)])
    f = frames(sfmt, n, ssize[1], ssize[0], rng.integers(1 << 30))
    mats = np.stack([quad_map(rng, ssize, dsize, (20 + 7 * k, 120 + 9 * k)) for k in range(20)])
    idx = rng.permutation(np.arange(n) % 20).astype(np.int32)  # ~n runs of one frame: > 16 per chunk
    assert _native.warp_host_rows(ssize, dsize, HORIZON, 16) == (0, ssize[1] - 1)
    cases = (("per-frame matrices", np.stack([mats[i % 20] for i in range(n)]), None, 0),
             ("mat_index", mats, idx, 0), ("horizon", HORIZON[None], None, 16))
    for what, Ms, ix, inverse in cases:
        for flags in (1 | inverse, inverse):
            poison(sfmt, dfmt, n, ssize, dsize, n)
            kw = {} if ix is None else {"mat_index": ix}
            out = homo.warp_perspective_video_host(f, Ms, dsize, sfmt, dfmt, flags=flags, **kw)
            check(out, f, sfmt, dfmt, Ms, ix, dsize, flags, 0, "%s -> %s %s flags %d" % (sfmt, dfmt, what, flags))


def test_band_edges():
    """Maps whose uploaded row band starts and ends on odd and even luma rows: the chroma band
    [r0 / 2, r1 / 2] must hold the chroma rows of both ends."""
    ssize, dsize, n = (480, 270), (96, 64), 3
    seen = set()
    for k, (y0, y1) in enumerate([(40, 100), (41, 100), (40, 101), (41, 101), (42, 160), (43, 161), (44, 163)]):
        # a scaled translation onto the rows [y0, y1]: bilinear windows reach one row past each end
        M = np.array([[3.0, 0.0, 20.0], [0.0, (y1 - y0 - 1.0) / (dsize[1] - 1), y0 + 0.5], [0.0, 0.0, 1.0]])
        for flags in (17, 16):
            r0, r1 = _native.warp_host_rows(ssize, dsize, M, flags)
            assert 0 < r0 and r1 < ssize[1] - 1
            seen.add((r0 % 2, r1 % 2))
            for sfmt in ("i420", "nv12"):
                f = frames(sfmt, n, ssize[1], ssize[0], [k, flags])
                for dfmt in FORMATS:
                    poison(sfmt, dfmt, n, ssize, dsize, k)
                    out = homo.warp_perspective_video_host(f, M, dsize, sfmt, dfmt, flags=flags)
                    check(out, f, sfmt, dfmt, M[None], None, dsize, flags, 0,
                          "%s -> %s rows [%d, %d] flags %d" % (sfmt, dfmt, r0, r1, flags))
    assert seen == {(0, 0), (0, 1), (1, 0), (1, 1)}, seen


def test_pinned_pageable_and_empty():
    """Pinned CPU tensors in and out (the fast route) and pageable numpy arrays give the same bytes;
    0 frames return an empty batch."""
    ssize, dsize, n = (1920, 1080), (512, 512), 9
    H = homo.homo_from_pts(np.array([[700, 420], [1220, 420], [1900, 1060], [20, 1060]], np.float64),
                           np.array([[0, 0], [512, 0], [512, 512], [0, 512]], np.float64))
    for sfmt, dfmt in (("i420", "i420"), ("nv12", "bgr"), ("bgr", "nv12")):
        f = frames(sfmt, n, ssize[1], ssize[0], 7)
        pageable = homo.warp_perspective_video_host(f, H, dsize, sfmt, dfmt)
        src = torch.from_numpy(f).pin_memory()
        dst = torch.empty(pageable.shape, dtype=torch.uint8).pin_memory()
        assert homo.warp_perspective_video_host(src, H, dsize, sfmt, dfmt, dst=dst) is dst
        assert np.array_equal(dst.numpy(), pageable)
        for i in (0, n - 1):
            assert np.array_equal(pageable[i], cv2_chain(f[i], sfmt, dfmt, H, dsize, 1)), (sfmt, dfmt, i)
        empty = homo.warp_perspective_video_host(f[:0], H, dsize, sfmt, dfmt)
        assert empty.shape == (0,) + pageable.shape[1:]


def test_bgr_to_bgr_is_the_host_warp():
    """BGR -> BGR takes the path of warp_perspective_host and gives its bytes."""
    ssize, dsize, n = (1920, 1080), (1024, 1024), 12
    rng = np.random.default_rng(5)
    f = frames("bgr", n, ssize[1], ssize[0], 5)
    H = quad_map(rng, ssize, dsize, (400, 1060))
    for flags in (0, 1):
        a = homo.warp_perspective_video_host(f, H, dsize, "bgr", "bgr", flags=flags, borderValue=BV)
        b = _native.warp_perspective_host(f, H, dsize, flags=flags, borderValue=BV)
        assert np.array_equal(a, b), flags


@pytest.mark.parametrize("flags", [0, 1])
def test_i420_source_equals_nv12_source(flags):
    """An I420 frame and its NV12 relayout give the same BEV through every destination format."""
    ssize, dsize, n = (962, 542), (322, 242), 6
    rng = np.random.default_rng(flags)
    i420 = frames("i420", n, ssize[1], ssize[0], 11)
    nv12 = np.stack([yo.i420_to_nv12(x) for x in i420])
    H = quad_map(rng, ssize, dsize, (100, 530))
    for dfmt in FORMATS:
        a = homo.warp_perspective_video_host(i420, H, dsize, "i420", dfmt, flags=flags, borderValue=BV)
        b = homo.warp_perspective_video_host(nv12, H, dsize, "nv12", dfmt, flags=flags, borderValue=BV)
        assert np.array_equal(a, b), dfmt
