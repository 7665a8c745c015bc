"""CPU: what the one-pass host video call with small frames (bevk_warp_perspective_video_host_small)
relies on and rejects without a GPU: the I420 resize equals the pinned NV12 resize oracles of the
I420 frame's NV12 relayout, and the C entry point and its Python binding refuse bad formats, shapes,
matrix tables, interpolations and small sizes before looking for a device."""
import ctypes

import cv2
import numpy as np
import pytest

from bev_b200 import _native, homo
from oracle import resize_area_oracle as ra
from oracle import resize_nv12_oracle as rno
from oracle import yuv420_oracle as yo

BGR, I420, NV12 = 2, 0, 1

# (h, w) of the I420 source, (dst_w, dst_h)
SHAPES = [
    ((1080, 1920), (852, 480)),   # the small frame of vis_homo.py:90, non-integer cells
    ((1080, 1920), (960, 540)),   # exact 2x
    ((1080, 1920), (640, 360)),   # integer 3x cells
    ((720, 1280), (320, 180)),    # integer 4x cells
    ((480, 852), (1920, 1080)),   # upscale
    ((270, 478), (239, 135)),     # exact 2x, W % 4 == 2
    ((34, 66), (22, 11)),         # integer 3x cells, W % 4 == 2
    ((60, 90), (36, 24)),         # 2.5x cells
    ((272, 482), (130, 98)),      # non-integer cells, W % 4 == 2
    ((540, 962), (481, 270)),
    ((96, 130), (1, 1)),          # 1-pixel dst axes
    ((96, 130), (130, 1)),
    ((96, 130), (1, 96)),
    ((2, 2), (1, 1)),
    ((2, 2), (7, 5)),
    ((4, 6), (1, 9)),
    ((64, 32), (16, 64)),         # one axis up, one down
    ((32, 64), (200, 17)),
    ((18, 10), (10, 18)),
    ((100, 200), (400, 50)),
]


@pytest.mark.parametrize("interp", [cv2.INTER_LINEAR, cv2.INTER_AREA], ids=["linear", "area"])
@pytest.mark.parametrize("hw,dsize", SHAPES, ids=lambda v: "x".join(map(str, v)))
def test_i420_resize_is_the_nv12_oracle_of_its_relayout(hw, dsize, interp):
    """The GPU tests hold the I420 resize to live cv2; this pins the reasoning behind the kernel:
    cv2.resize of an I420 frame's BGR equals the pinned NV12 oracle of the same frame as NV12."""
    h, w = hw
    f = np.random.default_rng([h, w, dsize[0], dsize[1]]).integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
    ref = cv2.resize(cv2.cvtColor(f, cv2.COLOR_YUV2BGR_I420), dsize, interpolation=interp)
    oracle = rno.resize_nv12 if interp == cv2.INTER_LINEAR else ra.resize_nv12
    got = oracle(yo.i420_to_nv12(f), dsize)
    assert got.shape == ref.shape and np.array_equal(got, ref)


def _call(src_fmt=I420, dst_fmt=I420, n=2, sh=8, sw=8, dh=4, dw=4, smh=4, smw=4, n_mats=1, idx=None, flags=1,
          interp=1, bm=0, null=()):
    lib = _native.lib()
    M = np.tile(np.eye(3), (max(n_mats, 1), 1, 1))
    b = np.zeros(4)
    buf = ctypes.create_string_buffer(4096)
    ptr = {k: (None if k in null else buf) for k in ("src", "dst", "small", "dst_small")}
    ip = None
    if idx is not None:
        idx = np.asarray(idx, np.int32)
        ip = idx.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
    dp = M.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    rc = lib.bevk_warp_perspective_video_host_small(
        ptr["src"], src_fmt, ptr["dst"], dst_fmt, ptr["small"], ptr["dst_small"], n, sh, sw, dh, dw, smh, smw, dp,
        None if "M_small" in null else dp, n_mats, ip, flags, interp, bm,
        b.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
    return rc, lib.bevk_last_error().decode()


@pytest.mark.parametrize("kw,msg", [
    (dict(src_fmt=3), "formats"),
    (dict(dst_fmt=-1), "formats"),
    (dict(src_fmt=I420, sh=7), "even"),
    (dict(src_fmt=NV12, sw=9), "even"),
    (dict(src_fmt=BGR, dst_fmt=I420, dh=5), "even"),
    (dict(src_fmt=BGR, dst_fmt=NV12, dw=3), "even"),
    (dict(n_mats=3, idx=[0, 3]), "mat_index"),
    (dict(n_mats=3, idx=[-1, 0]), "mat_index"),
    (dict(n_mats=3), "mat_index"),
    (dict(bm=1), "BORDER_CONSTANT"),
    (dict(flags=2), "INTER_"),
    (dict(n=-1), "n_frames"),
    (dict(src_fmt=NV12, sh=4000, sw=1000000), "4 GB"),
    (dict(interp=0), "INTER_AREA"),
    (dict(interp=2), "INTER_AREA"),
    (dict(smh=0), "positive"),
    (dict(smw=-4), "positive"),
    (dict(smh=32768), "32767"),
    (dict(smw=32768), "32767"),
    (dict(null=("M_small",)), "M_small"),
    (dict(null=("small",)), "small"),
    (dict(null=("dst_small",)), "dst_small"),
    (dict(null=("src",)), "null"),
    (dict(null=("dst",)), "null"),
])
def test_c_argument_errors(kw, msg):
    """Every rejection returns BEVK_E_ARG (-1) with a message, on a machine without a GPU too."""
    rc, err = _call(**kw)
    assert rc == -1, (kw, rc, err)
    assert msg in err, (kw, err)
    assert "warp_video_host_small" in err or "warp:" in err, err


def test_empty_batch_and_odd_sizes_on_bgr_sides():
    """0 frames need no output buffers; BGR sides and the small frames take odd sizes."""
    rc, err = _call(src_fmt=BGR, dst_fmt=BGR, n=0, sh=7, sw=9, dh=5, dw=3, smh=3, smw=5,
                    null=("src", "dst", "small", "dst_small"))
    assert rc in (0, -3), err  # BEVK_OK, or BEVK_E_NOGPU without a device


def test_python_validation():
    H = np.eye(3)
    i420 = np.zeros((12, 8), np.uint8)
    bgr = np.zeros((8, 8, 3), np.uint8)
    f = homo.warp_perspective_video_host_small
    with pytest.raises(ValueError, match="src_format"):
        f(i420, H, H, (4, 4), (4, 2), "yuv420p", "i420")
    with pytest.raises(ValueError, match="dst_format"):
        f(i420, H, H, (4, 4), (4, 2), "i420", "rgb")
    with pytest.raises(ValueError, match="H\\*3/2 rows"):
        f(np.zeros((13, 8), np.uint8), H, H, (4, 4), (4, 2), "i420", "i420")
    with pytest.raises(ValueError, match="\\(H, W, 3\\)"):
        f(i420, H, H, (4, 4), (4, 2), "bgr", "i420")
    with pytest.raises(ValueError, match="uint8"):
        f(i420.astype(np.float32), H, H, (4, 4), (4, 2), "i420", "i420")
    with pytest.raises(ValueError, match="even width and height"):
        f(bgr, H, H, (5, 4), (4, 2), "bgr", "nv12")
    with pytest.raises(ValueError, match="interpolation"):
        f(bgr, H, H, (4, 4), (4, 2), "bgr", "bgr", interpolation=0)
    with pytest.raises(ValueError, match="M_small"):
        f(np.zeros((2, 12, 8), np.uint8), np.stack([H] * 2), H, (4, 4), (4, 2), "i420", "i420")
    with pytest.raises(ValueError, match="mat_index"):
        f(np.zeros((2, 12, 8), np.uint8), np.stack([H] * 3), np.stack([H] * 3), (4, 4), (4, 2), "i420", "nv12")
    with pytest.raises(ValueError, match="small must be"):
        f(bgr, H, H, (4, 4), (4, 2), "bgr", "bgr", small=np.zeros((4, 4, 3), np.uint8))
    with pytest.raises(ValueError, match="dst_small must be"):
        f(bgr, H, H, (4, 4), (4, 2), "bgr", "i420", dst_small=np.zeros((4, 4, 3), np.uint8))
    with pytest.raises(ValueError, match="dst must be"):
        f(bgr, H, H, (4, 4), (4, 2), "bgr", "i420", dst=np.zeros((4, 4, 3), np.uint8))
