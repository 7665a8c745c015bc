"""CPU: what the host-buffer video warp (bevk_warp_perspective_video_host) relies on and rejects
without a GPU: cv2 converts I420 and NV12 with one arithmetic, and the C entry point and its Python
binding refuse bad formats, shapes, matrix tables and border modes before looking for a device."""
import ctypes

import cv2
import numpy as np
import pytest

from bev_b200 import _native, homo
from oracle import yuv420_oracle as yo

BGR, I420, NV12 = 2, 0, 1


@pytest.mark.parametrize("h,w", [(1080, 1920), (480, 852), (34, 66), (6, 10), (2, 2)])
def test_cv2_i420_and_nv12_conversions_agree(h, w):
    """An I420 frame differs from its NV12 relayout only in where the chroma bytes sit, so the NV12
    arithmetic of the kernels serves I420 sources unchanged."""
    rng = np.random.default_rng([h, w])
    f = rng.integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
    a = cv2.cvtColor(f, cv2.COLOR_YUV2BGR_I420)
    b = cv2.cvtColor(yo.i420_to_nv12(f), cv2.COLOR_YUV2BGR_NV12)
    assert a.tobytes() == b.tobytes()


def _call(src_fmt=I420, dst_fmt=I420, n=2, sh=8, sw=8, dh=4, dw=4, n_mats=1, idx=None, flags=1, bm=0):
    lib = _native.lib()
    M = np.tile(np.eye(3), (max(n_mats, 1), 1, 1))
    b = np.zeros(4)
    buf = ctypes.create_string_buffer(4096)
    ip = None
    if idx is not None:
        idx = np.asarray(idx, np.int32)
        ip = idx.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
    rc = lib.bevk_warp_perspective_video_host(buf, src_fmt, buf, dst_fmt, n, sh, sw, dh, dw,
                                              M.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), n_mats, ip, flags,
                                              bm, b.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
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
])
def test_c_argument_errors(kw, msg):
    """Every rejection returns BEVK_E_ARG (-1) with a message, on a machine without a GPU too."""
    rc, err = _call(**kw)
    assert rc == -1, (kw, rc, err)
    assert msg in err, (kw, err)


def test_odd_sizes_are_fine_on_bgr_sides():
    """Only YUV sides need even sizes: BGR -> BGR with odd sizes passes the checks (and then needs a
    device, or has no frames to warp)."""
    rc, err = _call(src_fmt=BGR, dst_fmt=BGR, n=0, sh=7, sw=9, dh=5, dw=3)
    assert rc in (0, -3), err  # BEVK_OK, or BEVK_E_NOGPU without a device


def test_python_validation():
    H = np.eye(3)
    i420 = np.zeros((12, 8), np.uint8)
    bgr = np.zeros((8, 8, 3), np.uint8)
    with pytest.raises(ValueError, match="src_format"):
        homo.warp_perspective_video_host(i420, H, (4, 4), "yuv420p", "i420")
    with pytest.raises(ValueError, match="dst_format"):
        homo.warp_perspective_video_host(i420, H, (4, 4), "i420", "rgb")
    with pytest.raises(ValueError, match="H\\*3/2 rows"):
        homo.warp_perspective_video_host(np.zeros((13, 8), np.uint8), H, (4, 4), "i420", "i420")
    with pytest.raises(ValueError, match="even width"):
        homo.warp_perspective_video_host(np.zeros((12, 7), np.uint8), H, (4, 4), "nv12", "bgr")
    with pytest.raises(ValueError, match="\\(H\\*3/2, W\\)"):
        homo.warp_perspective_video_host(bgr[None], H, (4, 4), "i420", "bgr")
    with pytest.raises(ValueError, match="\\(H, W, 3\\)"):
        homo.warp_perspective_video_host(i420, H, (4, 4), "bgr", "i420")
    with pytest.raises(ValueError, match="uint8"):
        homo.warp_perspective_video_host(i420.astype(np.float32), H, (4, 4), "i420", "i420")
    with pytest.raises(ValueError, match="C-contiguous"):
        homo.warp_perspective_video_host(np.zeros((12, 16), np.uint8)[:, ::2], H, (4, 4), "i420", "i420")
    with pytest.raises(ValueError, match="even width and height"):
        homo.warp_perspective_video_host(bgr, H, (5, 4), "bgr", "i420")
    with pytest.raises(ValueError, match="dst must be"):
        homo.warp_perspective_video_host(bgr, H, (4, 4), "bgr", "i420", dst=np.zeros((4, 4, 3), np.uint8))
    with pytest.raises(ValueError, match="mat_index"):
        homo.warp_perspective_video_host(np.zeros((2, 12, 8), np.uint8), np.stack([H] * 3), (4, 4), "i420", "nv12")
