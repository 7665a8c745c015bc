"""CPU: the device-matrix warps (bevk_*_dmat) reject bad arguments with BEVK_E_ARG before they look for
a device, as their host-matrix twins do, and the torch operator list stays as it was."""
import ctypes

import numpy as np
import pytest

from bev_b200 import _native, torch_ops

ARG, NOGPU = -1, -3
I420, NV12 = 0, 1
_buf = ctypes.create_string_buffer(4096)
_mats = np.zeros((4, 3, 3), np.float64)  # stands in for a device table: a rejected call never reads it


def _call(entry, n=2, sh=8, sw=8, dh=4, dw=4, c=3, dtype=0, M=True, n_mats=1, idx=None, flags=1, bm=0,
          pitch=None, layout=I420, dpitch=None):
    """One call of a _dmat entry point; returns (rc, error message)."""
    lib = _native.lib()
    m = _mats.ctypes.data_as(ctypes.POINTER(ctypes.c_double)) if M else None
    ip = np.ascontiguousarray(idx, np.int32).ctypes.data_as(ctypes.POINTER(ctypes.c_int32)) if idx is not None else None
    b = (ctypes.c_double * 4)()
    pitch = sw if pitch is None else pitch
    dpitch = dw if dpitch is None else dpitch
    if entry == "bevk_warp_perspective_dmat":
        args = (n, sh, sw, dh, dw, c, dtype, m, n_mats, ip, flags, bm, b)
    elif entry == "bevk_warp_perspective_nv12_dmat":
        args = (n, sh, sw, pitch, pitch * sh * 3 // 2, dh, dw, m, n_mats, ip, flags, bm, b)
    elif entry == "bevk_warp_perspective_yuv420_dmat":
        args = (n, sh, sw, dh, dw, layout, dpitch, dpitch * dh * 3 // 2, m, n_mats, ip, flags, bm, b)
    else:
        args = (n, sh, sw, pitch, pitch * sh * 3 // 2, dh, dw, layout, dpitch, dpitch * dh * 3 // 2, m, n_mats, ip,
                flags, bm, b)
    rc = getattr(lib, entry)(_buf, _buf, *args, None)
    return rc, lib.bevk_last_error().decode()


ENTRIES = ("bevk_warp_perspective_dmat", "bevk_warp_perspective_nv12_dmat", "bevk_warp_perspective_yuv420_dmat",
           "bevk_warp_perspective_nv12_yuv420_dmat")
COMMON = [
    (dict(M=False), "matrix"),
    (dict(n_mats=0), "matrix"),
    (dict(n_mats=-1), "matrix"),
    (dict(n_mats=2, idx=[0, 2]), "out of range"),
    (dict(n_mats=2, idx=[-1, 0]), "out of range"),
    (dict(n_mats=3), "needs a mat_index"),
    (dict(flags=2), "INTER_NEAREST and INTER_LINEAR"),   # INTER_CUBIC
    (dict(flags=2 | 16), "INTER_NEAREST and INTER_LINEAR"),
    (dict(bm=1), "BORDER_CONSTANT"),                     # BORDER_REPLICATE
    (dict(bm=4), "BORDER_CONSTANT"),
    (dict(n=-1), "n_frames"),
    (dict(sh=40000), "32767"),
]
NV12_SRC = [(dict(sh=7), "even"), (dict(sw=9, pitch=10), "even"), (dict(pitch=6), "pitch")]
YUV_DST = [(dict(dh=5), "even"), (dict(dw=6, dpitch=4), "pitch"), (dict(layout=2), "layout")]
CASES = [(e, kw, msg) for e in ENTRIES for kw, msg in COMMON]
CASES += [(e, kw, msg) for e in ENTRIES if "nv12" in e for kw, msg in NV12_SRC]
CASES += [(e, kw, msg) for e in ENTRIES if "yuv420" in e for kw, msg in YUV_DST]
CASES += [("bevk_warp_perspective_dmat", dict(c=5), "channels"), ("bevk_warp_perspective_dmat", dict(dtype=3), "dtype")]


@pytest.mark.parametrize("entry, kw, msg", CASES, ids=["%s-%d" % (c[0][5:], i) for i, c in enumerate(CASES)])
def test_c_argument_errors(entry, kw, msg):
    """BEVK_E_ARG with a message, before any device probe: also on a machine without a GPU."""
    rc, err = _call(entry, **kw)
    assert rc == ARG, (entry, kw, rc, err)
    assert msg in err, (entry, kw, err)


@pytest.mark.parametrize("entry", ENTRIES)
def test_good_arguments_reach_the_device_probe(entry):
    """Arguments that pass return BEVK_OK (0 frames: nothing to do) or, without an sm_100 device,
    BEVK_E_NOGPU: the checks above are the only ones made on the host."""
    for kw in (dict(n=0), dict(n=0, n_mats=3, idx=[])):
        rc, err = _call(entry, **kw)
        assert rc in (0, NOGPU), (entry, kw, err)


def test_dmat_entry_points_are_bound():
    for e in ENTRIES:
        twin = e[:-len("_dmat")]
        assert _native.SIGNATURES[e] == _native.SIGNATURES[twin], e  # the twin's arguments, M a device pointer


def test_operator_list_is_unchanged():
    """The four warps take CUDA matrices through their existing operators: no operator was added."""
    assert torch_ops.OPS == (
        "warp_perspective", "project_points", "rbox_corners_project", "corners_to_rbox", "rbox_similarity",
        "nv12_to_bgr", "warp_perspective_nv12", "resize_nv12", "bgr_to_yuv420", "warp_perspective_yuv420",
        "resize", "warp_perspective_nv12_yuv420", "composite", "composite_bev", "rbox_iou_matrix",
        "rboxtt_similarity", "rbox_zt2tt_world", "rbox_heading", "corners_heading", "angle_similarity",
        "dist_similarity", "v2yaw", "yaw2v", "yaw2mat")
