"""GPU: every warp / resize entry point against the live cv2 build, byte for byte, on the seeded
cases of tests/cv2_cases.py (the generators the CPU fuzz of the oracles uses).

The other GPU tests hold the kernels equal to the oracles; this file holds them equal to cv2 itself,
so an oracle and a kernel that read cv2 the same wrong way cannot both pass.  Frames go to and from
the device in whole batches of 5 to 9, so the staged kernel runs more than one frame per stage.
"""
import numpy as np
import pytest
import torch

from bev_b200 import _native, homo, torch_ops
from oracle import yuv420_oracle as yo
from tests import cv2_cases as cc
from tests import util

cv2 = pytest.importorskip("cv2")

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
WARP_SEED, N_WARP = 20261022, 480
RESIZE_SEED, N_RESIZE = 20261023, 300


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def cv2_warp(frame, H, case, border=None):
    border = case["border"] if border is None else border
    b = list(border) + [0.0] * (4 - len(border))
    dw, dh = case["dsize"]
    out = cv2.warpPerspective(frame, H, (dw, dh), flags=case["flags"], borderMode=cv2.BORDER_CONSTANT,
                              borderValue=b)
    return out.reshape(dh, dw, -1)


def check_frame(out, ref, src, H, case, dtype, what):
    msg = "%s, %s: %s" % (what, dtype, cc.describe(case))
    if cc.nearest_deviation_applies(dtype, case["flags"], ref.shape[2]):
        bad = cc.unexplained_nearest_deviations(out, ref, src, H, case["flags"], case["border"],
                                                case["geom"] in cc.DEGENERATE)
        assert len(bad) == 0, "kernel != cv2 beyond the documented nearest deviation at %d px (first " \
            "(y, x) %s); %s" % (len(bad), bad[:4].tolist(), msg)
    else:
        assert util.bits_equal(out, ref), "kernel != cv2 at %d px; %s" % (int(np.sum(out != ref)), msg)


def batch_size(case):
    return 5 + case["index"] % 5


def warp_batches():
    """(case, dtype, frames (n, h, w, c), table of matrices (K, 3, 3), mat_index or None)"""
    for case in cc.warp_cases(WARP_SEED, N_WARP):
        n = batch_size(case)
        src = cc.warp_src(case, n)
        dtypes = [case["dtype"]] + (["float16"] if case["dtype"] == "float32" and case["index"] % 2 else [])
        idx = None
        Ms = np.asarray(case["H"], np.float64)[None]
        if case["index"] % 4 == 3:  # a table of matrices chosen per frame
            other = cc.warp_case(WARP_SEED + 1, case["index"])["H"]
            if case["geom"] not in cc.DEGENERATE and not cc.nearest_deviation_applies(
                    case["dtype"], case["flags"], case["channels"]):
                Ms = np.stack([case["H"], other])
                idx = np.array([(i * 3) % 2 for i in range(n)], np.int32)
        for dt in dtypes:
            yield case, dt, (src.astype(np.float16) if dt == "float16" else src), Ms, idx


def cv2_refs(frames, Ms, idx, case, dtype):
    out = []
    for i in range(frames.shape[0]):
        H = Ms[0 if idx is None else idx[i]]
        f = frames[i].astype(np.float32) if dtype == "float16" else frames[i]
        r = cv2_warp(f, H, case)
        out.append((r.astype(np.float16) if dtype == "float16" else r, H))
    return out


@pytest.mark.parametrize("path", ["generic", "auto", "fast"])
def test_warp_perspective_vs_cv2(path):
    ran = 0
    for case, dt, frames, Ms, idx in warp_batches():
        t = cu(frames)
        try:
            out = homo.warp_perspective(t, Ms if Ms.shape[0] > 1 else Ms[0], case["dsize"],
                                        flags=case["flags"], borderValue=case["border"],
                                        mat_index=idx, path=path)
        except _native.NativeError as e:
            assert path == "fast" and "does not qualify" in str(e), (str(e), cc.describe(case))
            continue
        out = out.cpu().numpy()
        for i, (ref, H) in enumerate(cv2_refs(frames, Ms, idx, case, dt)):
            check_frame(out[i], ref, frames[i], H, case, dt, "%s path, frame %d" % (path, i))
        ran += 1
    assert ran > 0 if path == "fast" else ran >= N_WARP  # fast takes uint8 BGR, zero border


def test_torch_operator_vs_cv2():
    torch_ops.load()
    for case in cc.warp_cases(WARP_SEED, N_WARP)[::8]:
        n = batch_size(case)
        frames = cc.warp_src(case, n)
        bv = case["border"][0]  # the operator takes one border value for every channel
        out = torch.ops.bev_cuda.warp_perspective(cu(frames), torch.from_numpy(np.asarray(case["H"], np.float64)),
                                                  case["dsize"][0], case["dsize"][1], case["flags"], 0, bv,
                                                  None).cpu().numpy()
        border = [bv] * case["channels"]
        uniform = dict(case, border=tuple(border))
        for i in range(n):
            ref = cv2_warp(frames[i], case["H"], case, border)
            check_frame(out[i], ref, frames[i], case["H"], uniform, case["dtype"], "torch op, frame %d" % i)


def nv12_batch(case, n):
    h, w = (max(2, v + v % 2) for v in case["src_hw"])  # NV12 needs even sizes
    rng = np.random.default_rng([case["seed"], case["index"], 2])
    nv12 = rng.integers(0, 256, (n, h * 3 // 2, w), dtype=np.uint8)
    return nv12, [cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12) for f in nv12]


def test_warp_perspective_nv12_vs_cv2():
    for case in cc.warp_cases(WARP_SEED, N_WARP // 2, dtypes=("uint8",)):
        n = batch_size(case)
        nv12, bgr = nv12_batch(case, n)
        border = (list(case["border"]) + [0.0, 0.0])[:3]
        out = homo.warp_perspective_nv12(cu(nv12), case["H"], case["dsize"], flags=case["flags"],
                                         borderValue=border).cpu().numpy()
        for i in range(n):
            ref = cv2_warp(bgr[i], case["H"], case, border)
            assert util.bits_equal(out[i], ref), "nv12 warp != cv2 at %d px, frame %d: %s" % (
                int(np.sum(out[i] != ref)), i, cc.describe(case))


def test_warp_perspective_yuv420_vs_cv2():
    """The fused warps to YUV 4:2:0 from BGR and NV12 sources: 3 channels, dst sizes rounded up to
    even (so rows shorter than 16 give odd block widths, whose 2x2 dst blocks straddle two cv2 block
    columns), against cv2's warp followed by cv2's BGR -> I420 conversion (and its NV12 relayout)."""
    for case in cc.warp_cases(WARP_SEED, N_WARP // 2, dtypes=("uint8",)):
        n = batch_size(case)
        dw, dh = (v + v % 2 for v in case["dsize"])
        case = dict(case, channels=3, dsize=(dw, dh), bw0=cc.block_width(dw, dh))
        border = (list(case["border"]) + [0.0, 0.0])[:3]
        nv12, nv12_bgr = nv12_batch(case, n)
        bgr = cc.warp_src(case, n)
        for what, src, fn, refs in (("bgr", cu(bgr), homo.warp_perspective_yuv420, bgr),
                                    ("nv12", cu(nv12), homo.warp_perspective_nv12_yuv420, nv12_bgr)):
            i420 = [cv2.cvtColor(cv2_warp(f, case["H"], case, border), cv2.COLOR_BGR2YUV_I420) for f in refs]
            for layout in ("i420", "nv12"):
                out = fn(src, case["H"], (dw, dh), layout, flags=case["flags"], borderValue=border).cpu().numpy()
                for i in range(n):
                    ref = i420[i] if layout == "i420" else yo.i420_to_nv12(i420[i])
                    assert util.bits_equal(out[i], ref), "%s source, %s output != cv2 at %d bytes, frame %d: %s" % (
                        what, layout, int(np.sum(out[i] != ref)), i, cc.describe(case))


def test_resize_vs_cv2():
    for case in cc.resize_cases(RESIZE_SEED, N_RESIZE):
        n = batch_size(case)
        frames = cc.resize_src(case, n)
        out = homo.resize(cu(frames), case["dsize"]).cpu().numpy()
        for i in range(n):
            ref = cv2.resize(frames[i], case["dsize"]).reshape(out.shape[1:])
            assert util.bits_equal(out[i], ref), "resize != cv2 at %d bytes, frame %d: %s" % (
                int(np.sum(out[i] != ref)), i, cc.describe(case))


def test_resize_nv12_vs_cv2():
    for case in cc.resize_cases(RESIZE_SEED, N_RESIZE // 2):
        n = batch_size(case)
        nv12, bgr = nv12_batch(case, n)
        out = homo.resize_nv12(cu(nv12), case["dsize"]).cpu().numpy()
        for i in range(n):
            ref = cv2.resize(bgr[i], case["dsize"])
            assert util.bits_equal(out[i], ref), "nv12 resize != cv2 at %d bytes, frame %d: %s" % (
                int(np.sum(out[i] != ref)), i, cc.describe(case))


@pytest.mark.parametrize("flags", [0, 1])
def test_large_frames_vs_cv2(flags):
    """1080p frames at the eight cfg-4 camera homographies, and 4K frames at the canonical map."""
    cams = util.load_json("cfg4_cams.json")
    rng = np.random.default_rng(40 + flags)
    frames = rng.integers(0, 256, (3, 1080, 1920, 3), dtype=np.uint8)
    t = cu(frames)
    for cam in cams:
        H = np.array(cam["H_bev_img"], np.float64)
        dsize = (cam["bspec"]["u_size"], cam["bspec"]["v_size"])
        for path in ("generic", "auto", "fast"):
            out = homo.warp_perspective(t, H, dsize, flags=flags, path=path).cpu().numpy()
            for i in range(3):
                assert util.bits_equal(out[i], cv2.warpPerspective(frames[i], H, dsize, flags=flags)), \
                    (path, flags, i, repr(H))
    frames4k = rng.integers(0, 256, (2, 2160, 3840, 3), dtype=np.uint8)
    H4k = util.h_canon(4)
    out = homo.warp_perspective(cu(frames4k), H4k, (1024, 1024), flags=flags).cpu().numpy()
    for i in range(2):
        assert util.bits_equal(out[i], cv2.warpPerspective(frames4k[i], H4k, (1024, 1024), flags=flags)), \
            (flags, i, repr(H4k))
