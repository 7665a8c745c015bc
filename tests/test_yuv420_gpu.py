"""GPU: BGR -> YUV 4:2:0 conversion and the fused warps to YUV BEVs (csrc/yuv420.cu) against the
oracle (oracle/yuv420_oracle.py, oracle/nv12_oracle.py and oracle/warp_oracle.c, all pinned to
cv2 4.13), the committed cv2 hashes and the two-pass route on the device.  Every comparison is bit
for bit."""
import ctypes

import numpy as np
import pytest
import torch

from bev_b200 import _native, homo
from oracle import nv12_oracle as no
from oracle import warp_oracle as wo
from oracle import yuv420_oracle as yo
from tests import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LAYOUTS = ["i420", "nv12"]
HASHES = util.load_json("yuv420_hash.json")["cases"]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def random_bgr(n, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device=DEV, generator=g)


def random_nv12(n, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(0, 256, (n, h * 3 // 2, w), dtype=torch.uint8, device=DEV, generator=g)


def misaligned(t):
    """A contiguous copy of t whose data starts one byte past a 4-byte boundary."""
    buf = torch.empty(t.numel() + 4, dtype=torch.uint8, device=DEV)
    view = buf[1:1 + t.numel()].view(t.shape)
    view.copy_(t)
    return view


def laid_out(frames, pitch, gap_rows=0):
    """NV12 frames (N, H*3/2, W) as a decoder surface: rows `pitch` bytes apart, `gap_rows` unused rows
    after each frame."""
    n, rows, w = frames.shape
    buf = torch.full((n * (rows + gap_rows) * pitch + pitch,), 0xA5, dtype=torch.uint8, device=DEV)
    view = buf.as_strided((n, rows, w), ((rows + gap_rows) * pitch, pitch, 1))
    view.copy_(frames if isinstance(frames, torch.Tensor) else torch.from_numpy(frames))
    return view


def surface(n, h, w, pitch, gap_rows=0):
    """An encoder surface for n YUV 4:2:0 frames of h x w filled with 0xA5: the (N, H*3/2, W) view and
    a mask of the bytes outside it."""
    rows = h * 3 // 2
    buf = torch.full((n * (rows + gap_rows) * pitch,), 0xA5, dtype=torch.uint8, device=DEV)
    view = buf.as_strided((n, rows, w), ((rows + gap_rows) * pitch, pitch, 1))
    mask = torch.ones_like(buf, dtype=torch.bool)
    mask.as_strided((n, rows, w), ((rows + gap_rows) * pitch, pitch, 1)).fill_(False)
    return buf, view, mask


def ref_yuv(bgr, layout):
    return yo.convert(np.ascontiguousarray(bgr), layout)


def fwd(H, flags):
    return np.linalg.inv(H) if flags & 16 else H


def cfg4_mats():
    cams = util.load_json("cfg4_cams.json")
    return np.stack([np.diag([256.0 / c["bspec"]["u_size"], 512.0 / c["bspec"]["v_size"], 1.0])
                     @ np.array(c["H_bev_img"]) for c in cams])


# ---- conversion ---------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w,n", [(1080, 1920, 5), (2160, 3840, 3)])
def test_convert_batches(h, w, n, layout):
    t = random_bgr(n, h, w, h + n)
    out = homo.bgr_to_yuv420(t, layout)
    assert tuple(out.shape) == (n, h * 3 // 2, w) and out.dtype == torch.uint8
    for i in (0, n - 1):
        assert util.bits_equal(out[i].cpu().numpy(), ref_yuv(t[i].cpu().numpy(), layout)), i


@pytest.mark.parametrize("case", [c for c in HASHES if "H" not in c], ids=lambda c: c["name"])
def test_convert_cv2_hashes(case):
    h, w = case["shape"]
    out = homo.bgr_to_yuv420(dev(util.seeded_frame(case["seed"], h, w, 3, "uint8")))
    assert util.sha256(out.cpu().numpy()) == case["sha256"]


def test_convert_every_bgr_triple():
    for r0 in range(0, 4096, 1024):
        f = yo.all_triples_bgr(r0, 1024)
        for layout in LAYOUTS:
            assert util.bits_equal(homo.bgr_to_yuv420(dev(f), layout).cpu().numpy(), ref_yuv(f, layout)), (r0, layout)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w", [(2, 2), (2, 6), (6, 2), (4, 130), (10, 128), (30, 190), (480, 852), (480, 854),
                                 (270, 478), (1080, 1920)])
def test_convert_shapes_and_misaligned_sources(h, w, layout):
    """W % 4 == 2, partial and whole 64-column segments, and a source one byte off alignment."""
    frames = np.stack([util.seeded_frame(50 + i + h + w, h, w, 3, "uint8") for i in range(3)])
    for t in (dev(frames), misaligned(dev(frames))):
        out = homo.bgr_to_yuv420(t, layout).cpu().numpy()
        for i in range(3):
            assert util.bits_equal(out[i], ref_yuv(frames[i], layout)), (i, t.data_ptr() % 4)
    one = homo.bgr_to_yuv420(dev(frames[1]), layout)
    assert tuple(one.shape) == (h * 3 // 2, w) and util.bits_equal(one.cpu().numpy(), ref_yuv(frames[1], layout))


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w,pitch,gap", [(1080, 1920, 2048, 0), (1080, 1920, 2048, 3), (480, 854, 857, 1),
                                           (6, 10, 11, 0), (2, 2, 3, 2)])
def test_convert_to_pitched_surfaces(h, w, pitch, gap, layout):
    frames = random_bgr(3, h, w, pitch + gap)
    buf, view, pad = surface(3, h, w, pitch, gap)
    assert homo.bgr_to_yuv420(frames, layout, dst=view) is view
    for i in range(3):
        assert util.bits_equal(view[i].cpu().numpy(), ref_yuv(frames[i].cpu().numpy(), layout)), i
    assert bool((buf[pad] == 0xA5).all()), "padding bytes were written"


# ---- fused warps --------------------------------------------------------------------------------

@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("flags", [0, 1, 16, 17])
def test_cfg2_batch(flags, layout):
    """16 x 1080p -> 1024^2 BEVs (the cfg-2 map), BGR and NV12 sources."""
    H = fwd(util.h_canon(), flags)
    t = random_bgr(16, 1080, 1920, 100 + flags)
    out = homo.warp_perspective_yuv420(t, H, (1024, 1024), layout, flags=flags)
    assert tuple(out.shape) == (16, 1536, 1024)
    for i in (0, 15):
        ref = ref_yuv(wo.warp_perspective(t[i].cpu().numpy(), H, (1024, 1024), flags=flags), layout)
        assert util.bits_equal(out[i].cpu().numpy(), ref), (flags, i)
    v = random_nv12(16, 1080, 1920, 200 + flags)
    out = homo.warp_perspective_nv12_yuv420(v, H, (1024, 1024), layout, flags=flags)
    for i in (0, 15):
        bev = wo.warp_perspective(no.nv12_to_bgr(v[i].cpu().numpy()), H, (1024, 1024), flags=flags)
        assert util.bits_equal(out[i].cpu().numpy(), ref_yuv(bev, layout)), (flags, i)


@pytest.mark.parametrize("case", [c for c in HASHES if "H" in c], ids=lambda c: c["name"])
def test_warp_cv2_hashes(case):
    h, w = case["shape"]
    if case["format"] == "bgr":
        out = homo.warp_perspective_yuv420(dev(util.seeded_frame(case["seed"], h, w, 3, "uint8")), np.array(case["H"]),
                                           case["dsize"], flags=case["flags"])
    else:
        out = homo.warp_perspective_nv12_yuv420(dev(no.seeded_nv12(case["seed"], h, w)), np.array(case["H"]),
                                                case["dsize"], flags=case["flags"])
    assert util.sha256(out.cpu().numpy()) == case["sha256"]


MAPS = [  # (H, dsize) on a 96 x 128 source
    (np.array([[1.0, 0, 0.5], [0, 1.0, 0.5], [0, 0, 1.0]]), (128, 96)),      # last column / row half out
    (np.array([[1.0, 0, -0.5], [0, 1.0, -0.25], [0, 0, 1.0]]), (128, 96)),
    (np.array([[0.5, 0, 0], [0, 0.5, 0], [0, 0, 1.0]]), (62, 46)),           # minifying, W % 4 == 2
    (np.array([[3.0, 0.2, -7.0], [0.1, 2.7, -5.0], [0, 0, 1.0]]), (382, 290)),
    (np.array([[1.0, 0.2, -3.0], [0.1, 1.1, -2.0], [0.0, 0.03, -0.5]]), (130, 96)),  # horizon crossing
    (np.array([[1.0, 0, 2.0], [0, 1.0, 1.0], [0, 0, 1.0]]), (2, 2)),
    # rows shorter than 16: odd block widths 85 and 73, so some 2x2 dst blocks straddle two cv2 block columns
    (np.array([[0.7, 0.05, 3.5], [0.02, 0.9, 2.5], [0.0, 0.001, 1.0]]), (170, 12)),
    (np.array([[0.75, 0.0, 0.5], [0.0, 0.5, 0.5], [0.0, 0.0, 1.0]]), (146, 14)),
]


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("flags", [0, 1, 16, 17])
def test_every_kernel_variant(flags, layout):
    """BGR word gathers (aligned, width % 4 == 0) and byte gathers (width 130, a misaligned source,
    1-pixel wide and high sources), NV12 word and byte gathers, zero and non-zero borders: the fused
    output equals the two passes (warp to BGR, then bgr_to_yuv420) and the oracle."""
    h, w = 96, 128
    bgr = random_bgr(3, h, w, 7 + flags)
    narrow = random_bgr(3, h, 130, 8 + flags)
    sources = [("words", bgr), ("bytes_w130", narrow), ("bytes_misaligned", misaligned(bgr)),
               ("bytes_1xN", random_bgr(3, 1, 7, 9)), ("bytes_Nx1", random_bgr(3, 5, 1, 10))]
    v = random_nv12(3, h, w, 11 + flags)
    nv12_sources = [("nv12_words", v), ("nv12_bytes", laid_out(v, 131, 1)), ("nv12_misaligned", misaligned(v))]
    for k, (H, dsize) in enumerate(MAPS):
        M = fwd(H, flags)
        for bv in (0, (3, 50, 250)):
            for name, s in sources:
                out = homo.warp_perspective_yuv420(s, M, dsize, layout, flags=flags, borderValue=bv)
                bev = homo.warp_perspective(s.contiguous(), M, dsize, flags=flags, borderValue=bv)
                assert torch.equal(out, homo.bgr_to_yuv420(bev, layout)), (k, bv, name)
                ref = wo.warp_perspective(s[2].cpu().numpy(), M, dsize, flags=flags, borderValue=bv)
                assert util.bits_equal(out[2].cpu().numpy(), ref_yuv(ref, layout)), (k, bv, name)
            for name, s in nv12_sources:
                out = homo.warp_perspective_nv12_yuv420(s, M, dsize, layout, flags=flags, borderValue=bv)
                bev = homo.warp_perspective_nv12(s, M, dsize, flags=flags, borderValue=bv)
                assert torch.equal(out, homo.bgr_to_yuv420(bev, layout)), (k, bv, name)
                ref = wo.warp_perspective(no.nv12_to_bgr(v[2].cpu().numpy()), M, dsize, flags=flags, borderValue=bv)
                assert util.bits_equal(out[2].cpu().numpy(), ref_yuv(ref, layout)), (k, bv, name)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("h,w,pitch,gap", [(1080, 1920, 2048, 0), (1080, 1920, 2048, 5), (480, 852, 852, 0),
                                           (480, 854, 854, 2), (480, 852, 857, 1)])
def test_pitched_gapped_nv12_sources(h, w, pitch, gap, layout):
    frames = np.stack([no.seeded_nv12(600 + i, h, w) for i in range(3)])
    H = np.diag([0.5, 0.5, 1.0]) @ util.h_canon() @ np.diag([1920.0 / w, 1080.0 / h, 1.0])
    for flags in (0, 1):
        out = homo.warp_perspective_nv12_yuv420(laid_out(frames, pitch, gap), H, (512, 512), layout, flags=flags)
        for i in (0, 2):
            bev = wo.warp_perspective(no.nv12_to_bgr(frames[i]), H, (512, 512), flags=flags)
            assert util.bits_equal(out[i].cpu().numpy(), ref_yuv(bev, layout)), (flags, i)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_pitched_destinations_keep_their_padding(layout):
    H = np.diag([0.25, 0.25, 1.0]) @ util.h_canon()
    t = random_bgr(4, 1080, 1920, 21)
    v = random_nv12(4, 1080, 1920, 22)
    for pitch, gap in ((256, 0), (300, 3), (259, 1)):
        for flags in (0, 1):
            buf, view, pad = surface(4, 256, 254, pitch, gap)
            assert homo.warp_perspective_yuv420(t, H, (254, 256), layout, dst=view, flags=flags) is view
            assert torch.equal(view, homo.warp_perspective_yuv420(t, H, (254, 256), layout, flags=flags))
            assert bool((buf[pad] == 0xA5).all()), (pitch, gap, flags)
            buf, view, pad = surface(4, 256, 254, pitch, gap)
            homo.warp_perspective_nv12_yuv420(v, H, (254, 256), layout, dst=view, flags=flags)
            assert torch.equal(view, homo.warp_perspective_nv12_yuv420(v, H, (254, 256), layout, flags=flags))
            assert bool((buf[pad] == 0xA5).all()), (pitch, gap, flags)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("flags", [0, 1])
def test_matrices_per_frame_and_camera_table(flags, layout):
    """One matrix per frame, and the eight cfg-4 cameras interleaved through mat_index: fused equals
    the two passes for BGR and NV12 sources."""
    rng = np.random.default_rng(flags)
    quad = np.array([[0, 0], [479, 0], [479, 269], [0, 269]], np.float64)
    d = np.array([[0, 0], [199, 0], [199, 149], [0, 149]], np.float64)
    Hs = np.stack([homo.homo_from_pts(quad + rng.normal(size=(4, 2)) * 30, d) for _ in range(8)])
    t = random_bgr(8, 270, 480, 30 + flags)
    out = homo.warp_perspective_yuv420(t, Hs, (200, 150), layout, flags=flags)
    for i in range(8):
        ref = ref_yuv(wo.warp_perspective(t[i].cpu().numpy(), Hs[i], (200, 150), flags=flags), layout)
        assert util.bits_equal(out[i].cpu().numpy(), ref), i
    Hc, n = cfg4_mats(), 16
    idx = np.array([(5 * i) % 8 for i in range(n)], np.int32)
    t = random_bgr(n, 1080, 1920, 40 + flags)
    out = homo.warp_perspective_yuv420(t, Hc, (256, 512), layout, flags=flags, mat_index=idx)
    two = homo.bgr_to_yuv420(homo.warp_perspective(t, Hc, (256, 512), flags=flags, mat_index=idx), layout)
    assert torch.equal(out, two)
    ref = ref_yuv(wo.warp_perspective(t[3].cpu().numpy(), Hc[idx[3]], (256, 512), flags=flags), layout)
    assert util.bits_equal(out[3].cpu().numpy(), ref)
    v = random_nv12(n, 1080, 1920, 50 + flags)
    out = homo.warp_perspective_nv12_yuv420(v, Hc, (256, 512), layout, flags=flags, mat_index=idx)
    two = homo.bgr_to_yuv420(homo.warp_perspective_nv12(v, Hc, (256, 512), flags=flags, mat_index=idx), layout)
    assert torch.equal(out, two)


def test_cfg4_eight_cameras_fused_equals_two_pass():
    """The cfg-4 BEVs at their own sizes, 24 frames per camera, as the benchmark runs them."""
    cams = util.load_json("cfg4_cams.json")
    t = random_bgr(24, 1080, 1920, 60)
    v = random_nv12(24, 1080, 1920, 61)
    for c in cams:
        H, dsize = np.array(c["H_bev_img"]), (int(c["bspec"]["u_size"]), int(c["bspec"]["v_size"]))
        for layout in LAYOUTS:
            out = homo.warp_perspective_yuv420(t, H, dsize, layout)
            assert torch.equal(out, homo.bgr_to_yuv420(homo.warp_perspective(t, H, dsize), layout)), (c["k"], layout)
            out = homo.warp_perspective_nv12_yuv420(v, H, dsize, layout)
            two = homo.bgr_to_yuv420(homo.warp_perspective_nv12(v, H, dsize), layout)
            assert torch.equal(out, two), (c["k"], layout)


def test_batches_equal_single_frames():
    H = np.diag([0.5, 0.5, 1.0]) @ util.h_canon()
    t = random_bgr(7, 1080, 1920, 70)
    v = random_nv12(7, 1080, 1920, 71)
    for layout in LAYOUTS:
        for flags in (0, 1):
            out = homo.warp_perspective_yuv420(t, H, (512, 512), layout, flags=flags)
            outn = homo.warp_perspective_nv12_yuv420(v, H, (512, 512), layout, flags=flags)
            for i in (0, 3, 6):
                assert torch.equal(out[i], homo.warp_perspective_yuv420(t[i], H, (512, 512), layout, flags=flags))
                assert torch.equal(outn[i], homo.warp_perspective_nv12_yuv420(v[i], H, (512, 512), layout,
                                                                              flags=flags))
        conv = homo.bgr_to_yuv420(t, layout)
        assert all(torch.equal(conv[i], homo.bgr_to_yuv420(t[i], layout)) for i in (0, 6))


def test_calibration_helpers():
    from bev_b200.bev import BEVWorldSpec
    from bev_b200.calib import Calib
    cam = util.load_json("cfg4_cams.json")[0]
    calib = Calib(vp1=np.array(cam["vp1"]), vp2=np.array(cam["vp2"]), height=cam["height"], u_size=1920, v_size=1080)
    bspec = BEVWorldSpec(**{k: v for k, v in cam["bspec"].items() if v is not None and k not in ("x_max", "y_max")})
    t = random_bgr(3, 1080, 1920, 80)
    v = random_nv12(3, 1080, 1920, 81)
    for layout in LAYOUTS:
        for flags in (0, 1):
            out = homo.warp_img_to_bev_yuv420(t, calib, bspec, layout, flags=flags)
            assert torch.equal(out, homo.bgr_to_yuv420(homo.warp_img_to_bev(t, calib, bspec, flags=flags), layout))
            out = homo.warp_nv12_img_to_bev_yuv420(v, calib, bspec, layout, flags=flags)
            two = homo.bgr_to_yuv420(homo.warp_nv12_img_to_bev(v, calib, bspec, flags=flags), layout)
            assert torch.equal(out, two)


def test_side_streams_match_serial():
    H = util.h_canon()
    t = random_bgr(12, 1080, 1920, 90)
    v = random_nv12(12, 1080, 1920, 91)
    jobs = [lambda: homo.warp_perspective_yuv420(t, H, (1024, 1024), "nv12"),
            lambda: homo.warp_perspective_nv12_yuv420(v, H, (1024, 1024), flags=0),
            lambda: homo.bgr_to_yuv420(t)]
    serial = [j() for j in jobs]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=DEV) for _ in jobs]
    outs = []
    for rep in range(3):
        for j, st in enumerate(streams):
            with torch.cuda.stream(st):
                outs.append((j, jobs[j]()))
    for st in streams:
        st.synchronize()
    for j, o in outs:
        assert torch.equal(o, serial[j]), j


def test_empty_batch_and_argument_errors():
    empty = torch.zeros((0, 8, 6, 3), dtype=torch.uint8, device=DEV)
    assert tuple(homo.bgr_to_yuv420(empty).shape) == (0, 12, 6)
    assert tuple(homo.warp_perspective_yuv420(empty, np.eye(3), (4, 2)).shape) == (0, 3, 4)
    assert tuple(homo.warp_perspective_nv12_yuv420(torch.zeros((0, 12, 8), dtype=torch.uint8, device=DEV),
                                                   np.eye(3), (4, 2), "nv12").shape) == (0, 3, 4)
    lib = _native.lib()
    M = np.eye(3)
    dp = M.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    # no frames: nothing is launched, so null buffers are fine
    assert lib.bevk_bgr_to_yuv420(None, None, 0, 8, 8, 0, 8, 96, None) == 0
    assert lib.bevk_warp_perspective_yuv420(None, None, 0, 8, 8, 4, 4, 1, 4, 24, dp, 1, None, 1, 0, None, None) == 0
    assert lib.bevk_warp_perspective_nv12_yuv420(None, None, 0, 8, 8, 8, 96, 4, 4, 0, 4, 24, dp, 1, None, 1, 0, None,
                                                 None) == 0
    t = random_bgr(2, 8, 8, 1)
    with pytest.raises(ValueError):
        homo.bgr_to_yuv420(t[:, :7])                                         # odd height
    with pytest.raises(ValueError):
        homo.bgr_to_yuv420(t, "yuv444")
    with pytest.raises(ValueError):
        homo.bgr_to_yuv420(t.to(torch.int16))
    with pytest.raises(ValueError):
        homo.warp_perspective_yuv420(t, np.eye(3), (5, 4))                   # odd dst width
    with pytest.raises(ValueError):
        homo.bgr_to_yuv420(t, dst=torch.empty((2, 12, 8), dtype=torch.uint8, device=DEV)[:, :, ::2])
    with pytest.raises(ValueError):
        homo.bgr_to_yuv420(t, dst=torch.empty((2, 12, 7), dtype=torch.uint8, device=DEV))
    with pytest.raises(_native.NativeError):
        homo.warp_perspective_yuv420(t, np.eye(3), (4, 4), flags=2)          # INTER_CUBIC
    with pytest.raises(_native.NativeError):
        homo.warp_perspective_nv12_yuv420(random_nv12(2, 8, 8, 2), np.eye(3), (4, 4), borderMode=1)
    with pytest.raises(ValueError):
        homo.warp_perspective_yuv420(t, np.stack([np.eye(3)] * 3), (4, 4))
    torch.cuda.synchronize()


def test_torch_ops_route_matches_ctypes_route():
    from bev_b200 import torch_ops
    torch_ops.load()
    t = random_bgr(5, 270, 480, 95)
    H = np.diag([0.25, 0.25, 1.0]) @ util.h_canon() @ np.diag([4.0, 4.0, 1.0])
    Ht = torch.from_numpy(H)
    for code, layout in enumerate(LAYOUTS):
        assert torch.equal(torch.ops.bev_cuda.bgr_to_yuv420(t, code), homo.bgr_to_yuv420(t, layout))
        assert torch.equal(torch.ops.bev_cuda.bgr_to_yuv420(t[2], code), homo.bgr_to_yuv420(t[2], layout))
        for flags in (0, 1):
            out = torch.ops.bev_cuda.warp_perspective_yuv420(t, Ht, 256, 256, code, flags, 0, 7.0, None)
            ref = homo.warp_perspective_yuv420(t, H, (256, 256), layout, flags=flags, borderValue=(7, 7, 7))
            assert torch.equal(out, ref), (layout, flags)
    idx = torch.tensor([i % 2 for i in range(5)], dtype=torch.int32)
    Hs = torch.from_numpy(np.stack([H, H @ np.diag([1.0, 0.9, 1.0])]))
    out = torch.ops.bev_cuda.warp_perspective_yuv420(t, Hs, 256, 256, 1, 1, 0, 0.0, idx)
    assert torch.equal(out, homo.warp_perspective_yuv420(t, Hs.numpy(), (256, 256), "nv12", mat_index=idx.numpy()))
    one = torch.ops.bev_cuda.warp_perspective_yuv420(t[4], Ht, 256, 256)
    ref = ref_yuv(wo.warp_perspective(t[4].cpu().numpy(), H, (256, 256)), "i420")
    assert util.bits_equal(one.cpu().numpy(), ref)
