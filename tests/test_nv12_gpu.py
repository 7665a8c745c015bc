"""GPU: NV12 -> BGR conversion and the fused NV12 perspective warp (csrc/nv12.cu) against the oracle
(oracle/nv12_oracle.py + oracle/warp_oracle.c, both pinned to cv2 4.13), the committed cv2 hashes
and the BGR warp paths.  Every comparison is bit for bit."""
import ctypes

import numpy as np
import pytest
import torch

from bev_b200 import _native, homo
from oracle import nv12_oracle as no
from oracle import warp_oracle as wo
from tests import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FLAGS = [0, 1, 16, 17]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def laid_out(frames, pitch, gap_rows=0):
    """The (N, H*3/2, W) frames as a decoder surface: rows `pitch` bytes apart, `gap_rows` unused
    rows after each frame.  Returns the strided CUDA view."""
    n, rows, w = frames.shape
    buf = torch.full((n * (rows + gap_rows) * pitch + pitch,), 0xA5, dtype=torch.uint8, device=DEV)
    view = buf.as_strided((n, rows, w), ((rows + gap_rows) * pitch, pitch, 1))
    view.copy_(torch.from_numpy(frames))
    return view


def ref_warp(f, H, dsize, flags, bv=0):
    return wo.warp_perspective(no.nv12_to_bgr(f), H, dsize, flags=flags, borderValue=bv)


def random_nv12(n, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(0, 256, (n, h * 3 // 2, w), dtype=torch.uint8, device=DEV, generator=g)


def fwd(H, flags):
    return np.linalg.inv(H) if flags & 16 else H


# ---- conversion ---------------------------------------------------------------------------------

@pytest.mark.parametrize("h,w,n", [(1080, 1920, 5), (2160, 3840, 3)])
def test_convert_batches(h, w, n):
    t = random_nv12(n, h, w, h + n)
    out = homo.nv12_to_bgr(t)
    assert tuple(out.shape) == (n, h, w, 3) and out.dtype == torch.uint8
    for i in (0, n - 1):
        assert util.bits_equal(out[i].cpu().numpy(), no.nv12_to_bgr(t[i].cpu().numpy())), i


@pytest.mark.parametrize("case", [c for c in util.load_json("nv12_hash.json")["cases"] if "H" not in c],
                         ids=lambda c: c["name"])
def test_convert_cv2_hashes(case):
    h, w = case["shape"]
    out = homo.nv12_to_bgr(dev(no.seeded_nv12(case["seed"], h, w)))
    assert util.sha256(out.cpu().numpy()) == case["sha256"]


def test_convert_every_yuv_triple():
    f = no.all_triples_nv12()
    assert util.bits_equal(homo.nv12_to_bgr(dev(f)).cpu().numpy(), no.nv12_to_bgr(f))


@pytest.mark.parametrize("h,w,pitch,gap", [(480, 852, 852, 0), (480, 854, 854, 0), (1080, 1920, 2048, 0),
                                           (1080, 1920, 2048, 7), (270, 478, 481, 3), (2, 2, 2, 0),
                                           (4, 6, 9, 1)])
def test_convert_layouts(h, w, pitch, gap):
    frames = np.stack([no.seeded_nv12(40 + i, h, w) for i in range(3)])
    out = homo.nv12_to_bgr(laid_out(frames, pitch, gap)).cpu().numpy()
    for i in range(3):
        assert util.bits_equal(out[i], no.nv12_to_bgr(frames[i])), (h, w, pitch, gap, i)
    one = homo.nv12_to_bgr(laid_out(frames[1:2], pitch, gap)[0])
    assert util.bits_equal(one.cpu().numpy(), no.nv12_to_bgr(frames[1]))


# ---- fused warp ---------------------------------------------------------------------------------

@pytest.mark.parametrize("flags", FLAGS)
def test_cfg2_batch(flags):
    """32 x 1080p NV12 -> 1024^2 BEV (the cfg-2 map) in one call."""
    H = fwd(util.h_canon(), flags)
    t = random_nv12(32, 1080, 1920, 100 + flags)
    out = homo.warp_perspective_nv12(t, H, (1024, 1024), flags=flags)
    assert tuple(out.shape) == (32, 1024, 1024, 3)
    for i in (0, 17, 31):
        ref = ref_warp(t[i].cpu().numpy(), H, (1024, 1024), flags)
        assert util.bits_equal(out[i].cpu().numpy(), ref), (flags, i)


@pytest.mark.parametrize("case", [c for c in util.load_json("nv12_hash.json")["cases"] if "H" in c],
                         ids=lambda c: c["name"])
def test_warp_cv2_hashes(case):
    h, w = case["shape"]
    out = homo.warp_perspective_nv12(dev(no.seeded_nv12(case["seed"], h, w)), np.array(case["H"]),
                                     case["dsize"], flags=case["flags"])
    assert util.sha256(out.cpu().numpy()) == case["sha256"]


@pytest.mark.parametrize("flags", FLAGS)
def test_cfg5_4k(flags):
    H = fwd(util.h_canon(2), flags)
    t = random_nv12(4, 2160, 3840, 200 + flags)
    out = homo.warp_perspective_nv12(t, H, (2048, 2048), flags=flags)
    for i in (0, 3):
        assert util.bits_equal(out[i].cpu().numpy(), ref_warp(t[i].cpu().numpy(), H, (2048, 2048), flags)), i


@pytest.mark.parametrize("flags", FLAGS)
def test_per_frame_matrices_and_camera_table(flags):
    rng = np.random.default_rng(flags)
    frames = np.stack([no.seeded_nv12(300 + i, 270, 480) for i in range(8)])
    quad = np.array([[0, 0], [479, 0], [479, 269], [0, 269]], np.float64)
    d = np.array([[0, 0], [199, 0], [199, 149], [0, 149]], np.float64)
    Hs = np.stack([fwd(homo.homo_from_pts(quad + rng.normal(size=(4, 2)) * 30, d), flags) for _ in range(8)])
    out = homo.warp_perspective_nv12(dev(frames), Hs, (200, 150), flags=flags).cpu().numpy()
    for i in range(8):
        assert util.bits_equal(out[i], ref_warp(frames[i], Hs[i], (200, 150), flags)), i
    # the eight cfg-4 cameras, interleaved through mat_index in one call
    cams = util.load_json("cfg4_cams.json")
    Hc = np.stack([fwd(np.diag([256.0 / c["bspec"]["u_size"], 512.0 / c["bspec"]["v_size"], 1.0])
                       @ np.array(c["H_bev_img"]), flags) for c in cams])
    n = 16
    idx = np.array([(5 * i) % 8 for i in range(n)], np.int32)
    t = random_nv12(n, 1080, 1920, 300 + flags)
    out = homo.warp_perspective_nv12(t, Hc, (256, 512), flags=flags, mat_index=idx).cpu().numpy()
    for i in range(n):
        ref = ref_warp(t[i].cpu().numpy(), Hc[idx[i]], (256, 512), flags)
        assert util.bits_equal(out[i], ref), (i, int(idx[i]))


@pytest.mark.parametrize("flags", FLAGS)
def test_edges_border_and_odd_dst_widths(flags):
    """Windows on the last luma column / row (and past them), a horizon-crossing map, a non-zero
    BGR border and dst widths that are not multiples of 4."""
    h, w = 96, 128
    frames = np.stack([no.seeded_nv12(500 + i, h, w) for i in range(3)])
    t = dev(frames)
    maps = [
        (np.array([[1.0, 0, 0.5], [0, 1.0, 0.5], [0, 0, 1.0]]), (w, h)),      # last column / row half out
        (np.array([[1.0, 0, -0.5], [0, 1.0, -0.25], [0, 0, 1.0]]), (w, h)),
        (np.diag([63.0 / (w - 1), 47.0 / (h - 1), 1.0]), (64, 48)),          # last dst pixel on the last luma pixel
        (np.array([[0.5, 0, 0], [0, 0.5, 0], [0, 0, 1.0]]), (63, 47)),        # minifying to an odd width
        (np.array([[3.0, 0.2, -7.0], [0.1, 2.7, -5.0], [0, 0, 1.0]]), (381, 290)),
        (np.array([[1.0, 0.2, -3.0], [0.1, 1.1, -2.0], [0.0, 0.03, -0.5]]), (130, 96)),  # horizon crossing
        (np.array([[1.0, 0, 2.0], [0, 1.0, 1.0], [0, 0, 1.0]]), (3, 2)),
        (np.array([[1.0, 0, 0], [0, 1.0, 0], [0, 0, 1.0]]), (1, 1)),
    ]
    for k, (H, dsize) in enumerate(maps):
        for bv in (0, (3, 50, 250)):
            out = homo.warp_perspective_nv12(t, fwd(H, flags), dsize, flags=flags, borderValue=bv).cpu().numpy()
            for i in (0, 2):
                ref = ref_warp(frames[i], fwd(H, flags), dsize, flags, bv)
                assert util.bits_equal(out[i], ref), (k, bv, i)
    # nearest identity is the conversion itself
    if flags == 0:
        assert util.bits_equal(homo.warp_perspective_nv12(t, np.eye(3), (w, h), flags=0).cpu().numpy(),
                               homo.nv12_to_bgr(t).cpu().numpy())


@pytest.mark.parametrize("flags", FLAGS)
@pytest.mark.parametrize("h,w,pitch,gap", [(1080, 1920, 2048, 0), (1080, 1920, 2048, 5), (480, 852, 852, 0),
                                           (480, 854, 854, 2), (480, 852, 857, 1)])
def test_pitched_and_narrow_inputs(flags, h, w, pitch, gap):
    frames = np.stack([no.seeded_nv12(600 + i, h, w) for i in range(3)])
    # the cfg-2 map for this frame size, to a 512^2 BEV
    H = fwd(np.diag([0.5, 0.5, 1.0]) @ util.h_canon() @ np.diag([1920.0 / w, 1080.0 / h, 1.0]), flags)
    out = homo.warp_perspective_nv12(laid_out(frames, pitch, gap), H, (512, 512), flags=flags).cpu().numpy()
    for i in (0, 2):
        assert util.bits_equal(out[i], ref_warp(frames[i], H, (512, 512), flags)), i


def test_fuzz_against_every_bgr_path():
    """Random homographies: the fused warp gives the bytes of warp_perspective(nv12_to_bgr(f)) on
    each BGR path (the forced staged kernel where the shape qualifies for it)."""
    import cv2
    rng = np.random.default_rng(20261020)
    sizes = [(368, 640), (480, 852), (540, 960), (1080, 1920)]
    for case in range(24):
        sh, sw = sizes[int(rng.integers(len(sizes)))]
        dw, dh = int(rng.integers(16, 200)) * 4 - int(rng.integers(0, 2)) * 2, int(rng.integers(40, 600))
        n = int(rng.integers(3, 8))
        jit = float(rng.uniform(0.05, 0.45))
        s = np.float32([[0, 0], [sw, 0], [sw, sh], [0, sh]]) + (rng.uniform(-jit, jit, (4, 2)) * [sw, sh]).astype(np.float32)
        d = np.float32([[0, 0], [dw, 0], [dw, dh], [0, dh]]) + (rng.uniform(-jit, jit, (4, 2)) * [dw, dh]).astype(np.float32)
        H = cv2.getPerspectiveTransform(s, d).astype(np.float64)
        flags = int(rng.integers(0, 2)) | (16 if rng.random() < 0.3 else 0)
        H = fwd(H, flags)
        t = random_nv12(n, sh, sw, 7000 + case)
        fused = homo.warp_perspective_nv12(t, H, (dw, dh), flags=flags)
        bgr = homo.nv12_to_bgr(t)
        for pth in ("generic", "auto", "fast"):
            try:
                ref = homo.warp_perspective(bgr, H, (dw, dh), flags=flags, path=pth)
            except _native.NativeError as e:
                assert pth == "fast" and "does not qualify" in str(e)
                continue
            assert torch.equal(fused, ref), (case, pth, sh, sw, dw, dh, flags)


def test_empty_batch_and_argument_errors():
    empty = torch.zeros((0, 12, 8), dtype=torch.uint8, device=DEV)
    assert tuple(homo.warp_perspective_nv12(empty, np.eye(3), (5, 4)).shape) == (0, 4, 5, 3)
    assert tuple(homo.nv12_to_bgr(empty).shape) == (0, 8, 8, 3)
    lib = _native.lib()
    M = np.eye(3)
    dp = M.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    # no frames: nothing is launched, so null buffers are fine
    assert lib.bevk_nv12_to_bgr(None, None, 0, 8, 8, 8, 96, None) == 0
    assert lib.bevk_warp_perspective_nv12(None, None, 0, 8, 8, 8, 96, 4, 4, dp, 1, None, 1, 0, None, None) == 0
    f = random_nv12(2, 8, 8, 1)
    with pytest.raises(ValueError):
        homo.nv12_to_bgr(f[:, :11])                                   # rows not H * 3 / 2
    with pytest.raises(ValueError):
        homo.nv12_to_bgr(f[:, :, :7])                                 # odd width
    with pytest.raises(ValueError):
        homo.warp_perspective_nv12(f[:, :, ::2], np.eye(3), (4, 4))   # inner stride 2
    with pytest.raises(ValueError):
        homo.nv12_to_bgr(f.to(torch.int16))
    with pytest.raises(ValueError):
        homo.nv12_to_bgr(f.as_strided((2, 12, 8), (96, 6, 1)))        # pitch below the width
    with pytest.raises(_native.NativeError):
        homo.warp_perspective_nv12(f, np.eye(3), (4, 4), flags=2)     # INTER_CUBIC
    with pytest.raises(_native.NativeError):
        homo.warp_perspective_nv12(f, np.eye(3), (4, 4), borderMode=1)
    with pytest.raises(ValueError):
        homo.warp_perspective_nv12(f, np.stack([np.eye(3)] * 3), (4, 4))
    torch.cuda.synchronize()


def test_side_stream_matches_serial():
    H = util.h_canon()
    t = random_nv12(12, 1080, 1920, 9)
    serial = [homo.warp_perspective_nv12(t, H, (1024, 1024), flags=f) for f in (1, 0)] + [homo.nv12_to_bgr(t)]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=DEV) for _ in range(3)]
    outs = []
    for rep in range(3):
        for j, st in enumerate(streams):
            with torch.cuda.stream(st):
                outs.append((j, homo.warp_perspective_nv12(t, H, (1024, 1024), flags=1 - j) if j < 2
                             else homo.nv12_to_bgr(t)))
    for st in streams:
        st.synchronize()
    for j, o in outs:
        assert torch.equal(o, serial[j]), j


def test_torch_ops_route_matches_ctypes_route():
    from bev_b200 import torch_ops
    torch_ops.load()
    frames = np.stack([no.seeded_nv12(800 + i, 270, 480) for i in range(5)])
    t = laid_out(frames, 512, 2)
    H = np.diag([0.25, 0.25, 1.0]) @ util.h_canon() @ np.diag([4.0, 4.0, 1.0])
    Ht = torch.from_numpy(H)
    assert torch.equal(torch.ops.bev_cuda.nv12_to_bgr(t), homo.nv12_to_bgr(t))
    assert torch.equal(torch.ops.bev_cuda.nv12_to_bgr(t[2]), homo.nv12_to_bgr(t[2]))
    for flags in (0, 1):
        out = torch.ops.bev_cuda.warp_perspective_nv12(t, Ht, 256, 256, flags, 0, 7.0, None)
        assert torch.equal(out, homo.warp_perspective_nv12(t, H, (256, 256), flags=flags, borderValue=(7, 7, 7)))
    idx = torch.tensor([i % 2 for i in range(5)], dtype=torch.int32)
    Hs = torch.from_numpy(np.stack([H, H @ np.diag([1.0, 0.9, 1.0])]))
    out = torch.ops.bev_cuda.warp_perspective_nv12(t, Hs, 256, 256, 1, 0, 0.0, idx)
    assert torch.equal(out, homo.warp_perspective_nv12(t, Hs.numpy(), (256, 256), mat_index=idx.numpy()))
    one = torch.ops.bev_cuda.warp_perspective_nv12(t[4], Ht, 256, 256)
    assert util.bits_equal(one.cpu().numpy(), ref_warp(frames[4], H, (256, 256), 1))
