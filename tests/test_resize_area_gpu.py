"""GPU: cv2.resize(..., interpolation=cv2.INTER_AREA) through homo.resize and homo.resize_nv12
(csrc/resize.cu) against the oracle (oracle/resize_area_oracle.py, pinned to cv2 4.13), live
cv2 where it is installed, and the committed cv2 hashes of tests/golden/resize_area_hash.json.
Every comparison is bit for bit."""
import numpy as np
import pytest
import torch

from bev_b200 import _native, homo
from oracle import nv12_oracle as no
from oracle import resize_area_oracle as ra
from oracle import warp_oracle as wo
from oracle.synth import seeded_frame
from tests import area_cases as ac
from tests import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
AREA = homo.INTER_AREA
HASHES = util.load_json("resize_area_hash.json")["cases"]
SEED = 2027


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def decoder_layout(frames, pitch, gap_rows=0, offset=0):
    """The (N, H*3/2, W) frames as a decoder surface: rows `pitch` bytes apart, `gap_rows` unused
    rows after each frame, the first byte `offset` bytes into the allocation."""
    n, rows, w = frames.shape
    buf = torch.full((offset + n * (rows + gap_rows) * pitch + pitch,), 0xA5, dtype=torch.uint8, device=DEV)
    view = buf.as_strided((n, rows, w), ((rows + gap_rows) * pitch, pitch, 1), offset)
    view.copy_(torch.from_numpy(frames))
    return view


def random_frames(shape, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(0, 256, shape, dtype=torch.uint8, device=DEV, generator=g)


def oracle(case, f):
    return ra.resize_nv12(f, case["dsize"]) if case["nv12"] else ra.resize(f, case["dsize"])


@pytest.mark.parametrize("nv12", [False, True], ids=["bgr", "nv12"])
def test_fuzz_against_oracle_and_cv2(nv12):
    cv2 = None
    try:
        import cv2
    except ImportError:
        pass
    for case in ac.area_cases(SEED + nv12, 800, nv12=nv12):
        src = ac.area_src(case, n=2)
        if nv12:
            out = homo.resize_nv12(dev(src), case["dsize"], interpolation=AREA).cpu().numpy()
        else:
            out = homo.resize(dev(src), case["dsize"], interpolation=AREA).cpu().numpy()
        for i in range(2):
            ref = oracle(case, src[i])
            assert util.bits_equal(out[i], ref), (i, ac.describe(case))
            if cv2 is not None and i == 0:
                img = cv2.cvtColor(src[i], no.COLOR_YUV2BGR_NV12) if nv12 else src[i]
                want = cv2.resize(img, case["dsize"], interpolation=cv2.INTER_AREA).reshape(ref.shape)
                assert util.bits_equal(out[i], want), ac.describe(case)


@pytest.mark.parametrize("case", HASHES, ids=lambda c: c["name"])
def test_cv2_hashes(case):
    h, w = case["shape"]
    if case["format"] == "bgr":
        small = homo.resize(dev(seeded_frame(case["seed"], h, w, 3, "uint8")), case["dsize"], interpolation=AREA)
    else:
        small = homo.resize_nv12(dev(no.seeded_nv12(case["seed"], h, w)), case["dsize"], interpolation=AREA)
    assert tuple(small.shape) == (case["dsize"][1], case["dsize"][0], 3)
    assert util.sha256(small.cpu().numpy()) == case["sha256"]
    if "H" in case:
        bev = homo.warp_perspective(small, np.array(case["H"]), tuple(case["bev_size"]))
        assert util.sha256(bev.cpu().numpy()) == case["sha256_bev"]


# one shape per branch: (src h, w), dsize.  The upscaling branch runs the bilinear kernels: with
# src_w % 4 == 2 the byte gathers; with src_w and dst_w multiples of 4 ("words") the BGR word-gather
# kernel and the NV12 word-gather one with packed stores; and with dst_w % 4 == 2 the NV12
# word-gather one with unpacked stores.
BRANCH_SHAPES = {"fast": ((96, 130), (65, 32)), "area": ((96, 130), (57, 41)), "linear": ((40, 62), (97, 30)),
                 "linear_words": ((40, 64), (96, 30)), "linear_words_unpacked": ((40, 64), (98, 52))}


@pytest.mark.parametrize("branch", sorted(BRANCH_SHAPES))
@pytest.mark.parametrize("channels", [1, 2, 3, 4, "nv12"])
def test_every_kernel_variant(branch, channels):
    (h, w), dsize = BRANCH_SHAPES[branch]
    assert ra.branch((w, h), dsize) == branch.split("_")[0]
    rng = np.random.default_rng([7, h, w, dsize[0]])
    if channels == "nv12":
        frames = rng.integers(0, 256, (3, h * 3 // 2, w), dtype=np.uint8)
        out = homo.resize_nv12(dev(frames), dsize, interpolation=AREA).cpu().numpy()
        refs = [ra.resize_nv12(f, dsize) for f in frames]
    else:
        frames = rng.integers(0, 256, (3, h, w, channels), dtype=np.uint8)
        out = homo.resize(dev(frames), dsize, interpolation=AREA).cpu().numpy()
        refs = [ra.resize(f, dsize) for f in frames]
    for i in range(3):
        assert util.bits_equal(out[i], refs[i]), (branch, channels, i)


@pytest.mark.parametrize("dsize", [(852, 480), (960, 540), (640, 360), (1920, 1200)])
def test_batch_equals_single_frames(dsize):
    frames = random_frames((70, 108, 192, 3), 5)  # more frames than one chunk
    nv = random_frames((70, 162, 192), 6)
    small = tuple(max(1, d // 10) for d in dsize)
    out = homo.resize(frames, small, interpolation=AREA)
    out_nv = homo.resize_nv12(nv, small, interpolation=AREA)
    for i in (0, 1, 33, 63, 64, 69):
        assert torch.equal(out[i], homo.resize(frames[i], small, interpolation=AREA)), i
        assert torch.equal(out_nv[i], homo.resize_nv12(nv[i], small, interpolation=AREA)), i
        assert util.bits_equal(out[i].cpu().numpy(), ra.resize(frames[i].cpu().numpy(), small)), i


def test_2d_and_3d_inputs():
    g = random_frames((1, 60, 90), 8)[0]
    out = homo.resize(g, (40, 27), interpolation=AREA)
    assert tuple(out.shape) == (27, 40)
    assert util.bits_equal(out.cpu().numpy(), ra.resize(g.cpu().numpy(), (40, 27)))
    c = random_frames((60, 90, 4), 9)
    out = homo.resize(c, (40, 27), interpolation=AREA)
    assert util.bits_equal(out.cpu().numpy(), ra.resize(c.cpu().numpy(), (40, 27)))


@pytest.mark.parametrize("h,w,pitch,gap,offset", [
    (1080, 1920, 2048, 0, 0), (1080, 1920, 2048, 5, 0), (480, 852, 852, 0, 0), (480, 854, 854, 2, 0),
    (480, 852, 857, 1, 0), (270, 478, 512, 3, 1), (1080, 1920, 1920, 0, 1), (2, 2, 2, 0, 0), (4, 6, 9, 1, 1)])
def test_decoder_layouts(h, w, pitch, gap, offset):
    frames = np.stack([no.seeded_nv12(900 + i, h, w) for i in range(3)])
    t = decoder_layout(frames, pitch, gap, offset)
    for dsize in ((max(1, w * 4 // 9), max(1, h * 4 // 9)), (max(1, w // 2), max(1, h // 2)), (w // 3 + 1, h),
                  (2 * w + 4, 2 * h + 1)):
        out = homo.resize_nv12(t, dsize, interpolation=AREA).cpu().numpy()
        for i in range(3):
            assert util.bits_equal(out[i], ra.resize_nv12(frames[i], dsize)), (dsize, i)
        one = homo.resize_nv12(t[1], dsize, interpolation=AREA)
        assert util.bits_equal(one.cpu().numpy(), ra.resize_nv12(frames[1], dsize)), dsize


@pytest.mark.parametrize("dsize", [(852, 480), (960, 540), (640, 360), (1280, 720), (2400, 500)])
def test_fused_nv12_equals_two_pass_route(dsize):
    t = random_frames((8, 1620, 1920), 12)
    fused = homo.resize_nv12(t, dsize, interpolation=AREA)
    assert torch.equal(fused, homo.resize(homo.nv12_to_bgr(t), dsize, interpolation=AREA)), dsize


def test_full_batch_4k():
    t = random_frames((4, 2160, 3840, 3), 13)
    out = homo.resize(t, (1920, 1080), interpolation=AREA)
    for i in (0, 3):
        assert util.bits_equal(out[i].cpu().numpy(), ra.resize(t[i].cpu().numpy(), (1920, 1080))), i


def test_default_is_still_inter_linear():
    t = random_frames((2, 1080, 1920, 3), 14)
    nv = random_frames((2, 1620, 1920), 15)
    assert torch.equal(homo.resize(t, (852, 480)), homo.resize(t, (852, 480), interpolation=homo.INTER_LINEAR))
    assert torch.equal(homo.resize_nv12(nv, (852, 480)),
                       homo.resize_nv12(nv, (852, 480), interpolation=homo.INTER_LINEAR))
    assert not torch.equal(homo.resize(t, (852, 480)), homo.resize(t, (852, 480), interpolation=AREA))


def _cfg4_camera0():
    from bev_b200.bev import BEVWorldSpec
    from bev_b200.calib import Calib
    cam = util.load_json("cfg4_cams.json")[0]
    calib = Calib(vp1=np.array(cam["vp1"]), vp2=np.array(cam["vp2"]), height=cam["height"],
                  u_size=1920, v_size=1080)
    bspec = BEVWorldSpec(**{k: v for k, v in cam["bspec"].items() if v is not None and k not in ("x_max", "y_max")})
    return calib, bspec


def test_small_frame_helpers_match_hashes():
    calib, bspec = _cfg4_camera0()
    for case in (c for c in HASHES if "H" in c):
        if case["format"] == "bgr":
            f = dev(seeded_frame(case["seed"], 1080, 1920, 3, "uint8"))
            small, bev = homo.warp_small_img_to_bev(f, calib, bspec, 852, 480, interpolation=AREA)
        else:
            f = dev(no.seeded_nv12(case["seed"], 1080, 1920))
            small, bev = homo.warp_small_nv12_img_to_bev(f, calib, bspec, 852, 480, interpolation=AREA)
        assert util.sha256(small.cpu().numpy()) == case["sha256"], case["name"]
        assert util.sha256(bev.cpu().numpy()) == case["sha256_bev"], case["name"]
    # a batch through both helpers, against the oracle chain
    t = random_frames((4, 1620, 1920), 16)
    chain = [c for c in HASHES if "H" in c][0]
    for flags in (homo.INTER_LINEAR, homo.INTER_NEAREST):
        small, bev = homo.warp_small_nv12_img_to_bev(t, calib, bspec, 852, 480, flags=flags, interpolation=AREA)
        small_ref, bev_ref = homo.warp_small_img_to_bev(homo.nv12_to_bgr(t), calib, bspec, 852, 480, flags=flags,
                                                        interpolation=AREA)
        assert torch.equal(small, small_ref) and torch.equal(bev, bev_ref), flags
        ref = wo.warp_perspective(ra.resize_nv12(t[3].cpu().numpy(), (852, 480)), np.array(chain["H"]),
                                  chain["bev_size"], flags=flags)
        assert util.bits_equal(bev[3].cpu().numpy(), ref), flags


def test_side_streams_match_serial():
    t = random_frames((12, 1080, 1920, 3), 17)
    nv = random_frames((12, 1620, 1920), 18)
    sizes = ((852, 480), (960, 540), (853, 479))
    serial = [(homo.resize(t, d, interpolation=AREA), homo.resize_nv12(nv, d, interpolation=AREA)) for d in sizes]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=DEV) for _ in sizes]
    outs = []
    for rep in range(3):
        for j, st in enumerate(streams):
            with torch.cuda.stream(st):
                outs.append((j, homo.resize(t, sizes[j], interpolation=AREA),
                             homo.resize_nv12(nv, sizes[j], interpolation=AREA)))
    for st in streams:
        st.synchronize()
    for j, a, b in outs:
        assert torch.equal(a, serial[j][0]) and torch.equal(b, serial[j][1]), j


def test_empty_batch_and_argument_errors():
    assert tuple(homo.resize(torch.zeros((0, 8, 8, 3), dtype=torch.uint8, device=DEV), (4, 4),
                             interpolation=AREA).shape) == (0, 4, 4, 3)
    empty = torch.zeros((0, 12, 8), dtype=torch.uint8, device=DEV)
    assert tuple(homo.resize_nv12(empty, (5, 4), interpolation=AREA).shape) == (0, 4, 5, 3)
    assert _native.lib().bevk_resize_nv12_interp(None, None, 0, 8, 8, 8, 96, 4, 4, AREA, None) == 0
    t = torch.zeros(8, 8, 3, dtype=torch.uint8, device=DEV)
    f = random_frames((2, 12, 8), 1)
    for bad in (0, 2, 4, 5):
        with pytest.raises(_native.NativeError, match="INTER_LINEAR"):
            homo.resize(t, (4, 4), interpolation=bad)
        with pytest.raises(_native.NativeError, match="INTER_LINEAR"):
            homo.resize_nv12(f, (4, 4), interpolation=bad)
    with pytest.raises(_native.NativeError, match="positive"):
        homo.resize_nv12(f, (0, 4), interpolation=AREA)
    out = torch.empty((2, 4, 4, 3), dtype=torch.uint8, device=DEV)
    assert homo.resize_nv12(f, (4, 4), dst=out, interpolation=AREA) is out
    for i in range(2):
        assert util.bits_equal(out[i].cpu().numpy(), ra.resize_nv12(f[i].cpu().numpy(), (4, 4)))
    torch.cuda.synchronize()


def test_torch_ops_route_matches_ctypes_route():
    from bev_b200 import torch_ops
    torch_ops.load()
    frames = np.stack([no.seeded_nv12(950 + i, 270, 480) for i in range(5)])
    t = decoder_layout(frames, 512, 2)
    for w, h in ((240, 135), (213, 120), (160, 90), (960, 540)):
        out = torch.ops.bev_cuda.resize_nv12(t, w, h, AREA)
        assert torch.equal(out, homo.resize_nv12(t, (w, h), interpolation=AREA)), (w, h)
        one = torch.ops.bev_cuda.resize_nv12(t[3], w, h, interpolation=AREA)
        assert util.bits_equal(one.cpu().numpy(), ra.resize_nv12(frames[3], (w, h))), (w, h)
        assert torch.equal(torch.ops.bev_cuda.resize_nv12(t, w, h), homo.resize_nv12(t, (w, h))), (w, h)
    odd = decoder_layout(frames, 480, 0, 1)
    assert torch.equal(torch.ops.bev_cuda.resize_nv12(odd, 213, 120, 3),
                       homo.resize_nv12(odd, (213, 120), interpolation=AREA))
