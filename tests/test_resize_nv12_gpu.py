"""GPU: the NV12 resize (csrc/resize.cu, resize_nv12_kernel) against the composed oracle
(oracle/resize_nv12_oracle.py, pinned to cv2 4.13), the committed cv2 hashes of
tests/golden/nv12_resize_hash.json and the two-pass route nv12_to_bgr + resize.  Every comparison
is bit for bit."""
import numpy as np
import pytest
import torch

from bev_b200 import _native, homo
from oracle import nv12_oracle as no
from oracle import resize_nv12_oracle as rno
from oracle import warp_oracle as wo
from tests import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
HASHES = util.load_json("nv12_resize_hash.json")["cases"]


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def decoder_layout(frames, pitch, gap_rows=0, offset=0):
    """The (N, H*3/2, W) frames as a decoder surface: rows `pitch` bytes apart, `gap_rows` unused
    rows after each frame, the first byte `offset` bytes into the allocation.  Returns the strided
    CUDA view."""
    n, rows, w = frames.shape
    buf = torch.full((offset + n * (rows + gap_rows) * pitch + pitch,), 0xA5, dtype=torch.uint8, device=DEV)
    view = buf.as_strided((n, rows, w), ((rows + gap_rows) * pitch, pitch, 1), offset)
    view.copy_(torch.from_numpy(frames))
    return view


def random_nv12(n, h, w, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(0, 256, (n, h * 3 // 2, w), dtype=torch.uint8, device=DEV, generator=g)


def check_frames(out, frames, dsize, which=None):
    out = out.cpu().numpy()
    for i in (range(len(frames)) if which is None else which):
        assert util.bits_equal(out[i], rno.resize_nv12(frames[i], dsize)), (i, dsize)


@pytest.mark.parametrize("case", HASHES, ids=lambda c: c["name"])
def test_cv2_hashes(case):
    h, w = case["shape"]
    small = homo.resize_nv12(dev(no.seeded_nv12(case["seed"], h, w)), case["dsize"])
    assert tuple(small.shape) == (case["dsize"][1], case["dsize"][0], 3)
    assert util.sha256(small.cpu().numpy()) == case["sha256"]
    if "H" in case:
        bev = homo.warp_perspective(small, np.array(case["H"]), tuple(case["bev_size"]))
        assert util.sha256(bev.cpu().numpy()) == case["sha256_bev"]


@pytest.mark.parametrize("words", [True, False], ids=["words", "bytes"])
@pytest.mark.parametrize("packed", [True, False], ids=["packed", "unpacked"])
def test_random_shapes_on_each_kernel_variant(words, packed):
    """Word loads need a 4-byte aligned base, pitch and frame stride; the packed store a dst width
    that is a multiple of 4 (and an aligned dst, which torch allocations are)."""
    rng = np.random.default_rng(300 + 2 * words + packed)
    for k in range(10):
        h, w = 2 * int(rng.integers(1, 120)), 2 * int(rng.integers(1, 120))
        dw, dh = int(rng.integers(1, 300)), int(rng.integers(1, 300))
        dw = max(4, dw // 4 * 4) if packed else dw // 4 * 4 + int(rng.integers(1, 4))
        if words:
            pitch = (w + 3) // 4 * 4 + 4 * int(rng.integers(0, 3))
        else:
            pitch = w + int(rng.choice([0, 1, 3] if w % 4 == 2 else [1, 3]))
        n = int(rng.integers(1, 6))
        frames = np.stack([no.seeded_nv12(4000 + 10 * k + i, h, w) for i in range(n)])
        t = decoder_layout(frames, pitch)
        assert ((t.data_ptr() % 4 == 0 and pitch % 4 == 0) == words), (h, w, pitch)
        check_frames(homo.resize_nv12(t, (dw, dh)), frames, (dw, dh))


@pytest.mark.parametrize("h,w,pitch,gap,offset", [
    (1080, 1920, 2048, 0, 0), (1080, 1920, 2048, 5, 0), (480, 852, 852, 0, 0), (480, 854, 854, 2, 0),
    (480, 852, 857, 1, 0), (270, 478, 512, 3, 1), (1080, 1920, 1920, 0, 1), (2, 2, 2, 0, 0), (4, 6, 9, 1, 1)])
def test_decoder_layouts(h, w, pitch, gap, offset):
    frames = np.stack([no.seeded_nv12(600 + i, h, w) for i in range(3)])
    t = decoder_layout(frames, pitch, gap, offset)
    for dsize in ((max(1, w * 4 // 9), max(1, h * 4 // 9)), (w // 2 + 1, h // 2), (2 * w + 4, 2 * h + 1)):
        check_frames(homo.resize_nv12(t, dsize), frames, dsize)
        one = homo.resize_nv12(t[1], dsize)
        assert util.bits_equal(one.cpu().numpy(), rno.resize_nv12(frames[1], dsize)), dsize


def test_batch_equals_single_frames():
    frames = np.stack([no.seeded_nv12(700 + i, 90, 120) for i in range(70)])  # more frames than one chunk
    t = dev(frames)
    out = homo.resize_nv12(t, (52, 40))
    check_frames(out, frames, (52, 40), (0, 1, 33, 63, 64, 69))
    for i in range(70):
        assert torch.equal(out[i], homo.resize_nv12(t[i], (52, 40))), i


def test_full_batch_1080p():
    t = random_nv12(24, 1080, 1920, 3)
    out = homo.resize_nv12(t, (852, 480))
    assert tuple(out.shape) == (24, 480, 852, 3) and out.dtype == torch.uint8
    for i in (0, 11, 23):
        assert util.bits_equal(out[i].cpu().numpy(), rno.resize_nv12(t[i].cpu().numpy(), (852, 480))), i
    # the fused route gives the bytes of the two-pass route on the whole batch
    assert torch.equal(out, homo.resize(homo.nv12_to_bgr(t), (852, 480)))


def _cfg4_camera0():
    from bev_b200.bev import BEVWorldSpec
    from bev_b200.calib import Calib
    cam = util.load_json("cfg4_cams.json")[0]
    calib = Calib(vp1=np.array(cam["vp1"]), vp2=np.array(cam["vp2"]), height=cam["height"],
                  u_size=1920, v_size=1080)
    bspec = BEVWorldSpec(**{k: v for k, v in cam["bspec"].items() if v is not None and k not in ("x_max", "y_max")})
    return calib, bspec


def test_small_frame_helper_matches_hashes_and_bgr_route():
    calib, bspec = _cfg4_camera0()
    case = [c for c in HASHES if "H" in c][0]
    f = dev(no.seeded_nv12(case["seed"], 1080, 1920))
    small, bev = homo.warp_small_nv12_img_to_bev(f, calib, bspec, 852, 480)
    assert util.sha256(small.cpu().numpy()) == case["sha256"]
    assert util.sha256(bev.cpu().numpy()) == case["sha256_bev"]
    # a batch, against the BGR helper on converted frames
    t = random_nv12(6, 1080, 1920, 11)
    for flags in (homo.INTER_LINEAR, homo.INTER_NEAREST):
        small, bev = homo.warp_small_nv12_img_to_bev(t, calib, bspec, 852, 480, flags=flags)
        small_ref, bev_ref = homo.warp_small_img_to_bev(homo.nv12_to_bgr(t), calib, bspec, 852, 480, flags=flags)
        assert torch.equal(small, small_ref) and torch.equal(bev, bev_ref), flags
        ref = wo.warp_perspective(rno.resize_nv12(t[5].cpu().numpy(), (852, 480)), np.array(case["H"]),
                                  case["bev_size"], flags=flags)
        assert util.bits_equal(bev[5].cpu().numpy(), ref), flags


def test_side_stream_matches_serial():
    t = random_nv12(12, 1080, 1920, 9)
    sizes = ((852, 480), (960, 540), (853, 479))
    serial = [homo.resize_nv12(t, d) for d in sizes]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=DEV) for _ in sizes]
    outs = []
    for rep in range(3):
        for j, st in enumerate(streams):
            with torch.cuda.stream(st):
                outs.append((j, homo.resize_nv12(t, sizes[j])))
    for st in streams:
        st.synchronize()
    for j, o in outs:
        assert torch.equal(o, serial[j]), j


def test_empty_batch_and_argument_errors():
    empty = torch.zeros((0, 12, 8), dtype=torch.uint8, device=DEV)
    assert tuple(homo.resize_nv12(empty, (5, 4)).shape) == (0, 4, 5, 3)
    # no frames: nothing is launched, so null buffers are fine
    assert _native.lib().bevk_resize_nv12(None, None, 0, 8, 8, 8, 96, 4, 4, None) == 0
    f = random_nv12(2, 8, 8, 1)
    with pytest.raises(ValueError):
        homo.resize_nv12(f[:, :11], (4, 4))                            # rows not H * 3 / 2
    with pytest.raises(ValueError):
        homo.resize_nv12(f[:, :, :7], (4, 4))                          # odd width
    with pytest.raises(ValueError):
        homo.resize_nv12(f[:, :, ::2], (4, 4))                         # inner stride 2
    with pytest.raises(ValueError):
        homo.resize_nv12(f.to(torch.int16), (4, 4))
    with pytest.raises(ValueError):
        homo.resize_nv12(f.as_strided((2, 12, 8), (96, 6, 1)), (4, 4))  # pitch below the width
    with pytest.raises(ValueError):
        homo.resize_nv12(f, (4, 4), dst=torch.empty((2, 4, 5, 3), dtype=torch.uint8, device=DEV))
    with pytest.raises(ValueError):
        homo.resize_nv12(f[0], (4, 4), dst=torch.empty((1, 4, 4, 3), dtype=torch.uint8, device=DEV))
    with pytest.raises(_native.NativeError, match="positive"):
        homo.resize_nv12(f, (0, 4))
    with pytest.raises(_native.NativeError, match="32767"):
        homo.resize_nv12(f, (4, 32768))
    out = torch.empty((2, 4, 4, 3), dtype=torch.uint8, device=DEV)
    assert homo.resize_nv12(f, (4, 4), dst=out) is out
    check_frames(out, f.cpu().numpy(), (4, 4))
    torch.cuda.synchronize()


def test_torch_ops_route_matches_ctypes_route():
    from bev_b200 import torch_ops
    torch_ops.load()
    frames = np.stack([no.seeded_nv12(800 + i, 270, 480) for i in range(5)])
    t = decoder_layout(frames, 512, 2)
    for w, h in ((240, 135), (213, 120), (960, 540)):
        out = torch.ops.bev_cuda.resize_nv12(t, w, h)
        assert torch.equal(out, homo.resize_nv12(t, (w, h))), (w, h)
        one = torch.ops.bev_cuda.resize_nv12(t[3], w, h)
        assert util.bits_equal(one.cpu().numpy(), rno.resize_nv12(frames[3], (w, h))), (w, h)
    odd = decoder_layout(frames, 480, 0, 1)
    assert torch.equal(torch.ops.bev_cuda.resize_nv12(odd, 213, 120), homo.resize_nv12(odd, (213, 120)))
