"""CPU: pins the composed oracle of the NV12 resize (oracle/resize_nv12_oracle.py) against
cv2.resize(cv2.cvtColor(f, COLOR_YUV2BGR_NV12)) and the committed cv2 hashes, and checks that
bevk_resize_nv12 rejects bad arguments without a GPU."""
import ctypes

import numpy as np
import pytest

from bev_b200 import _native
from oracle import nv12_oracle as no
from oracle import resize_nv12_oracle as rno
from oracle import resize_oracle as ro
from oracle import warp_oracle as wo
from tests import util

HASHES = util.load_json("nv12_resize_hash.json")["cases"]

# (h, w) of the NV12 source, (dst_w, dst_h)
SHAPES = [
    ((1080, 1920), (852, 480)), ((1080, 1920), (960, 540)), ((1080, 1920), (640, 360)),
    ((1080, 1920), (1280, 720)), ((2160, 3840), (1920, 1080)), ((720, 1280), (640, 360)),
    ((480, 852), (1920, 1080)), ((480, 854), (853, 479)), ((2, 2), (1, 1)), ((2, 2), (7, 5)),
    ((2, 2), (2, 2)), ((4, 6), (1, 9)), ((96, 130), (1, 1)), ((96, 130), (130, 1)),
    ((96, 130), (1, 96)), ((270, 478), (239, 135)), ((64, 32), (16, 64)), ((32, 64), (200, 17)),
    ((18, 10), (10, 18)), ((100, 200), (400, 50)), ((540, 962), (481, 270)),
]


@pytest.mark.parametrize("hw,dsize", SHAPES, ids=lambda v: "x".join(map(str, v)))
def test_oracle_matches_live_cv2(hw, dsize):
    cv2 = pytest.importorskip("cv2")
    h, w = hw
    f = no.seeded_nv12(h * 11 + w + dsize[0], h, w)
    ref = cv2.resize(cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12), dsize)
    assert util.bits_equal(rno.resize_nv12(f, dsize), ref)


@pytest.mark.parametrize("case", HASHES, ids=lambda c: c["name"])
def test_oracle_matches_cv2_hashes(case):
    h, w = case["shape"]
    small = rno.resize_nv12(no.seeded_nv12(case["seed"], h, w), case["dsize"])
    assert small.shape == (case["dsize"][1], case["dsize"][0], 3)
    assert util.sha256(small) == case["sha256"]
    if "H" in case:
        bev = wo.warp_perspective(small, np.array(case["H"]), case["bev_size"])
        assert util.sha256(bev) == case["sha256_bev"]


def test_chain_case_uses_the_bgr_chain_map():
    chain = util.load_json("resize_kat.json")["small_frame_chain"]
    case = [c for c in HASHES if "H" in c][0]
    assert case["H"] == chain["H_bev_img_small"] and case["bev_size"] == chain["bev_size"]
    assert case["dsize"] == chain["new_uv"]


def test_resize_touched_samples():
    luma, chroma = rno.resize_touched_samples((1920, 1080), (852, 480))
    assert luma == ro.touched_pixels((1920, 1080), (852, 480))
    assert luma // 4 <= chroma <= luma
    # exact 2x: every tap has weight 1/2 on two neighbours, so every source pixel is read
    assert rno.resize_touched_samples((1920, 1080), (960, 540)) == (1920 * 1080, 960 * 540)
    # an upscale reads the whole frame
    assert rno.resize_touched_samples((852, 480), (1920, 1080)) == (852 * 480, 426 * 240)


def test_c_abi_rejects_bad_arguments():
    lib = _native.lib()
    buf = ctypes.create_string_buffer(4096)
    p = ctypes.cast(buf, ctypes.c_void_p)
    bad = [  # (src, dst, n, h, w, pitch, frame_stride, dst_h, dst_w)
        (p, p, 1, 8, 7, 8, 96, 4, 4),          # odd width
        (p, p, 1, 7, 8, 8, 96, 4, 4),          # odd height
        (p, p, 1, 0, 8, 8, 96, 4, 4),          # empty source
        (p, p, 1, 8, 8, 6, 96, 4, 4),          # pitch below the width
        (p, p, 2, 8, 8, 8, -1, 4, 4),          # negative frame stride
        (p, p, -1, 8, 8, 8, 96, 4, 4),         # negative batch
        (p, p, 1, 8, 8, 8, 96, 0, 4),          # empty dst
        (p, p, 1, 8, 8, 8, 96, 4, -3),
        (p, p, 1, 8, 8, 8, 96, 32768, 4),      # dst above 32767
        (p, p, 1, 8, 8, 8, 96, 4, 32768),
        (p, p, 1, 32768, 8, 8, 0, 4, 4),       # source above 32767
        (p, p, 1, 8, 32768, 32768, 0, 4, 4),
        (p, p, 1, 30000, 30000, 100000, 0, 4, 4),  # a frame of 4 GB or more
        (None, p, 1, 8, 8, 8, 96, 4, 4),       # null src
        (p, None, 1, 8, 8, 8, 96, 4, 4),       # null dst
    ]
    for args in bad:
        src, dst, rest = args[0], args[1], args[2:]
        assert lib.bevk_resize_nv12(src, dst, *rest, None) == -1, args[2:]
        assert lib.bevk_last_error(), args[2:]


def test_python_wrappers_reject_cpu_tensors():
    import torch
    from bev_b200 import homo
    f = torch.zeros((12, 8), dtype=torch.uint8)
    with pytest.raises(ValueError, match="no CPU fallback"):
        homo.resize_nv12(f, (4, 4))


def test_torch_extension_registers_the_resize_operator():
    import torch
    from bev_b200 import torch_ops
    torch_ops.load()
    assert hasattr(torch.ops.bev_cuda, "resize_nv12")
    with pytest.raises((RuntimeError, NotImplementedError)):
        torch.ops.bev_cuda.resize_nv12(torch.zeros((12, 8), dtype=torch.uint8), 4, 4)
