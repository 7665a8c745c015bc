"""CPU: pins the INTER_AREA oracle (oracle/resize_area_oracle.py) against live
cv2.resize(..., interpolation=cv2.INTER_AREA) on a seeded fuzz over cv2's three branches and 1 to 4
channels, and against the committed cv2 hashes of tests/golden/resize_area_hash.json; checks that
the C ABI rejects other interpolations and bad NV12 layouts without a GPU, and that the torch
operator is registered."""
import ctypes

import numpy as np
import pytest

from bev_b200 import _native
from oracle import nv12_oracle as no
from oracle import resize_area_oracle as ra
from oracle import warp_oracle as wo
from oracle.synth import seeded_frame
from tests import area_cases as ac
from tests import util

HASHES = util.load_json("resize_area_hash.json")["cases"]
SEED = 2026


def _cv2_area(cv2, img, dsize):
    return cv2.resize(img, tuple(dsize), interpolation=cv2.INTER_AREA)


@pytest.mark.parametrize("part", range(4))
def test_oracle_matches_live_cv2_fuzz(part):
    cv2 = pytest.importorskip("cv2")
    branches = set()
    for case in ac.area_cases(SEED, 4000)[1000 * part:1000 * (part + 1)]:
        src = ac.area_src(case)
        img = src[:, :, 0] if case["channels"] == 1 else src
        ref = _cv2_area(cv2, img, case["dsize"])
        assert util.bits_equal(ra.resize(img, case["dsize"]), ref), ac.describe(case)
        h, w = case["src_hw"]
        branches.add(ra.branch((w, h), case["dsize"]))
    assert branches == {"fast", "area", "linear"}


def test_nv12_oracle_matches_live_cv2_fuzz():
    cv2 = pytest.importorskip("cv2")
    for case in ac.area_cases(SEED + 1, 600, nv12=True):
        f = ac.area_src(case)
        ref = _cv2_area(cv2, cv2.cvtColor(f, no.COLOR_YUV2BGR_NV12), case["dsize"])
        assert util.bits_equal(ra.resize_nv12(f, case["dsize"]), ref), ac.describe(case)


@pytest.mark.parametrize("k", [2, 3, 4])
@pytest.mark.parametrize("channels", [1, 2, 3, 4])
def test_integer_cells_to_the_last_column(k, channels):
    """Integer factors per channel count at widths where a SIMD row would end in a scalar tail."""
    cv2 = pytest.importorskip("cv2")
    for dw in list(range(1, 40)) + [63, 64, 65, 127, 129, 852, 960]:
        for ky in (1, k):
            src = seeded_frame(100 * k + dw, 2 * ky, k * dw, channels, "uint8")
            img = src[:, :, 0] if channels == 1 else src
            ref = _cv2_area(cv2, img, (dw, 2))
            assert util.bits_equal(ra.resize(img, (dw, 2)), ref), (k, ky, channels, dw)


def test_branches():
    assert ra.branch((1920, 1080), (960, 540)) == "fast"
    assert ra.branch((1920, 1080), (1920, 1080)) == "fast"
    assert ra.branch((3840, 2160), (1920, 1080)) == "fast"
    assert ra.branch((1920, 1080), (852, 480)) == "area"
    assert ra.branch((1920, 1080), (2400, 500)) == "linear"
    assert ra.branch((852, 480), (1920, 1080)) == "linear"


@pytest.mark.parametrize("case", HASHES, ids=lambda c: c["name"])
def test_oracle_matches_cv2_hashes(case):
    h, w = case["shape"]
    if case["format"] == "bgr":
        small = ra.resize(seeded_frame(case["seed"], h, w, 3, "uint8"), case["dsize"])
    else:
        small = ra.resize_nv12(no.seeded_nv12(case["seed"], h, w), case["dsize"])
    assert small.shape == (case["dsize"][1], case["dsize"][0], 3)
    assert util.sha256(small) == case["sha256"]
    if "H" in case:
        bev = wo.warp_perspective(small, np.array(case["H"]), case["bev_size"])
        assert util.sha256(bev) == case["sha256_bev"]


def test_chain_cases_use_the_bgr_chain_map():
    chain = util.load_json("resize_kat.json")["small_frame_chain"]
    chains = [c for c in HASHES if "H" in c]
    assert {c["format"] for c in chains} == {"bgr", "nv12"}
    for c in chains:
        assert c["H"] == chain["H_bev_img_small"] and c["bev_size"] == chain["bev_size"]
        assert c["dsize"] == chain["new_uv"]


def test_touched_samples():
    # a downscale reads every source pixel, whichever branch it takes
    for dsize in ((852, 480), (960, 540), (640, 360)):
        assert ra.touched_pixels((1920, 1080), dsize) == 1920 * 1080, dsize
        assert ra.touched_samples_nv12((1920, 1080), dsize) == (1920 * 1080, 960 * 540), dsize
    assert ra.touched_pixels((3840, 2160), (1920, 1080)) == 3840 * 2160
    # an upscale reads the whole frame too; a 1-pixel dst reads a 2 x 2 window at most
    assert ra.touched_pixels((852, 480), (1920, 1080)) == 852 * 480
    assert ra.touched_pixels((10, 10), (1, 1)) == 100


def _buf():
    buf = ctypes.create_string_buffer(4096)
    return buf, ctypes.cast(buf, ctypes.c_void_p)


@pytest.mark.parametrize("interp", [0, 2, 4, 5])
def test_c_abi_rejects_other_interpolations(interp):
    lib = _native.lib()
    _keep, p = _buf()
    assert lib.bevk_resize(p, p, 1, 8, 8, 4, 4, 3, 0, interp, None) == -1
    assert b"INTER_LINEAR" in lib.bevk_last_error()
    assert lib.bevk_resize_nv12_interp(p, p, 1, 8, 8, 8, 96, 4, 4, interp, None) == -1
    assert b"INTER_LINEAR" in lib.bevk_last_error()


def test_c_abi_nv12_layout_rules():
    lib = _native.lib()
    _keep, p = _buf()
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
        (p, p, 1, 32768, 8, 8, 0, 4, 4),       # source above 32767
        (p, p, 1, 30000, 30000, 100000, 0, 4, 4),  # a frame of 4 GB or more
        (None, p, 1, 8, 8, 8, 96, 4, 4),       # null src
        (p, None, 1, 8, 8, 8, 96, 4, 4),       # null dst
    ]
    for interp in (1, 3):
        for args in bad:
            assert lib.bevk_resize_nv12_interp(*args, interp, None) == -1, (interp, args[2:])
            assert lib.bevk_last_error(), args[2:]


def test_python_constants_and_defaults():
    import inspect

    from bev_b200 import homo
    assert homo.INTER_AREA == 3 and homo.INTER_LINEAR == 1
    for fn in (homo.resize, homo.resize_nv12, homo.warp_small_img_to_bev, homo.warp_small_nv12_img_to_bev):
        assert inspect.signature(fn).parameters["interpolation"].default == homo.INTER_LINEAR, fn


def test_torch_extension_registers_the_resize_operator_with_interpolation():
    import torch
    from bev_b200 import torch_ops
    torch_ops.load()
    schema = str(torch.ops.bev_cuda.resize_nv12.default._schema)
    assert "int interpolation=1" in schema, schema
    with pytest.raises((RuntimeError, NotImplementedError)):
        torch.ops.bev_cuda.resize_nv12(torch.zeros((12, 8), dtype=torch.uint8), 4, 4, 3)
