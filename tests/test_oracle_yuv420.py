"""CPU: pins oracle/yuv420_oracle.py against cv2.cvtColor(COLOR_BGR2YUV_I420) and the committed cv2
hashes, and checks that the YUV 4:2:0 entry points reject bad arguments without a GPU."""
import ctypes

import numpy as np
import pytest

from bev_b200 import _native
from oracle import nv12_oracle as no
from oracle import warp_oracle as wo
from oracle import yuv420_oracle as yo
from tests import util


def test_oracle_matches_cv2_on_every_bgr_triple():
    cv2 = pytest.importorskip("cv2")
    seen = 0
    for r0 in range(0, 4096, 512):  # 512 block rows at a time keep the buffers small
        f = yo.all_triples_bgr(r0, 512)
        assert util.bits_equal(yo.bgr_to_i420(f), cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)), r0
        seen += 512 * 4096
    assert seen == 1 << 24


def test_all_triples_image_holds_every_triple_as_a_chroma_sample():
    f = yo.all_triples_bgr(0, 4096)[::2, ::2].reshape(-1, 3).astype(np.int64)
    assert np.unique((f[:, 0] << 16) | (f[:, 1] << 8) | f[:, 2]).size == 1 << 24


def random_shapes():
    rng = np.random.default_rng(20261021)
    shapes = [(2, 2), (2, 4), (4, 2), (2, 6), (6, 2), (4, 6), (8, 12), (480, 852), (480, 854), (1080, 1920)]
    while len(shapes) < 26:
        shapes.append((2 * int(rng.integers(1, 200)), 2 * int(rng.integers(1, 300))))
    return shapes


@pytest.mark.parametrize("h,w", random_shapes())
def test_oracle_matches_live_cv2_on_even_shapes(h, w):
    cv2 = pytest.importorskip("cv2")
    f = util.seeded_frame(h * 131 + w, h, w, 3, "uint8")
    ref = cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)
    assert ref.shape == (h * 3 // 2, w)
    assert util.bits_equal(yo.bgr_to_i420(f), ref)


def test_shapes_cover_both_chroma_row_phases():
    """W % 4 == 2 puts a U row boundary in the middle of a packed row; H % 4 == 2 starts V there."""
    shapes = random_shapes()
    assert any(w % 4 == 2 for _, w in shapes) and any(h % 4 == 2 for h, _ in shapes)


@pytest.mark.parametrize("h,w", [(2, 2), (6, 10), (8, 12), (480, 854)])
def test_nv12_layout_is_a_relayout_of_i420(h, w):
    f = util.seeded_frame(h + w, h, w, 3, "uint8")
    i420, nv12 = yo.bgr_to_i420(f), yo.bgr_to_nv12(f)
    assert util.bits_equal(nv12, yo.i420_to_nv12(i420))
    assert util.bits_equal(nv12[:h], i420[:h])
    uv = nv12[h:].reshape(h // 2, w // 2, 2)
    assert util.bits_equal(uv[..., 0].reshape(-1), i420[h:].reshape(-1)[:h * w // 4])
    assert util.bits_equal(uv[..., 1].reshape(-1), i420[h:].reshape(-1)[h * w // 4:])


def test_oracle_rejects_odd_sizes():
    for shape in ((3, 4, 3), (4, 3, 3), (4, 4, 4), (0, 4, 3)):
        with pytest.raises(ValueError):
            yo.bgr_to_i420(np.zeros(shape, np.uint8))


def case_bev(case):
    h, w = case["shape"]
    bgr = util.seeded_frame(case["seed"], h, w, 3, "uint8") if case["format"] == "bgr" else \
        no.nv12_to_bgr(no.seeded_nv12(case["seed"], h, w))
    if "H" in case:
        bgr = wo.warp_perspective(bgr, np.array(case["H"]), case["dsize"], flags=case["flags"])
    return bgr


@pytest.mark.parametrize("case", util.load_json("yuv420_hash.json")["cases"], ids=lambda c: c["name"])
def test_oracle_chain_matches_cv2_hashes(case):
    assert util.sha256(yo.bgr_to_i420(case_bev(case))) == case["sha256"]


def test_touched_bytes():
    assert yo.touched(2, 4, 6) == 2 * 4 * 6 * 3 + 2 * 4 * 6 * 3 // 2
    assert yo.touched(1, 4, 6, bgr_in=False) == 36


def test_c_abi_rejects_bad_arguments():
    lib = _native.lib()
    buf = ctypes.create_string_buffer(4096)
    p = ctypes.cast(buf, ctypes.c_void_p)
    M = np.eye(3)
    dp = M.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    bad = [  # (p_src, p_dst, n, h, w, layout, pitch, frame_stride)
        (p, p, 1, 8, 7, 0, 8, 96),      # odd width
        (p, p, 1, 7, 8, 0, 8, 96),      # odd height
        (p, p, 1, 0, 8, 0, 8, 96),      # empty
        (p, p, 1, 8, 8, 0, 6, 96),      # pitch below the width
        (p, p, 1, 8, 8, 2, 8, 96),      # unknown layout
        (p, p, 1, 8, 8, -1, 8, 96),     # unknown layout
        (p, p, 2, 8, 8, 1, 8, -1),      # negative frame stride
        (p, p, -1, 8, 8, 0, 8, 96),     # negative batch
        (None, p, 1, 8, 8, 0, 8, 96),   # null src
        (p, None, 1, 8, 8, 1, 8, 96),   # null dst
        (p, p, 1, 30000, 30000, 0, 100000, 0),  # a dst frame of 4 GB or more
    ]
    for s, d, n, h, w, layout, pitch, fs in bad:
        what = (s is None, d is None, n, h, w, layout, pitch, fs)
        assert lib.bevk_bgr_to_yuv420(s, d, n, h, w, layout, pitch, fs, None) == -1, what
        assert lib.bevk_last_error()
        assert lib.bevk_warp_perspective_yuv420(s, d, n, 8, 8, h, w, layout, pitch, fs, dp, 1, None, 1, 0, None,
                                                None) == -1, what
        assert lib.bevk_warp_perspective_nv12_yuv420(s, d, n, 8, 8, 8, 96, h, w, layout, pitch, fs, dp, 1, None, 1,
                                                     0, None, None) == -1, what
    assert lib.bevk_bgr_to_yuv420(p, p, 1, 40000, 8, 0, 8, 0, None) == -1  # cv2's SHRT_MAX limit
    # the warp rules: interpolation, border mode, matrices, source sizes and NV12 source layouts
    for flags, bm, n_mats, sh in ((2, 0, 1, 8), (1, 1, 1, 8), (1, 0, 2, 8), (1, 0, 1, 0)):
        assert lib.bevk_warp_perspective_yuv420(p, p, 3, sh, 8, 4, 4, 0, 4, 24, dp, n_mats, None, flags, bm, None,
                                                None) == -1, (flags, bm, n_mats, sh)
    for h, w, pitch, fs in ((8, 7, 8, 96), (7, 8, 8, 96), (8, 8, 6, 96), (8, 8, 8, -1), (30000, 30000, 100000, 0)):
        assert lib.bevk_warp_perspective_nv12_yuv420(p, p, 1, h, w, pitch, fs, 4, 4, 0, 4, 24, dp, 1, None, 1, 0,
                                                     None, None) == -1, (h, w, pitch, fs)


def test_python_wrappers_check_their_arguments():
    import torch
    from bev_b200 import homo
    f = torch.zeros((8, 8, 3), dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        homo.bgr_to_yuv420(f)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        homo.warp_perspective_yuv420(f, np.eye(3), (4, 4))
    with pytest.raises(ValueError, match="no CPU fallback"):
        homo.warp_perspective_nv12_yuv420(torch.zeros((12, 8), dtype=torch.uint8), np.eye(3), (4, 4))
    assert homo.COLOR_BGR2YUV_I420 == 128
    assert _native.YUV_LAYOUTS == {"i420": 0, "nv12": 1}


def test_torch_extension_registers_the_yuv420_operators():
    import torch
    from bev_b200 import torch_ops
    torch_ops.load()
    assert hasattr(torch.ops.bev_cuda, "bgr_to_yuv420")
    assert hasattr(torch.ops.bev_cuda, "warp_perspective_yuv420")
    f = torch.zeros((8, 8, 3), dtype=torch.uint8)
    with pytest.raises((RuntimeError, NotImplementedError)):
        torch.ops.bev_cuda.bgr_to_yuv420(f)
    with pytest.raises((RuntimeError, NotImplementedError)):
        torch.ops.bev_cuda.warp_perspective_yuv420(f, torch.eye(3, dtype=torch.float64), 4, 4)
