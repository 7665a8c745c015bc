"""CPU: pins oracle/nv12_oracle.py against cv2.cvtColor(COLOR_YUV2BGR_NV12) and the committed cv2
hashes, and checks that the NV12 entry points reject bad frame layouts without a GPU."""
import ctypes

import numpy as np
import pytest

from bev_b200 import _native
from oracle import nv12_oracle as no
from oracle import warp_oracle as wo
from tests import util


@pytest.mark.parametrize("h,w", [(1080, 1920), (2160, 3840), (2, 2), (2, 64), (480, 852), (480, 854), (6, 10)])
def test_oracle_matches_live_cv2(h, w):
    cv2 = pytest.importorskip("cv2")
    f = no.seeded_nv12(h * 7 + w, h, w)
    assert util.bits_equal(no.nv12_to_bgr(f), cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12))


def test_oracle_matches_cv2_on_every_yuv_triple():
    cv2 = pytest.importorskip("cv2")
    f = no.all_triples_nv12()
    h = f.shape[0] // 3 * 2
    seen = 0
    for r0 in range(0, h, 512):  # 512-row slices keep cv2's and the oracle's buffers small
        piece = np.concatenate([f[r0:r0 + 512], f[h + r0 // 2:h + (r0 + 512) // 2]])
        assert util.bits_equal(no.nv12_to_bgr(piece), cv2.cvtColor(piece, cv2.COLOR_YUV2BGR_NV12)), r0
        seen += 512 * f.shape[1]
    assert seen == 1 << 24


def test_all_triples_frame_holds_every_triple():
    f = no.all_triples_nv12()
    h, w = f.shape[0] // 3 * 2, f.shape[1]
    Y = f[:h].astype(np.int64)
    uv = f[h:].reshape(h // 2, w // 2, 2).astype(np.int64)
    U = np.repeat(np.repeat(uv[:, :, 0], 2, 0), 2, 1)
    V = np.repeat(np.repeat(uv[:, :, 1], 2, 0), 2, 1)
    key = (Y << 16) | (U << 8) | V
    assert np.unique(key).size == 1 << 24


@pytest.mark.parametrize("case", util.load_json("nv12_hash.json")["cases"], ids=lambda c: c["name"])
def test_oracle_chain_matches_cv2_hashes(case):
    h, w = case["shape"]
    bgr = no.nv12_to_bgr(no.seeded_nv12(case["seed"], h, w))
    if "H" in case:
        bgr = wo.warp_perspective(bgr, np.array(case["H"]), case["dsize"], flags=case["flags"])
    assert util.sha256(bgr) == case["sha256"]


def test_touched_samples_count_the_warp_footprint():
    H = util.h_canon()
    luma, chroma = no.touched_samples((1920, 1080), (1024, 1024), H, 1)
    assert luma == wo.touched_pixels((1920, 1080), (1024, 1024), H, 1)[0]
    assert luma // 4 <= chroma <= luma
    assert no.touched_samples((1920, 1080), (1024, 1024), H, 0)[0] == \
        wo.touched_pixels((1920, 1080), (1024, 1024), H, 0)[0]


def test_c_abi_rejects_bad_layouts():
    lib = _native.lib()
    buf = ctypes.create_string_buffer(4096)
    p = ctypes.cast(buf, ctypes.c_void_p)
    M = np.eye(3)
    dp = M.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    bad = [  # (n, h, w, pitch, frame_stride)
        (1, 8, 7, 8, 96),     # odd width
        (1, 7, 8, 8, 96),     # odd height
        (1, 0, 8, 8, 96),     # empty
        (1, 8, 8, 6, 96),     # pitch below the width
        (2, 8, 8, 8, -1),     # negative frame stride
        (-1, 8, 8, 8, 96),    # negative batch
    ]
    for n, h, w, pitch, fs in bad:
        assert lib.bevk_nv12_to_bgr(p, p, n, h, w, pitch, fs, None) == -1, (n, h, w, pitch, fs)
        assert lib.bevk_last_error()
        rc = lib.bevk_warp_perspective_nv12(p, p, n, h, w, pitch, fs, 4, 4, dp, 1, None, 1, 0, None, None)
        assert rc == -1, (n, h, w, pitch, fs)
    # the rules of bevk_warp_perspective: interpolation, border mode, matrices, sizes
    for flags, bm, n_mats, dh in ((2, 0, 1, 4), (1, 1, 1, 4), (1, 0, 2, 4), (1, 0, 1, 0)):
        rc = lib.bevk_warp_perspective_nv12(p, p, 3, 8, 8, 8, 96, dh, 4, dp, n_mats, None, flags, bm, None, None)
        assert rc == -1, (flags, bm, n_mats, dh)
    # a frame of 4 GB or more does not fit the kernel's 32-bit in-frame offsets
    assert lib.bevk_warp_perspective_nv12(p, p, 1, 30000, 30000, 100000, 0, 4, 4, dp, 1, None, 1, 0,
                                          None, None) == -1


def test_python_wrappers_reject_cpu_tensors():
    import torch
    from bev_b200 import homo
    f = torch.zeros((12, 8), dtype=torch.uint8)
    with pytest.raises(ValueError, match="no CPU fallback"):
        homo.nv12_to_bgr(f)
    with pytest.raises(ValueError, match="no CPU fallback"):
        homo.warp_perspective_nv12(f, np.eye(3), (4, 4))


def test_torch_extension_registers_the_nv12_operators():
    import torch
    from bev_b200 import torch_ops
    torch_ops.load()
    assert hasattr(torch.ops.bev_cuda, "nv12_to_bgr")
    assert hasattr(torch.ops.bev_cuda, "warp_perspective_nv12")
    f = torch.zeros((12, 8), dtype=torch.uint8)
    with pytest.raises((RuntimeError, NotImplementedError)):
        torch.ops.bev_cuda.nv12_to_bgr(f)
    with pytest.raises((RuntimeError, NotImplementedError)):
        torch.ops.bev_cuda.warp_perspective_nv12(f, torch.eye(3, dtype=torch.float64), 4, 4)
