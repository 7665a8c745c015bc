"""GPU parity: bev_b200.homo.resize (CUDA, through the C ABI) vs cv2.resize 4.13 hashes
(tests/golden/resize_kat.json) and the numpy oracle (oracle/resize_oracle.py).  Bar: bit-exact."""
import numpy as np
import pytest
import torch

from bev_b200 import homo
from bev_b200._native import NativeError
from oracle import resize_oracle as ro
from tests import util

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KAT = util.load_json("resize_kat.json")


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def case_input(case):
    h, w, c = case["shape"]
    src = util.seeded_frame(case["seed"], h, w, c, "uint8")
    return src[:, :, 0] if c == 1 else src


@pytest.mark.parametrize("case", KAT["cases"], ids=lambda c: "x".join(map(str, c["shape"] + c["dsize"])))
def test_golden_hashes(case):
    out = homo.resize(cu(case_input(case)), case["dsize"]).cpu().numpy()
    assert util.sha256(out) == case["sha256"]


@pytest.mark.parametrize("c", [1, 2, 3, 4])
def test_random_shapes_against_oracle(c):
    rng = np.random.default_rng(100 + c)
    for _ in range(12):
        h, w, dw, dh = (int(v) for v in rng.integers(1, 200, 4))
        if c == 3 and rng.random() < 0.6:  # steer BGR cases onto the word-gather kernel
            w, dw = max(4, w // 4 * 4), max(4, dw // 4 * 4)
        src = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
        out = homo.resize(cu(src), (dw, dh)).cpu().numpy()
        assert np.array_equal(out, ro.resize(src, (dw, dh))), (h, w, c, dw, dh)


def test_batch_equals_single_frames():
    rng = np.random.default_rng(7)
    frames = rng.integers(0, 256, (70, 90, 120, 3), dtype=np.uint8)  # more frames than one chunk
    out = homo.resize(cu(frames), (52, 40)).cpu().numpy()
    for i in (0, 1, 33, 69):
        assert np.array_equal(out[i], ro.resize(frames[i], (52, 40))), i
    g = rng.integers(0, 256, (5, 31, 45), dtype=np.uint8)  # a batch of single-channel frames
    out = homo.resize(cu(g[..., None]), (20, 50)).cpu().numpy()
    for i in range(5):
        assert np.array_equal(out[i, :, :, 0], ro.resize(g[i], (20, 50))), i


def test_small_frame_chain_1080p():
    """vis_homo.py:73-78,90-91: resize to 852x480, Calib.scale, warp to the BEV -- against cv2's
    hashes of both stages."""
    ch = KAT["small_frame_chain"]
    img = util.seeded_frame(ch["seed"], 1080, 1920, 3, "uint8")
    small = homo.resize(cu(img), ch["new_uv"])
    assert util.sha256(small.cpu().numpy()) == ch["sha256_small"]
    bev = homo.warp_perspective(small, np.array(ch["H_bev_img_small"]), tuple(ch["bev_size"]))
    assert util.sha256(bev.cpu().numpy()) == ch["sha256_bev_small"]


def test_small_frame_helper_matches_the_two_calls():
    from bev_b200.calib import Calib
    from bev_b200.bev import BEVWorldSpec
    cam = util.load_json("cfg4_cams.json")[0]
    calib = Calib(vp1=np.array(cam["vp1"]), vp2=np.array(cam["vp2"]), height=cam["height"],
                  u_size=1920, v_size=1080)
    bspec = BEVWorldSpec(**{k: v for k, v in cam["bspec"].items() if v is not None and k not in ("x_max", "y_max")})
    ch = KAT["small_frame_chain"]
    img = cu(util.seeded_frame(ch["seed"], 1080, 1920, 3, "uint8"))
    small, bev = homo.warp_small_img_to_bev(img, calib, bspec, 852, 480)
    assert util.sha256(small.cpu().numpy()) == ch["sha256_small"]
    H_small = np.linalg.inv(bspec.gen_H_world_bev()).dot(
        calib.scale(align_corners=False, new_u=852, new_v=480).gen_H_world_img())
    assert np.allclose(H_small, np.array(ch["H_bev_img_small"]), rtol=1e-9, atol=1e-9)
    assert torch.equal(bev, homo.warp_perspective(small, H_small, tuple(ch["bev_size"])))


def test_full_batch_1080p():
    g = torch.Generator(device=DEV).manual_seed(3)
    frames = torch.randint(0, 256, (24, 1080, 1920, 3), dtype=torch.uint8, device=DEV, generator=g)
    out = homo.resize(frames, (852, 480))
    for i in (0, 23):
        assert np.array_equal(out[i].cpu().numpy(), ro.resize(frames[i].cpu().numpy(), (852, 480)))


def test_argument_errors():
    t = torch.zeros(8, 8, 3, dtype=torch.uint8, device=DEV)
    with pytest.raises(TypeError):
        homo.resize(t.float(), (4, 4))
    with pytest.raises(NativeError, match="INTER_LINEAR"):
        homo.resize(t, (4, 4), interpolation=0)
    with pytest.raises(NativeError, match="positive"):
        homo.resize(t, (0, 4))
    with pytest.raises(RuntimeError):
        homo.resize(t.cpu(), (4, 4))
    assert homo.resize(torch.zeros(0, 8, 8, 3, dtype=torch.uint8, device=DEV), (4, 4)).shape == (0, 4, 4, 3)


def test_two_channel_exact_half_matches_cv2_hashes():
    """2-channel frames downscaled by exactly 2 take cv2's round-half-even 2x2 mean, batched."""
    for case in util.load_json("resize_c2_half_hash.json")["cases"]:
        h, w, c = case["shape"]
        src = util.seeded_frame(case["seed"], h, w, c, "uint8")
        out = homo.resize(cu(np.stack([src] * 3)), case["dsize"]).cpu().numpy()
        for i in range(3):
            assert util.sha256(out[i]) == case["sha256"], (case, i)
