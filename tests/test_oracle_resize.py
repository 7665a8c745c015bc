"""CPU: the resize oracle (oracle/resize_oracle.py) against cv2.resize 4.13 outputs hashed in the
build container (tests/golden/resize_kat.json, written by oracle/gen_golden.py), and the
small-frame chain of the reference (vis_homo.py:73-78,90-91)."""
import numpy as np

from oracle import resize_oracle as ro
from oracle import warp_oracle as wo
from tests import util

KAT = util.load_json("resize_kat.json")


def case_input(case):
    h, w, c = case["shape"]
    src = util.seeded_frame(case["seed"], h, w, c, "uint8")
    return src[:, :, 0] if c == 1 else src


def test_oracle_matches_cv2_hashes():
    for case in KAT["cases"]:
        out = ro.resize(case_input(case), case["dsize"])
        assert out.shape[:2] == (case["dsize"][1], case["dsize"][0])
        assert util.sha256(out) == case["sha256"], case


def test_small_frame_chain():
    ch = KAT["small_frame_chain"]
    img = util.seeded_frame(ch["seed"], 1080, 1920, 3, "uint8")
    small = ro.resize(img, ch["new_uv"])
    assert util.sha256(small) == ch["sha256_small"]
    bev = wo.warp_perspective(small, np.array(ch["H_bev_img_small"]), tuple(ch["bev_size"]))
    assert util.sha256(bev) == ch["sha256_bev_small"]


def test_identity_and_constant():
    img = util.seeded_frame(5, 40, 60, 3, "uint8")
    assert np.array_equal(ro.resize(img, (60, 40)), img)
    flat = np.full((13, 17, 3), 201, np.uint8)
    assert np.array_equal(ro.resize(flat, (40, 29)), np.full((29, 40, 3), 201, np.uint8))


def test_scaled_calibration_reproduces_the_small_homography():
    """Host mirror: Calib.scale(align_corners=False) (bev/calib.py:142-198) gives the reference's
    H_bev_img_small (vis_homo.py:73-78) for cfg-4 camera 0."""
    from bev_b200.calib import Calib
    from bev_b200.bev import BEVWorldSpec
    cam = util.load_json("cfg4_cams.json")[0]
    calib = Calib(vp1=np.array(cam["vp1"]), vp2=np.array(cam["vp2"]), height=cam["height"],
                  u_size=1920, v_size=1080)
    bspec = BEVWorldSpec(**{k: v for k, v in cam["bspec"].items() if v is not None and k not in ("x_max", "y_max")})
    ch = KAT["small_frame_chain"]
    small = calib.scale(align_corners=False, new_u=ch["new_uv"][0], new_v=ch["new_uv"][1])
    H = np.linalg.inv(bspec.gen_H_world_bev()).dot(small.gen_H_world_img())
    assert np.allclose(H, np.array(ch["H_bev_img_small"]), rtol=1e-9, atol=1e-9)


def test_two_channel_exact_half_matches_cv2_hashes():
    """cv2 sends an exact 2x downscale to INTER_AREA; for 2 channels that rounds the 2x2 mean half
    to even, which the bilinear formula does not (tests/golden/resize_c2_half_hash.json)."""
    for case in util.load_json("resize_c2_half_hash.json")["cases"]:
        h, w, c = case["shape"]
        out = ro.resize(util.seeded_frame(case["seed"], h, w, c, "uint8"), case["dsize"])
        assert util.sha256(out) == case["sha256"], case
