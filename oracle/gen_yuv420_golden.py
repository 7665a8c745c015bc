"""oracle/gen_yuv420_golden.py -- TEST INFRASTRUCTURE ONLY.  Writes tests/golden/yuv420_hash.json.

sha256 of cv2 4.13 outputs of cv2.cvtColor(..., COLOR_BGR2YUV_I420) on seeded frames
(oracle.synth.seeded_frame for BGR, oracle.nv12_oracle.seeded_nv12 for NV12): the conversion of a
1080p and a 4K frame; cv2.warpPerspective of a 1080p frame to the cfg-2 BEV (1024^2, the h_canon
map of homo_kat.json), bilinear and nearest, then the conversion; the same for cfg-4 camera 0
(H_bev_img and bspec of tests/golden/cfg4_cams.json); and the cfg-2 warp of an NV12 frame converted
with COLOR_YUV2BGR_NV12, then the conversion.  Before it stores anything it checks that
oracle.yuv420_oracle gives cv2's bytes on every case.  Needs only cv2 and numpy; the tests
regenerate the inputs from their seeds.

    python oracle/gen_yuv420_golden.py
"""
import hashlib
import json
import os
import sys

import cv2
import numpy as np

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, ROOT)
from oracle import yuv420_oracle as yo  # noqa: E402
from oracle.nv12_oracle import COLOR_YUV2BGR_NV12, seeded_nv12  # noqa: E402
from oracle.synth import seeded_frame  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "yuv420_hash.json")


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def i420(bgr):
    out = cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)
    assert np.array_equal(out, yo.bgr_to_i420(bgr)), "oracle differs from cv2"
    return out


def cases():
    H = json.load(open(os.path.join(ROOT, "tests", "golden", "homo_kat.json")))["h_canon"]
    cam = json.load(open(os.path.join(ROOT, "tests", "golden", "cfg4_cams.json")))[0]
    out = []
    for name, seed, (h, w) in (("convert_1080p", 4001, (1080, 1920)), ("convert_4k", 4002, (2160, 3840))):
        out.append({"name": name, "format": "bgr", "seed": seed, "shape": [h, w],
                    "sha256": sha256(i420(seeded_frame(seed, h, w, 3, "uint8")))})
    bgr = seeded_frame(4003, 1080, 1920, 3, "uint8")
    for name, flags in (("cfg2_warp_lin", cv2.INTER_LINEAR), ("cfg2_warp_nn", cv2.INTER_NEAREST)):
        bev = cv2.warpPerspective(bgr, np.array(H, np.float64), (1024, 1024), flags=flags)
        out.append({"name": name, "format": "bgr", "seed": 4003, "shape": [1080, 1920], "H": H,
                    "dsize": [1024, 1024], "flags": flags, "sha256": sha256(i420(bev))})
    dsize = [int(cam["bspec"]["u_size"]), int(cam["bspec"]["v_size"])]
    bev = cv2.warpPerspective(seeded_frame(4004, 1080, 1920, 3, "uint8"), np.array(cam["H_bev_img"]), tuple(dsize))
    out.append({"name": "cfg4_cam0_warp_lin", "format": "bgr", "seed": 4004, "shape": [1080, 1920],
                "H": cam["H_bev_img"], "dsize": dsize, "flags": cv2.INTER_LINEAR, "sha256": sha256(i420(bev))})
    bgr = cv2.cvtColor(seeded_nv12(4005, 1080, 1920), COLOR_YUV2BGR_NV12)
    bev = cv2.warpPerspective(bgr, np.array(H, np.float64), (1024, 1024))
    out.append({"name": "nv12_cfg2_warp_lin", "format": "nv12", "seed": 4005, "shape": [1080, 1920], "H": H,
                "dsize": [1024, 1024], "flags": cv2.INTER_LINEAR, "sha256": sha256(i420(bev))})
    return out


if __name__ == "__main__":
    c = cases()
    with open(OUT, "w") as f:
        json.dump({"cv2_version": cv2.__version__, "conversion": "COLOR_BGR2YUV_I420", "cases": c}, f, indent=1)
        f.write("\n")
    print("wrote", OUT)
