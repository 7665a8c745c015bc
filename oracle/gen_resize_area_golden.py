"""oracle/gen_resize_area_golden.py -- TEST INFRASTRUCTURE ONLY.  Writes
tests/golden/resize_area_hash.json.

sha256 of cv2 4.13 outputs of cv2.resize(..., interpolation=cv2.INTER_AREA) on seeded frames
(oracle.synth.seeded_frame for BGR, oracle.nv12_oracle.seeded_nv12 for NV12, converted with
cv2.cvtColor(f, COLOR_YUV2BGR_NV12)).  The shapes cover each of cv2's three INTER_AREA branches:
1080p -> 852x480 and a mixed-axis downscale (general area), the exact 2x to 960x540 and
4K -> 1080p and an exact 3x (integer cells), an upscale and an up/down mix (bilinear with area
coefficients); and the small-frame chain of cfg-4 camera 0 (vis_homo.py:90-91) with INTER_AREA:
the 852x480 small frame, then its warp with the H_bev_img_small and bev_size of resize_kat.json's
small_frame_chain.  Needs only cv2 and numpy; the tests regenerate the inputs from their seeds.

    python oracle/gen_resize_area_golden.py
"""
import hashlib
import json
import os
import sys

import cv2
import numpy as np

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, ROOT)
from oracle.nv12_oracle import COLOR_YUV2BGR_NV12, seeded_nv12  # noqa: E402
from oracle.synth import seeded_frame  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "resize_area_hash.json")

# (name, (h, w) of the source, (dst_w, dst_h)); case k takes the seeds SEED0 + k (BGR) and
# SEED0 + 50 + k (NV12)
SHAPES = [
    ("1080p_852x480", (1080, 1920), (852, 480)),
    ("1080p_960x540", (1080, 1920), (960, 540)),      # exact 2x
    ("4k_1920x1080", (2160, 3840), (1920, 1080)),     # exact 2x
    ("1080p_640x360", (1080, 1920), (640, 360)),      # exact 3x
    ("1080p_1280x360", (1080, 1920), (1280, 360)),    # 1.5x across, 3x down
    ("480x852_up_1920x1080", (480, 852), (1920, 1080)),
    ("1080p_2400x500", (1080, 1920), (2400, 500)),    # up across, down vertically
]
SEED0 = 3100


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def cases():
    out = []
    for k, (name, (h, w), dsize) in enumerate(SHAPES):
        seed = SEED0 + k
        small = cv2.resize(seeded_frame(seed, h, w, 3, "uint8"), dsize, interpolation=cv2.INTER_AREA)
        out.append({"name": "bgr_" + name, "format": "bgr", "seed": seed, "shape": [h, w], "dsize": list(dsize),
                    "sha256": sha256(small)})
        seed = SEED0 + 50 + k
        bgr = cv2.cvtColor(seeded_nv12(seed, h, w), COLOR_YUV2BGR_NV12)
        small = cv2.resize(bgr, dsize, interpolation=cv2.INTER_AREA)
        out.append({"name": "nv12_" + name, "format": "nv12", "seed": seed, "shape": [h, w], "dsize": list(dsize),
                    "sha256": sha256(small)})
    chain = json.load(open(os.path.join(ROOT, "tests", "golden", "resize_kat.json")))["small_frame_chain"]
    new_uv, H, bev_size = tuple(chain["new_uv"]), np.array(chain["H_bev_img_small"], np.float64), tuple(chain["bev_size"])
    for fmt, seed in (("bgr", SEED0 + 99), ("nv12", SEED0 + 98)):
        img = seeded_frame(seed, 1080, 1920, 3, "uint8") if fmt == "bgr" else \
            cv2.cvtColor(seeded_nv12(seed, 1080, 1920), COLOR_YUV2BGR_NV12)
        small = cv2.resize(img, new_uv, interpolation=cv2.INTER_AREA)
        bev = cv2.warpPerspective(small, H, bev_size)
        out.append({"name": fmt + "_cfg4_cam0_small_frame_chain", "format": fmt, "seed": seed, "shape": [1080, 1920],
                    "dsize": list(new_uv), "sha256": sha256(small), "H": chain["H_bev_img_small"],
                    "bev_size": chain["bev_size"], "sha256_bev": sha256(bev)})
    return out


if __name__ == "__main__":
    with open(OUT, "w") as f:
        json.dump({"cv2_version": cv2.__version__, "interpolation": "INTER_AREA", "cases": cases()}, f, indent=1)
        f.write("\n")
    print("wrote", OUT)
