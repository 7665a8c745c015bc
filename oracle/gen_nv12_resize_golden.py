"""oracle/gen_nv12_resize_golden.py -- TEST INFRASTRUCTURE ONLY.  Writes
tests/golden/nv12_resize_hash.json.

sha256 of cv2 4.13 outputs on seeded full-size NV12 frames (oracle.nv12_oracle.seeded_nv12):
cv2.resize of the converted frame (cv2.cvtColor(f, COLOR_YUV2BGR_NV12)) for downscales, the exact
2x, an upscale and a dst width that is not a multiple of 4, and the small-frame chain of cfg-4
camera 0 (vis_homo.py:90-91): the 852x480 small frame, then its warp with the H_bev_img_small
and bev_size of resize_kat.json's small_frame_chain.  Needs only cv2 and numpy; the inputs are
regenerated from their seeds by the tests.

    python oracle/gen_nv12_resize_golden.py
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

OUT = os.path.join(ROOT, "tests", "golden", "nv12_resize_hash.json")

# (name, seed, (h, w) of the source, (dst_w, dst_h))
CASES = [
    ("1080p_852x480", 2101, (1080, 1920), (852, 480)),
    ("1080p_960x540", 2102, (1080, 1920), (960, 540)),  # exact 2x
    ("1080p_1280x720", 2103, (1080, 1920), (1280, 720)),
    ("4k_1920x1080", 2104, (2160, 3840), (1920, 1080)),
    ("480x852_up_1920x1080", 2105, (480, 852), (1920, 1080)),
    ("1080p_853x479", 2106, (1080, 1920), (853, 479)),  # dst width not a multiple of 4
]


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def cases():
    out = []
    for name, seed, (h, w), dsize in CASES:
        small = cv2.resize(cv2.cvtColor(seeded_nv12(seed, h, w), COLOR_YUV2BGR_NV12), dsize)
        out.append({"name": name, "seed": seed, "shape": [h, w], "dsize": list(dsize), "sha256": sha256(small)})
    chain = json.load(open(os.path.join(ROOT, "tests", "golden", "resize_kat.json")))["small_frame_chain"]
    seed, new_uv = 2107, tuple(chain["new_uv"])
    small = cv2.resize(cv2.cvtColor(seeded_nv12(seed, 1080, 1920), COLOR_YUV2BGR_NV12), new_uv)
    bev = cv2.warpPerspective(small, np.array(chain["H_bev_img_small"], np.float64), tuple(chain["bev_size"]))
    out.append({"name": "cfg4_cam0_small_frame_chain", "seed": seed, "shape": [1080, 1920], "dsize": list(new_uv),
                "sha256": sha256(small), "H": chain["H_bev_img_small"], "bev_size": chain["bev_size"],
                "sha256_bev": sha256(bev)})
    return out


if __name__ == "__main__":
    with open(OUT, "w") as f:
        json.dump({"cv2_version": cv2.__version__, "cases": cases()}, f, indent=1)
        f.write("\n")
    print("wrote", OUT)
