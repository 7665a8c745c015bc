"""oracle/gen_nv12_golden.py -- TEST INFRASTRUCTURE ONLY.  Writes tests/golden/nv12_hash.json.

sha256 of cv2 4.13 outputs on seeded full-size NV12 frames (oracle.nv12_oracle.seeded_nv12):
cv2.cvtColor(f, COLOR_YUV2BGR_NV12) at 1080p and 4K, and cv2.warpPerspective of the converted
1080p frame to the cfg-2 BEV (1024^2, the h_canon map of homo_kat.json), bilinear and nearest.
Needs only cv2 and numpy; the inputs are regenerated from their seeds by the tests.

    python oracle/gen_nv12_golden.py
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

OUT = os.path.join(ROOT, "tests", "golden", "nv12_hash.json")


def sha256(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def cases():
    H = json.load(open(os.path.join(ROOT, "tests", "golden", "homo_kat.json")))["h_canon"]
    out = []
    for name, seed, (h, w) in (("convert_1080p", 2001, (1080, 1920)), ("convert_4k", 2002, (2160, 3840))):
        bgr = cv2.cvtColor(seeded_nv12(seed, h, w), COLOR_YUV2BGR_NV12)
        out.append({"name": name, "seed": seed, "shape": [h, w], "sha256": sha256(bgr)})
    bgr = cv2.cvtColor(seeded_nv12(2003, 1080, 1920), COLOR_YUV2BGR_NV12)
    for name, flags in (("cfg2_warp_lin", cv2.INTER_LINEAR), ("cfg2_warp_nn", cv2.INTER_NEAREST)):
        dst = cv2.warpPerspective(bgr, np.array(H, np.float64), (1024, 1024), flags=flags)
        out.append({"name": name, "seed": 2003, "shape": [1080, 1920], "H": H, "dsize": [1024, 1024],
                    "flags": flags, "sha256": sha256(dst)})
    return out


if __name__ == "__main__":
    with open(OUT, "w") as f:
        json.dump({"cv2_version": cv2.__version__, "cases": cases()}, f, indent=1)
        f.write("\n")
    print("wrote", OUT)
