"""oracle/resize_nv12_oracle.py -- TEST INFRASTRUCTURE ONLY.

``cv2.resize(cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12), dsize)`` (cv2 4.13, default INTER_LINEAR)
as the composition of two oracles that are already pinned to cv2: ``nv12_oracle.nv12_to_bgr``
and ``resize_oracle.resize``.  Pinned against live cv2 and against the cv2 hashes of
tests/golden/nv12_resize_hash.json by tests/test_oracle_resize_nv12.py.

Also the host-side count of the luma and chroma samples the resize reads, for the benchmark's
algorithmic bytes.
"""
import numpy as np

from . import nv12_oracle, resize_oracle


def resize_nv12(f, dsize):
    """cv2.resize(cv2.cvtColor(f, COLOR_YUV2BGR_NV12), dsize) (INTER_LINEAR) of one (H*3/2, W)
    NV12 frame; dsize = (width, height)."""
    return resize_oracle.resize(nv12_oracle.nv12_to_bgr(f), dsize)


def resize_touched_samples(ssize, dsize):
    """(luma, chroma): distinct luma pixels the resize's taps with a non-zero weight read, and the
    distinct chroma samples (U,V pairs) those pixels use.  ssize / dsize = (width, height)."""
    w, h = int(ssize[0]), int(ssize[1])
    sx, a0, a1 = resize_oracle.axis_coefficients(w, int(dsize[0]), True)
    sy, b0, b1 = resize_oracle.axis_coefficients(h, int(dsize[1]), False)
    cols = np.zeros(w, bool)
    cols[sx[a0 != 0]] = True
    cols[np.minimum(sx + 1, w - 1)[a1 != 0]] = True
    rows = np.zeros(h, bool)
    rows[np.clip(sy, 0, h - 1)[b0 != 0]] = True
    rows[np.clip(sy + 1, 0, h - 1)[b1 != 0]] = True
    luma = int(cols.sum()) * int(rows.sum())
    chroma = int(cols.reshape(-1, 2).any(1).sum()) * int(rows.reshape(-1, 2).any(1).sum())
    return luma, chroma
