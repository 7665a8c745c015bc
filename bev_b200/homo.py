"""Homography construction (host, float64) and the B200 warp entry points.

Host geometry mirrors /root/reference/bev/homo.py (same names, argument meaning, return values);
it runs once per camera and stays numpy (SURVEY.md 8a row a2).  The per-pixel work the reference
delegates to ``cv2.warpPerspective`` (/root/reference/vis_homo.py:89,91;
/root/reference/bev/tool/compo.py:38,46,47) is served by the CUDA kernels behind
``warp_perspective`` below -- there is no CPU fallback: CPU tensors / a missing native library raise.
"""
import math

import numpy as np

from . import _native

# flag values follow cv2 so existing call sites keep working unchanged
INTER_NEAREST = 0
INTER_LINEAR = 1
INTER_AREA = 3
WARP_INVERSE_MAP = 16
BORDER_CONSTANT = 0
COLOR_YUV2BGR_NV12 = 91
COLOR_BGR2YUV_I420 = 128


# ----------------------------------------------------------------------------- host geometry

def homo_from_KRt(K, R=None, t=None, Rt_homo=None):
    """H_img_world = K * [r1 r2 t] for the world plane z = 0 (reference homo.py:6-26).

    Either ``Rt_homo`` (3x4 or 4x4 [R|t]) or both ``R`` and ``t`` must be given; a 3x4 ``K`` is cut
    to its left 3x3 block.  The result is not normalised.
    """
    K = np.asarray(K)
    if K.shape[1] == 4:
        K = K[:, :3]
    if Rt_homo is not None:
        assert R is None and t is None
        cols = np.asarray(Rt_homo)[:3][:, [0, 1, 3]]
    else:
        assert R is not None and t is not None
        t = np.asarray(t)
        cols = np.concatenate((np.asarray(R)[:, [0, 1]], t.reshape(-1, 1)), axis=1)
    return K.dot(cols)


def _dlt_normalised(src, dst):
    """Hartley-normalised DLT (least squares over all points), h22 scaled to 1."""
    def norm(p):
        c = p.mean(0)
        s = np.abs(p - c).mean(0)
        s = np.where(s < 1e-12, 1.0, s)
        T = np.array([[1 / s[0], 0, -c[0] / s[0]], [0, 1 / s[1], -c[1] / s[1]], [0, 0, 1.0]])
        return (p - c) / s, T
    a, Ta = norm(src)
    b, Tb = norm(dst)
    n = len(a)
    A = np.zeros((2 * n, 9))
    A[0::2, 0:2], A[0::2, 2] = a, 1
    A[0::2, 6:8], A[0::2, 8] = -b[:, :1] * a, -b[:, 0]
    A[1::2, 3:5], A[1::2, 5] = a, 1
    A[1::2, 6:8], A[1::2, 8] = -b[:, 1:] * a, -b[:, 1]
    _, _, vt = np.linalg.svd(A)
    H = np.linalg.inv(Tb).dot(vt[-1].reshape(3, 3)).dot(Ta)
    return H / H[2, 2]


def _refine_reprojection(H, src, dst, iters=30):
    """Gauss-Newton on the 8 free parameters minimising the reprojection error (n > 4 points)."""
    h = (H / H[2, 2]).reshape(-1)[:8].copy()
    for _ in range(iters):
        w = h[6] * src[:, 0] + h[7] * src[:, 1] + 1.0
        u = (h[0] * src[:, 0] + h[1] * src[:, 1] + h[2]) / w
        v = (h[3] * src[:, 0] + h[4] * src[:, 1] + h[5]) / w
        r = np.concatenate((u - dst[:, 0], v - dst[:, 1]))
        n = len(src)
        J = np.zeros((2 * n, 8))
        J[:n, 0], J[:n, 1], J[:n, 2] = src[:, 0] / w, src[:, 1] / w, 1 / w
        J[:n, 6], J[:n, 7] = -u * src[:, 0] / w, -u * src[:, 1] / w
        J[n:, 3], J[n:, 4], J[n:, 5] = src[:, 0] / w, src[:, 1] / w, 1 / w
        J[n:, 6], J[n:, 7] = -v * src[:, 0] / w, -v * src[:, 1] / w
        step = np.linalg.lstsq(J, -r, rcond=None)[0]
        h += step
        if np.abs(step).max() < 1e-14 * max(1.0, np.abs(h).max()):
            break
    return np.append(h, 1.0).reshape(3, 3)


def homo_from_pts(pts_src, pts_tgt):
    """H with pts_tgt ~ H * pts_src; both (n, 2) arrays, n >= 4 (reference homo.py:29-38).

    The reference calls ``cv2.findHomography`` with default arguments; when cv2 is importable the
    same call is made (bit-identical matrices), otherwise an equivalent normalised DLT with
    reprojection refinement is used.
    """
    pts_src = np.asarray(pts_src)
    pts_tgt = np.asarray(pts_tgt)
    assert pts_src.ndim == 2 and pts_src.shape[1] == 2, pts_src.shape
    assert pts_tgt.ndim == 2 and pts_tgt.shape[1] == 2, pts_tgt.shape
    try:
        import cv2
    except ImportError:
        cv2 = None
    if cv2 is not None:
        H, _ = cv2.findHomography(pts_src, pts_tgt)
        return H
    return homo_from_pts_numpy(pts_src, pts_tgt)


def homo_from_pts_numpy(pts_src, pts_tgt):
    """cv2-free path of :func:`homo_from_pts`."""
    s = np.asarray(pts_src, np.float64)
    d = np.asarray(pts_tgt, np.float64)
    H = _dlt_normalised(s, d)
    if len(s) > 4:
        H = _refine_reprojection(H, s, d)
    return H


def get_focal(vp1, vp2, pp):
    """Focal length from two orthogonal vanishing points and the principal point (homo.py:40-41)."""
    return math.sqrt(-np.dot(vp1[0:2] - pp[0:2], vp2[0:2] - pp[0:2]))


def get_K_from_f_pp(focal, pp):
    return np.array([[focal, 0, pp[0]], [0, focal, pp[1]], [0, 0, 1]])


def get_K_from_vps(vp1, vp2, pp):
    focal = get_focal(vp1, vp2, pp)
    return get_K_from_f_pp(focal, pp), focal


def homo_from_vps(vp1, vp2, height, u_size, v_size, pp=None):
    """H_img_world from two vanishing points and camera height (reference homo.py:52-96;
    Dubska et al. 2015).  ``pp`` defaults to the image centre ((u-1)/2, (v-1)/2)."""
    vp1 = np.asarray(vp1, dtype=np.float64)
    vp2 = np.asarray(vp2, dtype=np.float64)
    if pp is None:
        pp = np.array([(u_size - 1) * 0.5, (v_size - 1) * 0.5])
    K, f = get_K_from_vps(vp1, vp2, pp)

    pp3 = np.array([pp[0], pp[1], 0.0])
    d1 = np.array([vp1[0], vp1[1], f]) - pp3
    d2 = np.array([vp2[0], vp2[1], f]) - pp3
    n = np.cross(d1, d2)
    vp3 = n[0:2] / n[2] * f + pp            # third vanishing point on the image plane
    d3 = np.array([vp3[0], vp3[1], f]) - pp3

    d1 = d1 / np.linalg.norm(d1)
    d2 = d2 / np.linalg.norm(d2)
    d3 = d3 / np.linalg.norm(d3)

    # rows: the two road axes, the road normal with the camera height as offset, homogeneous row
    M = np.stack((np.append(d1, 0.0), np.append(d2, 0.0), np.append(d3, -1 * height),
                  [0, 0, 0, 1]), axis=0)
    M_inv = np.linalg.inv(M)
    K34 = np.concatenate((K, np.zeros((3, 1))), axis=1)
    return np.dot(K34, M_inv[:, [0, 1, 3]])


def get_vps_from_homo(H_img_world):
    H = H_img_world
    vp1 = np.array([H[0, 0] / H[2, 0], H[1, 0] / H[2, 0]])
    vp2 = np.array([H[0, 1] / H[2, 1], H[1, 1] / H[2, 1]])
    return vp1, vp2


def Rt_from_homo_K(H_img_world, K):
    """Decompose H = K [r1 r2 t] -> (R, t); R is orthonormalised by SVD (homo.py:111-128)."""
    G = np.linalg.inv(K).dot(H_img_world)
    G = G / np.sqrt((G[:, 0] ** 2).sum())
    r1, r2, tvec = G[:, 0], G[:, 1], G[:, 2]
    R = np.stack((r1, r2, np.cross(r1, r2)), axis=1)
    u, _, vt = np.linalg.svd(R)
    return np.matmul(u, vt), tvec


def get_KRt_from_homo(H_img_world, pp):
    vp1, vp2 = get_vps_from_homo(H_img_world)
    K, focal = get_K_from_vps(vp1, vp2, pp)
    R, t = Rt_from_homo_K(H_img_world, K)
    return K, focal, R, t


def Rt_from_pts_K_dist(pts_world, pts_img, K, dist_coeffs):
    """PnP pose (reference homo.py:130-135).  Needs cv2 (host-only helper, not on the hot path)."""
    import cv2
    _, rvec, tvec = cv2.solvePnP(pts_world, pts_img, K, dist_coeffs)
    R, _ = cv2.Rodrigues(rvec)
    return R, tvec


# ----------------------------------------------------------------------------- warp (hot path)

def invert_homography(H):
    """3x3 adjugate inverse evaluated like ``cv2.invert`` (bit-equal; ``np.linalg.inv`` is not).

    The warp kernel consumes the dst->src map; computing it this way is what keeps exact-tie
    pixels identical to cv2 (SURVEY.md App. A note 1).  Done by the native library on the host.
    """
    return _native.invert3x3(np.asarray(H, dtype=np.float64))


def compose_H_bev_img(calib, bspec):
    """H_bev_img = inv(H_world_bev) . H_world_img, exactly as /root/reference/vis_homo.py:61-63."""
    H_world_img = calib.gen_H_world_img()
    H_world_bev = bspec.gen_H_world_bev()
    return np.linalg.inv(H_world_bev).dot(H_world_img)


def warp_perspective(src, M, dsize, dst=None, flags=INTER_LINEAR, borderMode=BORDER_CONSTANT,
                     borderValue=0, mat_index=None, path=None):
    """Drop-in for ``cv2.warpPerspective(src, M, dsize[, dst, flags, borderMode, borderValue])``
    on CUDA tensors, batched.

    src   : cuda tensor, uint8 / float16 / float32, contiguous, shape (H, W), (H, W, C) or
            (N, H, W, C) with C in 1..4 (channels interleaved, as cv2 / the video reader gives).
    M     : float64 3x3 (numpy or CPU tensor), or (K, 3, 3) with ``mat_index`` (length N, values in
            [0, K)) choosing the matrix per frame; K == N without ``mat_index`` means one per frame.
            Forward (src->dst) unless ``flags`` has WARP_INVERSE_MAP -- same as cv2.
    dsize : (width, height) of the output, e.g. ``(bspec.u_size, bspec.v_size)``.
    Returns a new tensor (..., height, width[, C]) of src's dtype on src's device; the kernel is
    launched asynchronously on the current CUDA stream.

    uint8/float32 results are bit-identical to cv2 4.13 (nearest and bilinear); float16 equals
    float16(cv2(float32(src))).  Exception: float nearest warps of 1 or 4 channels follow cv2's own
    remap, not the IPP path cv2 takes for most of those shapes (DESIGN.md section 4).  Only BORDER_CONSTANT is implemented (all reference call sites
    use the default).  ``path`` ("auto" / "generic" / "fast") pins the kernel family for this call
    (tests and benchmarks); None leaves the choice to the library.
    """
    return _native.warp_perspective(src, M, dsize, dst, flags, borderMode, borderValue, mat_index, path)


def warp_img_to_bev(frames, calib, bspec, flags=INTER_LINEAR):
    """Image -> BEV warp of a frame batch with the calibration objects (vis_homo.py:61-63,89)."""
    H = compose_H_bev_img(calib, bspec)
    return warp_perspective(frames, H, (int(bspec.u_size), int(bspec.v_size)), flags=flags)


def nv12_to_bgr(src, dst=None):
    """Drop-in for ``cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)`` on CUDA tensors, batched: NV12 frames
    as a GPU video decoder gives them, (H*3/2, W) or (N, H*3/2, W) uint8 with H and W even, to
    (H, W, 3) / (N, H, W, 3) BGR, byte-identical to cv2 4.13.  Rows may be padded (a row stride,
    the decoder's pitch, larger than W) and frames may lie apart; the strides are read from the
    tensor."""
    return _native.nv12_to_bgr(src, dst)


def warp_perspective_nv12(src, M, dsize, dst=None, flags=INTER_LINEAR, borderMode=BORDER_CONSTANT,
                          borderValue=0, mat_index=None):
    """``warp_perspective(nv12_to_bgr(src), M, dsize, ...)`` in one pass, without the BGR copy of
    the frames: byte-identical to ``cv2.warpPerspective(cv2.cvtColor(f, COLOR_YUV2BGR_NV12), M,
    dsize, flags=flags, borderValue=borderValue)``.  src as for :func:`nv12_to_bgr`; M, mat_index,
    flags and borderValue (B, G, R) as for :func:`warp_perspective`.  Returns (h, w, 3) or
    (N, h, w, 3) BGR uint8; the kernel is launched asynchronously on the current CUDA stream."""
    return _native.warp_perspective_nv12(src, M, dsize, dst, flags, borderMode, borderValue, mat_index)


def warp_nv12_img_to_bev(frames, calib, bspec, flags=INTER_LINEAR):
    """:func:`warp_img_to_bev` for NV12 frames from a GPU video decoder (vis_homo.py:61-63,89)."""
    H = compose_H_bev_img(calib, bspec)
    return warp_perspective_nv12(frames, H, (int(bspec.u_size), int(bspec.v_size)), flags=flags)


def bgr_to_yuv420(src, layout="i420", dst=None):
    """Drop-in for ``cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)`` on CUDA tensors, batched: the colour
    conversion a video writer does to every BEV (vis_homo.py:110-111), on the GPU, so that 1.5
    instead of 3 bytes per pixel leave it.  src (H, W, 3) or (N, H, W, 3) uint8 BGR with H and W
    even; returns (H*3/2, W) or (N, H*3/2, W) uint8, byte-identical to cv2 4.13 for layout "i420"
    (libx264 / PyAV ``yuv420p``), or the same Y rows followed by H/2 rows of interleaved U, V for
    layout "nv12" (what GPU encoders take).  ``dst`` may have padded rows (a row stride, the
    encoder's pitch, larger than W) and frames that lie apart: it is written in place, the padding
    is left as it is."""
    return _native.bgr_to_yuv420(src, layout, dst)


def warp_perspective_yuv420(src, M, dsize, layout="i420", dst=None, flags=INTER_LINEAR,
                            borderMode=BORDER_CONSTANT, borderValue=0, mat_index=None):
    """``bgr_to_yuv420(warp_perspective(src, M, dsize, ...), layout)`` in one pass, without the BGR
    BEV: byte-identical to ``cv2.cvtColor(cv2.warpPerspective(f, M, dsize, flags=flags,
    borderValue=borderValue), COLOR_BGR2YUV_I420)`` (or its NV12 relayout).  src (H, W, 3) or
    (N, H, W, 3) uint8 BGR; M, mat_index, flags and borderValue (B, G, R) as for
    :func:`warp_perspective`; dsize = (w, h), both even; dst as for :func:`bgr_to_yuv420`.  Returns
    (h*3/2, w) or (N, h*3/2, w) uint8; the kernel is launched asynchronously on the current CUDA
    stream."""
    return _native.warp_perspective_yuv420(src, M, dsize, layout, dst, flags, borderMode, borderValue, mat_index)


def warp_perspective_nv12_yuv420(src, M, dsize, layout="i420", dst=None, flags=INTER_LINEAR,
                                 borderMode=BORDER_CONSTANT, borderValue=0, mat_index=None):
    """:func:`warp_perspective_yuv420` of NV12 frames from a GPU video decoder (src as for
    :func:`nv12_to_bgr`): decoder frames to encoder frames in one pass, byte-identical to
    ``cv2.cvtColor(cv2.warpPerspective(cv2.cvtColor(f, COLOR_YUV2BGR_NV12), M, dsize, ...),
    COLOR_BGR2YUV_I420)`` (or its NV12 relayout)."""
    return _native.warp_perspective_nv12_yuv420(src, M, dsize, layout, dst, flags, borderMode, borderValue,
                                                mat_index)


def warp_img_to_bev_yuv420(frames, calib, bspec, layout="i420", flags=INTER_LINEAR):
    """:func:`warp_img_to_bev` with YUV 4:2:0 BEVs for a video encoder (vis_homo.py:61-63,89,110-111)."""
    H = compose_H_bev_img(calib, bspec)
    return warp_perspective_yuv420(frames, H, (int(bspec.u_size), int(bspec.v_size)), layout, flags=flags)


def warp_nv12_img_to_bev_yuv420(frames, calib, bspec, layout="i420", flags=INTER_LINEAR):
    """:func:`warp_nv12_img_to_bev` with YUV 4:2:0 BEVs for a video encoder (vis_homo.py:61-63,89,110-111)."""
    H = compose_H_bev_img(calib, bspec)
    return warp_perspective_nv12_yuv420(frames, H, (int(bspec.u_size), int(bspec.v_size)), layout, flags=flags)


def warp_perspective_video_host(src, M, dsize, src_format="bgr", dst_format="i420", dst=None, flags=INTER_LINEAR,
                                borderMode=BORDER_CONSTANT, borderValue=0, mat_index=None):
    """The frame loop of vis_homo.py:85-111 for a CPU decoder and / or encoder: host frames in,
    host BEVs out, each format "bgr", "i420" (planar yuv420p, what PyAV's ``to_ndarray(format=
    "yuv420p")`` and ffmpeg ``-pix_fmt yuv420p`` pipes give and take) or "nv12".  Byte-identical to
    cv2's chain for the pair: ``cv2.cvtColor(f, COLOR_YUV2BGR_I420 / _NV12)`` for a YUV source,
    then ``cv2.warpPerspective(..., M, dsize, flags=flags, borderValue=borderValue)``, then
    ``cv2.cvtColor(..., COLOR_BGR2YUV_I420)`` (or its NV12 relayout) for a YUV destination.

    src / dst: numpy arrays or CPU tensors, uint8, contiguous; BGR (H, W, 3) / (N, H, W, 3), YUV
    (H*3/2, W) / (N, H*3/2, W) with H and W even.  Pinned memory gives full speed; pageable works.
    M, mat_index, flags and borderValue (B, G, R) as for :func:`warp_perspective`; dsize = (w, h),
    both even for a YUV destination.  Only the source rows the homographies reference (and the
    chroma rows under them) are uploaded, so a YUV frame moves half the bytes of a BGR one; copies
    and kernels overlap.  Synchronous: returns when the BEVs are in the host buffer."""
    return _native.warp_perspective_video_host(src, M, dsize, src_format, dst_format, dst, flags, borderMode,
                                               borderValue, mat_index)


def warp_img_to_bev_video_host(frames, calib, bspec, src_format="i420", dst_format="i420", flags=INTER_LINEAR):
    """:func:`warp_img_to_bev` on host video frames for a CPU codec (vis_homo.py:61-63,85-111):
    see :func:`warp_perspective_video_host`."""
    H = compose_H_bev_img(calib, bspec)
    return warp_perspective_video_host(frames, H, (int(bspec.u_size), int(bspec.v_size)), src_format, dst_format,
                                       flags=flags)


def warp_bev_to_img(bev_frames, calib, bspec, flags=INTER_LINEAR):
    """Inverse BEV -> image warp (north_star extension; same kernel, H inverted on the host)."""
    H = np.linalg.inv(compose_H_bev_img(calib, bspec))
    return warp_perspective(bev_frames, H, (int(calib.u_size), int(calib.v_size)), flags=flags)


def resize(src, dsize, dst=None, interpolation=INTER_LINEAR):
    """Drop-in for ``cv2.resize(src, dsize, interpolation=...)`` (uint8) on CUDA tensors, batched:
    the small-frame copy of the reference's frame loop (vis_homo.py:90).  src (H, W), (H, W, C)
    or (N, H, W, C); dsize = (width, height); interpolation INTER_LINEAR (cv2's default) or
    INTER_AREA (what OpenCV recommends for downscaling: no aliasing of fine texture).
    Bit-identical to cv2 4.13."""
    return _native.resize(src, dsize, interpolation, dst)


def warp_small_img_to_bev(frames, calib, bspec, new_u, new_v, flags=INTER_LINEAR, interpolation=INTER_LINEAR):
    """The small-frame path of vis_homo.py:73-78,90-91 on a frame batch: resize to (new_u, new_v)
    with ``interpolation``, rescale the calibration with ``Calib.scale(align_corners=False)`` and
    warp the small frames to the same BEV with ``flags``.  Returns (small_frames, bev_small)."""
    calib_small = calib.scale(align_corners=False, new_u=new_u, new_v=new_v)
    H_small = np.linalg.inv(bspec.gen_H_world_bev()).dot(calib_small.gen_H_world_img())
    small = resize(frames, (int(new_u), int(new_v)), interpolation=interpolation)
    return small, warp_perspective(small, H_small, (int(bspec.u_size), int(bspec.v_size)), flags=flags)


def resize_nv12(src, dsize, dst=None, interpolation=INTER_LINEAR):
    """``resize(nv12_to_bgr(src), dsize, interpolation=interpolation)`` in one pass, without the
    BGR copy of the frames: byte-identical to
    ``cv2.resize(cv2.cvtColor(f, COLOR_YUV2BGR_NV12), dsize, interpolation=interpolation)`` with
    INTER_LINEAR (the default) or INTER_AREA.  src as for :func:`nv12_to_bgr`; dsize = (width,
    height), 1..32767 each.  Returns (h, w, 3) or (N, h, w, 3) BGR uint8; the kernel is launched
    asynchronously on the current CUDA stream."""
    return _native.resize_nv12(src, dsize, dst, interpolation)


def warp_small_nv12_img_to_bev(frames, calib, bspec, new_u, new_v, flags=INTER_LINEAR,
                               interpolation=INTER_LINEAR):
    """:func:`warp_small_img_to_bev` for NV12 frames from a GPU video decoder (vis_homo.py:73-78,
    90-91): the small BGR frames come from :func:`resize_nv12` with ``interpolation``, without a
    full-size BGR copy.  Returns (small_frames, bev_small)."""
    calib_small = calib.scale(align_corners=False, new_u=new_u, new_v=new_v)
    H_small = np.linalg.inv(bspec.gen_H_world_bev()).dot(calib_small.gen_H_world_img())
    small = resize_nv12(frames, (int(new_u), int(new_v)), interpolation=interpolation)
    return small, warp_perspective(small, H_small, (int(bspec.u_size), int(bspec.v_size)), flags=flags)
