"""ctypes binding of libbev_b200.so (the C ABI declared in include/bev_b200.h).

PyTorch is only the plumbing here -- device memory, the current CUDA stream -- and every compute
call goes through the C ABI with raw pointers.  There is no CPU fallback: a missing library, a CPU
tensor or a non-sm_100 device raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libbev_b200.so")

U8, F16, F32, F64 = 0, 1, 2, 3
MODE = {"bev": 0, "world": 1}

_lib = None

_c_int = ctypes.c_int
_c_i64 = ctypes.c_int64
_vp = ctypes.c_void_p
_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)
_i32p = ctypes.POINTER(ctypes.c_int32)
_fp = ctypes.POINTER(ctypes.c_float)

# name -> (restype, argtypes); kept in step with include/bev_b200.h (tests/test_capi_symbols.py)
SIGNATURES = {
    "bevk_version": (_c_int, []),
    "bevk_last_error": (ctypes.c_char_p, []),
    "bevk_device_info": (_c_int, [_ip, _ip, _ip]),
    "bevk_invert3x3": (_c_int, [_dp, _dp]),
    "bevk_warp_perspective": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                       _c_int, _dp, _c_int, _i32p, _c_int, _c_int, _dp, _vp]),
    "bevk_warp_perspective_path": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                            _c_int, _dp, _c_int, _i32p, _c_int, _c_int, _dp, _c_int, _vp]),
    "bevk_warp_perspective_host": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int,
                                            _c_int, _c_int, _dp, _c_int, _i32p, _c_int, _c_int,
                                            _dp]),
    "bevk_warp_perspective_video_host": (_c_int, [_vp, _c_int, _vp, _c_int] + [_c_int] * 5 + [_dp, _c_int, _i32p,
                                                                                       _c_int, _c_int, _dp]),
    "bevk_warp_perspective_video_host_small": (_c_int, [_vp, _c_int, _vp, _c_int, _vp, _vp] + [_c_int] * 7
                                               + [_dp, _dp, _c_int, _i32p, _c_int, _c_int, _c_int, _dp]),
    "bevk_warp_host_rows": (_c_int, [_c_int, _c_int, _c_int, _c_int, _dp, _c_int, _c_int, _ip]),
    "bevk_warp_set_path": (_c_int, [_c_int]),
    "bevk_warp_touched_pixels": (_c_i64, [_c_int, _c_int, _c_int, _c_int, _dp, _c_int, _ip]),
    "bevk_nv12_to_bgr": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _vp]),
    "bevk_warp_perspective_nv12": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _c_int, _c_int,
                                            _dp, _c_int, _i32p, _c_int, _c_int, _dp, _vp]),
    "bevk_bgr_to_yuv420": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_i64, _vp]),
    "bevk_warp_perspective_yuv420": (_c_int, [_vp, _vp] + [_c_int] * 6 + [_c_int, _c_i64, _dp, _c_int, _i32p, _c_int,
                                                                          _c_int, _dp, _vp]),
    "bevk_warp_perspective_nv12_yuv420": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _c_int, _c_int,
                                                   _c_int, _c_int, _c_i64, _dp, _c_int, _i32p, _c_int, _c_int, _dp,
                                                   _vp]),
    "bevk_warp_perspective_dmat": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int,
                                            _c_int, _dp, _c_int, _i32p, _c_int, _c_int, _dp, _vp]),
    "bevk_warp_perspective_nv12_dmat": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _c_int, _c_int,
                                                 _dp, _c_int, _i32p, _c_int, _c_int, _dp, _vp]),
    "bevk_warp_perspective_yuv420_dmat": (_c_int, [_vp, _vp] + [_c_int] * 6 + [_c_int, _c_i64, _dp, _c_int, _i32p,
                                                                               _c_int, _c_int, _dp, _vp]),
    "bevk_warp_perspective_nv12_yuv420_dmat": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _c_int,
                                                        _c_int, _c_int, _c_int, _c_i64, _dp, _c_int, _i32p, _c_int,
                                                        _c_int, _dp, _vp]),
    "bevk_resize": (_c_int, [_vp, _vp] + [_c_int] * 8 + [_vp]),
    "bevk_resize_nv12": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _c_int, _c_int, _vp]),
    "bevk_resize_nv12_interp": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _c_int, _c_int, _c_int,
                                         _vp]),
    "bevk_composite_u8c3": (_c_int, [_vp, _vp, _vp, _vp, _c_i64, _c_int, _vp]),
    "bevk_composite_bev_u8c3": (_c_int, [_vp, _vp, _vp, _vp] + [_c_int] * 8 + [_dp, _dp, _c_int, _vp]),
    "bevk_composite_bev_u8c3_dmat": (_c_int, [_vp, _vp, _vp, _vp] + [_c_int] * 8 + [_dp, _dp, _c_int, _vp]),
    "bevk_pts_project": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _dp, _vp]),
    "bevk_xywhr2xyxy": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _dp, _vp]),
    "bevk_xy82xywhr": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _dp, _vp]),
    "bevk_rbox_world_bev": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _dp, _vp]),
    "bevk_rboxtt_world_bev": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _dp, _vp]),
    "bevk_rbox_zt2tt_world": (_c_int, [_vp, _vp, _c_i64, _c_int, _dp, _dp, _vp]),
    "bevk_angle_world_bev": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _dp, _vp]),
    "bevk_dist_world_bev": (_c_int, [_vp, _vp, _c_i64, _c_int, _dp, _vp]),
    "bevk_xywhr2xyvec": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _vp]),
    "bevk_xy82xyvec": (_c_int, [_vp, _vp, _c_i64, _c_int, _vp]),
    "bevk_v2yaw": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _vp]),
    "bevk_yaw2v": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _vp]),
    "bevk_yaw2mat": (_c_int, [_vp, _vp, _c_i64, _c_int, _c_int, _vp]),
    "bevk_rbox_iou_matrix": (_c_int, [_vp, _c_i64, _c_int, _vp, _c_i64, _c_int, _vp, _c_int,
                                      ctypes.c_double, _vp]),
    "bevk_xywhr2xyxy_host": (_c_int, [_fp, _fp, _c_i64, _c_int, _dp]),
    "bevk_xy82xywhr_host": (_c_int, [_fp, _fp, _c_i64, _c_int, _dp]),
}


class NativeError(RuntimeError):
    """An entry point of libbev_b200.so returned an error code."""


def lib():
    """Load libbev_b200.so (once).  Raises if it has not been built -- never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "bev_b200: native library %s is missing. Build it with "
                "`python -c 'import __graft_entry__ as g; g.build()'` or `make -C bev_b200/csrc`. "
                "There is no CPU fallback." % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def _check(rc, what):
    if rc != 0:
        msg = lib().bevk_last_error().decode("utf-8", "replace")
        if rc == -4:
            # the reference raises AssertionError here (rbox_torch.py:140,161)
            raise AssertionError(msg)
        raise NativeError("%s failed (code %d): %s" % (what, rc, msg))


def _mat(H, what="H"):
    a = np.ascontiguousarray(_to_numpy(H), dtype=np.float64)
    if a.shape != (3, 3):
        raise ValueError("%s must be 3x3, got %s" % (what, a.shape))
    return a


def _to_numpy(a):
    if hasattr(a, "detach"):  # torch tensor: homographies live on the host (SURVEY.md 8b)
        if a.is_cuda:
            a = a.cpu()       # explicit sync, same as the reference's assert on a CUDA H
        return a.detach().numpy()
    return np.asarray(a)


def _dptr(a):
    return a.ctypes.data_as(_dp)


def invert3x3(H):
    H = _mat(H)
    M = np.empty((3, 3), np.float64)
    lib().bevk_invert3x3(_dptr(H), _dptr(M))
    return M


def device_info():
    sm, mj, mn = _c_int(), _c_int(), _c_int()
    _check(lib().bevk_device_info(ctypes.byref(sm), ctypes.byref(mj), ctypes.byref(mn)),
           "bevk_device_info")
    return sm.value, mj.value, mn.value


def _stream_ptr(t):
    import torch
    return _vp(torch.cuda.current_stream(t.device).cuda_stream)


def _require_cuda(t, what):
    import torch
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor, got %s" % (what, type(t).__name__))
    if not t.is_cuda:
        raise RuntimeError("%s is on %s: bev_b200 runs on CUDA (sm_100a) only, there is no CPU "
                           "fallback" % (what, t.device))


def _aligned(t, align=4):
    """Contiguous tensor whose data pointer is `align`-byte aligned (a contiguous VIEW at an odd
    byte offset -- e.g. the second half of a concatenated uint8 batch -- is copied)."""
    t = t.contiguous()
    if t.data_ptr() % align:
        t = t.clone()
    return t


def _out(out, shape, dtype, device, what="dst"):
    """A new tensor of this shape, dtype and device, or `out` after checking that it is a contiguous one."""
    import torch
    shape = tuple(shape)
    if out is None:
        return torch.empty(shape, dtype=dtype, device=device)
    _require_cuda(out, what)
    if tuple(out.shape) != shape or out.dtype != dtype or out.device != device or not out.is_contiguous():
        raise ValueError("%s must be a contiguous %s tensor of shape %s on %s, got %s %s on %s"
                         % (what, dtype, shape, device, out.dtype, tuple(out.shape), out.device))
    return out


def _warp_dtype(t):
    import torch
    code = {torch.uint8: U8, torch.float16: F16, torch.float32: F32}.get(t.dtype)
    if code is None:
        raise TypeError("warp_perspective supports uint8 / float16 / float32, got %s" % t.dtype)
    return code


class _Mats:
    """The matrices of one warp call as the C ABI takes them: ptr (host, or with dmat device, float64
    3x3 matrices), n (their count) and idx (host int32 mat_index or None).  keep holds what ptr points
    into for the length of the call."""

    def __init__(self, M, n_frames, mat_index, dmat, device):
        if dmat:
            import torch
            if not isinstance(M, torch.Tensor) or not M.is_cuda:
                raise TypeError("M must be a CUDA tensor for the device-matrix warps, got %s"
                                % (getattr(M, "device", type(M).__name__),))
            if M.device != device:
                raise ValueError("M is on %s, the frames on %s" % (M.device, device))
            if M.dtype != torch.float64:
                raise TypeError("M must be float64, got %s" % (M.dtype,))
            Ms = (M[None] if M.dim() == 2 else M).contiguous()  # stream-ordered; no host read
            if Ms.dim() != 3 or tuple(Ms.shape[1:]) != (3, 3) or Ms.shape[0] == 0:
                raise ValueError("M must be 3x3 or (K,3,3), got %s" % (tuple(M.shape),))
        else:
            Ms = np.ascontiguousarray(_to_numpy(M), dtype=np.float64)
            Ms = Ms[None] if Ms.ndim == 2 else Ms
            if Ms.ndim != 3 or Ms.shape[1:] != (3, 3):
                raise ValueError("M must be 3x3 or (K,3,3), got %s" % (Ms.shape,))
        self.ptr = ctypes.cast(Ms.data_ptr(), _dp) if dmat else _dptr(Ms)
        self.keep, self.n, self.idx = Ms, Ms.shape[0], None
        # the indices are planned on the host, for device matrices too
        if mat_index is not None:
            self.idx = np.ascontiguousarray(_to_numpy(mat_index), dtype=np.int32).reshape(-1)
            if self.idx.shape[0] != n_frames:
                raise ValueError("mat_index has %d entries for %d frames" % (self.idx.shape[0], n_frames))
        elif self.n not in (1, n_frames):
            raise ValueError("%d matrices for %d frames needs mat_index" % (self.n, n_frames))

    def idx_ptr(self):
        return self.idx.ctypes.data_as(_i32p) if self.idx is not None else None


def _border(borderValue):
    b = np.zeros(4, np.float64)
    v = np.atleast_1d(np.asarray(borderValue, dtype=np.float64)).reshape(-1)[:4]
    b[:len(v)] = v  # cv2.Scalar semantics: missing channels are 0
    return b


def _frames_view(src):
    """(N, H, W, C) view of a (H,W) / (H,W,C) / (N,H,W,C) tensor or array + how to undo it."""
    if src.ndim == 2:
        return src[None, :, :, None], lambda o: o[0, :, :, 0]
    if src.ndim == 3:
        return src[None], lambda o: o[0]
    if src.ndim == 4:
        return src, lambda o: o
    raise ValueError("src must be (H,W), (H,W,C) or (N,H,W,C); got shape %s" % (tuple(src.shape),))


_PATHS = {None: -1, "auto": 0, "generic": 1, "fast": 2}


def warp_perspective(src, M, dsize, dst=None, flags=1, borderMode=0, borderValue=0,
                     mat_index=None, path=None):
    """path: None (the calling thread's default, see set_warp_path), "auto", "generic" (direct-gather
    kernels) or "fast" (staged kernel; raises if the shape does not qualify)."""
    return _warp(src, "frames", M, dsize, dst, "frames", flags, borderMode, borderValue, mat_index, False,
                 path=_PATHS.get(path, path))


def warp_perspective_dmat(src, M, dsize, dst=None, flags=1, borderMode=0, borderValue=0, mat_index=None):
    """warp_perspective with M a CUDA float64 tensor (3,3) or (K,3,3) on src's device, read by the
    kernels when they run on the current stream: no host sync, and a captured CUDA graph replays the
    matrices last written into M.  Always the direct-gather kernels; mat_index stays on the host."""
    return _warp(src, "frames", M, dsize, dst, "frames", flags, borderMode, borderValue, mat_index, True)


def warp_perspective_host(src, M, dsize, dst=None, flags=1, borderMode=0, borderValue=0,
                          mat_index=None):
    """Host-buffer form: src / dst are numpy arrays or CPU tensors (pinned for full PCIe speed)."""
    s = _to_numpy(src) if not isinstance(src, np.ndarray) else src
    code = {np.dtype("uint8"): U8, np.dtype("float16"): F16, np.dtype("float32"): F32}.get(s.dtype)
    if code is None:
        raise TypeError("warp_perspective_host supports uint8/float16/float32, got %s" % s.dtype)
    s4, undo = _frames_view(s)
    s4 = np.ascontiguousarray(s4)
    n, h, w, c = s4.shape
    dw, dh = int(dsize[0]), int(dsize[1])
    m = _Mats(M, n, mat_index, False, None)
    if dst is None:
        out4 = np.empty((n, dh, dw, c), s4.dtype)
    else:
        out4 = _to_numpy(dst).reshape(n, dh, dw, c)
        if out4.dtype != s4.dtype or not out4.flags["C_CONTIGUOUS"]:
            raise ValueError("dst must be C-contiguous with src's dtype")
    b = _border(borderValue)
    rc = lib().bevk_warp_perspective_host(
        _vp(s4.ctypes.data), _vp(out4.ctypes.data), n, h, w, dh, dw, c, code, m.ptr, m.n, m.idx_ptr(),
        int(flags), int(borderMode), _dptr(b))
    _check(rc, "bevk_warp_perspective_host")
    return dst if dst is not None else undo(out4)


def _nv12_frames(src):
    """(frames view (N, H*3/2, W), N, H, W, (pitch, frame stride)) of an NV12 tensor (H*3/2, W) or
    (N, H*3/2, W).  Pitch and frame stride come from the tensor's strides, so a decoder surface
    with padded rows is used as it is."""
    import torch
    if not isinstance(src, torch.Tensor):
        raise TypeError("src must be a torch.Tensor, got %s" % type(src).__name__)
    if not src.is_cuda:
        raise ValueError("src is on %s: bev_b200 runs on CUDA (sm_100a) only, there is no CPU fallback"
                         % (src.device,))
    if src.dtype != torch.uint8:
        raise ValueError("NV12 frames are uint8, got %s" % (src.dtype,))
    if src.dim() not in (2, 3):
        raise ValueError("NV12 frames must be (H*3/2, W) or (N, H*3/2, W); got shape %s" % (tuple(src.shape),))
    s3 = src[None] if src.dim() == 2 else src
    n, rows, w = s3.shape
    if rows == 0 or rows % 3 or w % 2:
        raise ValueError("NV12 frames need H*3/2 rows for an even H and an even width W; got %d rows x %d"
                         % (rows, w))
    if s3.stride(2) != 1:
        raise ValueError("NV12 rows must be contiguous (inner stride 1), got stride %d" % s3.stride(2))
    pitch = s3.stride(1)
    if pitch < w:
        raise ValueError("NV12 row pitch %d is smaller than the width %d" % (pitch, w))
    fstride = s3.stride(0) if n > 1 else pitch * rows
    return s3, n, rows // 3 * 2, w, (pitch, fstride)


def nv12_to_bgr(src, dst=None):
    """cv2.cvtColor(f, COLOR_YUV2BGR_NV12) on CUDA uint8 NV12 frames (H*3/2, W) or (N, H*3/2, W)
    -> (H, W, 3) or (N, H, W, 3) BGR."""
    import torch
    s3, n, h, w, (pitch, fstride) = _nv12_frames(src)
    dst = _out(dst, (n, h, w, 3) if src.dim() == 3 else (h, w, 3), torch.uint8, src.device)
    with torch.cuda.device(src.device):
        rc = lib().bevk_nv12_to_bgr(_vp(s3.data_ptr()), _vp(dst.data_ptr()), n, h, w, pitch, fstride,
                                    _stream_ptr(src))
    _check(rc, "bevk_nv12_to_bgr")
    return dst


def warp_perspective_nv12(src, M, dsize, dst=None, flags=1, borderMode=0, borderValue=0, mat_index=None):
    """warp_perspective of nv12_to_bgr(src) in one pass: (H*3/2, W) -> (h, w, 3), (N, H*3/2, W) ->
    (N, h, w, 3) BGR uint8.  M / mat_index as for warp_perspective."""
    return _warp(src, "nv12", M, dsize, dst, "bgr", flags, borderMode, borderValue, mat_index, False)


def warp_perspective_nv12_dmat(src, M, dsize, dst=None, flags=1, borderMode=0, borderValue=0, mat_index=None):
    """warp_perspective_nv12 with M a CUDA float64 tensor, as for warp_perspective_dmat."""
    return _warp(src, "nv12", M, dsize, dst, "bgr", flags, borderMode, borderValue, mat_index, True)


YUV_LAYOUTS = {"i420": 0, "nv12": 1}


def _yuv_layout(layout):
    code = YUV_LAYOUTS.get(layout)
    if code is None:
        raise ValueError("layout must be 'i420' or 'nv12', got %r" % (layout,))
    return code


def bgr_to_yuv420(src, layout="i420", dst=None):
    """cv2.cvtColor(f, COLOR_BGR2YUV_I420) (layout "i420") or its NV12 relayout ("nv12") on CUDA
    uint8 BGR frames (H, W, 3) or (N, H, W, 3) -> (H*3/2, W) or (N, H*3/2, W)."""
    import torch
    s4, n, h, w, batched, _ = _warp_src(src, "bgr")
    code = _yuv_layout(layout)
    dst, d3, dst_args = _warp_dst(dst, "yuv", src, s4, n, h, w, batched, code)
    with torch.cuda.device(src.device):
        rc = lib().bevk_bgr_to_yuv420(_vp(s4.data_ptr()), _vp(d3.data_ptr()), n, h, w, *dst_args, _stream_ptr(src))
    _check(rc, "bevk_bgr_to_yuv420")
    return dst


def warp_perspective_yuv420(src, M, dsize, layout="i420", dst=None, flags=1, borderMode=0, borderValue=0,
                            mat_index=None):
    """bgr_to_yuv420(warp_perspective(src, M, dsize, ...), layout) in one pass: CUDA uint8 BGR
    frames (H, W, 3) or (N, H, W, 3) -> (h*3/2, w) or (N, h*3/2, w)."""
    return _warp(src, "bgr", M, dsize, dst, "yuv", flags, borderMode, borderValue, mat_index, False, layout)


def warp_perspective_yuv420_dmat(src, M, dsize, layout="i420", dst=None, flags=1, borderMode=0, borderValue=0,
                                 mat_index=None):
    """warp_perspective_yuv420 with M a CUDA float64 tensor, as for warp_perspective_dmat."""
    return _warp(src, "bgr", M, dsize, dst, "yuv", flags, borderMode, borderValue, mat_index, True, layout)


def warp_perspective_nv12_yuv420(src, M, dsize, layout="i420", dst=None, flags=1, borderMode=0, borderValue=0,
                                 mat_index=None):
    """bgr_to_yuv420(warp_perspective_nv12(src, M, dsize, ...), layout) in one pass: CUDA uint8 NV12
    frames (H*3/2, W) or (N, H*3/2, W), any pitch and frame stride -> (h*3/2, w) or (N, h*3/2, w)."""
    return _warp(src, "nv12", M, dsize, dst, "yuv", flags, borderMode, borderValue, mat_index, False, layout)


def warp_perspective_nv12_yuv420_dmat(src, M, dsize, layout="i420", dst=None, flags=1, borderMode=0,
                                      borderValue=0, mat_index=None):
    """warp_perspective_nv12_yuv420 with M a CUDA float64 tensor, as for warp_perspective_dmat."""
    return _warp(src, "nv12", M, dsize, dst, "yuv", flags, borderMode, borderValue, mat_index, True, layout)


def _warp_src(src, kind):
    """(frames view, n, h, w, whether src has a frame axis, C arguments) of CUDA frames of a warp dtype
    (H,W), (H,W,C) or (N,H,W,C) ("frames"), uint8 BGR (H, W, 3) or (N, H, W, 3) ("bgr") or NV12 ("nv12")."""
    import torch
    if kind == "nv12":
        s3, n, h, w, args = _nv12_frames(src)
        return s3, n, h, w, src.dim() == 3, args
    _require_cuda(src, "src")
    if kind == "bgr" and (src.dtype != torch.uint8 or src.dim() not in (3, 4) or src.shape[-1] != 3):
        raise ValueError("src must be uint8 (H, W, 3) or (N, H, W, 3), got %s %s" % (src.dtype, tuple(src.shape)))
    _warp_dtype(src)
    s4 = _frames_view(src)[0].contiguous()
    return s4, s4.shape[0], s4.shape[1], s4.shape[2], src.dim() == 4, ()


def _warp_dst(dst, kind, src, s, n, h, w, batched, layout):
    """(what the call returns, frames view written, C arguments) of a new or given dst of n h x w frames,
    batched as src: frames shaped as src ("frames"), uint8 BGR ("bgr") or YUV 4:2:0 of this layout code
    ("yuv"; pitch and frame stride from the strides, so padded encoder surfaces are written in place)."""
    import torch
    if kind == "frames":  # a given dst may have any rank whose (N, H, W, C) view has the output's shape
        if dst is not None:
            _require_cuda(dst, "dst")
        out4 = _out(None if dst is None else _frames_view(dst)[0], (n, h, w, s.shape[3]), src.dtype, src.device)
        return dst if dst is not None else _frames_view(src)[1](out4), out4, (s.shape[3], _warp_dtype(src))
    if kind == "bgr":
        dst = _out(dst, (n, h, w, 3) if batched else (h, w, 3), torch.uint8, src.device)
        return dst, dst, ()
    if h % 2 or w % 2:
        raise ValueError("YUV 4:2:0 frames need an even width and height, got %dx%d" % (w, h))
    shape = (n, h * 3 // 2, w) if batched else (h * 3 // 2, w)
    if dst is None:
        dst = torch.empty(shape, dtype=torch.uint8, device=src.device)
    _require_cuda(dst, "dst")
    if tuple(dst.shape) != shape or dst.dtype != torch.uint8 or dst.device != src.device:
        raise ValueError("dst must be a uint8 tensor of shape %s on %s, got %s %s on %s"
                         % (shape, src.device, dst.dtype, tuple(dst.shape), dst.device))
    d3 = dst if batched else dst[None]
    if d3.stride(2) != 1 or d3.stride(1) < w:
        raise ValueError("dst rows must be contiguous and at least %d bytes apart, got strides %s"
                         % (w, tuple(d3.stride())))
    pitch = d3.stride(1)
    return dst, d3, (layout, pitch, d3.stride(0) if n > 1 else pitch * (h * 3 // 2))


# (source kind, destination kind, device matrices) -> entry point
_WARPS = {
    ("frames", "frames", False): "bevk_warp_perspective",
    ("frames", "frames", True): "bevk_warp_perspective_dmat",
    ("nv12", "bgr", False): "bevk_warp_perspective_nv12",
    ("nv12", "bgr", True): "bevk_warp_perspective_nv12_dmat",
    ("bgr", "yuv", False): "bevk_warp_perspective_yuv420",
    ("bgr", "yuv", True): "bevk_warp_perspective_yuv420_dmat",
    ("nv12", "yuv", False): "bevk_warp_perspective_nv12_yuv420",
    ("nv12", "yuv", True): "bevk_warp_perspective_nv12_yuv420_dmat",
}


def _warp(src, src_kind, M, dsize, dst, dst_kind, flags, borderMode, borderValue, mat_index, dmat, layout=None,
          path=None):
    """The device warps.  layout: a YUV destination's layout name; path: the BGR warp's kernel family
    code, passed to the entry point's _path form.  The C arguments compose as (src, dst, n, h, w)
    + the source's + (dh, dw) + the destination's + (M, n_mats, mat_index, flags, border) [+ path]."""
    import torch
    s, n, h, w, batched, src_args = _warp_src(src, src_kind)
    code = _yuv_layout(layout) if dst_kind == "yuv" else None
    dw, dh = int(dsize[0]), int(dsize[1])
    m = _Mats(M, n, mat_index, dmat, src.device)
    out, d, dst_args = _warp_dst(dst, dst_kind, src, s, n, dh, dw, batched, code)
    b = _border(borderValue)
    name = _WARPS[src_kind, dst_kind, dmat]
    args = ((_vp(s.data_ptr()), _vp(d.data_ptr()), n, h, w) + src_args + (dh, dw) + dst_args
            + (m.ptr, m.n, m.idx_ptr(), int(flags), int(borderMode), _dptr(b)) + (() if path is None else (path,)))
    with torch.cuda.device(src.device):
        rc = getattr(lib(), name if path is None else name + "_path")(*args, _stream_ptr(src))
    _check(rc, name)
    return out


VIDEO_FORMATS = {"i420": 0, "nv12": 1, "bgr": 2}


def _video_call(src, src_format, dst_format, sizes, caller="warp_perspective_video_host"):
    """The first checks of the host video calls, in order: format names, the host source frames (BGR or
    YUV 4:2:0 uint8), the (width, height) sizes, dsize first and even for YUV BEVs.  Returns (frames
    view, n, h, w, leading dims of the outputs, BEV frame shape, the sizes as ints)."""
    for name, fmt in (("src_format", src_format), ("dst_format", dst_format)):
        if fmt not in VIDEO_FORMATS:
            raise ValueError("%s must be 'bgr', 'i420' or 'nv12', got %r" % (name, fmt))
    if hasattr(src, "detach"):
        if src.is_cuda:
            raise ValueError("src is on %s: %s takes host buffers" % (src.device, caller))
        src = src.detach().numpy()
    a = np.asarray(src)
    if a.dtype != np.uint8:
        raise ValueError("src frames are uint8, got %s" % (a.dtype,))
    if not a.flags["C_CONTIGUOUS"]:
        raise ValueError("src must be C-contiguous")
    batched = a.ndim == (4 if src_format == "bgr" else 3)
    f = a if batched else a[None]
    if src_format == "bgr":
        if a.ndim not in (3, 4) or a.shape[-1] != 3:
            raise ValueError("src BGR frames must be (H, W, 3) or (N, H, W, 3), got shape %s" % (a.shape,))
        h, w = f.shape[1], f.shape[2]
    else:
        if a.ndim not in (2, 3):
            raise ValueError("src %s frames must be (H*3/2, W) or (N, H*3/2, W), got shape %s"
                             % (src_format.upper(), a.shape))
        rows, w = f.shape[1], f.shape[2]
        if rows == 0 or rows % 3 or w % 2 or w == 0:
            raise ValueError("src %s frames need H*3/2 rows for an even H and an even width W, got %d rows x %d"
                             % (src_format.upper(), rows, w))
        h = rows // 3 * 2
    sizes = [(int(z[0]), int(z[1])) for z in sizes]
    dw, dh = sizes[0]
    if dst_format != "bgr" and (dw % 2 or dh % 2):
        raise ValueError("YUV 4:2:0 frames need an even width and height, got dsize %dx%d" % (dw, dh))
    frame = (dh, dw, 3) if dst_format == "bgr" else (dh * 3 // 2, dw)
    return f, f.shape[0], h, w, f.shape[:1] if batched else (), frame, sizes


def _host_out(dst, shape, what, caller="warp_perspective_video_host"):
    """A new uint8 host array of this shape, or dst after checking that it is one."""
    if dst is None:
        return np.empty(shape, np.uint8)
    if getattr(dst, "is_cuda", False):
        raise ValueError("%s is on %s: %s takes host buffers" % (what, dst.device, caller))
    out = _to_numpy(dst) if not isinstance(dst, np.ndarray) else dst
    if out.shape != shape or out.dtype != np.uint8 or not out.flags["C_CONTIGUOUS"]:
        raise ValueError("%s must be a C-contiguous uint8 array of shape %s, got %s %s"
                         % (what, shape, out.dtype, out.shape))
    return out


def warp_perspective_video_host(src, M, dsize, src_format="bgr", dst_format="i420", dst=None, flags=1,
                                borderMode=0, borderValue=0, mat_index=None):
    """Host-buffer warp between video frame formats ("bgr", "i420", "nv12"): src / dst are numpy
    arrays or CPU tensors (pinned for full speed), BGR (H, W, 3) / (N, H, W, 3) or YUV 4:2:0
    (H*3/2, W) / (N, H*3/2, W) uint8."""
    s, n, h, w, lead, frame, [(dw, dh)] = _video_call(src, src_format, dst_format, [dsize])
    m = _Mats(M, n, mat_index, False, None)
    out = _host_out(dst, lead + frame, "dst")
    b = _border(borderValue)
    rc = lib().bevk_warp_perspective_video_host(
        _vp(s.ctypes.data), VIDEO_FORMATS[src_format], _vp(out.ctypes.data), VIDEO_FORMATS[dst_format], n, h, w,
        dh, dw, m.ptr, m.n, m.idx_ptr(), int(flags), int(borderMode), _dptr(b))
    _check(rc, "bevk_warp_perspective_video_host")
    return dst if dst is not None else out


def warp_perspective_video_host_small(src, M, M_small, dsize, small_size, src_format="bgr", dst_format="i420",
                                      flags=1, interpolation=1, borderMode=0, borderValue=0, mat_index=None,
                                      dst=None, small=None, dst_small=None):
    """warp_perspective_video_host plus the small frames (BGR, small_size = (w, h)) and their BEVs
    through M_small, from one upload of each frame.  Returns (dst, small, dst_small)."""
    caller = "warp_perspective_video_host_small"
    s, n, h, w, lead, frame, [(dw, dh), (sw, sh)] = _video_call(src, src_format, dst_format, [dsize, small_size],
                                                                 caller)
    if interpolation not in (1, 3):
        raise ValueError("interpolation must be INTER_LINEAR (1) or INTER_AREA (3), got %r" % (interpolation,))
    m = _Mats(M, n, mat_index, False, None)
    Mss = np.ascontiguousarray(_to_numpy(M_small), dtype=np.float64)
    Mss = Mss[None] if Mss.ndim == 2 else Mss
    if Mss.shape != m.keep.shape:
        raise ValueError("M_small must hold one 3x3 matrix per matrix of M, shape %s, got %s"
                         % (m.keep.shape, Mss.shape))
    out = _host_out(dst, lead + frame, "dst", caller)
    out_small = _host_out(small, lead + (sh, sw, 3), "small", caller)
    out_bev_small = _host_out(dst_small, lead + frame, "dst_small", caller)
    b = _border(borderValue)
    rc = lib().bevk_warp_perspective_video_host_small(
        _vp(s.ctypes.data), VIDEO_FORMATS[src_format], _vp(out.ctypes.data), VIDEO_FORMATS[dst_format],
        _vp(out_small.ctypes.data), _vp(out_bev_small.ctypes.data), n, h, w, dh, dw, sh, sw, m.ptr, _dptr(Mss),
        m.n, m.idx_ptr(), int(flags), int(interpolation), int(borderMode), _dptr(b))
    _check(rc, "bevk_warp_perspective_video_host_small")
    return (dst if dst is not None else out, small if small is not None else out_small,
            dst_small if dst_small is not None else out_bev_small)


def warp_touched_pixels(ssize, dsize, M, flags=1):
    """(T, row_min, row_max) of SURVEY.md 8d, computed on the device."""
    Mm = _mat(M, "M")
    rr = (_c_int * 2)()
    t = lib().bevk_warp_touched_pixels(int(ssize[1]), int(ssize[0]), int(dsize[1]), int(dsize[0]),
                                       _dptr(Mm), int(flags), rr)
    if t < 0:
        _check(int(t), "bevk_warp_touched_pixels")
    return int(t), int(rr[0]), int(rr[1])


def warp_host_rows(ssize, dsize, M, flags=1):
    """[first, last] source row that warp_perspective_host uploads for these matrices."""
    Ms = np.ascontiguousarray(_to_numpy(M), dtype=np.float64).reshape(-1, 3, 3)
    rr = (_c_int * 2)()
    _check(lib().bevk_warp_host_rows(int(ssize[1]), int(ssize[0]), int(dsize[1]), int(dsize[0]),
                                     _dptr(Ms), Ms.shape[0], int(flags), rr), "bevk_warp_host_rows")
    return int(rr[0]), int(rr[1])


def set_warp_path(path):
    _check(lib().bevk_warp_set_path({"auto": 0, "generic": 1, "fast": 2}.get(path, path)),
           "bevk_warp_set_path")


# ----------------------------------------------------------------------------- projection plumbing

def _proj_dtype(t):
    import torch
    code = {torch.float32: F32, torch.float64: F64}.get(t.dtype)
    if code is None:
        raise TypeError("projection kernels take float32 / float64 tensors, got %s" % t.dtype)
    return code


def rows_op(name, x, in_cols, out_shape_tail, *extra, H=None, has_H=False):
    """Run a row-wise projection entry point: x (N, in_cols) -> (N, *out_shape_tail)."""
    import torch
    _require_cuda(x, "input")
    code = _proj_dtype(x)
    if in_cols == 1:
        x2 = x.reshape(-1).contiguous()
        n = x2.shape[0]
    else:
        if x.dim() != 2 or x.shape[1] != in_cols:
            raise ValueError("%s expects shape (N, %d), got %s" % (name, in_cols, tuple(x.shape)))
        x2 = x.contiguous()
        n = x2.shape[0]
    out = torch.empty((n,) + tuple(out_shape_tail), dtype=x.dtype, device=x.device)
    args = [_vp(x2.data_ptr()), _vp(out.data_ptr()), n] + [int(e) for e in extra] + [code]
    if has_H:
        args.append(_dptr(_mat(H)) if H is not None else None)
    with torch.cuda.device(x.device):
        args.append(_stream_ptr(x))
        rc = getattr(lib(), name)(*args)
    _check(rc, name)
    return out


def resize(src, dsize, interpolation=1, dst=None):
    """cv2.resize(src, dsize, interpolation=interpolation) (INTER_LINEAR = 1 or INTER_AREA = 3) on
    uint8 CUDA frames (H,W), (H,W,C) or (N,H,W,C); dsize = (width, height).  Replaces the
    per-frame call at vis_homo.py:90."""
    import torch
    _require_cuda(src, "src")
    if src.dtype != torch.uint8:
        raise TypeError("resize: only uint8 frames are implemented, got %s" % (src.dtype,))
    s4, _ = _frames_view(src)
    s4 = s4.contiguous()
    n, sh, sw, c = s4.shape
    w, h = int(dsize[0]), int(dsize[1])
    dst = _out(dst, {2: (h, w), 3: (h, w, c), 4: (n, h, w, c)}[src.dim()], torch.uint8, src.device)
    with torch.cuda.device(src.device):
        rc = lib().bevk_resize(_vp(s4.data_ptr()), _vp(dst.data_ptr()), n, sh, sw, h, w, c, 0,
                               int(interpolation), _stream_ptr(src))
    _check(rc, "bevk_resize")
    return dst


def resize_nv12(src, dsize, dst=None, interpolation=1):
    """resize(nv12_to_bgr(src), dsize, interpolation) in one pass: CUDA uint8 NV12 frames
    (H*3/2, W) or (N, H*3/2, W) -> (h, w, 3) or (N, h, w, 3) BGR; dsize = (width, height);
    interpolation INTER_LINEAR = 1 or INTER_AREA = 3."""
    import torch
    s3, n, h, w, (pitch, fstride) = _nv12_frames(src)
    dw, dh = int(dsize[0]), int(dsize[1])
    dst = _out(dst, (n, dh, dw, 3) if src.dim() == 3 else (dh, dw, 3), torch.uint8, src.device)
    with torch.cuda.device(src.device):
        rc = lib().bevk_resize_nv12_interp(_vp(s3.data_ptr()), _vp(dst.data_ptr()), n, h, w, pitch, fstride, dh,
                                           dw, int(interpolation), _stream_ptr(src))
    _check(rc, "bevk_resize_nv12_interp")
    return dst


def composite_u8c3(bg, fg, fg_mask, bw_mode=False, out=None):
    """out = uint8(round(fg * mask/255 + bg * (1 - mask/255))) on CUDA uint8 tensors of one shape
    (..., 3); bit-identical to the reference's numpy float64 blend (bev/tool/compo.py:16-23)."""
    import torch
    for name, t in (("bg", bg), ("fg", fg), ("fg_mask", fg_mask)):
        _require_cuda(t, name)
        if t.dtype != torch.uint8:
            raise TypeError("%s must be uint8, got %s" % (name, t.dtype))
    if not (tuple(bg.shape) == tuple(fg.shape) == tuple(fg_mask.shape)) or bg.shape[-1] != 3:
        raise ValueError("bg, fg and fg_mask must share one (..., 3) shape; got %s %s %s"
                         % (tuple(bg.shape), tuple(fg.shape), tuple(fg_mask.shape)))
    if not (bg.device == fg.device == fg_mask.device):
        raise ValueError("bg, fg and fg_mask must be on one device; got %s %s %s"
                         % (bg.device, fg.device, fg_mask.device))
    # the kernel reads 4-byte words: views at an odd byte offset (the mask half of a concatenated
    # warp output, user slices) are realigned by a copy
    bg, fg, fg_mask = _aligned(bg), _aligned(fg), _aligned(fg_mask)
    out = _out(out, bg.shape, torch.uint8, bg.device, "out")
    if out.data_ptr() % 4:
        raise ValueError("out must be 4-byte aligned")
    n_pixels = bg.numel() // 3
    with torch.cuda.device(bg.device):
        rc = lib().bevk_composite_u8c3(_vp(bg.data_ptr()), _vp(fg.data_ptr()), _vp(fg_mask.data_ptr()),
                                       _vp(out.data_ptr()), n_pixels, int(bool(bw_mode)), _stream_ptr(bg))
    _check(rc, "bevk_composite_u8c3")
    return out


def composite_bev_fusable(bg, fg, dsize):
    """Shapes bevk_composite_bev_u8c3 takes: all widths multiples of 4, sources at least 2x2."""
    return (bg.shape[-2] % 4 == 0 and fg.shape[-2] % 4 == 0 and int(dsize[0]) % 4 == 0
            and min(bg.shape[-3], bg.shape[-2], fg.shape[-3], fg.shape[-2]) >= 2)


def composite_bev_u8c3(bg, fg, fg_mask, H_bg, H_fg, dsize, out=None):
    """Fused warp + warp + warp + blend (bev/tool/compo.py:26-50).  bg: (Hb,Wb,3) or (N,Hb,Wb,3);
    fg, fg_mask: (N,Hf,Wf,3) uint8 CUDA; H_bg, H_fg: forward 3x3 (or (N,3,3)) float64 on the host;
    dsize = (width, height) of the BEV.  Returns (N, height, width, 3)."""
    return _composite_bev(bg, fg, fg_mask, H_bg, H_fg, dsize, out, False)


def composite_bev_u8c3_dmat(bg, fg, fg_mask, H_bg, H_fg, dsize, out=None):
    """composite_bev_u8c3 with H_bg, H_fg CUDA tensors (3,3) or (N,3,3) on fg's device, converted to
    contiguous float64 on the current stream and read by the kernels when they run: no host sync, and
    a captured CUDA graph replays the matrices last written into them.  Same bytes as the host call."""
    return _composite_bev(bg, fg, fg_mask, H_bg, H_fg, dsize, out, True)


def _composite_mats(H, what, device):
    """(K, 9) float64 device matrices for bevk_composite_bev_u8c3_dmat, converted in stream order"""
    import torch
    if not isinstance(H, torch.Tensor) or not H.is_cuda:
        raise TypeError("%s must be a CUDA tensor for the device-matrix compositor, got %s"
                        % (what, getattr(H, "device", type(H).__name__)))
    if H.device != device:
        raise ValueError("%s is on %s, the frames on %s" % (what, H.device, device))
    if H.numel() == 0 or H.numel() % 9:
        raise ValueError("%s must be 3x3 or (N,3,3), got %s" % (what, tuple(H.shape)))
    return H.to(torch.float64).contiguous().reshape(-1, 9)


def _composite_bev(bg, fg, fg_mask, H_bg, H_fg, dsize, out, dmat):
    import torch
    for name, t in (("bg", bg), ("fg", fg), ("fg_mask", fg_mask)):
        _require_cuda(t, name)
        if t.dtype != torch.uint8 or t.shape[-1] != 3:
            raise TypeError("%s must be uint8 (..., 3), got %s %s" % (name, t.dtype, tuple(t.shape)))
    if fg.dim() != 4 or tuple(fg.shape) != tuple(fg_mask.shape):
        raise ValueError("fg and fg_mask must share one (N, H, W, 3) shape; got %s %s"
                         % (tuple(fg.shape), tuple(fg_mask.shape)))
    n = fg.shape[0]
    if bg.dim() == 3:
        bg = bg[None]
    if bg.dim() != 4 or bg.shape[0] not in (1, n):
        raise ValueError("bg must be (H, W, 3) or (N, H, W, 3) with N = %d; got %s" % (n, tuple(bg.shape)))
    if dmat:
        Hb, Hf = _composite_mats(H_bg, "H_bg", fg.device), _composite_mats(H_fg, "H_fg", fg.device)
        pb, pf = ctypes.cast(Hb.data_ptr(), _dp), ctypes.cast(Hf.data_ptr(), _dp)
    else:
        Hb = np.ascontiguousarray(np.asarray(_to_numpy(H_bg), np.float64).reshape(-1, 9))
        Hf = np.ascontiguousarray(np.asarray(_to_numpy(H_fg), np.float64).reshape(-1, 9))
        pb, pf = _dptr(Hb), _dptr(Hf)
    if Hb.shape[0] != Hf.shape[0] or Hb.shape[0] not in (1, n):
        raise ValueError("need 1 or %d homography pairs, got %d / %d" % (n, Hb.shape[0], Hf.shape[0]))
    if not (bg.device == fg.device == fg_mask.device):
        raise ValueError("bg, fg and fg_mask must be on one device; got %s %s %s"
                         % (bg.device, fg.device, fg_mask.device))
    bg, fg, fg_mask = _aligned(bg, 16), _aligned(fg, 16), _aligned(fg_mask, 16)
    w, h = int(dsize[0]), int(dsize[1])
    out = _out(out, (n, h, w, 3), torch.uint8, fg.device, "out")
    if out.data_ptr() % 4:
        raise ValueError("out must be 4-byte aligned")
    name = "bevk_composite_bev_u8c3_dmat" if dmat else "bevk_composite_bev_u8c3"
    with torch.cuda.device(fg.device):
        rc = getattr(lib(), name)(
            _vp(bg.data_ptr()), _vp(fg.data_ptr()), _vp(fg_mask.data_ptr()), _vp(out.data_ptr()),
            n, bg.shape[0], bg.shape[1], bg.shape[2], fg.shape[1], fg.shape[2], h, w,
            pb, pf, Hb.shape[0], _stream_ptr(fg))
    _check(rc, name)
    return out


def rbox_zt2tt_world(x, K, Rt):
    """(N,7) world boxes with height -> (N,7) ground boxes with a projected height tail."""
    import torch
    _require_cuda(x, "input")
    code = _proj_dtype(x)
    if x.dim() != 2 or x.shape[1] != 7:
        raise ValueError("rbox_zt2tt_world expects shape (N, 7), got %s" % (tuple(x.shape),))
    Kn = np.ascontiguousarray(np.asarray(_to_numpy(K), np.float64)[:3, :3])
    Rn = np.ascontiguousarray(np.asarray(_to_numpy(Rt), np.float64)[:3, :4])
    if Kn.shape != (3, 3) or Rn.shape != (3, 4):
        raise ValueError("K must be 3x3 (or 3x4) and Rt 3x4 (or 4x4)")
    x2 = x.contiguous()
    out = torch.empty_like(x2)
    with torch.cuda.device(x.device):
        rc = lib().bevk_rbox_zt2tt_world(_vp(x2.data_ptr()), _vp(out.data_ptr()), x2.shape[0], code,
                                         _dptr(Kn), _dptr(Rn), _stream_ptr(x))
    _check(rc, "bevk_rbox_zt2tt_world")
    return out


def rbox_iou_matrix(boxes1, boxes2, yaw_offset=0.0):
    """(N, >=5), (M, >=5) CUDA float32/float64 boxes [x, y, w, h, r, ...] -> (N, M) IoU matrix
    (w along (cos r, sin r)); replaces d3d.box.box2d_iou(..., method="rbox")
    (bev/tracker/rbox_tracker.py:87-92)."""
    import torch
    _require_cuda(boxes1, "boxes1")
    _require_cuda(boxes2, "boxes2")
    code = _proj_dtype(boxes1)
    if boxes2.dtype != boxes1.dtype or boxes2.device != boxes1.device:
        raise TypeError("boxes1 and boxes2 must share dtype and device")
    for name, b in (("boxes1", boxes1), ("boxes2", boxes2)):
        if b.dim() != 2 or b.shape[1] < 5:
            raise ValueError("%s must be (N, >=5) rows [x, y, w, h, r, ...], got %s" % (name, tuple(b.shape)))
    b1, b2 = boxes1.contiguous(), boxes2.contiguous()
    out = torch.empty((b1.shape[0], b2.shape[0]), dtype=b1.dtype, device=b1.device)
    with torch.cuda.device(b1.device):
        rc = lib().bevk_rbox_iou_matrix(_vp(b1.data_ptr()), b1.shape[0], b1.shape[1], _vp(b2.data_ptr()),
                                        b2.shape[0], b2.shape[1], _vp(out.data_ptr()), code,
                                        float(yaw_offset), _stream_ptr(b1))
    _check(rc, "bevk_rbox_iou_matrix")
    return out
