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
    "bevk_warp_host_rows": (_c_int, [_c_int, _c_int, _c_int, _c_int, _dp, _c_int, _c_int, _ip]),
    "bevk_warp_set_path": (_c_int, [_c_int]),
    "bevk_warp_touched_pixels": (_c_i64, [_c_int, _c_int, _c_int, _c_int, _dp, _c_int, _ip]),
    "bevk_nv12_to_bgr": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _vp]),
    "bevk_warp_perspective_nv12": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _c_int, _c_int,
                                            _dp, _c_int, _i32p, _c_int, _c_int, _dp, _vp]),
    "bevk_resize": (_c_int, [_vp, _vp] + [_c_int] * 8 + [_vp]),
    "bevk_resize_nv12": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _c_int, _c_int, _vp]),
    "bevk_resize_nv12_interp": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_i64, _c_int, _c_int, _c_int,
                                         _vp]),
    "bevk_composite_u8c3": (_c_int, [_vp, _vp, _vp, _vp, _c_i64, _c_int, _vp]),
    "bevk_composite_bev_u8c3": (_c_int, [_vp, _vp, _vp, _vp] + [_c_int] * 8 + [_dp, _dp, _c_int, _vp]),
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


def _check_out(out, like, what):
    """`out` must be a contiguous tensor of `like`'s shape, dtype and device."""
    _require_cuda(out, what)
    if tuple(out.shape) != tuple(like.shape) or out.dtype != like.dtype or out.device != like.device \
            or not out.is_contiguous():
        raise ValueError("%s must be a contiguous %s tensor of shape %s on %s"
                         % (what, like.dtype, tuple(like.shape), like.device))


def _warp_dtype(t):
    import torch
    code = {torch.uint8: U8, torch.float16: F16, torch.float32: F32}.get(t.dtype)
    if code is None:
        raise TypeError("warp_perspective supports uint8 / float16 / float32, got %s" % t.dtype)
    return code


def _prep_mats(M, n_frames, mat_index):
    Ms = np.ascontiguousarray(_to_numpy(M), dtype=np.float64)
    if Ms.ndim == 2:
        Ms = Ms[None]
    if Ms.ndim != 3 or Ms.shape[1:] != (3, 3):
        raise ValueError("M must be 3x3 or (K,3,3), got %s" % (Ms.shape,))
    idx = None
    if mat_index is not None:
        idx = np.ascontiguousarray(_to_numpy(mat_index), dtype=np.int32).reshape(-1)
        if idx.shape[0] != n_frames:
            raise ValueError("mat_index has %d entries for %d frames" % (idx.shape[0], n_frames))
    elif Ms.shape[0] not in (1, n_frames):
        raise ValueError("%d matrices for %d frames needs mat_index" % (Ms.shape[0], n_frames))
    return Ms, idx


def _border(borderValue):
    b = np.zeros(4, np.float64)
    v = np.atleast_1d(np.asarray(borderValue, dtype=np.float64)).reshape(-1)[:4]
    b[:len(v)] = v  # cv2.Scalar semantics: missing channels are 0
    return b


def _frames_view(src):
    """(N, H, W, C) view of a (H,W) / (H,W,C) / (N,H,W,C) tensor + how to undo it."""
    if src.dim() == 2:
        return src[None, :, :, None], lambda o: o[0, :, :, 0]
    if src.dim() == 3:
        return src[None], lambda o: o[0]
    if src.dim() == 4:
        return src, lambda o: o
    raise ValueError("src must be (H,W), (H,W,C) or (N,H,W,C); got shape %s" % (tuple(src.shape),))


_PATHS = {None: -1, "auto": 0, "generic": 1, "fast": 2}


def warp_perspective(src, M, dsize, dst=None, flags=1, borderMode=0, borderValue=0,
                     mat_index=None, path=None):
    """path: None (the calling thread's default, see set_warp_path), "auto", "generic" (direct-gather
    kernels) or "fast" (staged kernel; raises if the shape does not qualify)."""
    import torch
    _require_cuda(src, "src")
    code = _warp_dtype(src)
    s4, undo = _frames_view(src)
    s4 = s4.contiguous()
    n, h, w, c = s4.shape
    dw, dh = int(dsize[0]), int(dsize[1])
    Ms, idx = _prep_mats(M, n, mat_index)
    if dst is not None:
        _require_cuda(dst, "dst")
        d4, _ = _frames_view(dst)
        if tuple(d4.shape) != (n, dh, dw, c) or dst.dtype != src.dtype or not dst.is_contiguous() \
                or dst.device != src.device:
            raise ValueError("dst must be a contiguous %s tensor of shape %s on %s"
                             % (src.dtype, (n, dh, dw, c), src.device))
        out4 = d4
    else:
        out4 = torch.empty((n, dh, dw, c), dtype=src.dtype, device=src.device)
    b = _border(borderValue)
    with torch.cuda.device(src.device):
        rc = lib().bevk_warp_perspective_path(
            _vp(s4.data_ptr()), _vp(out4.data_ptr()), n, h, w, dh, dw, c, code, _dptr(Ms),
            Ms.shape[0], idx.ctypes.data_as(_i32p) if idx is not None else None, int(flags),
            int(borderMode), _dptr(b), _PATHS.get(path, path), _stream_ptr(src))
    _check(rc, "bevk_warp_perspective")
    return dst if dst is not None else undo(out4)


def warp_perspective_host(src, M, dsize, dst=None, flags=1, borderMode=0, borderValue=0,
                          mat_index=None):
    """Host-buffer form: src / dst are numpy arrays or CPU tensors (pinned for full PCIe speed)."""
    s = _to_numpy(src) if not isinstance(src, np.ndarray) else src
    code = {np.dtype("uint8"): U8, np.dtype("float16"): F16, np.dtype("float32"): F32}.get(s.dtype)
    if code is None:
        raise TypeError("warp_perspective_host supports uint8/float16/float32, got %s" % s.dtype)
    if s.ndim == 2:
        s4, undo = s[None, :, :, None], (lambda o: o[0, :, :, 0])
    elif s.ndim == 3:
        s4, undo = s[None], (lambda o: o[0])
    elif s.ndim == 4:
        s4, undo = s, (lambda o: o)
    else:
        raise ValueError("src must be (H,W), (H,W,C) or (N,H,W,C)")
    s4 = np.ascontiguousarray(s4)
    n, h, w, c = s4.shape
    dw, dh = int(dsize[0]), int(dsize[1])
    Ms, idx = _prep_mats(M, n, mat_index)
    if dst is None:
        out4 = np.empty((n, dh, dw, c), s4.dtype)
    else:
        out4 = _to_numpy(dst) if not isinstance(dst, np.ndarray) else dst
        out4 = out4.reshape(n, dh, dw, c)
        if out4.dtype != s4.dtype or not out4.flags["C_CONTIGUOUS"]:
            raise ValueError("dst must be C-contiguous with src's dtype")
    b = _border(borderValue)
    rc = lib().bevk_warp_perspective_host(
        _vp(s4.ctypes.data), _vp(out4.ctypes.data), n, h, w, dh, dw, c, code, _dptr(Ms),
        Ms.shape[0], idx.ctypes.data_as(_i32p) if idx is not None else None, int(flags),
        int(borderMode), _dptr(b))
    _check(rc, "bevk_warp_perspective_host")
    return dst if dst is not None else undo(out4)


def _nv12_frames(src):
    """(frames view (N, H*3/2, W), N, H, W, pitch, frame stride) of an NV12 tensor (H*3/2, W) or
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
    return s3, n, rows // 3 * 2, w, pitch, fstride


def nv12_to_bgr(src, dst=None):
    """cv2.cvtColor(f, COLOR_YUV2BGR_NV12) on CUDA uint8 NV12 frames (H*3/2, W) or (N, H*3/2, W)
    -> (H, W, 3) or (N, H, W, 3) BGR."""
    import torch
    s3, n, h, w, pitch, fstride = _nv12_frames(src)
    want = (n, h, w, 3) if src.dim() == 3 else (h, w, 3)
    if dst is None:
        dst = torch.empty(want, dtype=torch.uint8, device=src.device)
    else:
        _require_cuda(dst, "dst")
        if tuple(dst.shape) != want or dst.dtype != torch.uint8 or not dst.is_contiguous() \
                or dst.device != src.device:
            raise ValueError("dst must be a contiguous uint8 tensor of shape %s on %s" % (want, src.device))
    with torch.cuda.device(src.device):
        rc = lib().bevk_nv12_to_bgr(_vp(s3.data_ptr()), _vp(dst.data_ptr()), n, h, w, pitch, fstride,
                                    _stream_ptr(src))
    _check(rc, "bevk_nv12_to_bgr")
    return dst


def warp_perspective_nv12(src, M, dsize, dst=None, flags=1, borderMode=0, borderValue=0, mat_index=None):
    """warp_perspective of nv12_to_bgr(src) in one pass: (H*3/2, W) -> (h, w, 3), (N, H*3/2, W) ->
    (N, h, w, 3) BGR uint8.  M / mat_index as for warp_perspective."""
    import torch
    s3, n, h, w, pitch, fstride = _nv12_frames(src)
    dw, dh = int(dsize[0]), int(dsize[1])
    Ms, idx = _prep_mats(M, n, mat_index)
    want = (n, dh, dw, 3) if src.dim() == 3 else (dh, dw, 3)
    if dst is None:
        dst = torch.empty(want, dtype=torch.uint8, device=src.device)
    else:
        _require_cuda(dst, "dst")
        if tuple(dst.shape) != want or dst.dtype != torch.uint8 or not dst.is_contiguous() \
                or dst.device != src.device:
            raise ValueError("dst must be a contiguous uint8 tensor of shape %s on %s" % (want, src.device))
    b = _border(borderValue)
    with torch.cuda.device(src.device):
        rc = lib().bevk_warp_perspective_nv12(
            _vp(s3.data_ptr()), _vp(dst.data_ptr()), n, h, w, pitch, fstride, dh, dw, _dptr(Ms), Ms.shape[0],
            idx.ctypes.data_as(_i32p) if idx is not None else None, int(flags), int(borderMode), _dptr(b),
            _stream_ptr(src))
    _check(rc, "bevk_warp_perspective_nv12")
    return dst


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
    if src.dim() not in (2, 3, 4):
        raise ValueError("resize: src must be (H,W), (H,W,C) or (N,H,W,C); got %s" % (tuple(src.shape),))
    w, h = int(dsize[0]), int(dsize[1])
    s4 = src.contiguous()
    if src.dim() == 2:
        s4 = s4[None, :, :, None]
    elif src.dim() == 3:
        s4 = s4[None]
    n, sh, sw, c = s4.shape
    want = {2: (h, w), 3: (h, w, c), 4: (n, h, w, c)}[src.dim()]
    if dst is None:
        dst = torch.empty((n, h, w, c), dtype=torch.uint8, device=src.device)
    else:
        _require_cuda(dst, "dst")
        if tuple(dst.shape) != want or dst.dtype != torch.uint8 or not dst.is_contiguous() \
                or dst.device != src.device:
            raise ValueError("resize: dst must be a contiguous uint8 tensor of shape %s on %s, got %s %s on %s"
                             % (want, src.device, dst.dtype, tuple(dst.shape), dst.device))
    with torch.cuda.device(src.device):
        rc = lib().bevk_resize(_vp(s4.data_ptr()), _vp(dst.data_ptr()), n, sh, sw, h, w, c, 0,
                               int(interpolation), _stream_ptr(src))
    _check(rc, "bevk_resize")
    if src.dim() == 2:
        return dst.reshape(h, w)
    if src.dim() == 3:
        return dst.reshape(h, w, c)
    return dst


def resize_nv12(src, dsize, dst=None, interpolation=1):
    """resize(nv12_to_bgr(src), dsize, interpolation) in one pass: CUDA uint8 NV12 frames
    (H*3/2, W) or (N, H*3/2, W) -> (h, w, 3) or (N, h, w, 3) BGR; dsize = (width, height);
    interpolation INTER_LINEAR = 1 or INTER_AREA = 3."""
    import torch
    s3, n, h, w, pitch, fstride = _nv12_frames(src)
    dw, dh = int(dsize[0]), int(dsize[1])
    want = (n, dh, dw, 3) if src.dim() == 3 else (dh, dw, 3)
    if dst is None:
        dst = torch.empty(want, dtype=torch.uint8, device=src.device)
    else:
        _require_cuda(dst, "dst")
        if tuple(dst.shape) != want or dst.dtype != torch.uint8 or not dst.is_contiguous() \
                or dst.device != src.device:
            raise ValueError("dst must be a contiguous uint8 tensor of shape %s on %s" % (want, src.device))
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
    if out is None:
        out = torch.empty_like(bg)
    else:
        _check_out(out, bg, "out")
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
    Hb = np.ascontiguousarray(np.asarray(_to_numpy(H_bg), np.float64).reshape(-1, 9))
    Hf = np.ascontiguousarray(np.asarray(_to_numpy(H_fg), np.float64).reshape(-1, 9))
    if Hb.shape[0] != Hf.shape[0] or Hb.shape[0] not in (1, n):
        raise ValueError("need 1 or %d homography pairs, got %d / %d" % (n, Hb.shape[0], Hf.shape[0]))
    if not (bg.device == fg.device == fg_mask.device):
        raise ValueError("bg, fg and fg_mask must be on one device; got %s %s %s"
                         % (bg.device, fg.device, fg_mask.device))
    bg, fg, fg_mask = _aligned(bg, 16), _aligned(fg, 16), _aligned(fg_mask, 16)
    w, h = int(dsize[0]), int(dsize[1])
    if out is None:
        out = torch.empty((n, h, w, 3), dtype=torch.uint8, device=fg.device)
    else:
        _require_cuda(out, "out")
        if tuple(out.shape) != (n, h, w, 3) or out.dtype != torch.uint8 or not out.is_contiguous() \
                or out.device != fg.device or out.data_ptr() % 4:
            raise ValueError("out must be a contiguous, 4-byte aligned uint8 tensor of shape %s on %s"
                             % ((n, h, w, 3), fg.device))
    with torch.cuda.device(fg.device):
        rc = lib().bevk_composite_bev_u8c3(
            _vp(bg.data_ptr()), _vp(fg.data_ptr()), _vp(fg_mask.data_ptr()), _vp(out.data_ptr()),
            n, bg.shape[0], bg.shape[1], bg.shape[2], fg.shape[1], fg.shape[2], h, w,
            _dptr(Hb), _dptr(Hf), Hb.shape[0], _stream_ptr(fg))
    _check(rc, "bevk_composite_bev_u8c3")
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
