"""torch.ops.bev_cuda -- the hot path as registered PyTorch operators (SURVEY.md 8b).

``load()`` loads bev_b200/libbev_torch_ops.so (built by bev_b200/csrc/build_torch_ops.py, part of
``__graft_entry__.build()``): a thin C++ extension whose operators check tensors, allocate the
output with torch's caching allocator, take the current CUDA stream and call the extern "C" entry
points of libbev_b200.so.  After ``load()`` (frames are CUDA tensors; M, H, K, Rt are CPU float64
tensors, and the M of the four warps and the H_bg / H_fg of composite_bev may also be CUDA tensors on
the frames' device; shapes with a leading N also take one unbatched frame and then return one):

  frames (uint8 BGR (N,H,W,3); NV12 / YUV 4:2:0 (N,H*3/2,W), NV12 with any row pitch / frame stride)
    warp_perspective(src, M, w, h, flags=1, border_mode=0, border_val=0., mat_index=None)
                                        (H,W) / (H,W,C) / (N,H,W,C) u8/f16/f32 -> same rank, h x w
    resize(src, w, h, interpolation=1)  (H,W) / (H,W,C) / (N,H,W,C) uint8, C 1..4 -> same rank, h x w
    nv12_to_bgr(src)                    NV12 -> BGR
    warp_perspective_nv12(src, M, w, h, flags=1, border_mode=0, border_val=0., mat_index=None)
                                        NV12 -> BGR h x w
    resize_nv12(src, w, h, interpolation=1)                               NV12 -> BGR h x w
    bgr_to_yuv420(src, layout=0)        BGR -> YUV 4:2:0 (layout 0 I420, 1 NV12)
    warp_perspective_yuv420(src, M, w, h, layout=0, flags=1, border_mode=0, border_val=0., mat_index=None)
                                        BGR -> YUV 4:2:0 h x w
    warp_perspective_nv12_yuv420(src, M, w, h, layout=0, flags=1, border_mode=0, border_val=0.,
                                 mat_index=None)                      NV12 -> YUV 4:2:0 h x w
  compositing (bev/tool/compo.py)
    composite(bg, fg, mask, bw_mode=0)  three uint8 (..., 3) of one shape -> that shape
    composite_bev(bg, fg, mask, H_bg, H_fg, w, h)
                                        fg, mask (N,Hf,Wf,3), bg (1 or N,Hb,Wb,3) -> (N,h,w,3)
  boxes and points (float32 / float64; mode / src_mode 0 "bev", 1 "world")
    project_points(pts, H)              (N,2) -> (N,2), (N,3) -> (N,3)
    rbox_corners_project(xywhr, H_or_None, mode)                          (N,5) -> (N,8)
    corners_to_rbox(xy8, H_or_None, mode)                                 (N,8) -> (N,5)
    rbox_similarity(rbox, H, src_mode)                                    (N,5) -> (N,5)
    rboxtt_similarity(rboxtt, H, src_mode)                                (N,7) -> (N,7)
    rbox_zt2tt_world(rboxzt, K, Rt)     K 3x3, Rt 3x4                     (N,7) -> (N,7)
    rbox_heading(xywhr, mode)                                             (N,5) -> (N,4)
    corners_heading(xy8)                                                  (N,8) -> (N,4)
    angle_similarity(yaw, H, src_mode)  any shape -> (numel,)
    dist_similarity(d, H)               any shape -> same shape
    v2yaw(v, mode)                      (N,2) -> (N,)
    yaw2v(yaw, mode)                    any shape -> (numel, 2)
    yaw2mat(yaw, mode)                  any shape -> (numel, 2, 2)
    rbox_iou_matrix(boxes1, boxes2, yaw_offset=0.)    (N,>=5) x (M,>=5) -> (N,M)

Only CUDA and Meta implementations are registered; there is no CPU fallback.  The Python modules
(bev_b200.homo, bev_b200.rbox_torch, bev_b200.compo) reach the same entry points through ctypes;
both routes run the same kernels and give identical bytes (tests/test_torch_ops_gpu.py,
tests/test_torch_ops_compile_gpu.py).

The operators work under FakeTensor, ``torch.compile(fullgraph=True)`` (also with dynamic batch
sizes), ``torch.export`` and ``torch.library.opcheck``, and they can be captured in a
``torch.cuda.graph``.  Where the homographies live decides what a captured graph replays:

  * CPU M / H: read on the host when the call is made, so fixed at capture time.
  * CUDA M (warp_perspective, warp_perspective_nv12, warp_perspective_yuv420,
    warp_perspective_nv12_yuv420): read by the kernels when they run, in stream order (a non-float64
    one is converted on the stream).  A graph captured once replays whatever matrices were last
    written into M (``M.copy_(new)`` between replays), and homographies made on the GPU cost no sync.
    These calls always take the direct-gather warp kernels, not the staged one.
  * CUDA H_bg and H_fg (composite_bev; both, not one of them): the same, through the fused
    compositor's device-matrix kernels.

mat_index is planned on the host and stays fixed at capture time; a CUDA mat_index cannot be
captured (reading it synchronises): pass a CPU one.  The box and point operators take CPU H only.
"""
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
OPS_PATH = os.path.join(_HERE, "libbev_torch_ops.so")
_loaded = False

# every operator the extension registers (tests/test_torch_ops_meta.py holds the two lists equal)
OPS = ("warp_perspective", "project_points", "rbox_corners_project", "corners_to_rbox", "rbox_similarity",
       "nv12_to_bgr", "warp_perspective_nv12", "resize_nv12", "bgr_to_yuv420", "warp_perspective_yuv420",
       "resize", "warp_perspective_nv12_yuv420", "composite", "composite_bev", "rbox_iou_matrix",
       "rboxtt_similarity", "rbox_zt2tt_world", "rbox_heading", "corners_heading", "angle_similarity",
       "dist_similarity", "v2yaw", "yaw2v", "yaw2mat")


def _fake_kernel(op):
    """FakeTensor rule of one operator: its C++ Meta kernel, with the result placed on the device of
    the first tensor argument (the frames or boxes).

    FakeTensor's default device rule refuses an operator whose arguments mix a CUDA tensor with a
    CPU tensor of more than zero dimensions, which every operator taking a homography does.  The
    shapes still come from the Meta kernel alone (the same C++ function as the CUDA kernel)."""
    import torch
    from torch._subclasses.fake_tensor import in_kernel_invocation_manager

    def fake(*args, **kwargs):
        device = next(a.device for a in args if isinstance(a, torch.Tensor))
        if device.type != "cuda":
            raise NotImplementedError("bev_cuda::%s has no kernel for %s tensors (CUDA only, no CPU fallback)"
                                      % (op._schema.name.split("::")[1], device.type))
        mode = torch.library.get_ctx()._fake_mode
        with in_kernel_invocation_manager(mode):
            out = op(*args, **kwargs)
        return mode.fake_tensor_converter.from_meta_and_device(mode, out, device)
    return fake


def load():
    """Register torch.ops.bev_cuda.* (idempotent).  Raises if the extension has not been built."""
    global _loaded
    if _loaded:
        return
    import torch
    if not os.path.exists(OPS_PATH):
        raise ImportError("bev_b200: %s is missing; build it with `python bev_b200/csrc/build_torch_ops.py` "
                          "(or __graft_entry__.build())" % OPS_PATH)
    torch.ops.load_library(OPS_PATH)
    # The fake rule goes straight into FakeTensor's registry of custom-op rules:
    # torch.library.register_fake would also replace the C++ Meta kernel, which the rule runs.
    from torch._library.simple_registry import singleton
    from torch._library.utils import Kernel
    for name in OPS:
        op = getattr(torch.ops.bev_cuda, name).default
        singleton.find(op.name()).fake_impl.kernels.append(Kernel(_fake_kernel(op), __name__))
    _loaded = True
