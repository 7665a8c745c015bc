// torch_ops.cpp -- the thin PyTorch C++ extension in front of libbev_b200.so (SURVEY.md 8b,
// "C-ABI / extension" row): registers the hot-path operators with the dispatcher as
//
//   torch.ops.bev_cuda.warp_perspective(Tensor src, Tensor M, int w, int h, int flags, int border_mode,
//                                       float border_val, Tensor? mat_index) -> Tensor
//   torch.ops.bev_cuda.project_points(Tensor pts, Tensor H) -> Tensor
//   torch.ops.bev_cuda.rbox_corners_project(Tensor xywhr, Tensor? H, int mode) -> Tensor
//   torch.ops.bev_cuda.corners_to_rbox(Tensor xy8, Tensor? H, int mode) -> Tensor
//   torch.ops.bev_cuda.rbox_similarity(Tensor rbox, Tensor H, int src_mode) -> Tensor
//   torch.ops.bev_cuda.nv12_to_bgr(Tensor src) -> Tensor
//   torch.ops.bev_cuda.warp_perspective_nv12(Tensor src, Tensor M, int w, int h, int flags, int border_mode,
//                                            float border_val, Tensor? mat_index) -> Tensor
//   torch.ops.bev_cuda.resize_nv12(Tensor src, int w, int h, int interpolation=1) -> Tensor
//
// Every implementation only checks tensors, allocates the result with torch's caching allocator,
// takes the current CUDA stream and calls the extern "C" entry point of include/bev_b200.h with raw
// pointers -- no arithmetic lives here.  Homographies are CPU float64 tensors (they stay on the
// host, SURVEY.md 8b "Matrix ownership").  Only a CUDA implementation is registered: CPU tensors
// fail in the dispatcher, there is no CPU fallback.
//
// Reference interfaces replaced: cv2.warpPerspective at vis_homo.py:85-91, rbox.pts_world_bev
// (bev/rbox.py:136-151), rbox_torch.xywhr2xyxy (bev/rbox_torch.py:52-99) + the projection of
// rbox_vis.py:38-55, rbox.xy82xywhr (bev/rbox.py:50-63), rbox_torch.rbox_world_bev (:123-168); the NV12
// operators serve the frame loop of vis_homo.py:85-91 with frames from a GPU video decoder
// (resize_nv12: its small-frame copy, vis_homo.py:90).
#include <ATen/ATen.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>

#include "../../include/bev_b200.h"

namespace {

void *current_stream(const at::Tensor &t)
{
    return (void *)at::cuda::getCurrentCUDAStream(t.get_device()).stream();
}

void check_rc(int rc, const char *what)
{
    if (rc == BEVK_E_AFFINE)  // where the reference asserts (rbox_torch.py:140,161)
        TORCH_CHECK(false, "AssertionError: ", bevk_last_error());
    TORCH_CHECK(rc == BEVK_OK, what, " failed (code ", rc, "): ", bevk_last_error());
}

int elem_dtype(const at::Tensor &t, bool allow_bytes)
{
    switch (t.scalar_type()) {
    case at::kByte: TORCH_CHECK(allow_bytes, "uint8 tensors are frames, not boxes"); return BEVK_U8;
    case at::kHalf: TORCH_CHECK(allow_bytes, "float16 tensors are frames, not boxes"); return BEVK_F16;
    case at::kFloat: return BEVK_F32;
    case at::kDouble: TORCH_CHECK(!allow_bytes, "float64 frames are not supported"); return BEVK_F64;
    default: TORCH_CHECK(false, "unsupported dtype ", t.scalar_type());
    }
}

// homography / matrix table on the host as contiguous float64
at::Tensor host_f64(const at::Tensor &m, const char *what)
{
    TORCH_CHECK(!m.is_cuda(), what, " must be a CPU tensor (homographies stay on the host)");
    return m.to(at::kDouble).contiguous();
}

at::Tensor warp_perspective(const at::Tensor &src, const at::Tensor &M, int64_t w, int64_t h, int64_t flags,
                            int64_t border_mode, double border_val, const c10::optional<at::Tensor> &mat_index)
{
    TORCH_CHECK(src.is_cuda(), "src must be a CUDA tensor");
    TORCH_CHECK(src.dim() >= 2 && src.dim() <= 4, "src must be (H,W), (H,W,C) or (N,H,W,C)");
    const int dtype = elem_dtype(src, true);
    at::Tensor s4 = src.contiguous();
    if (src.dim() == 2) s4 = s4.unsqueeze(0).unsqueeze(-1);
    else if (src.dim() == 3) s4 = s4.unsqueeze(0);
    const int64_t n = s4.size(0), sh = s4.size(1), sw = s4.size(2), c = s4.size(3);
    at::Tensor Ms = host_f64(M, "M").reshape({-1, 3, 3});
    at::Tensor idx;
    const int32_t *idx_ptr = nullptr;
    if (mat_index.has_value()) {
        idx = mat_index->to(at::kCPU, at::kInt).contiguous();
        TORCH_CHECK(idx.numel() == n, "mat_index has ", idx.numel(), " entries for ", n, " frames");
        idx_ptr = idx.data_ptr<int32_t>();
    }
    at::Tensor out = at::empty({n, h, w, c}, s4.options());
    const double border[4] = {border_val, border_val, border_val, border_val};
    c10::cuda::CUDAGuard guard(src.device());
    check_rc(bevk_warp_perspective(s4.data_ptr(), out.data_ptr(), (int)n, (int)sh, (int)sw, (int)h, (int)w, (int)c,
                                   dtype, Ms.data_ptr<double>(), (int)Ms.size(0), idx_ptr, (int)flags,
                                   (int)border_mode, border, current_stream(src)),
             "bevk_warp_perspective");
    if (src.dim() == 2) return out.squeeze(-1).squeeze(0);
    if (src.dim() == 3) return out.squeeze(0);
    return out;
}

// NV12 frames (H*3/2, W) or (N, H*3/2, W): row pitch and frame stride from the tensor's strides
struct Nv12View {
    at::Tensor s3;
    int64_t n, h, w, pitch, frame_stride;
};

Nv12View nv12_view(const at::Tensor &src)
{
    TORCH_CHECK(src.is_cuda(), "src must be a CUDA tensor");
    TORCH_CHECK(src.scalar_type() == at::kByte, "NV12 frames are uint8, got ", src.scalar_type());
    TORCH_CHECK(src.dim() == 2 || src.dim() == 3, "NV12 frames must be (H*3/2, W) or (N, H*3/2, W)");
    Nv12View v;
    v.s3 = src.dim() == 2 ? src.unsqueeze(0) : src;
    v.n = v.s3.size(0);
    const int64_t rows = v.s3.size(1);
    v.w = v.s3.size(2);
    TORCH_CHECK(rows > 0 && rows % 3 == 0 && v.w % 2 == 0,
                "NV12 frames need H*3/2 rows for an even H and an even width; got ", rows, " x ", v.w);
    TORCH_CHECK(v.s3.stride(2) == 1, "NV12 rows must be contiguous (inner stride 1)");
    v.h = rows / 3 * 2;
    v.pitch = v.s3.stride(1);
    v.frame_stride = v.n > 1 ? v.s3.stride(0) : v.pitch * rows;
    return v;
}

at::Tensor nv12_to_bgr(const at::Tensor &src)
{
    Nv12View v = nv12_view(src);
    at::Tensor out = at::empty({v.n, v.h, v.w, 3}, v.s3.options());
    c10::cuda::CUDAGuard guard(src.device());
    check_rc(bevk_nv12_to_bgr(v.s3.data_ptr(), out.data_ptr(), (int)v.n, (int)v.h, (int)v.w, (int)v.pitch,
                              v.frame_stride, current_stream(src)),
             "bevk_nv12_to_bgr");
    return src.dim() == 2 ? out.squeeze(0) : out;
}

at::Tensor warp_perspective_nv12(const at::Tensor &src, const at::Tensor &M, int64_t w, int64_t h, int64_t flags,
                                 int64_t border_mode, double border_val,
                                 const c10::optional<at::Tensor> &mat_index)
{
    Nv12View v = nv12_view(src);
    at::Tensor Ms = host_f64(M, "M").reshape({-1, 3, 3});
    at::Tensor idx;
    const int32_t *idx_ptr = nullptr;
    if (mat_index.has_value()) {
        idx = mat_index->to(at::kCPU, at::kInt).contiguous();
        TORCH_CHECK(idx.numel() == v.n, "mat_index has ", idx.numel(), " entries for ", v.n, " frames");
        idx_ptr = idx.data_ptr<int32_t>();
    }
    at::Tensor out = at::empty({v.n, h, w, 3}, v.s3.options());
    const double border[4] = {border_val, border_val, border_val, border_val};
    c10::cuda::CUDAGuard guard(src.device());
    check_rc(bevk_warp_perspective_nv12(v.s3.data_ptr(), out.data_ptr(), (int)v.n, (int)v.h, (int)v.w,
                                        (int)v.pitch, v.frame_stride, (int)h, (int)w, Ms.data_ptr<double>(),
                                        (int)Ms.size(0), idx_ptr, (int)flags, (int)border_mode, border,
                                        current_stream(src)),
             "bevk_warp_perspective_nv12");
    return src.dim() == 2 ? out.squeeze(0) : out;
}

at::Tensor resize_nv12(const at::Tensor &src, int64_t w, int64_t h, int64_t interpolation)
{
    Nv12View v = nv12_view(src);
    at::Tensor out = at::empty({v.n, h, w, 3}, v.s3.options());
    c10::cuda::CUDAGuard guard(src.device());
    check_rc(bevk_resize_nv12_interp(v.s3.data_ptr(), out.data_ptr(), (int)v.n, (int)v.h, (int)v.w, (int)v.pitch,
                                     v.frame_stride, (int)h, (int)w, (int)interpolation, current_stream(src)),
             "bevk_resize_nv12_interp");
    return src.dim() == 2 ? out.squeeze(0) : out;
}

// rows (N, in_cols) -> (N, out_cols) through fn(in, out, n, ..., stream)
template <typename FN> at::Tensor rows(const at::Tensor &x, int64_t in_cols, int64_t out_cols, FN fn, const char *what)
{
    TORCH_CHECK(x.is_cuda(), "input must be a CUDA tensor");
    TORCH_CHECK(x.dim() == 2 && x.size(1) == in_cols, what, " expects shape (N, ", in_cols, ")");
    const int dtype = elem_dtype(x, false);
    at::Tensor xc = x.contiguous();
    at::Tensor out = at::empty({xc.size(0), out_cols}, xc.options());
    c10::cuda::CUDAGuard guard(x.device());
    check_rc(fn(xc.data_ptr(), out.data_ptr(), xc.size(0), dtype, current_stream(x)), what);
    return out;
}

at::Tensor project_points(const at::Tensor &pts, const at::Tensor &H)
{
    TORCH_CHECK(pts.dim() == 2 && (pts.size(1) == 2 || pts.size(1) == 3), "pts must be (N, 2) or (N, 3)");
    at::Tensor Hh = host_f64(H, "H");
    const int dim = (int)pts.size(1);
    return rows(pts, dim, dim, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_pts_project(i, o, n, dim, dt, Hh.data_ptr<double>(), st);
    }, "bevk_pts_project");
}

at::Tensor rbox_corners_project(const at::Tensor &xywhr, const c10::optional<at::Tensor> &H, int64_t mode)
{
    at::Tensor Hh = H.has_value() ? host_f64(*H, "H") : at::Tensor();
    return rows(xywhr, 5, 8, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_xywhr2xyxy(i, o, n, (int)mode, dt, Hh.defined() ? Hh.data_ptr<double>() : nullptr, st);
    }, "bevk_xywhr2xyxy");
}

at::Tensor corners_to_rbox(const at::Tensor &xy8, const c10::optional<at::Tensor> &H, int64_t mode)
{
    at::Tensor Hh = H.has_value() ? host_f64(*H, "H") : at::Tensor();
    return rows(xy8, 8, 5, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_xy82xywhr(i, o, n, (int)mode, dt, Hh.defined() ? Hh.data_ptr<double>() : nullptr, st);
    }, "bevk_xy82xywhr");
}

at::Tensor rbox_similarity(const at::Tensor &rbox, const at::Tensor &H, int64_t src_mode)
{
    at::Tensor Hh = host_f64(H, "H");
    return rows(rbox, 5, 5, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_rbox_world_bev(i, o, n, (int)src_mode, dt, Hh.data_ptr<double>(), st);
    }, "bevk_rbox_world_bev");
}

}  // namespace

TORCH_LIBRARY(bev_cuda, m)
{
    m.def("warp_perspective(Tensor src, Tensor M, int w, int h, int flags=1, int border_mode=0, "
          "float border_val=0., Tensor? mat_index=None) -> Tensor");
    m.def("project_points(Tensor pts, Tensor H) -> Tensor");
    m.def("rbox_corners_project(Tensor xywhr, Tensor? H, int mode) -> Tensor");
    m.def("corners_to_rbox(Tensor xy8, Tensor? H, int mode) -> Tensor");
    m.def("rbox_similarity(Tensor rbox, Tensor H, int src_mode) -> Tensor");
    m.def("nv12_to_bgr(Tensor src) -> Tensor");
    m.def("warp_perspective_nv12(Tensor src, Tensor M, int w, int h, int flags=1, int border_mode=0, "
          "float border_val=0., Tensor? mat_index=None) -> Tensor");
    m.def("resize_nv12(Tensor src, int w, int h, int interpolation=1) -> Tensor");
}

TORCH_LIBRARY_IMPL(bev_cuda, CUDA, m)
{
    m.impl("warp_perspective", &warp_perspective);
    m.impl("project_points", &project_points);
    m.impl("rbox_corners_project", &rbox_corners_project);
    m.impl("corners_to_rbox", &corners_to_rbox);
    m.impl("rbox_similarity", &rbox_similarity);
    m.impl("nv12_to_bgr", &nv12_to_bgr);
    m.impl("warp_perspective_nv12", &warp_perspective_nv12);
    m.impl("resize_nv12", &resize_nv12);
}
