// torch_ops.cpp -- the thin PyTorch C++ extension in front of libbev_b200.so (SURVEY.md 8b,
// "C-ABI / extension" row): registers every stream-ordered device entry point of
// include/bev_b200.h with the dispatcher as torch.ops.bev_cuda.* (the schemas are the m.def lines at
// the end of this file; bev_b200/torch_ops.py lists them with their shapes).
//
// Every CUDA implementation only checks tensors, allocates the result with torch's caching
// allocator, takes the current CUDA stream and calls the extern "C" entry point with raw pointers --
// no arithmetic lives here.  Homographies, K and Rt are CPU float64 tensors (they stay on the host,
// SURVEY.md 8b "Matrix ownership"), and so is a mat_index during CUDA-graph capture -- except the M of
// the four warps and the H_bg / H_fg of composite_bev, which may also be CUDA tensors on the frames'
// device: the kernels then read them when they run (the *_dmat entry points), so nothing synchronises
// and a captured graph replays whatever matrices were last written into them.  No CPU implementation
// is registered: CPU tensors fail in the dispatcher, there is no CPU fallback.
//
// Each operator is ONE function, registered for both the CUDA and the Meta dispatch key: it checks
// shapes and dtypes and allocates the output with SymInt sizes, and returns there for meta tensors
// (FakeTensor, torch.compile, torch.export, opcheck), so the two can never disagree on a shape.  A
// symbolic batch dimension only flows into the output's size (no guard on its value).  Checks that
// need values, or that the C library makes itself (BEVK_E_ARG), run on the CUDA side only.
//
// Reference interfaces replaced: cv2.warpPerspective at vis_homo.py:85-91, cv2.resize at
// vis_homo.py:90, rbox.pts_world_bev (bev/rbox.py:136-151), rbox_torch.xywhr2xyxy
// (bev/rbox_torch.py:52-99) + the projection of rbox_vis.py:38-55, rbox.xy82xywhr (bev/rbox.py:50-63),
// rbox_torch.rbox_world_bev (:123-168) and the other rbox_torch / rbox helpers, the compositor of
// bev/tool/compo.py, the tracker's iou_batch_rbox (rbox_tracker.py:87-92); the NV12 operators serve
// the frame loop of vis_homo.py:85-91 with frames from a GPU video decoder; the YUV 4:2:0 operators
// serve its VideoWriter.write (vis_homo.py:110-111) with frames for a video encoder.
#include <ATen/ATen.h>
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGraphsC10Utils.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/library.h>

#include "../../include/bev_b200.h"

namespace {

using c10::SymInt;
using Shape = c10::SymDimVector;

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

int64_t I(const SymInt &s) { return s.expect_int(); }

// a device operand of the CUDA side: on the device of `ref`
void check_cuda(const at::Tensor &t, const at::Tensor &ref, const char *what)
{
    TORCH_CHECK(t.is_cuda(), what, " must be a CUDA tensor");
    TORCH_CHECK(t.device() == ref.device(), what, " is on ", t.device(), ", expected ", ref.device());
}

// homography / matrix table on the host as contiguous float64
at::Tensor host_f64(const at::Tensor &m, const char *what)
{
    TORCH_CHECK(!m.is_cuda(), what, " must be a CPU tensor (homographies stay on the host)");
    return m.to(at::kDouble).contiguous();
}

// one 3x3 matrix
void check_mat3(const at::Tensor &H, const char *what)
{
    TORCH_SYM_CHECK(H.sym_numel().sym_eq(9), what, " must be 3x3, got shape ", H.sym_sizes());
}

void check_mats(const at::Tensor &M, const char *what)
{
    TORCH_SYM_CHECK(M.sym_numel().sym_gt(0).sym_and((M.sym_numel() % 9).sym_eq(0)), what,
                    " must hold 3x3 matrices (a multiple of 9 elements), got shape ", M.sym_sizes());
}

// ---- shape and validation helpers, one per operator family ----------------------------------------

// Warp matrices of n frames: (K, 3, 3) float64, on the host or (device) on the frames' device, and
// the optional per-frame index.  During CUDA-graph capture a CUDA mat_index cannot be read (the copy to
// the host synchronises): the captured graph would bake in the index of capture time anyway, so a CPU
// one is asked for.
struct WarpMats {
    at::Tensor M, idx;
    bool device;  // M is a CUDA tensor: call the *_dmat twin of the entry point
    const int32_t *idx_ptr() const { return idx.defined() ? idx.data_ptr<int32_t>() : nullptr; }
    // the entry point for M: host (host_fn) or device (dmat_fn) matrices; the twins share a signature
    template <typename FN> FN *pick(FN *host_fn, FN *dmat_fn) const { return device ? dmat_fn : host_fn; }
};

void check_warp_mats(const at::Tensor &M, const c10::optional<at::Tensor> &mat_index, const SymInt &n)
{
    check_mats(M, "M");
    if (mat_index.has_value())
        TORCH_SYM_CHECK(mat_index->sym_numel().sym_eq(n), "mat_index has ", mat_index->sym_numel(), " entries for ",
                        n, " frames");
}

WarpMats warp_mats(const at::Tensor &M, const c10::optional<at::Tensor> &mat_index, const at::Tensor &src)
{
    WarpMats m;
    m.device = M.is_cuda();
    if (m.device) {
        check_cuda(M, src, "M");
        m.M = M.to(at::kDouble).contiguous().reshape({-1, 3, 3});  // on the current stream, no host read
    } else {
        m.M = host_f64(M, "M").reshape({-1, 3, 3});
    }
    if (mat_index.has_value()) {
        TORCH_CHECK(!mat_index->is_cuda() ||
                        c10::cuda::currentStreamCaptureStatusMayInitCtx() == c10::cuda::CaptureStatus::None,
                    "mat_index is a CUDA tensor during CUDA-graph capture: reading it would synchronise the "
                    "capturing stream.  Pass mat_index as a CPU int32 tensor (it is fixed at capture time, like "
                    "the matrices)");
        m.idx = mat_index->to(at::kCPU, at::kInt).contiguous();
    }
    return m;
}

// Packed frames (H,W), (H,W,C) or (N,H,W,C), seen as (N,H,W,C); out() is a result of the same rank
struct Frames {
    int64_t dim;
    SymInt n, h, w, c;
    Shape out(const SymInt &oh, const SymInt &ow) const
    {
        if (dim == 2) return {oh, ow};
        if (dim == 3) return {oh, ow, c};
        return {n, oh, ow, c};
    }
};

Frames frames(const at::Tensor &src)
{
    TORCH_CHECK(src.dim() >= 2 && src.dim() <= 4, "src must be (H,W), (H,W,C) or (N,H,W,C)");
    const auto s = src.sym_sizes();
    const int64_t d = src.dim();
    return Frames{d, d == 4 ? s[0] : SymInt(1), s[d == 4 ? 1 : 0], s[d == 4 ? 2 : 1],
                  d == 2 ? SymInt(1) : s[d - 1]};
}

// BGR frames (H, W, 3) or (N, H, W, 3) uint8
Frames bgr_frames(const at::Tensor &src)
{
    TORCH_CHECK(src.scalar_type() == at::kByte, "BGR frames are uint8, got ", src.scalar_type());
    TORCH_CHECK((src.dim() == 3 || src.dim() == 4) && src.sym_size(-1) == 3, "src must be (H, W, 3) or (N, H, W, 3)");
    return frames(src);
}

// YUV 4:2:0 frames of h x w pixels, (h*3/2, w) or (N, h*3/2, w)
Shape yuv420_shape(bool batched, const SymInt &n, const SymInt &h, const SymInt &w)
{
    TORCH_SYM_CHECK((h % 2).sym_eq(0).sym_and((w % 2).sym_eq(0)),
                    "YUV 4:2:0 frames need an even width and height, got ", w, "x", h);
    if (batched) return {n, h / 2 * 3, w};
    return {h / 2 * 3, w};
}

// NV12 frames (H*3/2, W) or (N, H*3/2, W): uint8 with contiguous rows; pitch and frame stride are
// the tensor's (a decoder surface with padded rows is used as it is)
struct Nv12 {
    bool batched;
    SymInt n, h, w;
    Shape bgr(const SymInt &oh, const SymInt &ow) const
    {
        if (batched) return {n, oh, ow, 3};
        return {oh, ow, 3};
    }
};

Nv12 nv12_frames(const at::Tensor &src)
{
    TORCH_CHECK(src.scalar_type() == at::kByte, "NV12 frames are uint8, got ", src.scalar_type());
    TORCH_CHECK(src.dim() == 2 || src.dim() == 3, "NV12 frames must be (H*3/2, W) or (N, H*3/2, W)");
    const bool batched = src.dim() == 3;
    const SymInt rows = src.sym_size(-2), w = src.sym_size(-1);
    TORCH_SYM_CHECK(rows.sym_gt(0).sym_and((rows % 3).sym_eq(0)).sym_and((w % 2).sym_eq(0)),
                    "NV12 frames need H*3/2 rows for an even H and an even width; got ", rows, " x ", w);
    TORCH_SYM_CHECK(src.sym_stride(-1).sym_eq(1), "NV12 rows must be contiguous (inner stride 1)");
    return Nv12{batched, batched ? src.sym_size(0) : SymInt(1), rows / 3 * 2, w};
}

// the CUDA side of NV12 frames: the (N, H*3/2, W) view, row pitch and frame stride in bytes
struct Nv12View {
    at::Tensor s3;
    int64_t n, h, w, pitch, frame_stride;
};

Nv12View nv12_view(const at::Tensor &src, const Nv12 &f)
{
    Nv12View v;
    v.s3 = f.batched ? src : src.unsqueeze(0);
    v.n = I(f.n);
    v.h = I(f.h);
    v.w = I(f.w);
    v.pitch = v.s3.stride(1);
    v.frame_stride = v.n > 1 ? v.s3.stride(0) : v.pitch * v.s3.size(1);
    return v;
}

// Rows of boxes or points, float32 / float64: (N, in_cols), or any shape read flat when in_cols is 0
SymInt rows_n(const at::Tensor &x, int64_t in_cols, const char *what)
{
    elem_dtype(x, false);
    if (in_cols == 0) return x.sym_numel();
    TORCH_CHECK(x.dim() == 2 && x.sym_size(1) == in_cols, what, " expects shape (N, ", in_cols, ")");
    return x.sym_size(0);
}

// rows -> (N, *out_tail) through fn(in, out, n, dtype, stream), which calls one row-wise entry
// point; keep_shape: the output has x's shape (one value per element)
template <typename FN>
at::Tensor rows(const at::Tensor &x, int64_t in_cols, Shape out_tail, FN fn, const char *what,
                bool keep_shape = false)
{
    const SymInt n = rows_n(x, in_cols, what);
    Shape shape{n};
    shape.append(out_tail.begin(), out_tail.end());
    at::Tensor out = at::empty_symint(keep_shape ? Shape(x.sym_sizes()) : shape, x.options());
    if (x.is_meta()) return out;
    TORCH_CHECK(x.is_cuda(), "input must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(x.device());
    at::Tensor xc = x.contiguous();
    check_rc(fn(xc.data_ptr(), out.data_ptr(), I(n), elem_dtype(x, false), current_stream(x)), what);
    return out;
}

// ---- frame operators --------------------------------------------------------------------------------

at::Tensor warp_perspective(const at::Tensor &src, const at::Tensor &M, int64_t w, int64_t h, int64_t flags,
                            int64_t border_mode, double border_val, const c10::optional<at::Tensor> &mat_index)
{
    const int dtype = elem_dtype(src, true);
    const Frames f = frames(src);
    check_warp_mats(M, mat_index, f.n);
    at::Tensor out = at::empty_symint(f.out(h, w), src.options());
    if (src.is_meta()) return out;
    TORCH_CHECK(src.is_cuda(), "src must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(src.device());
    const at::Tensor s = src.contiguous();
    const WarpMats m = warp_mats(M, mat_index, src);
    const double border[4] = {border_val, border_val, border_val, border_val};
    check_rc(m.pick(bevk_warp_perspective, bevk_warp_perspective_dmat)(s.data_ptr(), out.data_ptr(), (int)I(f.n), (int)I(f.h), (int)I(f.w), (int)h,
                                   (int)w, (int)I(f.c), dtype, m.M.data_ptr<double>(), (int)m.M.size(0),
                                   m.idx_ptr(), (int)flags, (int)border_mode, border, current_stream(src)),
             "bevk_warp_perspective");
    return out;
}

at::Tensor resize(const at::Tensor &src, int64_t w, int64_t h, int64_t interpolation)
{
    TORCH_CHECK(src.scalar_type() == at::kByte, "resize takes uint8 frames, got ", src.scalar_type());
    const Frames f = frames(src);
    TORCH_SYM_CHECK(f.c.sym_ge(1).sym_and(f.c.sym_le(4)), "resize takes 1 to 4 channels, got ", f.c);
    at::Tensor out = at::empty_symint(f.out(h, w), src.options());
    if (src.is_meta()) return out;
    TORCH_CHECK(src.is_cuda(), "src must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(src.device());
    const at::Tensor s = src.contiguous();
    check_rc(bevk_resize(s.data_ptr(), out.data_ptr(), (int)I(f.n), (int)I(f.h), (int)I(f.w), (int)h, (int)w,
                         (int)I(f.c), BEVK_U8, (int)interpolation, current_stream(src)),
             "bevk_resize");
    return out;
}

at::Tensor nv12_to_bgr(const at::Tensor &src)
{
    const Nv12 f = nv12_frames(src);
    at::Tensor out = at::empty_symint(f.bgr(f.h, f.w), src.options());
    if (src.is_meta()) return out;
    TORCH_CHECK(src.is_cuda(), "src must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(src.device());
    const Nv12View v = nv12_view(src, f);
    check_rc(bevk_nv12_to_bgr(v.s3.data_ptr(), out.data_ptr(), (int)v.n, (int)v.h, (int)v.w, (int)v.pitch,
                              v.frame_stride, current_stream(src)),
             "bevk_nv12_to_bgr");
    return out;
}

at::Tensor warp_perspective_nv12(const at::Tensor &src, const at::Tensor &M, int64_t w, int64_t h, int64_t flags,
                                 int64_t border_mode, double border_val,
                                 const c10::optional<at::Tensor> &mat_index)
{
    const Nv12 f = nv12_frames(src);
    check_warp_mats(M, mat_index, f.n);
    at::Tensor out = at::empty_symint(f.bgr(h, w), src.options());
    if (src.is_meta()) return out;
    TORCH_CHECK(src.is_cuda(), "src must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(src.device());
    const Nv12View v = nv12_view(src, f);
    const WarpMats m = warp_mats(M, mat_index, src);
    const double border[4] = {border_val, border_val, border_val, border_val};
    check_rc(m.pick(bevk_warp_perspective_nv12, bevk_warp_perspective_nv12_dmat)(v.s3.data_ptr(), out.data_ptr(), (int)v.n, (int)v.h, (int)v.w,
                                        (int)v.pitch, v.frame_stride, (int)h, (int)w, m.M.data_ptr<double>(),
                                        (int)m.M.size(0), m.idx_ptr(), (int)flags, (int)border_mode, border,
                                        current_stream(src)),
             "bevk_warp_perspective_nv12");
    return out;
}

at::Tensor resize_nv12(const at::Tensor &src, int64_t w, int64_t h, int64_t interpolation)
{
    const Nv12 f = nv12_frames(src);
    at::Tensor out = at::empty_symint(f.bgr(h, w), src.options());
    if (src.is_meta()) return out;
    TORCH_CHECK(src.is_cuda(), "src must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(src.device());
    const Nv12View v = nv12_view(src, f);
    check_rc(bevk_resize_nv12_interp(v.s3.data_ptr(), out.data_ptr(), (int)v.n, (int)v.h, (int)v.w, (int)v.pitch,
                                     v.frame_stride, (int)h, (int)w, (int)interpolation, current_stream(src)),
             "bevk_resize_nv12_interp");
    return out;
}

at::Tensor bgr_to_yuv420(const at::Tensor &src, int64_t layout)
{
    const Frames f = bgr_frames(src);
    at::Tensor out = at::empty_symint(yuv420_shape(f.dim == 4, f.n, f.h, f.w), src.options());
    if (src.is_meta()) return out;
    TORCH_CHECK(src.is_cuda(), "src must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(src.device());
    const at::Tensor s = src.contiguous();
    const int64_t h = I(f.h), w = I(f.w);
    check_rc(bevk_bgr_to_yuv420(s.data_ptr(), out.data_ptr(), (int)I(f.n), (int)h, (int)w, (int)layout, (int)w,
                                w * (h / 2 * 3), current_stream(src)),
             "bevk_bgr_to_yuv420");
    return out;
}

at::Tensor warp_perspective_yuv420(const at::Tensor &src, const at::Tensor &M, int64_t w, int64_t h, int64_t layout,
                                   int64_t flags, int64_t border_mode, double border_val,
                                   const c10::optional<at::Tensor> &mat_index)
{
    const Frames f = bgr_frames(src);
    check_warp_mats(M, mat_index, f.n);
    at::Tensor out = at::empty_symint(yuv420_shape(f.dim == 4, f.n, h, w), src.options());
    if (src.is_meta()) return out;
    TORCH_CHECK(src.is_cuda(), "src must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(src.device());
    const at::Tensor s = src.contiguous();
    const WarpMats m = warp_mats(M, mat_index, src);
    const double border[4] = {border_val, border_val, border_val, border_val};
    check_rc(m.pick(bevk_warp_perspective_yuv420, bevk_warp_perspective_yuv420_dmat)(s.data_ptr(), out.data_ptr(), (int)I(f.n), (int)I(f.h), (int)I(f.w),
                                          (int)h, (int)w, (int)layout, (int)w, w * (h / 2 * 3),
                                          m.M.data_ptr<double>(), (int)m.M.size(0), m.idx_ptr(), (int)flags,
                                          (int)border_mode, border, current_stream(src)),
             "bevk_warp_perspective_yuv420");
    return out;
}

at::Tensor warp_perspective_nv12_yuv420(const at::Tensor &src, const at::Tensor &M, int64_t w, int64_t h,
                                        int64_t layout, int64_t flags, int64_t border_mode, double border_val,
                                        const c10::optional<at::Tensor> &mat_index)
{
    const Nv12 f = nv12_frames(src);
    check_warp_mats(M, mat_index, f.n);
    at::Tensor out = at::empty_symint(yuv420_shape(f.batched, f.n, h, w), src.options());
    if (src.is_meta()) return out;
    TORCH_CHECK(src.is_cuda(), "src must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(src.device());
    const Nv12View v = nv12_view(src, f);
    const WarpMats m = warp_mats(M, mat_index, src);
    const double border[4] = {border_val, border_val, border_val, border_val};
    check_rc(m.pick(bevk_warp_perspective_nv12_yuv420, bevk_warp_perspective_nv12_yuv420_dmat)(v.s3.data_ptr(), out.data_ptr(), (int)v.n, (int)v.h, (int)v.w,
                                               (int)v.pitch, v.frame_stride, (int)h, (int)w, (int)layout, (int)w,
                                               w * (h / 2 * 3), m.M.data_ptr<double>(), (int)m.M.size(0),
                                               m.idx_ptr(), (int)flags, (int)border_mode, border,
                                               current_stream(src)),
             "bevk_warp_perspective_nv12_yuv420");
    return out;
}

// ---- compositing --------------------------------------------------------------------------------------

void check_bgr_bytes(const at::Tensor &t, const char *what)
{
    TORCH_CHECK(t.scalar_type() == at::kByte, what, " must be uint8, got ", t.scalar_type());
    TORCH_CHECK(t.dim() >= 1 && t.sym_size(-1) == 3, what, " must be (..., 3) BGR, got shape ", t.sym_sizes());
}

// contiguous, with a data pointer aligned to `align` bytes (the kernels read words; a view at an odd
// byte offset is copied)
at::Tensor aligned(const at::Tensor &t, int64_t align)
{
    at::Tensor c = t.contiguous();
    return (reinterpret_cast<uintptr_t>(c.data_ptr()) % align) ? c.clone() : c;
}

at::Tensor composite(const at::Tensor &bg, const at::Tensor &fg, const at::Tensor &mask, int64_t bw_mode)
{
    check_bgr_bytes(bg, "bg");
    check_bgr_bytes(fg, "fg");
    check_bgr_bytes(mask, "mask");
    TORCH_SYM_CHECK(c10::sym_equals(bg.sym_sizes(), fg.sym_sizes()).sym_and(
                        c10::sym_equals(bg.sym_sizes(), mask.sym_sizes())),
                    "bg, fg and mask must share one shape; got ", bg.sym_sizes(), " ", fg.sym_sizes(), " ",
                    mask.sym_sizes());
    at::Tensor out = at::empty_symint(bg.sym_sizes(), bg.options());
    if (bg.is_meta()) return out;
    TORCH_CHECK(bg.is_cuda(), "bg must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(bg.device());
    check_cuda(fg, bg, "fg");
    check_cuda(mask, bg, "mask");
    const at::Tensor b = aligned(bg, 4), f = aligned(fg, 4), k = aligned(mask, 4);
    check_rc(bevk_composite_u8c3(b.data_ptr(), f.data_ptr(), k.data_ptr(), out.data_ptr(), out.numel() / 3,
                                 (int)(bw_mode != 0), current_stream(bg)),
             "bevk_composite_u8c3");
    return out;
}

// The compositor's forward matrices as contiguous float64: on the host, or (device) on fg's device,
// converted on the current stream with no host read
at::Tensor composite_mats(const at::Tensor &H, bool device, const at::Tensor &fg, const char *what)
{
    if (!device) return host_f64(H, what);
    check_cuda(H, fg, what);
    return H.to(at::kDouble).contiguous();
}

// fg, mask (H, W, 3) or (N, H, W, 3); bg (H, W, 3), (1, H, W, 3) or (N, H, W, 3); H_bg, H_fg 1 or N
// forward 3x3 matrices each, both on the host or both on fg's device -> (h, w, 3) or (N, h, w, 3)
at::Tensor composite_bev(const at::Tensor &bg, const at::Tensor &fg, const at::Tensor &mask, const at::Tensor &H_bg,
                         const at::Tensor &H_fg, int64_t w, int64_t h)
{
    check_bgr_bytes(bg, "bg");
    check_bgr_bytes(fg, "fg");
    check_bgr_bytes(mask, "mask");
    TORCH_CHECK(fg.dim() == 3 || fg.dim() == 4, "fg must be (H, W, 3) or (N, H, W, 3)");
    TORCH_SYM_CHECK(c10::sym_equals(fg.sym_sizes(), mask.sym_sizes()), "fg and mask must share one shape; got ",
                    fg.sym_sizes(), " ", mask.sym_sizes());
    TORCH_CHECK(bg.dim() == 3 || bg.dim() == 4, "bg must be (H, W, 3) or (N, H, W, 3)");
    const Frames fr = frames(fg);
    if (bg.dim() == 4)
        TORCH_SYM_CHECK(bg.sym_size(0).sym_eq(fr.n).sym_or(bg.sym_size(0).sym_eq(1)), "bg has ", bg.sym_size(0),
                        " frames for ", fr.n, " foregrounds (need 1 or one each)");
    check_mats(H_bg, "H_bg");
    check_mats(H_fg, "H_fg");
    TORCH_SYM_CHECK(H_bg.sym_numel().sym_eq(H_fg.sym_numel()), "H_bg and H_fg must hold as many matrices; got ",
                    H_bg.sym_sizes(), " and ", H_fg.sym_sizes());
    at::Tensor out = at::empty_symint(fr.out(h, w), fg.options());
    if (fg.is_meta()) return out;
    TORCH_CHECK(fg.is_cuda(), "fg must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(fg.device());
    check_cuda(bg, fg, "bg");
    check_cuda(mask, fg, "mask");
    const at::Tensor b = aligned(bg.dim() == 3 ? bg.unsqueeze(0) : bg, 16), f = aligned(fg, 16),
                     k = aligned(mask, 16);
    const bool device = H_bg.is_cuda() || H_fg.is_cuda();
    TORCH_CHECK(H_bg.is_cuda() == H_fg.is_cuda(), "H_bg is on ", H_bg.device(), " and H_fg on ", H_fg.device(),
                ": pass both homographies on the host or both on the frames' CUDA device");
    const at::Tensor Hb = composite_mats(H_bg, device, fg, "H_bg"), Hf = composite_mats(H_fg, device, fg, "H_fg");
    check_rc((device ? bevk_composite_bev_u8c3_dmat : bevk_composite_bev_u8c3)(
                 b.data_ptr(), f.data_ptr(), k.data_ptr(), out.data_ptr(), (int)I(fr.n), (int)b.size(0),
                 (int)b.size(1), (int)b.size(2), (int)I(fr.h), (int)I(fr.w), (int)h, (int)w, Hb.data_ptr<double>(),
                 Hf.data_ptr<double>(), (int)(Hb.numel() / 9), current_stream(fg)),
             device ? "bevk_composite_bev_u8c3_dmat" : "bevk_composite_bev_u8c3");
    return out;
}

// ---- boxes and points -------------------------------------------------------------------------------

at::Tensor project_points(const at::Tensor &pts, const at::Tensor &H)
{
    TORCH_CHECK(pts.dim() == 2 && (pts.sym_size(1) == 2 || pts.sym_size(1) == 3), "pts must be (N, 2) or (N, 3)");
    check_mat3(H, "H");
    const int64_t dim = pts.sym_size(1).guard_int(__FILE__, __LINE__);
    return rows(pts, dim, {dim}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_pts_project(i, o, n, (int)dim, dt, host_f64(H, "H").data_ptr<double>(), st);
    }, "bevk_pts_project");
}

const double *opt_host_f64(const c10::optional<at::Tensor> &H, at::Tensor &keep)
{
    if (!H.has_value()) return nullptr;
    keep = host_f64(*H, "H");
    return keep.data_ptr<double>();
}

at::Tensor rbox_corners_project(const at::Tensor &xywhr, const c10::optional<at::Tensor> &H, int64_t mode)
{
    if (H.has_value()) check_mat3(*H, "H");
    return rows(xywhr, 5, {8}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        at::Tensor keep;
        return bevk_xywhr2xyxy(i, o, n, (int)mode, dt, opt_host_f64(H, keep), st);
    }, "bevk_xywhr2xyxy");
}

at::Tensor corners_to_rbox(const at::Tensor &xy8, const c10::optional<at::Tensor> &H, int64_t mode)
{
    if (H.has_value()) check_mat3(*H, "H");
    return rows(xy8, 8, {5}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        at::Tensor keep;
        return bevk_xy82xywhr(i, o, n, (int)mode, dt, opt_host_f64(H, keep), st);
    }, "bevk_xy82xywhr");
}

at::Tensor rbox_similarity(const at::Tensor &rbox, const at::Tensor &H, int64_t src_mode)
{
    check_mat3(H, "H");
    return rows(rbox, 5, {5}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_rbox_world_bev(i, o, n, (int)src_mode, dt, host_f64(H, "H").data_ptr<double>(), st);
    }, "bevk_rbox_world_bev");
}

at::Tensor rboxtt_similarity(const at::Tensor &rboxtt, const at::Tensor &H, int64_t src_mode)
{
    check_mat3(H, "H");
    return rows(rboxtt, 7, {7}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_rboxtt_world_bev(i, o, n, (int)src_mode, dt, host_f64(H, "H").data_ptr<double>(), st);
    }, "bevk_rboxtt_world_bev");
}

// K (3, 3) or (3, 4), Rt (3, 4) or (4, 4): the entry point reads K's 3x3 and Rt's 3x4 block
at::Tensor rbox_zt2tt_world(const at::Tensor &rboxzt, const at::Tensor &K, const at::Tensor &Rt)
{
    TORCH_CHECK(K.dim() == 2 && K.sym_size(0) == 3 && (K.sym_size(1) == 3 || K.sym_size(1) == 4),
                "K must be 3x3 (or 3x4), got shape ", K.sym_sizes());
    TORCH_CHECK(Rt.dim() == 2 && (Rt.sym_size(0) == 3 || Rt.sym_size(0) == 4) && Rt.sym_size(1) == 4,
                "Rt must be 3x4 (or 4x4), got shape ", Rt.sym_sizes());
    return rows(rboxzt, 7, {7}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        const at::Tensor k = host_f64(K, "K").slice(1, 0, 3).contiguous();
        const at::Tensor rt = host_f64(Rt, "Rt").slice(0, 0, 3).contiguous();
        return bevk_rbox_zt2tt_world(i, o, n, dt, k.data_ptr<double>(), rt.data_ptr<double>(), st);
    }, "bevk_rbox_zt2tt_world");
}

at::Tensor rbox_heading(const at::Tensor &xywhr, int64_t mode)
{
    return rows(xywhr, 5, {4}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_xywhr2xyvec(i, o, n, (int)mode, dt, st);
    }, "bevk_xywhr2xyvec");
}

at::Tensor corners_heading(const at::Tensor &xy8)
{
    return rows(xy8, 8, {4}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_xy82xyvec(i, o, n, dt, st);
    }, "bevk_xy82xyvec");
}

// yaw angles of any shape, flattened like the reference
at::Tensor angle_similarity(const at::Tensor &yaw, const at::Tensor &H, int64_t src_mode)
{
    check_mat3(H, "H");
    return rows(yaw, 0, {}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_angle_world_bev(i, o, n, (int)src_mode, dt, host_f64(H, "H").data_ptr<double>(), st);
    }, "bevk_angle_world_bev");
}

// lengths of any shape, in the same shape
at::Tensor dist_similarity(const at::Tensor &d, const at::Tensor &H)
{
    check_mat3(H, "H");
    return rows(d, 0, {}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_dist_world_bev(i, o, n, dt, host_f64(H, "H").data_ptr<double>(), st);
    }, "bevk_dist_world_bev", true);
}

at::Tensor v2yaw(const at::Tensor &v, int64_t mode)
{
    return rows(v, 2, {}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_v2yaw(i, o, n, (int)mode, dt, st);
    }, "bevk_v2yaw");
}

at::Tensor yaw2v(const at::Tensor &yaw, int64_t mode)
{
    return rows(yaw, 0, {2}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_yaw2v(i, o, n, (int)mode, dt, st);
    }, "bevk_yaw2v");
}

at::Tensor yaw2mat(const at::Tensor &yaw, int64_t mode)
{
    return rows(yaw, 0, {2, 2}, [&](const void *i, void *o, int64_t n, int dt, void *st) {
        return bevk_yaw2mat(i, o, n, (int)mode, dt, st);
    }, "bevk_yaw2mat");
}

// (N, >=5) x (M, >=5) rows [x, y, w, h, r, ...] -> (N, M).  Rows are passed with their own stride, so
// a view of the first columns of wider rows (a score column) needs no copy.
at::Tensor rbox_iou_matrix(const at::Tensor &boxes1, const at::Tensor &boxes2, double yaw_offset)
{
    const int dtype = elem_dtype(boxes1, false);
    TORCH_CHECK(boxes2.scalar_type() == boxes1.scalar_type(), "boxes1 and boxes2 must share a dtype, got ",
                boxes1.scalar_type(), " and ", boxes2.scalar_type());
    for (const at::Tensor *b : {&boxes1, &boxes2})
        TORCH_CHECK(b->dim() == 2 && b->sym_size(1) >= 5, "boxes must be (N, >=5) rows [x, y, w, h, r, ...], got shape ",
                    b->sym_sizes());
    at::Tensor out = at::empty_symint({boxes1.sym_size(0), boxes2.sym_size(0)}, boxes1.options());
    if (boxes1.is_meta()) return out;
    TORCH_CHECK(boxes1.is_cuda(), "boxes1 must be a CUDA tensor");
    c10::cuda::CUDAGuard guard(boxes1.device());
    check_cuda(boxes2, boxes1, "boxes2");
    auto strided = [](const at::Tensor &b) {
        return (b.stride(1) == 1 && b.stride(0) >= 5 && b.stride(0) <= INT32_MAX) ? b : b.contiguous();
    };
    const at::Tensor b1 = strided(boxes1), b2 = strided(boxes2);
    check_rc(bevk_rbox_iou_matrix(b1.data_ptr(), b1.size(0), (int)b1.stride(0), b2.data_ptr(), b2.size(0),
                                  (int)b2.stride(0), out.data_ptr(), dtype, yaw_offset, current_stream(boxes1)),
             "bevk_rbox_iou_matrix");
    return out;
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
    m.def("bgr_to_yuv420(Tensor src, int layout=0) -> Tensor");
    m.def("warp_perspective_yuv420(Tensor src, Tensor M, int w, int h, int layout=0, int flags=1, "
          "int border_mode=0, float border_val=0., Tensor? mat_index=None) -> Tensor");
    m.def("resize(Tensor src, int w, int h, int interpolation=1) -> Tensor");
    m.def("warp_perspective_nv12_yuv420(Tensor src, Tensor M, int w, int h, int layout=0, int flags=1, "
          "int border_mode=0, float border_val=0., Tensor? mat_index=None) -> Tensor");
    m.def("composite(Tensor bg, Tensor fg, Tensor mask, int bw_mode=0) -> Tensor");
    m.def("composite_bev(Tensor bg, Tensor fg, Tensor mask, Tensor H_bg, Tensor H_fg, int w, int h) -> Tensor");
    m.def("rbox_iou_matrix(Tensor boxes1, Tensor boxes2, float yaw_offset=0.) -> Tensor");
    m.def("rboxtt_similarity(Tensor rboxtt, Tensor H, int src_mode) -> Tensor");
    m.def("rbox_zt2tt_world(Tensor rboxzt, Tensor K, Tensor Rt) -> Tensor");
    m.def("rbox_heading(Tensor xywhr, int mode) -> Tensor");
    m.def("corners_heading(Tensor xy8) -> Tensor");
    m.def("angle_similarity(Tensor yaw, Tensor H, int src_mode) -> Tensor");
    m.def("dist_similarity(Tensor d, Tensor H) -> Tensor");
    m.def("v2yaw(Tensor v, int mode) -> Tensor");
    m.def("yaw2v(Tensor yaw, int mode) -> Tensor");
    m.def("yaw2mat(Tensor yaw, int mode) -> Tensor");
}

#define BEV_CUDA_OPS(m)                                                  \
    m.impl("warp_perspective", &warp_perspective);                       \
    m.impl("project_points", &project_points);                           \
    m.impl("rbox_corners_project", &rbox_corners_project);               \
    m.impl("corners_to_rbox", &corners_to_rbox);                         \
    m.impl("rbox_similarity", &rbox_similarity);                         \
    m.impl("nv12_to_bgr", &nv12_to_bgr);                                 \
    m.impl("warp_perspective_nv12", &warp_perspective_nv12);             \
    m.impl("resize_nv12", &resize_nv12);                                 \
    m.impl("bgr_to_yuv420", &bgr_to_yuv420);                             \
    m.impl("warp_perspective_yuv420", &warp_perspective_yuv420);         \
    m.impl("resize", &resize);                                           \
    m.impl("warp_perspective_nv12_yuv420", &warp_perspective_nv12_yuv420); \
    m.impl("composite", &composite);                                     \
    m.impl("composite_bev", &composite_bev);                             \
    m.impl("rbox_iou_matrix", &rbox_iou_matrix);                         \
    m.impl("rboxtt_similarity", &rboxtt_similarity);                     \
    m.impl("rbox_zt2tt_world", &rbox_zt2tt_world);                       \
    m.impl("rbox_heading", &rbox_heading);                               \
    m.impl("corners_heading", &corners_heading);                         \
    m.impl("angle_similarity", &angle_similarity);                       \
    m.impl("dist_similarity", &dist_similarity);                         \
    m.impl("v2yaw", &v2yaw);                                             \
    m.impl("yaw2v", &yaw2v);                                             \
    m.impl("yaw2mat", &yaw2mat)

TORCH_LIBRARY_IMPL(bev_cuda, CUDA, m) { BEV_CUDA_OPS(m); }

// the same functions: they return after the shape checks and the SymInt allocation for meta tensors
TORCH_LIBRARY_IMPL(bev_cuda, Meta, m) { BEV_CUDA_OPS(m); }
