// resize_coef.cuh -- the coefficient arithmetic of cv2.resize's 8-bit bilinear resize, with
// INTER_LINEAR's rule and with INTER_AREA's for a resize with an upscaling axis, and the parameter
// block and launch plan of every resize kernel (resize.cu).  Semantics: see resize.cu.
#pragma once
#include "bevk_common.cuh"

constexpr int kCoefScale = 2048;  // INTER_RESIZE_COEF_SCALE

// (index, w0, w1) of dst position d along one axis; `clamp` = the column rule
__device__ __forceinline__ void axis_coef(int d, double scale, int ssize, bool clamp, int &s, int &w0, int &w1)
{
    float f = __double2float_rn(__dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), 0.5));
    int si = __float2int_rd(f);  // cvFloor
    f = __fsub_rn(f, (float)si);
    if (clamp) {
        if (si < 0) {
            f = 0.f;
            si = 0;
        }
        if (si >= ssize - 1) {
            f = 0.f;
            si = ssize - 1;
        }
    }
    w0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), (float)kCoefScale));
    w1 = __float2int_rn(__fmul_rn(f, (float)kCoefScale));
    s = si;
}

// (index, w0, w1) of dst position d in cv2's bilinear emulation of INTER_AREA; `clamp` = the
// column rule (at / right of the last pixel: (ssize - 1, 0))
__device__ __forceinline__ void linear_area_coef(int d, double scale, double inv, int ssize, bool clamp, int &s,
                                                 int &w0, int &w1)
{
    int si = __double2int_rd(__dmul_rn((double)d, scale));
    float f = __double2float_rn(__dsub_rn((double)(d + 1), __dmul_rn((double)(si + 1), inv)));
    f = f <= 0.f ? 0.f : __fsub_rn(f, floorf(f));
    if (clamp && si >= ssize - 1) {
        f = 0.f;
        si = ssize - 1;
    }
    w0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), (float)kCoefScale));
    w1 = __float2int_rn(__fmul_rn(f, (float)kCoefScale));
    s = si;
}

__device__ __forceinline__ uint32_t vpass(int b0, int b1, int s0, int s1)
{
    return (uint32_t)((((b0 * (s0 >> 4)) >> 16) + ((b1 * (s1 >> 4)) >> 16) + 2) >> 2);
}

// A resize of n_frames > 0 frames, as every resize kernel reads it.  The fields up to
// frames_per_chunk are those the INTER_LINEAR kernels of BGR frames read, in the order they
// always had.
struct BevkResizeParams {
    const uint8_t *src;              // frame 0; NV12: its first luma byte
    uint8_t *dst;
    int src_h, src_w, dst_h, dst_w;  // NV12: the luma size
    long long src_frame, dst_frame;  // bytes from one source / dst frame to the next
    double scale_x, scale_y;         // cv2: scale = 1. / inv_scale
    int n_frames, frames_per_chunk;  // frames_per_chunk: at most 64, fewer until the grid fills the SMs
    long long pitch;                 // bytes from one source row to the next (NV12: luma or chroma row)
    double inv_x, inv_y;             // cv2: inv_scale = (double)dsize / ssize
    int kx, ky;                      // INTER_AREA integer cells only: the integer scales
    float inv_area;                  // INTER_AREA integer cells only: 1.f / (kx * ky)
};

// The column (sx, a0, a1) and row (sy, b0, b1) coefficients of dst pixel (x, y): INTER_LINEAR's
// rule, or with AREA INTER_AREA's bilinear emulation
template <bool AREA>
__device__ __forceinline__ void bilinear_coef(const BevkResizeParams &p, int x, int y, int &sx, int &a0, int &a1,
                                              int &sy, int &b0, int &b1)
{
    if constexpr (AREA) {
        linear_area_coef(x, p.scale_x, p.inv_x, p.src_w, true, sx, a0, a1);
        linear_area_coef(y, p.scale_y, p.inv_y, p.src_h, false, sy, b0, b1);
    } else {
        axis_coef(x, p.scale_x, p.src_w, true, sx, a0, a1);
        axis_coef(y, p.scale_y, p.src_h, false, sy, b0, b1);
    }
}

// Fills p for n_frames > 0 frames and the grid of 32 x 8 pixel blocks that runs it, one thread per
// dst pixel of every frame of its chunk (grid z); leaves kx, ky and inv_area 0.
inline int bevk_plan_resize(const void *src, void *dst, int n_frames, int src_h, int src_w, int channels,
                            long long pitch, long long frame_stride, int dst_h, int dst_w, BevkResizeParams &p,
                            dim3 &grid)
{
    p = BevkResizeParams{};
    p.src = (const uint8_t *)src;
    p.dst = (uint8_t *)dst;
    p.src_h = src_h;
    p.src_w = src_w;
    p.dst_h = dst_h;
    p.dst_w = dst_w;
    p.src_frame = frame_stride;
    p.dst_frame = (long long)dst_h * dst_w * channels;
    p.pitch = pitch;
    p.inv_x = (double)dst_w / (double)src_w;
    p.inv_y = (double)dst_h / (double)src_h;
    p.scale_x = 1.0 / p.inv_x;
    p.scale_y = 1.0 / p.inv_y;
    const long long tiles = (long long)((dst_w + 31) / 32) * ((dst_h + 7) / 8);
    const long long want_blocks = (long long)bevk_sm_count() * 8 * 2;
    int fpc = n_frames < 64 ? n_frames : 64;
    while (fpc > 1 && tiles * ((n_frames + fpc - 1) / fpc) < want_blocks) fpc = (fpc + 1) / 2;
    // ~12 waves of blocks while a chunk keeps 8 frames: few long blocks leave a costly last wave
    while (fpc >= 16 && tiles * ((n_frames + fpc - 1) / fpc) < 6 * want_blocks) fpc = (fpc + 1) / 2;
    p.n_frames = n_frames;
    p.frames_per_chunk = fpc;
    const int z = (n_frames + fpc - 1) / fpc;
    if (z > 65535) BEVK_FAIL(BEVK_E_ARG, "resize: too many frame chunks (%d) for one launch", z);
    grid = dim3((dst_w + 31) / 32, (dst_h + 7) / 8, z);
    return BEVK_OK;
}
