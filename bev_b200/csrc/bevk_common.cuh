// bevk_common.cuh -- shared declarations of libbev_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>

#include "../../include/bev_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libbev_b200 is written for sm_100a (B200) only"
#endif

#define BEVK_HD __host__ __device__ __forceinline__

// ----------------------------------------------------------------------------- errors
void bevk_set_error(const char *fmt, ...);
#define BEVK_FAIL(code, ...)          \
    do {                              \
        bevk_set_error(__VA_ARGS__);  \
        return (code);                \
    } while (0)
#define BEVK_CUDA(expr)                                                                   \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            bevk_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                           __LINE__);                                                     \
            return BEVK_E_CUDA;                                                           \
        }                                                                                 \
    } while (0)

int bevk_require_device(void);  // BEVK_OK or BEVK_E_NOGPU (+ message); caches the probe
int bevk_sm_count(void);

// ----------------------------------------------------------------------------- warp geometry
// The dst->src coordinate pipeline of cv2.warpPerspective 4.13 (SURVEY.md Appendix A), which the
// reference reaches at vis_homo.py:89.  All of it is IEEE double with NO fused multiply-add:
// device code spells every operation with a round-to-nearest intrinsic, host code is compiled
// with -ffp-contract=off.  The column is split into a block base xb (multiples of bw0) plus an
// in-block offset x1 because cv2 evaluates it that way and exact-tie pixels flip otherwise.

BEVK_HD double bevk_mul(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
BEVK_HD double bevk_add(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
BEVK_HD double bevk_div(double a, double b)
{
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}
BEVK_HD int bevk_round_sat(double v)
{
    // clamp to int32 then round half to even
    v = v < -2147483648.0 ? -2147483648.0 : v;
    v = v > 2147483647.0 ? 2147483647.0 : v;
#ifdef __CUDA_ARCH__
    return __double2int_rn(v);
#else
    return (int)__builtin_lrint(v);
#endif
}
BEVK_HD int bevk_sat16(int v) { return v < -32768 ? -32768 : (v > 32767 ? 32767 : v); }

// cv2's block width for a dsize: min(16,h) rows -> 1024/rows columns, clipped to the width.
BEVK_HD int bevk_block_width(int dst_w, int dst_h)
{
    int bh0 = dst_h < 16 ? dst_h : 16;
    int bw0 = 1024 / bh0;
    return bw0 > dst_w ? dst_w : bw0;
}

// Quantised source coordinate of dst pixel (xb + x1, y), xb = start of its cv2 block column.
// scale = 32 (bilinear, 1/32 px) or 1 (nearest).
BEVK_HD void bevk_map_pixel_xb(const double *M, int xb, int x1, int y, double scale, int &X, int &Y)
{
    const double dxb = (double)xb, dx1 = (double)x1, dy = (double)y;
    const double X0 = bevk_add(bevk_add(bevk_mul(M[0], dxb), bevk_mul(M[1], dy)), M[2]);
    const double Y0 = bevk_add(bevk_add(bevk_mul(M[3], dxb), bevk_mul(M[4], dy)), M[5]);
    const double W0 = bevk_add(bevk_add(bevk_mul(M[6], dxb), bevk_mul(M[7], dy)), M[8]);
    double w = bevk_add(W0, bevk_mul(M[6], dx1));
    w = (w != 0.0) ? bevk_div(scale, w) : 0.0;
    X = bevk_round_sat(bevk_mul(bevk_add(X0, bevk_mul(M[0], dx1)), w));
    Y = bevk_round_sat(bevk_mul(bevk_add(Y0, bevk_mul(M[3], dx1)), w));
}
BEVK_HD void bevk_map_pixel(const double *M, int x, int y, int bw0, double scale, int &X, int &Y)
{
    const int xb = (x / bw0) * bw0;
    bevk_map_pixel_xb(M, xb, x - xb, y, scale, X, Y);
}

// ----------------------------------------------------------------------------- warp launch plan
// One launch serves up to BEVK_MAX_GROUPS (matrix, frame-run) pairs: "many frames and many
// homographies in one launch".  A run is frames first, first+stride, ... (count of them).
#define BEVK_MAX_GROUPS 16

struct BevkWarpGroup {
    double M[9];     // dst->src map (already inverted on the host)
    int first;       // first frame of the run
    int count;       // frames in the run
    int stride;      // frame index step
    int chunk0;      // first z-block (generic) / first work item (fast path) of this group
};

struct BevkWarpParams {
    const void *src;
    void *dst;
    int src_h, src_w, dst_h, dst_w;
    long long src_frame_elems, dst_frame_elems;  // elements (not bytes) per frame
    int bw0;                                     // cv2 block width for (dst_w, dst_h)
    int frames_per_chunk;
    int n_groups;
    int total_chunks;
    float border[4];
    // Split launches (staged kernel + direct-gather kernel over the tiles the first one could not
    // stage): one byte per (group, staged tile), index = group * hard_tiles + tile_x * hard_ty +
    // tile_y.  The staged kernel sets the byte and skips the tile; the direct kernel, when the
    // pointer is set, only works on 32x8 blocks whose staged tile (hard_tw x hard_th pixels) is
    // marked.  NULL: no split.
    unsigned char *hard;
    int hard_tw, hard_th, hard_ty, hard_tiles;
    BevkWarpGroup g[BEVK_MAX_GROUPS];
};

// The warp of NV12 or I420 frames to BGR (nv12.cu): w.src is frame 0's first luma byte, w.src_h /
// w.src_w the luma size; w.src_frame_elems is unused, the two strides below replace it.
struct BevkNv12Params {
    BevkWarpParams w;
    int pitch;               // bytes from one luma or chroma row to the next
    long long frame_stride;  // bytes from one frame to the next
};

// The warps to YUV 4:2:0 (yuv420.cu): w.dst is frame 0's first luma byte, w.src_frame_elems and
// w.dst_frame_elems are unused; BGR sources have pitch = 3 * src_w and frame_stride = pitch * src_h.
struct BevkYuvParams {
    BevkWarpParams w;
    int pitch;                   // source bytes from one (luma or chroma) row to the next
    long long frame_stride;      // source bytes from one frame to the next
    int dst_pitch;               // dst bytes from one luma or chroma row to the next
    long long dst_frame_stride;  // dst bytes from one frame to the next
};

// kernels-side entry points implemented in the .cu files
int bevk_launch_warp_generic(const BevkWarpParams &p, int channels, int dtype, int linear,
                             cudaStream_t stream);
// fills frames_per_chunk, total_chunks and the groups' chunk0 for the direct-gather kernels
int bevk_plan_generic_chunks(BevkWarpParams &p, int channels);
// returns 1 if it launched, 0 if the shape does not qualify for the staged path (or, unless
// `force`, is too small a batch to amortise its per-tile set-up), <0 on error
int bevk_launch_warp_fast(const BevkWarpParams &p, int channels, int dtype, int linear, int force,
                          cudaStream_t stream);
// NV12 or I420 (src_format BEVK_YUV_NV12 / BEVK_YUV_I420) -> BGR warp over the chunks
// bevk_plan_generic_chunks planned for P.w
int bevk_launch_warp_nv12(const BevkNv12Params &P, int src_format, int linear, cudaStream_t stream);
int bevk_launch_nv12_to_bgr(const void *src, void *dst, int n_frames, int h, int w, int pitch,
                            long long frame_stride, cudaStream_t stream);
// cv2.resize of n_frames > 0 frames with `interpolation` (BEVK_INTER_LINEAR or BEVK_INTER_AREA):
// uint8 frames with `channels` channels, or (nv12, channels 3) NV12 frames converted to BGR; rows
// `pitch` and frames `frame_stride` bytes apart; arguments already checked by the entry points
int bevk_launch_resize(const void *src, void *dst, int n_frames, int src_h, int src_w, int channels, int nv12,
                       long long pitch, long long frame_stride, int dst_h, int dst_w, int interpolation,
                       cudaStream_t stream);
// BGR, NV12 or I420 frames (src_format BEVK_BGR / BEVK_YUV_NV12 / BEVK_YUV_I420) warped to YUV
// 4:2:0 (nv12_out: NV12, else I420) over the chunks planned for P.w on the grid of 2x2 dst blocks
int bevk_launch_warp_yuv420(const BevkYuvParams &P, int src_format, int nv12_out, int linear, cudaStream_t stream);
// n_frames > 0 contiguous BGR frames of h x w (both even) to YUV 4:2:0 (nv12_out: NV12, else I420)
int bevk_launch_bgr_to_yuv420(const void *src, void *dst, int n_frames, int h, int w, int nv12_out, int dst_pitch,
                              long long dst_frame_stride, cudaStream_t stream);
