// resize_coef.cuh -- the coefficient arithmetic of cv2.resize (uint8, INTER_LINEAR) and the frame
// chunking of its launches, shared by the BGR resize (resize.cu) and the NV12 resize (nv12.cu).
// Semantics: see resize.cu.
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

__device__ __forceinline__ uint32_t vpass(int b0, int b1, int s0, int s1)
{
    return (uint32_t)((((b0 * (s0 >> 4)) >> 16) + ((b1 * (s1 >> 4)) >> 16) + 2) >> 2);
}

// Frames per chunk (grid z) of a resize launch with 32 x 8 pixel blocks, one thread per dst pixel
// of every frame of its chunk: at most 64, fewer until the grid fills the SMs.
inline int bevk_resize_frames_per_chunk(int n_frames, int dst_h, int dst_w)
{
    const long long tiles = (long long)((dst_w + 31) / 32) * ((dst_h + 7) / 8);
    const long long want_blocks = (long long)bevk_sm_count() * 8 * 2;
    int fpc = n_frames < 64 ? n_frames : 64;
    while (fpc > 1 && tiles * ((n_frames + fpc - 1) / fpc) < want_blocks) fpc = (fpc + 1) / 2;
    // ~12 waves of blocks while a chunk keeps 8 frames: few long blocks leave a costly last wave
    while (fpc >= 16 && tiles * ((n_frames + fpc - 1) / fpc) < 6 * want_blocks) fpc = (fpc + 1) / 2;
    return fpc;
}
