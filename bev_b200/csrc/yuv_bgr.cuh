// yuv_bgr.cuh -- one NV12 sample to BGR, cv2.cvtColor(COLOR_YUV2BGR_NV12)'s arithmetic (BT.601
// limited range, 20-bit fixed point), shared by the NV12 conversion and warp (nv12.cu) and the NV12
// resizes (resize.cu).
#pragma once
#include "bevk_common.cuh"

namespace {

__device__ __forceinline__ uint32_t byte_of(uint32_t w, int i) { return (w >> (8 * i)) & 0xffu; }

__device__ __forceinline__ int clamp8(int v) { return min(max(v, 0), 255); }

// One sample to [B, G, R, 0].  Every term fits in int32: |y| <= 239 * 1220542, |chroma| <= 128 *
// 2116026.
__device__ __forceinline__ uint32_t yuv_to_bgr(uint32_t Y, uint32_t U, uint32_t V)
{
    const int y = max((int)Y - 16, 0) * 1220542;
    const int u = (int)U - 128, v = (int)V - 128;
    const int r = clamp8((y + 1673527 * v + (1 << 19)) >> 20);
    const int g = clamp8((y - 852492 * v - 409993 * u + (1 << 19)) >> 20);
    const int b = clamp8((y + 2116026 * u + (1 << 19)) >> 20);
    return (uint32_t)b | ((uint32_t)g << 8) | ((uint32_t)r << 16);
}

}  // namespace
