// resize_area.cu -- batched cv2.resize(img, dsize, interpolation=INTER_AREA) on uint8 frames with 1
// to 4 channels, and the same fused with the NV12 -> BGR conversion for frames from a GPU video
// decoder: cv2.resize(cv2.cvtColor(f, COLOR_YUV2BGR_NV12), dsize, interpolation=INTER_AREA).
// INTER_AREA is what OpenCV recommends for a small frame: every source pixel contributes to the
// dst pixel whose cell it lies in, so fine texture such as lane markings does not alias.
//
// Semantics: OpenCV 4.13, bit for bit (oracle/resize_area_oracle.py restates it and is pinned
// against cv2).  With scale = 1 / (dsize / ssize) in double per axis, cv2 takes one of three
// branches, and each is a kernel variant here (MODE):
//   kFast   both scales >= 1 and integer (kx, ky): the integer sum s of the kx x ky cell, then
//           rint(s * (1.f / (kx * ky))) in float; (s + 2) >> 2 at kx = ky = 2 unless 2 channels.
//   kArea   both scales >= 1 otherwise: per axis cv2's computeResizeAreaTab in double -- an
//           optional partial first cell, full cells of weight 1 / cellWidth, an optional partial
//           last cell, 1e-3 thresholds, cellWidth = min(scale, ssize - fsx1).  The entries of one
//           dst position are consecutive source indices, so a thread keeps (first index, count,
//           first / middle / last alpha) per axis instead of a table.  Per source row
//           buf += S * alpha in table order, then sum = beta * buf for the first row and
//           sum += beta * buf for the others, float32 and unfused; rint and saturate at the end.
//   kLinear any axis upscales: cv2's bilinear fixed-point machinery (resize.cu) with the area
//           coefficients sx = floor(dx * scale), fx = float((dx + 1) - (sx + 1) / scale),
//           fx = fx <= 0 ? 0 : fx - floor(fx).
// One thread per dst pixel; its coefficients are computed once, with IEEE double / float
// intrinsics, and reused for every frame of its chunk.  An NV12 pixel is converted to BGR with
// cv2's arithmetic (yuv_bgr.cuh) where the thread reads it.
#include <cfloat>
#include <cmath>

#include "bevk_common.cuh"
#include "resize_coef.cuh"
#include "yuv_bgr.cuh"

namespace {

enum { kFast = 0, kArea = 1, kLinear = 2 };

struct AreaParams {
    const uint8_t *src;
    uint8_t *dst;
    int src_h, src_w, dst_h, dst_w;  // NV12: the luma size
    long long pitch, src_frame, dst_frame;  // bytes from one source row / source frame / dst frame to the next
    double scale_x, scale_y;         // cv2: 1 / (dsize / ssize)
    double inv_x, inv_y;             // cv2: dsize / ssize
    int kx, ky;                      // kFast: the integer scales
    float inv_area;                  // kFast: 1.f / (kx * ky)
    int n_frames, frames_per_chunk;
};

// The entries of computeResizeAreaTab for dst position d along one axis: source indices s0 ..
// s0 + n - 1, alpha a_first for the first, a_last for the last and a_mid for the others.
struct AreaAxis {
    int s0, n;
    float a_first, a_mid, a_last;
};

__device__ __forceinline__ AreaAxis area_axis(int d, double scale, int ssize)
{
    const double f1 = __dmul_rn((double)d, scale), f2 = __dadd_rn(f1, scale);
    const double cw = fmin(scale, __dsub_rn((double)ssize, f1));
    const int s2 = min(__double2int_rd(f2), ssize - 1);
    const int s1 = min(__double2int_ru(f1), s2);
    const bool first = __dsub_rn((double)s1, f1) > 1e-3, last = __dsub_rn(f2, (double)s2) > 1e-3;
    const float mid = __double2float_rn(__ddiv_rn(1.0, cw));
    const float af = __double2float_rn(__ddiv_rn(__dsub_rn((double)s1, f1), cw));
    const float al = __double2float_rn(__ddiv_rn(fmin(fmin(__dsub_rn(f2, (double)s2), 1.0), cw), cw));
    AreaAxis a;
    a.s0 = first ? s1 - 1 : s1;
    a.n = s2 - s1 + (first ? 1 : 0) + (last ? 1 : 0);
    // with no full cell the single partial cell is both the first and the last entry
    a.a_first = first ? af : (s2 > s1 ? mid : al);
    a.a_last = last ? al : (s2 > s1 ? mid : af);
    a.a_mid = mid;
    return a;
}

__device__ __forceinline__ float area_alpha(const AreaAxis &a, int i)
{
    return i == 0 ? a.a_first : (i == a.n - 1 ? a.a_last : a.a_mid);
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

// One source row of a frame: the bytes of row y, and for NV12 the chroma row under it.
template <int C, bool NV12> struct Row {
    const uint8_t *l, *c;
    __device__ __forceinline__ Row(const uint8_t *s, const AreaParams &p, int y)
    {
        l = s + (long long)y * p.pitch;
        c = NV12 ? s + (long long)(p.src_h + (y >> 1)) * p.pitch : nullptr;
    }
    __device__ __forceinline__ void px(int x, int (&v)[C]) const
    {
        if constexpr (NV12) {
            const uint8_t *uv = c + (x & ~1);
            const uint32_t bgr = yuv_to_bgr(__ldg(l + x), __ldg(uv), __ldg(uv + 1));
            v[0] = (int)(bgr & 0xffu);
            v[1] = (int)((bgr >> 8) & 0xffu);
            v[2] = (int)(bgr >> 16);
        } else {
#pragma unroll
            for (int k = 0; k < C; ++k) v[k] = (int)__ldg(l + x * C + k);
        }
    }
};

__device__ __forceinline__ uint8_t sat_round(float v) { return (uint8_t)min(max(__float2int_rn(v), 0), 255); }

template <int C, bool NV12, int MODE>
__global__ void __launch_bounds__(256) resize_area_kernel(const __grid_constant__ AreaParams p)
{
    static_assert(!NV12 || C == 3, "NV12 frames convert to BGR");
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= p.dst_w || y >= p.dst_h) return;
    const long long od = ((long long)y * p.dst_w + x) * C;
    const int f0 = blockIdx.z * p.frames_per_chunk, f1 = min(f0 + p.frames_per_chunk, p.n_frames);

    if constexpr (MODE == kFast) {
        const int sx0 = x * p.kx, sy0 = y * p.ky;
        const bool shift = p.kx == 2 && p.ky == 2 && C != 2;  // cv2's SIMD row for 2x2 cells
        for (int f = f0; f < f1; ++f) {
            const uint8_t *s = p.src + f * p.src_frame;
            int acc[C] = {};
            for (int j = 0; j < p.ky; ++j) {
                const Row<C, NV12> r(s, p, sy0 + j);
                for (int i = 0; i < p.kx; ++i) {
                    int v[C];
                    r.px(sx0 + i, v);
#pragma unroll
                    for (int k = 0; k < C; ++k) acc[k] += v[k];
                }
            }
            uint8_t *d = p.dst + f * p.dst_frame + od;
#pragma unroll
            for (int k = 0; k < C; ++k)
                d[k] = shift ? (uint8_t)((acc[k] + 2) >> 2) : sat_round(__fmul_rn((float)acc[k], p.inv_area));
        }
    } else if constexpr (MODE == kArea) {
        const AreaAxis ax = area_axis(x, p.scale_x, p.src_w), ay = area_axis(y, p.scale_y, p.src_h);
        for (int f = f0; f < f1; ++f) {
            const uint8_t *s = p.src + f * p.src_frame;
            float sum[C] = {};
            for (int j = 0; j < ay.n; ++j) {
                const Row<C, NV12> r(s, p, ay.s0 + j);
                float buf[C] = {};
                for (int i = 0; i < ax.n; ++i) {
                    const float alpha = area_alpha(ax, i);
                    int v[C];
                    r.px(ax.s0 + i, v);
#pragma unroll
                    for (int k = 0; k < C; ++k) buf[k] = __fadd_rn(buf[k], __fmul_rn((float)v[k], alpha));
                }
                const float beta = area_alpha(ay, j);
#pragma unroll
                for (int k = 0; k < C; ++k)
                    sum[k] = j == 0 ? __fmul_rn(beta, buf[k]) : __fadd_rn(sum[k], __fmul_rn(beta, buf[k]));
            }
            uint8_t *d = p.dst + f * p.dst_frame + od;
#pragma unroll
            for (int k = 0; k < C; ++k) d[k] = sat_round(sum[k]);
        }
    } else {
        int sx, a0, a1, sy, b0, b1;
        linear_area_coef(x, p.scale_x, p.inv_x, p.src_w, true, sx, a0, a1);
        linear_area_coef(y, p.scale_y, p.inv_y, p.src_h, false, sy, b0, b1);
        const int sx1 = min(sx + 1, p.src_w - 1);
        const int r0 = min(max(sy, 0), p.src_h - 1), r1 = min(max(sy + 1, 0), p.src_h - 1);
        for (int f = f0; f < f1; ++f) {
            const uint8_t *s = p.src + f * p.src_frame;
            const Row<C, NV12> ra(s, p, r0), rb(s, p, r1);
            int v00[C], v01[C], v10[C], v11[C];
            ra.px(sx, v00);
            ra.px(sx1, v01);
            rb.px(sx, v10);
            rb.px(sx1, v11);
            uint8_t *d = p.dst + f * p.dst_frame + od;
#pragma unroll
            for (int k = 0; k < C; ++k)
                d[k] = (uint8_t)vpass(b0, b1, v00[k] * a0 + v01[k] * a1, v10[k] * a0 + v11[k] * a1);
        }
    }
}

template <int C, bool NV12> void launch(const AreaParams &p, int mode, dim3 grid, cudaStream_t st)
{
    const dim3 block(32, 8, 1);
    if (mode == kFast)
        resize_area_kernel<C, NV12, kFast><<<grid, block, 0, st>>>(p);
    else if (mode == kArea)
        resize_area_kernel<C, NV12, kArea><<<grid, block, 0, st>>>(p);
    else
        resize_area_kernel<C, NV12, kLinear><<<grid, block, 0, st>>>(p);
}

// cvRound(scale) within DBL_EPSILON of scale, as cv2's is_area_fast
bool integer_scale(double scale, int &k)
{
    k = (int)std::lround(scale);
    return std::fabs(scale - k) < DBL_EPSILON;
}

}  // namespace

int bevk_launch_resize_area(const void *src, void *dst, int n_frames, int src_h, int src_w, int channels,
                            int nv12, long long pitch, long long frame_stride, int dst_h, int dst_w,
                            cudaStream_t stream)
{
    AreaParams p;
    p.src = (const uint8_t *)src;
    p.dst = (uint8_t *)dst;
    p.src_h = src_h;
    p.src_w = src_w;
    p.dst_h = dst_h;
    p.dst_w = dst_w;
    p.pitch = pitch;
    p.src_frame = frame_stride;
    p.dst_frame = (long long)dst_h * dst_w * channels;
    p.inv_x = (double)dst_w / (double)src_w;
    p.inv_y = (double)dst_h / (double)src_h;
    p.scale_x = 1.0 / p.inv_x;
    p.scale_y = 1.0 / p.inv_y;
    int mode = kLinear;
    p.kx = p.ky = 1;
    if (p.scale_x >= 1 && p.scale_y >= 1)
        mode = integer_scale(p.scale_x, p.kx) && integer_scale(p.scale_y, p.ky) ? kFast : kArea;
    p.inv_area = 1.f / (float)(p.kx * p.ky);
    p.n_frames = n_frames;
    p.frames_per_chunk = bevk_resize_frames_per_chunk(n_frames, dst_h, dst_w);
    const int z = (n_frames + p.frames_per_chunk - 1) / p.frames_per_chunk;
    if (z > 65535) BEVK_FAIL(BEVK_E_ARG, "resize: too many frame chunks (%d) for one launch", z);
    const dim3 grid((dst_w + 31) / 32, (dst_h + 7) / 8, z);
    if (nv12) {
        launch<3, true>(p, mode, grid, stream);
    } else {
        switch (channels) {
        case 1: launch<1, false>(p, mode, grid, stream); break;
        case 2: launch<2, false>(p, mode, grid, stream); break;
        case 3: launch<3, false>(p, mode, grid, stream); break;
        default: launch<4, false>(p, mode, grid, stream); break;
        }
    }
    BEVK_CUDA(cudaGetLastError());
    return BEVK_OK;
}
