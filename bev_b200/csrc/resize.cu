// resize.cu -- batched cv2.resize (uint8, INTER_LINEAR) for sm_100a: the small-frame path of the
// reference's frame loop, `img_small = cv2.resize(img, (new_u, new_v))` (vis_homo.py:90), whose
// result feeds the second warp at vis_homo.py:91 through the homography of
// Calib.scale(align_corners=False) (bev/calib.py:142-198).
//
// Semantics: OpenCV 4.13's 8-bit bilinear resize, bit for bit (oracle/resize_oracle.py restates it
// and is pinned against cv2):
//   column dx: fx = float((dx + 0.5) * scale_x - 0.5), sx = floor(fx), fx -= sx; left of the image
//   (sx, fx) = (0, 0), at / right of the last pixel (src_w - 1, 0); weights rint((1 - fx) * 2048),
//   rint(fx * 2048) in float.  Row dy: the same without that clamp, the two row indices clipped
//   into the image instead.  S = p[sx] * a0 + p[sx + 1] * a1 per row, then
//   (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2.
//   2-channel frames downscaled by exactly 2 in both axes take the round-half-even mean of each
//   2x2 block instead (cv2's INTER_AREA special case).
// The coefficients are recomputed per thread from (dx, dy) with unfused IEEE float / double
// operations (the library is built with -fmad=false) -- no tables to upload, nothing to keep alive
// across the asynchronous launch -- and amortised over the frames of the thread's chunk.
//
// HBM-bound: every source row a dst row references is read once (sector-wise), the small frame
// written once.  Two kernels: a word-gather one for BGR frames (3 aligned words per window row,
// dp2a for the horizontal pass, 32 pixels packed into one 96-byte store per warp) and a byte-wise
// one for every other channel count / width.
#include "bevk_common.cuh"
#include "resize_coef.cuh"
#include "warp_u8c3.cuh"

namespace {

// word load with a 256-byte L2 prefetch hint: the resize reads (nearly) every byte of the rows it
// touches, so the neighbouring lines are wanted anyway (3 % faster than the plain read-only load)
__device__ __forceinline__ uint32_t ldg_dense(const uint32_t *p)
{
    uint32_t v;
    asm("ld.global.nc.L2::256B.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

struct ResizeParams {
    const uint8_t *src;
    uint8_t *dst;
    int src_h, src_w, dst_h, dst_w;
    long long src_frame, dst_frame;  // bytes per frame
    double scale_x, scale_y;
    int n_frames, frames_per_chunk;
};

// ---- any channel count: one thread per dst pixel, byte loads -----------------------------------
template <int C>
__global__ void __launch_bounds__(256) resize_bytes_kernel(const __grid_constant__ ResizeParams p)
{
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= p.dst_w || y >= p.dst_h) return;
    int sx, a0, a1, sy, b0, b1;
    axis_coef(x, p.scale_x, p.src_w, true, sx, a0, a1);
    axis_coef(y, p.scale_y, p.src_h, false, sy, b0, b1);
    const int sx1 = min(sx + 1, p.src_w - 1);
    const int r0 = min(max(sy, 0), p.src_h - 1), r1 = min(max(sy + 1, 0), p.src_h - 1);
    const long long o00 = ((long long)r0 * p.src_w + sx) * C, o01 = ((long long)r0 * p.src_w + sx1) * C;
    const long long o10 = ((long long)r1 * p.src_w + sx) * C, o11 = ((long long)r1 * p.src_w + sx1) * C;
    const long long od = ((long long)y * p.dst_w + x) * C;
    const int f0 = blockIdx.z * p.frames_per_chunk, f1 = min(f0 + p.frames_per_chunk, p.n_frames);
    if constexpr (C == 2) {
        // cv2 sends an exact 2x downscale to INTER_AREA, which for 2 channels rounds the mean of
        // the 2x2 block half to even (for 1, 3, 4 channels it equals the bilinear result).  The
        // window above is then exactly that block.
        if (p.src_w == 2 * p.dst_w && p.src_h == 2 * p.dst_h) {
            for (int f = f0; f < f1; ++f) {
                const uint8_t *s = p.src + f * p.src_frame;
                uint8_t *d = p.dst + f * p.dst_frame + od;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const int sum = (int)__ldg(s + o00 + c) + (int)__ldg(s + o01 + c) +
                                    (int)__ldg(s + o10 + c) + (int)__ldg(s + o11 + c);
                    const int q = sum >> 2;
                    d[c] = (uint8_t)(q + ((sum & 3) + (q & 1) > 2));
                }
            }
            return;
        }
    }
    for (int f = f0; f < f1; ++f) {
        const uint8_t *s = p.src + f * p.src_frame;
        uint8_t *d = p.dst + f * p.dst_frame + od;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int s0 = (int)__ldg(s + o00 + c) * a0 + (int)__ldg(s + o01 + c) * a1;
            const int s1 = (int)__ldg(s + o10 + c) * a0 + (int)__ldg(s + o11 + c) * a1;
            d[c] = (uint8_t)vpass(b0, b1, s0, s1);
        }
    }
}

// ---- BGR frames: word gathers + packed stores ---------------------------------------------------
// Needs src_w % 4 == 0 (both window rows share one word alignment), dst_w % 4 == 0 (whole words
// per 4 pixels) and src_w >= 2.
__global__ void __launch_bounds__(256) resize_u8c3_kernel(const __grid_constant__ ResizeParams p)
{
    const int lane = threadIdx.x, x0 = blockIdx.x * 32;
    const int x = min(x0 + lane, p.dst_w - 1), y = blockIdx.y * 8 + threadIdx.y;
    if (y >= p.dst_h) return;  // a warp is one dst row segment: uniform exit, shuffles stay legal
    int sx, a0, a1, sy, b0, b1;
    axis_coef(x, p.scale_x, p.src_w, true, sx, a0, a1);
    axis_coef(y, p.scale_y, p.src_h, false, sy, b0, b1);
    // 2-pixel window starting inside the image: the last column moves one left and swaps weights
    const int cs = min(sx, p.src_w - 2);
    const int wa = cs == sx ? a0 : a1, wb = cs == sx ? a1 : a0;  // sx == src_w - 1 has a1 == 0
    const int r0 = min(max(sy, 0), p.src_h - 1), r1 = min(max(sy + 1, 0), p.src_h - 1);
    const uint32_t row_bytes = (uint32_t)p.src_w * 3u;
    const uint32_t A = 3u * (uint32_t)cs;          // window start inside a row
    const uint32_t addr = A & ~3u, sh = 8 * (A & 3);
    const uint32_t off2 = min(addr + 8u, row_bytes - 4u);  // third word, only some alignments use it
    const uint32_t w16 = (uint32_t)wa | ((uint32_t)wb << 16);
    const long long ra = (long long)r0 * row_bytes, rb = (long long)r1 * row_bytes;

    const int j = lane >> 2, r4 = lane & 3;
    const uint32_t sel_pack = r4 == 0 ? 0x4210u : (r4 == 1 ? 0x5421u : 0x6542u);
    const bool st_ok = r4 < 3 && 4 * j < min(32, p.dst_w - x0);
    uint8_t *dst = p.dst + ((long long)y * p.dst_w + x0) * 3 + (3 * j + r4) * 4;
    const int f0 = blockIdx.z * p.frames_per_chunk, f1 = min(f0 + p.frames_per_chunk, p.n_frames);
#pragma unroll 4
    for (int f = f0; f < f1; ++f) {
        const uint8_t *s = p.src + f * p.src_frame;
        const uint8_t *pa = s + ra, *pb = s + rb;
        const uint32_t u0 = ldg_dense((const uint32_t *)(pa + addr)), u1 = ldg_dense((const uint32_t *)(pa + addr + 4));
        const uint32_t u2 = ldg_dense((const uint32_t *)(pa + off2));
        const uint32_t v0 = ldg_dense((const uint32_t *)(pb + addr)), v1 = ldg_dense((const uint32_t *)(pb + addr + 4));
        const uint32_t v2 = ldg_dense((const uint32_t *)(pb + off2));
        // byte-aligned windows: f = [B0 B1 B2 B3], g = [B4 B5 . .] of each row
        const uint32_t fa = __funnelshift_r(u0, u1, sh), ga = __funnelshift_r(u1, u2, sh);
        const uint32_t fb = __funnelshift_r(v0, v1, sh), gb = __funnelshift_r(v1, v2, sh);
        // channel c pairs bytes (c, c + 3): [B0 B3 . .], [B1 B4 . .], [B2 B5 . .]
        const int s00 = __dp2a_lo(w16, prmt(fa, ga, 0x0030u), 0u), s01 = __dp2a_lo(w16, prmt(fa, ga, 0x0041u), 0u);
        const int s02 = __dp2a_lo(w16, prmt(fa, ga, 0x0052u), 0u);
        const int s10 = __dp2a_lo(w16, prmt(fb, gb, 0x0030u), 0u), s11 = __dp2a_lo(w16, prmt(fb, gb, 0x0041u), 0u);
        const int s12 = __dp2a_lo(w16, prmt(fb, gb, 0x0052u), 0u);
        const uint32_t P = vpass(b0, b1, s00, s10) | (vpass(b0, b1, s01, s11) << 8) | (vpass(b0, b1, s02, s12) << 16);
        const uint32_t word = prmt(P, __shfl_down_sync(0xffffffffu, P, 1), sel_pack);
        if (st_ok) st_stream_free(reinterpret_cast<uint32_t *>(dst + f * p.dst_frame), word);
    }
}

template <int C> void launch_bytes(const ResizeParams &p, dim3 grid, cudaStream_t st)
{
    resize_bytes_kernel<C><<<grid, dim3(32, 8, 1), 0, st>>>(p);
}

}  // namespace

int bevk_launch_resize(const void *src, void *dst, int n_frames, int src_h, int src_w, int channels, int dst_h,
                       int dst_w, cudaStream_t stream)
{
    BevkResizePlan plan;
    int rc = bevk_plan_resize(n_frames, src_h, src_w, dst_h, dst_w, plan);
    if (rc) return rc;
    ResizeParams p;
    p.src = (const uint8_t *)src;
    p.dst = (uint8_t *)dst;
    p.src_h = src_h;
    p.src_w = src_w;
    p.dst_h = dst_h;
    p.dst_w = dst_w;
    p.src_frame = (long long)src_h * src_w * channels;
    p.dst_frame = (long long)dst_h * dst_w * channels;
    p.scale_x = plan.scale_x;
    p.scale_y = plan.scale_y;
    p.n_frames = n_frames;
    p.frames_per_chunk = plan.frames_per_chunk;
    const bool words = channels == 3 && src_w >= 2 && (src_w % 4) == 0 && (dst_w % 4) == 0 &&
                       ((uintptr_t)src % 4) == 0 && ((uintptr_t)dst % 4) == 0;
    if (words) {
        resize_u8c3_kernel<<<plan.grid, dim3(32, 8, 1), 0, stream>>>(p);
    } else {
        switch (channels) {
        case 1: launch_bytes<1>(p, plan.grid, stream); break;
        case 2: launch_bytes<2>(p, plan.grid, stream); break;
        case 3: launch_bytes<3>(p, plan.grid, stream); break;
        default: launch_bytes<4>(p, plan.grid, stream); break;
        }
    }
    BEVK_CUDA(cudaGetLastError());
    return BEVK_OK;
}
