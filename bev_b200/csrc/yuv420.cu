// yuv420.cu -- BGR to YUV 4:2:0 (I420 or NV12), the layouts video encoders take: the conversion
// cv2.cvtColor(bgr, COLOR_BGR2YUV_I420) on frame batches, and the perspective warps of BGR and NV12
// frames fused with it, so that a BEV reaches the encoder's surface without a BGR copy of it
// (reference frame loop vis_homo.py:85-111, whose VideoWriter.write at :110-111 converts every BGR
// BEV on the CPU).
//
// Semantics: cv2 4.13.  BT.601 limited range in 20-bit fixed point; Y per pixel, U and V of a 2x2
// block from its top-left pixel alone.  The warps compute each BEV pixel's BGR bit-exactly as
// warp_generic.cu / nv12.cu do (cv2.warpPerspective, border colour included) and convert it in
// registers.  Sources: BGR, NV12 or I420 frames.
//
// dst layout of frame n (both layouts): h luma rows, then h / 2 rows of chroma, each row `pitch`
// bytes after the previous one, the frame at dst + n * frame_stride bytes.  NV12 chroma row r holds
// the U, V pairs of block row r.  I420 chroma follows cv2's packing with a row step: U of block row
// r at row h + r / 2, column (r % 2) * w / 2; V of block row r as U of block row r + h / 2.
#include "bevk_common.cuh"
#include "yuv_src.cuh"

namespace {

// ---- BGR -> Y, U, V (cv2's RGB2YUV420p arithmetic) ------------------------------------------------
__device__ __forceinline__ uint32_t bgr_y(uint32_t p)  // p = [B G R .]
{
    const int v = 269484 * (int)byte_of(p, 2) + 528482 * (int)byte_of(p, 1) + 102760 * (int)byte_of(p, 0) +
                  (1 << 19) + (16 << 20);
    return (uint32_t)clamp8(v >> 20);
}
// [U V 0 0] of p
__device__ __forceinline__ uint32_t bgr_uv(uint32_t p)
{
    const int r = (int)byte_of(p, 2), g = (int)byte_of(p, 1), b = (int)byte_of(p, 0);
    const int u = -155188 * r - 305135 * g + 460324 * b + (1 << 19) + (128 << 20);
    const int v = 460324 * r - 385875 * g - 74448 * b + (1 << 19) + (128 << 20);
    return (uint32_t)clamp8(u >> 20) | ((uint32_t)clamp8(v >> 20) << 8);
}

__device__ __forceinline__ void st_u16(uint8_t *d, uint32_t v)
{
    if (((uintptr_t)d & 1u) == 0) {
        __stcs(reinterpret_cast<unsigned short *>(d), (unsigned short)v);
    } else {
        d[0] = (uint8_t)v;
        d[1] = (uint8_t)(v >> 8);
    }
}

// The 2x2 block (bx, by) of a frame whose dst starts at d: luma [Y00 Y01] and [Y10 Y11] (16 bits
// each), chroma uv = [U V] of the top-left pixel.
template <bool NV12_OUT>
__device__ __forceinline__ void store_block(uint8_t *d, long long pitch, int h, int w, int bx, int by,
                                            uint32_t y0, uint32_t y1, uint32_t uv)
{
    uint8_t *l = d + (long long)(2 * by) * pitch + 2 * bx;
    st_u16(l, y0);
    st_u16(l + pitch, y1);
    if (NV12_OUT) {
        st_u16(d + (long long)(h + by) * pitch + 2 * bx, uv);
    } else {
        const int vb = by + h / 2;  // V of block row by is laid out as U of block row by + h / 2
        __stcs(d + (long long)(h + by / 2) * pitch + (by & 1) * (w / 2) + bx, (uint8_t)uv);
        __stcs(d + (long long)(h + vb / 2) * pitch + (vb & 1) * (w / 2) + bx, (uint8_t)(uv >> 8));
    }
}

// ---- conversion -------------------------------------------------------------------------------
// A thread owns a 2x2 block for kRowPairs block rows 4 apart (all loads issued before the first
// conversion); a warp covers 64 columns, i.e. 192 BGR bytes of a row, read as 48 coalesced words
// staged through shared memory when the segment is whole and 4-byte aligned, else byte by byte.
constexpr int kConvThreadsX = 64, kConvThreadsY = 4, kRowPairs = 4;

// The 6 bytes of this lane's two pixels in one BGR row segment (seg = the warp's first byte):
// p0, p1 = [B G R 0].
__device__ __forceinline__ void load_six(const uint8_t *seg, bool whole, uint32_t *stage, int lane, bool valid,
                                         uint32_t &p0, uint32_t &p1)
{
    if (whole && ((uintptr_t)seg & 3u) == 0) {  // warp-uniform
        const uint32_t *g = reinterpret_cast<const uint32_t *>(seg);
        stage[lane] = __ldcs(g + lane);
        if (lane < 16) stage[32 + lane] = __ldcs(g + 32 + lane);
        __syncwarp();
        const unsigned short *s16 = reinterpret_cast<const unsigned short *>(stage) + 3 * lane;
        const uint32_t lo = (uint32_t)s16[0] | ((uint32_t)s16[1] << 16), hi = s16[2];  // [B G R B'], [G' R']
        __syncwarp();
        p0 = lo & 0xffffffu;
        p1 = prmt(lo, hi, 0x7543u);
    } else {
        const uint8_t *s = seg + 6 * lane;
        p0 = p1 = 0;
        if (valid) {
            p0 = (uint32_t)__ldg(s) | ((uint32_t)__ldg(s + 1) << 8) | ((uint32_t)__ldg(s + 2) << 16);
            p1 = (uint32_t)__ldg(s + 3) | ((uint32_t)__ldg(s + 4) << 8) | ((uint32_t)__ldg(s + 5) << 16);
        }
    }
}

template <bool NV12_OUT>
__global__ void __launch_bounds__(kConvThreadsX *kConvThreadsY)
bgr_to_yuv420_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int n_frames, int h, int w,
                     int pitch, long long frame_stride)
{
    __shared__ uint32_t stage[kConvThreadsX * kConvThreadsY / 32][2 * kRowPairs][48];
    const int lane = threadIdx.x & 31;
    const int bx = blockIdx.x * kConvThreadsX + threadIdx.x;  // 2x2 block column
    const int bx0 = bx - lane;                                // the warp's first one
    const bool valid = 2 * bx < w, whole = 2 * (bx0 + 32) <= w;
    auto &st = stage[(threadIdx.y * kConvThreadsX + threadIdx.x) / 32];
    const int rp0 = blockIdx.y * kConvThreadsY * kRowPairs + threadIdx.y;  // first block row
    const long long src_row = 3LL * w;
    for (int f = blockIdx.z; f < n_frames; f += gridDim.z) {
        const uint8_t *s = src + (long long)f * h * src_row + 6LL * bx0;
        uint8_t *d = dst + (long long)f * frame_stride;
        uint32_t a0[kRowPairs], a1[kRowPairs], b0[kRowPairs], b1[kRowPairs];
#pragma unroll
        for (int k = 0; k < kRowPairs; ++k) {
            const int rp = min(rp0 + k * kConvThreadsY, h / 2 - 1);  // rows past the end reload the last pair
            load_six(s + (long long)(2 * rp) * src_row, whole, st[2 * k], lane, valid, a0[k], a1[k]);
            load_six(s + (long long)(2 * rp + 1) * src_row, whole, st[2 * k + 1], lane, valid, b0[k], b1[k]);
        }
#pragma unroll
        for (int k = 0; k < kRowPairs; ++k) {
            const int rp = rp0 + k * kConvThreadsY;
            if (rp >= h / 2) break;  // warp-uniform
            if (valid)
                store_block<NV12_OUT>(d, pitch, h, w, bx, rp, bgr_y(a0[k]) | (bgr_y(a1[k]) << 8),
                                      bgr_y(b0[k]) | (bgr_y(b1[k]) << 8), bgr_uv(a0[k]));
        }
    }
}

// ---- fused warps -------------------------------------------------------------------------------
// One lane per 2x2 dst block (a 32 x 8 CTA covers 64 x 16 dst pixels).  Each of its four pixels
// takes its source coordinate once per frame chunk (bevk_map_pixel) and then, for every frame of
// the chunk, its BGR value with the arithmetic of the BGR-output kernel for its source format; the
// four values are converted in registers and only Y and the top-left pixel's U, V are stored.
// A source format S provides the frame-invariant state of one pixel (S::Tap, S::make), the window
// loads of one frame (S::load, S::kWords words) and the BGR value (S::math); the YUV sources
// Nv12Src and I420Src are in yuv_src.cuh.

// BGR frames, src, row and frame 4-byte aligned: warp_u8c3_direct_kernel's aligned word gathers
template <bool LINEAR> struct BgrWords {
    static constexpr int kWords = LINEAR ? 6 : 2;
    struct Tap {
        uint32_t A;     // byte offset of the window's first byte (row 0)
        uint32_t off2;  // third (nearest: second) window word of row 0, clamped into the frame
        uint32_t w0, w1, k;  // dp2a weights of rows 0 / 1 and the border weight; nearest: k = kInside / border
    };
    static __device__ __forceinline__ Tap make(const BevkYuvParams &P, const double *M, int x, int y, uint32_t bpx)
    {
        int cs, rs, wc0, wc1, wr0, wr1;
        const bool act = clamped_window<LINEAR>(P.w, M, x, y, cs, rs, wc0, wc1, wr0, wr1);
        const uint32_t row = (uint32_t)P.pitch, last_word = (uint32_t)P.frame_stride - 4u;
        Tap t;
        t.A = (uint32_t)rs * row + 3u * (uint32_t)cs;
        t.off2 = LINEAR ? min((t.A & ~3u) + 8u, last_word - row) : min((t.A & ~3u) + 4u, last_word);
        t.w0 = tap_weight(wc0, wr0) | (tap_weight(wc1, wr0) << 16);
        t.w1 = tap_weight(wc0, wr1) | (tap_weight(wc1, wr1) << 16);
        t.k = LINEAR ? 64u * (uint32_t)(1024 - (wc0 + wc1) * (wr0 + wr1)) : (act ? kInside : bpx);
        return t;
    }
    static __device__ __forceinline__ void load(const BevkYuvParams &P, const uint8_t *s, const Tap &t,
                                                uint32_t (&w)[kWords])
    {
        auto LD = [](const uint8_t *a) { return ldg_sparse(reinterpret_cast<const uint32_t *>(a)); };
        const uint8_t *ra = s + (t.A & ~3u);
        w[0] = LD(ra);
        if (LINEAR) {
            const uint8_t *rb = ra + P.pitch;
            w[1] = LD(ra + 4);
            w[2] = LD(s + t.off2);
            w[3] = LD(rb);
            w[4] = LD(rb + 4);
            w[5] = LD(s + t.off2 + P.pitch);
        } else {
            w[1] = LD(s + t.off2);
        }
    }
    static __device__ __forceinline__ uint32_t math(const Tap &t, const uint32_t (&w)[kWords], uint32_t bpx)
    {
        const uint32_t sh = 8 * (t.A & 3u);
        if (!LINEAR) return t.k == kInside ? __funnelshift_r(w[0], w[1], sh) & 0xffffffu : t.k;
        const uint32_t f0 = __funnelshift_r(w[0], w[1], sh), f1 = __funnelshift_r(w[1], w[2], sh);
        const uint32_t g0 = __funnelshift_r(w[3], w[4], sh), g1 = __funnelshift_r(w[4], w[5], sh);
        return lerp_border(t.w0, t.w1, t.k, bpx, prmt(f0, f1, 0x4130u), prmt(f0, f1, 0x0052u), prmt(g0, g1, 0x4130u),
                           prmt(g0, g1, 0x0052u));
    }
};

// any other BGR frames: the per-tap byte arithmetic of warp_linear_kernel<uint8_t, 3> /
// warp_nearest_kernel (warp_generic.cu), which also serves 1-pixel wide or high frames
template <bool LINEAR> struct BgrBytes {
    static constexpr int kWords = LINEAR ? 4 : 1;  // [B G R 0] of taps 00, 01, 10, 11
    struct Tap {
        long long o;  // byte offset of tap 00 (it may lie outside the frame when another tap is inside)
        uint32_t in;  // bit 2j + i: tap (i, j) is inside
        uint32_t w0, w1, k;  // w00 | w01 << 16, w10 | w11 << 16 of the inside taps, the outside weight;
                             // nearest: k = kInside / border
    };
    static __device__ __forceinline__ Tap make(const BevkYuvParams &P, const double *M, int x, int y, uint32_t bpx)
    {
        const BevkWarpParams &p = P.w;
        int X, Y;
        bevk_map_pixel(M, x, y, p.bw0, LINEAR ? 32.0 : 1.0, X, Y);
        const int sx = bevk_sat16(LINEAR ? (X >> 5) : X), sy = bevk_sat16(LINEAR ? (Y >> 5) : Y);
        Tap t;
        t.in = 0;
#pragma unroll
        for (int j = 0; j < (LINEAR ? 2 : 1); ++j)
#pragma unroll
            for (int i = 0; i < (LINEAR ? 2 : 1); ++i)
                if (sx + i >= 0 && sx + i < p.src_w && sy + j >= 0 && sy + j < p.src_h) t.in |= 1u << (2 * j + i);
        t.o = t.in ? (long long)sy * P.pitch + 3LL * sx : 0;
        if (LINEAR) {
            const uint32_t ax = X & 31, ay = Y & 31;
            const uint32_t w00 = (32 - ax) * (32 - ay) * 32, w01 = ax * (32 - ay) * 32;
            const uint32_t w10 = (32 - ax) * ay * 32, w11 = ax * ay * 32;
            t.w0 = (t.in & 1 ? w00 : 0) | ((t.in & 2 ? w01 : 0) << 16);
            t.w1 = (t.in & 4 ? w10 : 0) | ((t.in & 8 ? w11 : 0) << 16);
            t.k = (t.in & 1 ? 0 : w00) + (t.in & 2 ? 0 : w01) + (t.in & 4 ? 0 : w10) + (t.in & 8 ? 0 : w11);
        } else {
            t.w0 = t.w1 = 0;
            t.k = t.in ? kInside : bpx;
        }
        return t;
    }
    static __device__ __forceinline__ uint32_t px(const uint8_t *a)
    {
        return (uint32_t)__ldg(a) | ((uint32_t)__ldg(a + 1) << 8) | ((uint32_t)__ldg(a + 2) << 16);
    }
    static __device__ __forceinline__ void load(const BevkYuvParams &P, const uint8_t *s, const Tap &t,
                                                uint32_t (&w)[kWords])
    {
        const uint8_t *a = s + t.o;
        if (LINEAR) {
            w[0] = (t.in & 1) ? px(a) : 0u;
            w[1] = (t.in & 2) ? px(a + 3) : 0u;
            w[2] = (t.in & 4) ? px(a + P.pitch) : 0u;
            w[3] = (t.in & 8) ? px(a + P.pitch + 3) : 0u;
        } else {
            w[0] = t.in ? px(a) : 0u;
        }
    }
    static __device__ __forceinline__ uint32_t math(const Tap &t, const uint32_t (&w)[kWords], uint32_t bpx)
    {
        if (!LINEAR) return t.k == kInside ? w[0] : t.k;
        uint32_t out = 0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const uint32_t acc = 16384u + byte_of(bpx, c) * t.k + (t.w0 & 0xffffu) * byte_of(w[0], c) +
                                 (t.w0 >> 16) * byte_of(w[1], c) + (t.w1 & 0xffffu) * byte_of(w[2], c) +
                                 (t.w1 >> 16) * byte_of(w[3], c);
            out |= (acc >> 15) << (8 * c);
        }
        return out;
    }
};

template <class S, bool NV12_OUT, int kBatch>
__global__ void __launch_bounds__(256) warp_yuv420_kernel(const __grid_constant__ BevkYuvParams P)
{
    const BevkWarpParams &p = P.w;
    const int bx = blockIdx.x * 32 + threadIdx.x, by = blockIdx.y * 8 + threadIdx.y;  // the lane's 2x2 block
    if (2 * bx >= p.dst_w || 2 * by >= p.dst_h) return;  // no shuffles: lanes may leave on their own
    int gi;
    const BevkWarpGroup &g = find_group(p, blockIdx.z, gi);
    const int c_local = blockIdx.z - g.chunk0;
    const int f0 = c_local * p.frames_per_chunk;
    const int f1 = min(f0 + p.frames_per_chunk, g.count);
    const uint32_t bpx = border_bgr(p.border);
    typename S::Tap t[4];  // pixels (0,0), (1,0), (0,1), (1,1) of the block
#pragma unroll
    for (int q = 0; q < 4; ++q) t[q] = S::make(P, g.M, 2 * bx + (q & 1), 2 * by + (q >> 1), bpx);
    const uint8_t *src = (const uint8_t *)p.src;
    uint8_t *dst = (uint8_t *)p.dst;

    auto load = [&](int f, uint32_t(&w)[4][S::kWords]) {
        const uint8_t *s = src + (long long)(g.first + f * g.stride) * P.frame_stride;
#pragma unroll
        for (int q = 0; q < 4; ++q) S::load(P, s, t[q], w[q]);
    };
    auto finish = [&](int f, const uint32_t(&w)[4][S::kWords]) {
        uint32_t px[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) px[q] = S::math(t[q], w[q], bpx);
        store_block<NV12_OUT>(dst + (long long)(g.first + f * g.stride) * P.dst_frame_stride, P.dst_pitch, p.dst_h,
                              p.dst_w, bx, by, bgr_y(px[0]) | (bgr_y(px[1]) << 8),
                              bgr_y(px[2]) | (bgr_y(px[3]) << 8), bgr_uv(px[0]));
    };
    // the windows of kBatch frames are requested before the first one is converted
    int f = f0;
    for (; f + kBatch <= f1; f += kBatch) {
        uint32_t w[kBatch][4][S::kWords];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) load(f + u, w[u]);
#pragma unroll
        for (int u = 0; u < kBatch; ++u) finish(f + u, w[u]);
    }
    for (; f < f1; ++f) {
        uint32_t w[4][S::kWords];
        load(f, w);
        finish(f, w);
    }
}

template <class S, int kBatch>
void launch_warp(const BevkYuvParams &P, bool nv12_out, cudaStream_t stream)
{
    dim3 block(32, 8, 1);
    dim3 grid((P.w.dst_w / 2 + 31) / 32, (P.w.dst_h / 2 + 7) / 8, P.w.total_chunks);
    if (nv12_out)
        warp_yuv420_kernel<S, true, kBatch><<<grid, block, 0, stream>>>(P);
    else
        warp_yuv420_kernel<S, false, kBatch><<<grid, block, 0, stream>>>(P);
}

// the four kernels of a YUV source format: bilinear / nearest, word / byte gathers
template <template <bool, bool> class S>
void launch_yuv_src(const BevkYuvParams &P, bool aligned, bool out, int linear, cudaStream_t stream)
{
    if (linear)
        aligned ? launch_warp<S<true, true>, 1>(P, out, stream) : launch_warp<S<true, false>, 1>(P, out, stream);
    else
        aligned ? launch_warp<S<false, true>, 2>(P, out, stream) : launch_warp<S<false, false>, 2>(P, out, stream);
}

}  // namespace

int bevk_launch_warp_yuv420(const BevkYuvParams &P, int src_format, int nv12_out, int linear, cudaStream_t stream)
{
    const bool out = nv12_out != 0;
    const bool aligned = ((uintptr_t)P.w.src % 4) == 0 && (P.pitch % 4) == 0 && (P.frame_stride % 4) == 0;
    if (src_format == BEVK_YUV_NV12) {
        launch_yuv_src<Nv12Src>(P, aligned, out, linear, stream);
    } else if (src_format == BEVK_YUV_I420) {
        launch_yuv_src<I420Src>(P, aligned, out, linear, stream);
    } else {
        // word gathers: rows of a multiple of 4 bytes (both window rows share one word alignment)
        // and a 2x2 window inside the frame
        const bool words = aligned && P.w.src_w >= 2 && P.w.src_h >= 2;
        if (linear)
            words ? launch_warp<BgrWords<true>, 1>(P, out, stream) : launch_warp<BgrBytes<true>, 1>(P, out, stream);
        else
            words ? launch_warp<BgrWords<false>, 2>(P, out, stream) : launch_warp<BgrBytes<false>, 2>(P, out, stream);
    }
    BEVK_CUDA(cudaGetLastError());
    return BEVK_OK;
}

int bevk_launch_bgr_to_yuv420(const void *src, void *dst, int n_frames, int h, int w, int nv12_out, int dst_pitch,
                              long long dst_frame_stride, cudaStream_t stream)
{
    dim3 block(kConvThreadsX, kConvThreadsY, 1);
    dim3 grid((w / 2 + kConvThreadsX - 1) / kConvThreadsX,
              (h / 2 + kConvThreadsY * kRowPairs - 1) / (kConvThreadsY * kRowPairs),
              n_frames < 65535 ? n_frames : 65535);
    if (nv12_out)
        bgr_to_yuv420_kernel<true><<<grid, block, 0, stream>>>((const uint8_t *)src, (uint8_t *)dst, n_frames, h, w,
                                                               dst_pitch, dst_frame_stride);
    else
        bgr_to_yuv420_kernel<false><<<grid, block, 0, stream>>>((const uint8_t *)src, (uint8_t *)dst, n_frames, h, w,
                                                                dst_pitch, dst_frame_stride);
    BEVK_CUDA(cudaGetLastError());
    return BEVK_OK;
}
