// nv12.cu -- NV12 video frames (what a GPU video decoder hands out) to BGR: the conversion
// cv2.cvtColor(f, COLOR_YUV2BGR_NV12) on frame batches, and the perspective warp of NV12 frames
// fused with it, so that decoded frames reach the BEV without a BGR copy of every frame.
//
// Semantics: cv2 4.13.  The conversion is BT.601 limited range in 20-bit fixed point with chroma
// replicated over each 2x2 luma block; the warp equals cv2.warpPerspective of the converted frame
// (reference frame loop vis_homo.py:85-91), i.e. every bilinear tap is converted on its own and
// the four are then interpolated with the uint8 x 3 arithmetic of warp_u8c3.cuh.  A tap outside
// the frame takes the BGR border colour; it is never converted from YUV.
//
// The resize equals cv2.resize of the converted frame with INTER_LINEAR (the small frame of
// vis_homo.py:90): the four taps of a dst pixel are converted on their own and then interpolated
// with the arithmetic of resize.cu.
//
// Layout of frame n: luma rows 0..H-1 then chroma rows 0..H/2-1 (interleaved U, V bytes), each
// row `pitch` bytes after the previous one, the frame at src + n * frame_stride bytes.
#include "bevk_common.cuh"
#include "resize_coef.cuh"
#include "warp_u8c3.cuh"
#include "yuv_bgr.cuh"

namespace {

__device__ __forceinline__ uint32_t byte_of(uint32_t w, int i) { return (w >> (8 * i)) & 0xffu; }

__device__ __forceinline__ uint32_t border_bgr(const float *b)
{
    uint32_t px = 0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        // cv2: saturate_cast<uchar>(borderValue[c])
        const int v = __float2int_rn(b[c]);
        px |= (uint32_t)(v < 0 ? 0 : (v > 255 ? 255 : v)) << (8 * c);
    }
    return px;
}

__device__ __forceinline__ const BevkWarpGroup &find_group(const BevkWarpParams &p, int z)
{
    int gi = 0;
#pragma unroll 1
    for (int i = 1; i < p.n_groups; ++i)
        if (z >= p.g[i].chunk0) gi = i;
    return p.g[gi];
}

// ---- fused warp -------------------------------------------------------------------------------
// One lane per dst pixel, as warp_u8c3_direct_kernel (warp_generic.cu): the coordinate is computed
// once per frame chunk with bevk_map_pixel, then every frame of the chunk gathers the window's two
// luma rows (2 bytes each) and the one or two chroma rows under them (4 bytes each: the U,V pairs
// of the window's one or two chroma columns).  WORDS (pitch, frame stride and src 4-byte aligned):
// aligned 32-bit words + funnel shifts, the second word of a row only when the window straddles
// it; otherwise byte loads.  PACKED (dst_w % 4 == 0): the warp packs 32 pixels into one coalesced
// 96-byte store, otherwise every lane stores its 3 bytes.
template <bool LINEAR, bool WORDS, bool PACKED, int kBatch>
__global__ void __launch_bounds__(256) warp_nv12_kernel(const __grid_constant__ BevkNv12Params P)
{
    const BevkWarpParams &p = P.w;
    const int lane = threadIdx.x, x0 = blockIdx.x * 32;
    const int x = x0 + lane, y = blockIdx.y * 8 + threadIdx.y;
    if (y >= p.dst_h) return;  // a warp is one dst row segment: uniform exit, shuffles stay legal
    const BevkWarpGroup &g = find_group(p, blockIdx.z);
    const int c_local = blockIdx.z - g.chunk0;
    const int f0 = c_local * p.frames_per_chunk;
    const int f1 = min(f0 + p.frames_per_chunk, g.count);

    int X, Y;
    bevk_map_pixel(g.M, min(x, p.dst_w - 1), y, p.bw0, LINEAR ? 32.0 : 1.0, X, Y);
    int cs, rs, wc0, wc1, wr0, wr1;
    if (LINEAR) {
        window(bevk_sat16(X >> 5), X & 31, p.src_w, cs, wc0, wc1);
        window(bevk_sat16(Y >> 5), Y & 31, p.src_h, rs, wr0, wr1);
    } else {
        const int sx = bevk_sat16(X), sy = bevk_sat16(Y);
        const bool in = sx >= 0 && sx < p.src_w && sy >= 0 && sy < p.src_h;
        cs = min(max(sx, 0), p.src_w - 1);
        rs = min(max(sy, 0), p.src_h - 1);
        wc0 = wr0 = in ? 1 : 0;
        wc1 = wr1 = 0;
    }
    const bool act = (wc0 | wc1) != 0 && (wr0 | wr1) != 0;
    if (!act) cs = rs = 0;  // the loads of an all-border pixel hit one cached line
    const uint32_t pitch = (uint32_t)P.pitch;
    // byte offsets inside a frame: luma row rs at column cs; chroma row rs/2 at the U of column cs
    const uint32_t lo = (uint32_t)rs * pitch + (uint32_t)cs;
    const uint32_t co = ((uint32_t)p.src_h + (uint32_t)(rs >> 1)) * pitch + 2u * (uint32_t)(cs >> 1);
    // the window's lower luma row uses the next chroma row when rs is odd; its right column the
    // next chroma column when cs is odd (else both columns share one U,V pair: duplicate it)
    const uint32_t co_b = co + ((rs & 1) ? pitch : 0u);
    const uint32_t csel = (cs & 1) ? 0x3210u : 0x1010u;
    // WORDS: the second word of a row is needed when the 2 luma / 4 chroma bytes straddle it
    const bool l_two = LINEAR && (lo & 3u) == 3u;
    const bool c_two = LINEAR && (co & 3u) == 2u && (cs & 1);

    uint32_t w0 = 0, w1 = 0, kB = 32768u, kG = 32768u, kR = 32768u, bpx = 0;
    if (LINEAR) {
        w0 = tap_weight(wc0, wr0) | (tap_weight(wc1, wr0) << 16);
        w1 = tap_weight(wc0, wr1) | (tap_weight(wc1, wr1) << 16);
        // taps outside the frame: border colour x their weight, folded into the rounding constant
        const uint32_t wout = 64u * (uint32_t)(1024 - (wc0 + wc1) * (wr0 + wr1));
        const uint32_t b = border_bgr(p.border);
        kB += byte_of(b, 0) * wout;
        kG += byte_of(b, 1) * wout;
        kR += byte_of(b, 2) * wout;
    } else {
        bpx = act ? 0xffffffffu : border_bgr(p.border);  // nearest: all-ones marks "convert the tap"
    }

    const int j = lane >> 2, r4 = lane & 3;
    const uint32_t sel_pack = r4 == 0 ? 0x4210u : (r4 == 1 ? 0x5421u : 0x6542u);
    const bool st_ok = PACKED ? (r4 < 3 && 4 * j < min(32, p.dst_w - x0)) : x < p.dst_w;
    uint8_t *dst = (uint8_t *)p.dst + ((long long)y * p.dst_w + x0) * 3 + (PACKED ? (3 * j + r4) * 4 : 3 * lane);
    const uint8_t *src = (const uint8_t *)p.src;

    constexpr int kWords = LINEAR ? (WORDS ? 8 : 4) : 2;
    auto LD = [](const uint8_t *a) { return ldg_sparse(reinterpret_cast<const uint32_t *>(a)); };
    auto B = [](const uint8_t *a) { return (uint32_t)__ldg(a); };
    auto load = [&](int f, uint32_t(&w)[kWords]) {
        const uint8_t *s = src + (long long)(g.first + f * g.stride) * P.frame_stride;
        if (LINEAR && WORDS) {
            const uint8_t *la = s + (lo & ~3u), *ca = s + (co & ~3u), *cb = s + (co_b & ~3u);
            w[0] = LD(la);
            w[1] = l_two ? LD(la + 4) : 0u;
            w[2] = LD(la + pitch);
            w[3] = l_two ? LD(la + pitch + 4) : 0u;
            w[4] = LD(ca);
            w[5] = c_two ? LD(ca + 4) : 0u;
            w[6] = LD(cb);
            w[7] = c_two ? LD(cb + 4) : 0u;
        } else if (LINEAR) {
            const uint8_t *la = s + lo, *ca = s + co, *cb = s + co_b;
            const uint32_t cn = (cs & 1) ? 2u : 0u;  // offset of the right column's U,V pair
            w[0] = B(la) | (B(la + 1) << 8);
            w[1] = B(la + pitch) | (B(la + pitch + 1) << 8);
            w[2] = B(ca) | (B(ca + 1) << 8) | (B(ca + cn) << 16) | (B(ca + cn + 1) << 24);
            w[3] = B(cb) | (B(cb + 1) << 8) | (B(cb + cn) << 16) | (B(cb + cn + 1) << 24);
        } else if (WORDS) {
            w[0] = LD(s + (lo & ~3u));
            w[1] = LD(s + (co & ~3u));
        } else {
            w[0] = B(s + lo);
            w[1] = B(s + co) | (B(s + co + 1) << 8);
        }
    };
    auto finish = [&](int f, const uint32_t(&w)[kWords]) {
        uint32_t P0;
        if (LINEAR) {
            uint32_t L0, L1, C0, C1;  // [Y Y' . .] of window rows 0 / 1, [U V U' V'] under them
            if (WORDS) {
                L0 = __funnelshift_r(w[0], w[1], 8 * (lo & 3u));
                L1 = __funnelshift_r(w[2], w[3], 8 * (lo & 3u));
                C0 = prmt(__funnelshift_r(w[4], w[5], 8 * (co & 3u)), 0u, csel);
                C1 = prmt(__funnelshift_r(w[6], w[7], 8 * (co_b & 3u)), 0u, csel);
            } else {
                L0 = w[0];
                L1 = w[1];
                C0 = w[2];
                C1 = w[3];
            }
            const uint32_t p00 = yuv_to_bgr(byte_of(L0, 0), byte_of(C0, 0), byte_of(C0, 1));
            const uint32_t p01 = yuv_to_bgr(byte_of(L0, 1), byte_of(C0, 2), byte_of(C0, 3));
            const uint32_t p10 = yuv_to_bgr(byte_of(L1, 0), byte_of(C1, 0), byte_of(C1, 1));
            const uint32_t p11 = yuv_to_bgr(byte_of(L1, 1), byte_of(C1, 2), byte_of(C1, 3));
            // the dp2a operands of lerp_xy: [B0 B0' G0 G0'] and [R0 R0' . .] per window row
            const uint32_t xa = prmt(p00, p01, 0x5140u), ya = prmt(p00, p01, 0x0062u);
            const uint32_t xb = prmt(p10, p11, 0x5140u), yb = prmt(p10, p11, 0x0062u);
            const uint32_t t0 = __dp2a_lo(w1, xb, __dp2a_lo(w0, xa, kB));
            const uint32_t t1 = __dp2a_hi(w1, xb, __dp2a_hi(w0, xa, kG));
            const uint32_t t2 = __dp2a_lo(w1, yb, __dp2a_lo(w0, ya, kR));
            P0 = prmt(prmt(t0, t1, 0x4462u), t2, 0x7610u);
        } else {
            const uint32_t Yw = WORDS ? byte_of(w[0], lo & 3u) : w[0];
            const uint32_t Cw = WORDS ? (w[1] >> (8 * (co & 2u))) : w[1];
            P0 = bpx == 0xffffffffu ? yuv_to_bgr(Yw, byte_of(Cw, 0), byte_of(Cw, 1)) : bpx;
        }
        uint8_t *d = dst + (long long)(g.first + f * g.stride) * p.dst_frame_elems;
        if (PACKED) {
            const uint32_t word = prmt(P0, __shfl_down_sync(0xffffffffu, P0, 1), sel_pack);
            if (st_ok) st_stream_free(reinterpret_cast<uint32_t *>(d), word);
        } else if (st_ok) {
            d[0] = (uint8_t)P0;
            d[1] = (uint8_t)(P0 >> 8);
            d[2] = (uint8_t)(P0 >> 16);
        }
    };
    // the windows of kBatch frames are requested before the first one is converted
    int f = f0;
    for (; f + kBatch <= f1; f += kBatch) {
        uint32_t w[kBatch][kWords];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) load(f + u, w[u]);
#pragma unroll
        for (int u = 0; u < kBatch; ++u) finish(f + u, w[u]);
    }
    for (; f < f1; ++f) {
        uint32_t w[kWords];
        load(f, w);
        finish(f, w);
    }
}

template <bool LINEAR, bool WORDS>
void launch_warp(const BevkNv12Params &P, bool packed, cudaStream_t stream)
{
    constexpr int kBatch = LINEAR ? 2 : 4;
    dim3 block(32, 8, 1);
    dim3 grid((P.w.dst_w + 31) / 32, (P.w.dst_h + 7) / 8, P.w.total_chunks);
    if (packed)
        warp_nv12_kernel<LINEAR, WORDS, true, kBatch><<<grid, block, 0, stream>>>(P);
    else
        warp_nv12_kernel<LINEAR, WORDS, false, kBatch><<<grid, block, 0, stream>>>(P);
}

// ---- resize -----------------------------------------------------------------------------------
struct ResizeNv12Params {
    const uint8_t *src;
    uint8_t *dst;
    int src_h, src_w, dst_h, dst_w;  // luma size of a source frame; dst size
    uint32_t pitch;                  // bytes from one luma or chroma row to the next
    long long frame_stride, dst_frame;  // bytes from one source / dst frame to the next
    double scale_x, scale_y;
    int n_frames, frames_per_chunk;
};

// One lane per dst pixel, as resize_u8c3_kernel (resize.cu): the coefficients are computed once
// per frame chunk with axis_coef, and the 2-pixel window starts inside the frame (cs = min(sx,
// src_w - 2), weights swapped when it moved).  Every frame gathers two luma rows r0, r1 (2 bytes
// at cs each; one row twice at the top and bottom edges) and the chroma rows r0 / 2, r1 / 2 under
// them (4 bytes each: the U,V pairs of columns cs and cs + 1, one pair twice when cs is even),
// converts the 4 taps on their own, then runs cv2's horizontal pass per channel as one dp2a on
// the weight pair and its vertical pass.  WORDS and PACKED as in warp_nv12_kernel.
// The gather is that kernel's with the second luma row at r1 instead of the next row.  It is kept
// separate: moving it into a helper both kernels call changed the register allocation and SASS
// of warp_nv12_kernel's bilinear variants.
template <bool WORDS, bool PACKED, int kBatch>
__global__ void __launch_bounds__(256) resize_nv12_kernel(const __grid_constant__ ResizeNv12Params p)
{
    const int lane = threadIdx.x, x0 = blockIdx.x * 32;
    const int x = x0 + lane, y = blockIdx.y * 8 + threadIdx.y;
    if (y >= p.dst_h) return;  // a warp is one dst row segment: uniform exit, shuffles stay legal
    int sx, a0, a1, sy, b0, b1;
    axis_coef(min(x, p.dst_w - 1), p.scale_x, p.src_w, true, sx, a0, a1);
    axis_coef(y, p.scale_y, p.src_h, false, sy, b0, b1);
    const int cs = min(sx, p.src_w - 2);
    const int wa = cs == sx ? a0 : a1, wb = cs == sx ? a1 : a0;  // sx == src_w - 1 has a1 == 0
    const uint32_t w16 = (uint32_t)wa | ((uint32_t)wb << 16);
    const int r0 = min(max(sy, 0), p.src_h - 1), r1 = min(max(sy + 1, 0), p.src_h - 1);
    const uint32_t pitch = p.pitch;
    // byte offsets inside a frame: luma row r0 at column cs, and from it to row r1 (0 or pitch);
    // chroma rows r0 / 2 and r1 / 2 at the U of column cs
    const uint32_t lo = (uint32_t)r0 * pitch + (uint32_t)cs;
    const uint32_t l1 = (uint32_t)(r1 - r0) * pitch;
    const uint32_t cx = 2u * (uint32_t)(cs >> 1);
    const uint32_t co = ((uint32_t)p.src_h + (uint32_t)(r0 >> 1)) * pitch + cx;
    const uint32_t co_b = ((uint32_t)p.src_h + (uint32_t)(r1 >> 1)) * pitch + cx;
    // the right column uses the next chroma column when cs is odd (else duplicate the one pair)
    const uint32_t csel = (cs & 1) ? 0x3210u : 0x1010u;
    // WORDS: the second word of a row is needed when the 2 luma / 4 chroma bytes straddle it
    const bool l_two = (lo & 3u) == 3u;
    const bool c_two = (co & 3u) == 2u && (cs & 1);

    const int j = lane >> 2, r4 = lane & 3;
    const uint32_t sel_pack = r4 == 0 ? 0x4210u : (r4 == 1 ? 0x5421u : 0x6542u);
    const bool st_ok = PACKED ? (r4 < 3 && 4 * j < min(32, p.dst_w - x0)) : x < p.dst_w;
    uint8_t *dst = p.dst + ((long long)y * p.dst_w + x0) * 3 + (PACKED ? (3 * j + r4) * 4 : 3 * lane);

    constexpr int kWords = WORDS ? 8 : 4;
    auto LD = [](const uint8_t *a) { return ldg_sparse(reinterpret_cast<const uint32_t *>(a)); };
    auto B = [](const uint8_t *a) { return (uint32_t)__ldg(a); };
    auto load = [&](int f, uint32_t(&w)[kWords]) {
        const uint8_t *s = p.src + (long long)f * p.frame_stride;
        if (WORDS) {
            const uint8_t *la = s + (lo & ~3u), *ca = s + (co & ~3u), *cb = s + (co_b & ~3u);
            w[0] = LD(la);
            w[1] = l_two ? LD(la + 4) : 0u;
            w[2] = LD(la + l1);
            w[3] = l_two ? LD(la + l1 + 4) : 0u;
            w[4] = LD(ca);
            w[5] = c_two ? LD(ca + 4) : 0u;
            w[6] = LD(cb);
            w[7] = c_two ? LD(cb + 4) : 0u;
        } else {
            const uint8_t *la = s + lo, *ca = s + co, *cb = s + co_b;
            const uint32_t cn = (cs & 1) ? 2u : 0u;  // offset of the right column's U,V pair
            w[0] = B(la) | (B(la + 1) << 8);
            w[1] = B(la + l1) | (B(la + l1 + 1) << 8);
            w[2] = B(ca) | (B(ca + 1) << 8) | (B(ca + cn) << 16) | (B(ca + cn + 1) << 24);
            w[3] = B(cb) | (B(cb + 1) << 8) | (B(cb + cn) << 16) | (B(cb + cn + 1) << 24);
        }
    };
    auto finish = [&](int f, const uint32_t(&w)[kWords]) {
        uint32_t L0, L1, C0, C1;  // [Y Y' . .] of window rows 0 / 1, [U V U' V'] under them
        if (WORDS) {
            L0 = __funnelshift_r(w[0], w[1], 8 * (lo & 3u));
            L1 = __funnelshift_r(w[2], w[3], 8 * (lo & 3u));
            C0 = prmt(__funnelshift_r(w[4], w[5], 8 * (co & 3u)), 0u, csel);
            C1 = prmt(__funnelshift_r(w[6], w[7], 8 * (co_b & 3u)), 0u, csel);
        } else {
            L0 = w[0];
            L1 = w[1];
            C0 = w[2];
            C1 = w[3];
        }
        const uint32_t p00 = yuv_to_bgr(byte_of(L0, 0), byte_of(C0, 0), byte_of(C0, 1));
        const uint32_t p01 = yuv_to_bgr(byte_of(L0, 1), byte_of(C0, 2), byte_of(C0, 3));
        const uint32_t p10 = yuv_to_bgr(byte_of(L1, 0), byte_of(C1, 0), byte_of(C1, 1));
        const uint32_t p11 = yuv_to_bgr(byte_of(L1, 1), byte_of(C1, 2), byte_of(C1, 3));
        // per window row [B B' G G'] and [R R' . .]: channel c of the horizontal pass is
        // p[cs][c] * wa + p[cs + 1][c] * wb, one dp2a on the low or high byte pair
        const uint32_t xa = prmt(p00, p01, 0x5140u), ya = prmt(p00, p01, 0x0062u);
        const uint32_t xb = prmt(p10, p11, 0x5140u), yb = prmt(p10, p11, 0x0062u);
        const int s00 = __dp2a_lo(w16, xa, 0u), s01 = __dp2a_hi(w16, xa, 0u), s02 = __dp2a_lo(w16, ya, 0u);
        const int s10 = __dp2a_lo(w16, xb, 0u), s11 = __dp2a_hi(w16, xb, 0u), s12 = __dp2a_lo(w16, yb, 0u);
        const uint32_t P0 = vpass(b0, b1, s00, s10) | (vpass(b0, b1, s01, s11) << 8) | (vpass(b0, b1, s02, s12) << 16);
        uint8_t *d = dst + (long long)f * p.dst_frame;
        if (PACKED) {
            const uint32_t word = prmt(P0, __shfl_down_sync(0xffffffffu, P0, 1), sel_pack);
            if (st_ok) st_stream_free(reinterpret_cast<uint32_t *>(d), word);
        } else if (st_ok) {
            d[0] = (uint8_t)P0;
            d[1] = (uint8_t)(P0 >> 8);
            d[2] = (uint8_t)(P0 >> 16);
        }
    };
    // the windows of kBatch frames are requested before the first one is converted
    const int f0 = blockIdx.z * p.frames_per_chunk, f1 = min(f0 + p.frames_per_chunk, p.n_frames);
    int f = f0;
    for (; f + kBatch <= f1; f += kBatch) {
        uint32_t w[kBatch][kWords];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) load(f + u, w[u]);
#pragma unroll
        for (int u = 0; u < kBatch; ++u) finish(f + u, w[u]);
    }
    for (; f < f1; ++f) {
        uint32_t w[kWords];
        load(f, w);
        finish(f, w);
    }
}

template <bool WORDS>
void launch_resize(const ResizeNv12Params &p, bool packed, dim3 grid, cudaStream_t stream)
{
    constexpr int kBatch = 2;
    if (packed)
        resize_nv12_kernel<WORDS, true, kBatch><<<grid, dim3(32, 8, 1), 0, stream>>>(p);
    else
        resize_nv12_kernel<WORDS, false, kBatch><<<grid, dim3(32, 8, 1), 0, stream>>>(p);
}

// ---- conversion -------------------------------------------------------------------------------
// A thread owns a 2x2 luma block and its one U,V pair, for kRowPairs block rows 4 apart (all
// loads issued before the first conversion); a warp covers 64 columns, i.e. 64 luma bytes per
// row read and 192 BGR bytes per row written, as 48 coalesced words staged through shared memory
// (measured on one B200 at 1000 W: 256 x 1080p in 0.90 ms when every lane stored its own 6 bytes).
constexpr int kConvThreadsX = 64, kConvThreadsY = 4, kRowPairs = 4;

__device__ __forceinline__ uint32_t ld_pair(const uint8_t *a)
{
    if (((uintptr_t)a & 1u) == 0) return __ldg(reinterpret_cast<const uint16_t *>(a));
    return (uint32_t)__ldg(a) | ((uint32_t)__ldg(a + 1) << 8);
}

__device__ __forceinline__ void st_six(uint8_t *d, uint32_t p0, uint32_t p1)
{
    // p0, p1 = [B G R 0] of two neighbouring pixels -> 6 bytes at d
    const uint32_t lo = prmt(p0, p1, 0x4210u), hi = prmt(p1, 0u, 0x4421u) & 0xffffu;  // [B G R B'], [G' R']
    const uintptr_t a = (uintptr_t)d;
    if ((a & 3u) == 0) {
        __stcs(reinterpret_cast<uint32_t *>(d), lo);
        __stcs(reinterpret_cast<unsigned short *>(d + 4), (unsigned short)hi);
    } else if ((a & 1u) == 0) {
        __stcs(reinterpret_cast<unsigned short *>(d), (unsigned short)(lo & 0xffffu));
        __stcs(reinterpret_cast<uint32_t *>(d + 2), (lo >> 16) | (hi << 16));
    } else {
        d[0] = (uint8_t)lo;
        d[1] = (uint8_t)(lo >> 8);
        d[2] = (uint8_t)(lo >> 16);
        d[3] = (uint8_t)(lo >> 24);
        d[4] = (uint8_t)hi;
        d[5] = (uint8_t)(hi >> 8);
    }
}

// One output row of a warp: a whole 192-byte segment at a 4-byte aligned address goes through
// shared memory and out as 48 coalesced words; a partial or misaligned one as st_six per lane.
__device__ __forceinline__ void store_row(uint8_t *seg, bool whole, uint32_t *stage, int lane, uint32_t p0,
                                          uint32_t p1, bool valid)
{
    if (whole && ((uintptr_t)seg & 3u) == 0) {  // warp-uniform
        unsigned short *s16 = reinterpret_cast<unsigned short *>(stage) + 3 * lane;
        const uint32_t lo = prmt(p0, p1, 0x4210u), hi = prmt(p1, 0u, 0x4421u);
        s16[0] = (unsigned short)lo;
        s16[1] = (unsigned short)(lo >> 16);
        s16[2] = (unsigned short)hi;
        __syncwarp();
        uint32_t *g = reinterpret_cast<uint32_t *>(seg);
        __stcs(g + lane, stage[lane]);
        if (lane < 16) __stcs(g + 32 + lane, stage[32 + lane]);
        __syncwarp();
    } else if (valid) {
        st_six(seg + 6 * lane, p0, p1);
    }
}

__global__ void __launch_bounds__(kConvThreadsX *kConvThreadsY)
nv12_to_bgr_kernel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int n_frames, int h, int w,
                   int pitch, long long frame_stride)
{
    __shared__ uint32_t stage[kConvThreadsX * kConvThreadsY / 32][48];
    const int lane = threadIdx.x & 31;
    const int bx = blockIdx.x * kConvThreadsX + threadIdx.x;  // 2x2 block column
    const int bx0 = bx - lane;                                // the warp's first one
    const bool valid = 2 * bx < w, whole = 2 * (bx0 + 32) <= w;
    const int bxl = valid ? bx : w / 2 - 1;                   // loads of lanes past the edge stay inside
    uint32_t *st = stage[(threadIdx.y * kConvThreadsX + threadIdx.x) / 32];
    const int rp0 = blockIdx.y * kConvThreadsY * kRowPairs + threadIdx.y;  // first block row
    const long long dst_row = 3LL * w;
    for (int f = blockIdx.z; f < n_frames; f += gridDim.z) {
        const uint8_t *s = src + (long long)f * frame_stride;
        uint8_t *d = dst + (long long)f * h * dst_row;
        uint32_t ya[kRowPairs], yb[kRowPairs], uv[kRowPairs];
#pragma unroll
        for (int k = 0; k < kRowPairs; ++k) {
            const int rp = min(rp0 + k * kConvThreadsY, h / 2 - 1);
            const uint8_t *l = s + (long long)(2 * rp) * pitch + 2 * bxl;
            ya[k] = ld_pair(l);
            yb[k] = ld_pair(l + pitch);
            uv[k] = ld_pair(s + (long long)(h + rp) * pitch + 2 * bxl);
        }
#pragma unroll
        for (int k = 0; k < kRowPairs; ++k) {
            const int rp = rp0 + k * kConvThreadsY;
            if (rp >= h / 2) break;  // warp-uniform: one block row per warp
            const uint32_t U = uv[k] & 0xffu, V = uv[k] >> 8;
            uint8_t *seg = d + (long long)(2 * rp) * dst_row + 6LL * bx0;
            store_row(seg, whole, st, lane, yuv_to_bgr(ya[k] & 0xffu, U, V), yuv_to_bgr(ya[k] >> 8, U, V), valid);
            store_row(seg + dst_row, whole, st, lane, yuv_to_bgr(yb[k] & 0xffu, U, V),
                      yuv_to_bgr(yb[k] >> 8, U, V), valid);
        }
    }
}

}  // namespace

int bevk_launch_warp_nv12(const BevkNv12Params &P, int linear, cudaStream_t stream)
{
    const bool words = ((uintptr_t)P.w.src % 4) == 0 && (P.pitch % 4) == 0 && (P.frame_stride % 4) == 0;
    const bool packed = (P.w.dst_w % 4) == 0 && ((uintptr_t)P.w.dst % 4) == 0;
    if (linear)
        words ? launch_warp<true, true>(P, packed, stream) : launch_warp<true, false>(P, packed, stream);
    else
        words ? launch_warp<false, true>(P, packed, stream) : launch_warp<false, false>(P, packed, stream);
    BEVK_CUDA(cudaGetLastError());
    return BEVK_OK;
}

int bevk_launch_nv12_to_bgr(const void *src, void *dst, int n_frames, int h, int w, int pitch,
                            long long frame_stride, cudaStream_t stream)
{
    dim3 block(kConvThreadsX, kConvThreadsY, 1);
    dim3 grid((w / 2 + kConvThreadsX - 1) / kConvThreadsX,
              (h / 2 + kConvThreadsY * kRowPairs - 1) / (kConvThreadsY * kRowPairs),
              n_frames < 65535 ? n_frames : 65535);
    nv12_to_bgr_kernel<<<grid, block, 0, stream>>>((const uint8_t *)src, (uint8_t *)dst, n_frames, h, w, pitch,
                                                   frame_stride);
    BEVK_CUDA(cudaGetLastError());
    return BEVK_OK;
}

int bevk_launch_resize_nv12(const void *src, void *dst, int n_frames, int src_h, int src_w, int pitch,
                            long long frame_stride, int dst_h, int dst_w, cudaStream_t stream)
{
    ResizeNv12Params p;
    p.src = (const uint8_t *)src;
    p.dst = (uint8_t *)dst;
    p.src_h = src_h;
    p.src_w = src_w;
    p.dst_h = dst_h;
    p.dst_w = dst_w;
    p.pitch = (uint32_t)pitch;
    p.frame_stride = frame_stride;
    p.dst_frame = (long long)dst_h * dst_w * 3;
    // cv2: inv_scale = (double)dsize / ssize; scale = 1. / inv_scale
    p.scale_x = 1.0 / ((double)dst_w / (double)src_w);
    p.scale_y = 1.0 / ((double)dst_h / (double)src_h);
    p.n_frames = n_frames;
    p.frames_per_chunk = bevk_resize_frames_per_chunk(n_frames, dst_h, dst_w);
    const int z = (n_frames + p.frames_per_chunk - 1) / p.frames_per_chunk;
    if (z > 65535) BEVK_FAIL(BEVK_E_ARG, "resize_nv12: too many frame chunks (%d) for one launch", z);
    const dim3 grid((dst_w + 31) / 32, (dst_h + 7) / 8, z);
    const bool words = ((uintptr_t)src % 4) == 0 && (pitch % 4) == 0 && (frame_stride % 4) == 0;
    const bool packed = (dst_w % 4) == 0 && ((uintptr_t)dst % 4) == 0;
    words ? launch_resize<true>(p, packed, grid, stream) : launch_resize<false>(p, packed, grid, stream);
    BEVK_CUDA(cudaGetLastError());
    return BEVK_OK;
}
