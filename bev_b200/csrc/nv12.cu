// nv12.cu -- NV12 video frames (what a GPU video decoder hands out) to BGR: the conversion
// cv2.cvtColor(f, COLOR_YUV2BGR_NV12) on frame batches, and the perspective warp of NV12 or I420
// frames (what CPU decoders hand out) fused with it, so that decoded frames reach the BEV without a
// BGR copy of every frame.
//
// Semantics: cv2 4.13.  The conversion is BT.601 limited range in 20-bit fixed point with chroma
// replicated over each 2x2 luma block; the warp equals cv2.warpPerspective of the converted frame
// (reference frame loop vis_homo.py:85-91), i.e. every bilinear tap is converted on its own and
// the four are then interpolated with the uint8 x 3 arithmetic of warp_u8c3.cuh.  A tap outside
// the frame takes the BGR border colour; it is never converted from YUV.  The resize of NV12
// frames is in resize.cu.
//
// Layout of frame n: luma rows 0..H-1 then chroma rows 0..H/2-1 (NV12: interleaved U, V bytes;
// I420: the U plane then the V plane, see yuv_src.cuh), each row `pitch` bytes after the previous
// one, the frame at src + n * frame_stride bytes.
#include "bevk_common.cuh"
#include "yuv_src.cuh"

namespace {

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
    int gi;
    const BevkWarpGroup &g = find_group(p, blockIdx.z, gi);
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

// warp_nv12_kernel over a source format S of yuv_src.cuh (S::make, S::load, S::math): the warp of
// I420 frames.  NV12 frames keep warp_nv12_kernel, which holds the NV12 addressing of Nv12Src with
// the window's border constants and straddle flags computed once per pixel; through Nv12Src the
// bilinear instances took 48 instead of 40 registers and ran 3-7 % slower (DESIGN.md 3.11).
template <class S, bool PACKED, int kBatch>
__global__ void __launch_bounds__(256) warp_yuv_src_kernel(const __grid_constant__ BevkNv12Params P)
{
    const BevkWarpParams &p = P.w;
    const int lane = threadIdx.x, x0 = blockIdx.x * 32;
    const int x = x0 + lane, y = blockIdx.y * 8 + threadIdx.y;
    if (y >= p.dst_h) return;  // a warp is one dst row segment: uniform exit, shuffles stay legal
    int gi;
    const BevkWarpGroup &g = find_group(p, blockIdx.z, gi);
    const int c_local = blockIdx.z - g.chunk0;
    const int f0 = c_local * p.frames_per_chunk;
    const int f1 = min(f0 + p.frames_per_chunk, g.count);

    const uint32_t bpx = border_bgr(p.border);
    const typename S::Tap t = S::make(P, g.M, min(x, p.dst_w - 1), y, bpx);

    const int j = lane >> 2, r4 = lane & 3;
    const uint32_t sel_pack = r4 == 0 ? 0x4210u : (r4 == 1 ? 0x5421u : 0x6542u);
    const bool st_ok = PACKED ? (r4 < 3 && 4 * j < min(32, p.dst_w - x0)) : x < p.dst_w;
    uint8_t *dst = (uint8_t *)p.dst + ((long long)y * p.dst_w + x0) * 3 + (PACKED ? (3 * j + r4) * 4 : 3 * lane);
    const uint8_t *src = (const uint8_t *)p.src;

    auto load = [&](int f, uint32_t(&w)[S::kWords]) {
        S::load(P, src + (long long)(g.first + f * g.stride) * P.frame_stride, t, w);
    };
    auto finish = [&](int f, const uint32_t(&w)[S::kWords]) {
        const uint32_t P0 = S::math(t, w, bpx);
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
        uint32_t w[kBatch][S::kWords];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) load(f + u, w[u]);
#pragma unroll
        for (int u = 0; u < kBatch; ++u) finish(f + u, w[u]);
    }
    for (; f < f1; ++f) {
        uint32_t w[S::kWords];
        load(f, w);
        finish(f, w);
    }
}

template <class S, int kBatch>
void launch_yuv_warp(const BevkNv12Params &P, bool packed, cudaStream_t stream)
{
    dim3 block(32, 8, 1);
    dim3 grid((P.w.dst_w + 31) / 32, (P.w.dst_h + 7) / 8, P.w.total_chunks);
    if (packed)
        warp_yuv_src_kernel<S, true, kBatch><<<grid, block, 0, stream>>>(P);
    else
        warp_yuv_src_kernel<S, false, kBatch><<<grid, block, 0, stream>>>(P);
}

// the four kernels of a YUV source format: bilinear / nearest, word / byte gathers
template <template <bool, bool> class S>
void launch_yuv_src(const BevkNv12Params &P, bool words, bool packed, int linear, cudaStream_t stream)
{
    if (linear)
        words ? launch_yuv_warp<S<true, true>, 2>(P, packed, stream)
              : launch_yuv_warp<S<true, false>, 2>(P, packed, stream);
    else
        words ? launch_yuv_warp<S<false, true>, 4>(P, packed, stream)
              : launch_yuv_warp<S<false, false>, 4>(P, packed, stream);
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

int bevk_launch_warp_nv12(const BevkNv12Params &P, int src_format, int linear, cudaStream_t stream)
{
    const bool words = ((uintptr_t)P.w.src % 4) == 0 && (P.pitch % 4) == 0 && (P.frame_stride % 4) == 0;
    const bool packed = (P.w.dst_w % 4) == 0 && ((uintptr_t)P.w.dst % 4) == 0;
    if (src_format == BEVK_YUV_I420)
        launch_yuv_src<I420Src>(P, words, packed, linear, stream);
    else if (linear)
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
