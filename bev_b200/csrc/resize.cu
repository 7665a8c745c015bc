// resize.cu -- batched cv2.resize of uint8 frames for sm_100a, INTER_LINEAR and INTER_AREA, from 1 to
// 4-channel frames or fused with the NV12 -> BGR conversion for frames from a GPU video decoder:
// cv2.resize(cv2.cvtColor(f, COLOR_YUV2BGR_NV12), dsize, interpolation).  INTER_LINEAR is the
// small-frame path of the reference's frame loop, `img_small = cv2.resize(img, (new_u, new_v))`
// (vis_homo.py:90), whose result feeds the second warp at vis_homo.py:91 through the homography of
// Calib.scale(align_corners=False) (bev/calib.py:142-198).  INTER_AREA is what OpenCV recommends
// for a small frame: every source pixel contributes to the dst pixel whose cell it lies in, so fine
// texture such as lane markings does not alias.
//
// Semantics: OpenCV 4.13, bit for bit (oracle/resize_oracle.py and oracle/resize_area_oracle.py
// restate it and are pinned against cv2).  INTER_LINEAR is cv2's 8-bit bilinear resize:
//   column dx: fx = float((dx + 0.5) * scale_x - 0.5), sx = floor(fx), fx -= sx; left of the image
//   (sx, fx) = (0, 0), at / right of the last pixel (src_w - 1, 0); weights rint((1 - fx) * 2048),
//   rint(fx * 2048) in float.  Row dy: the same without that clamp, the two row indices clipped
//   into the image instead.  S = p[sx] * a0 + p[sx + 1] * a1 per row, then
//   (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2.
//   2-channel frames downscaled by exactly 2 in both axes take the round-half-even mean of each
//   2x2 block instead (cv2's INTER_AREA special case).
// For INTER_AREA, with scale = 1 / (dsize / ssize) in double per axis, cv2 takes one of three
// branches:
//   integer cells  both scales >= 1 and integer (kx, ky): the integer sum s of the kx x ky cell,
//           then rint(s * (1.f / (kx * ky))) in float; (s + 2) >> 2 at kx = ky = 2 unless 2 channels.
//   area    both scales >= 1 otherwise: per axis cv2's computeResizeAreaTab in double -- an
//           optional partial first cell, full cells of weight 1 / cellWidth, an optional partial
//           last cell, 1e-3 thresholds, cellWidth = min(scale, ssize - fsx1).  The entries of one
//           dst position are consecutive source indices, so a thread keeps (first index, count,
//           first / middle / last alpha) per axis instead of a table.  Per source row
//           buf += S * alpha in table order, then sum = beta * buf for the first row and
//           sum += beta * buf for the others, float32 and unfused; rint and saturate at the end.
//   any axis upscales: the bilinear resize above with the area coefficients
//           sx = floor(dx * scale), fx = float((dx + 1) - (sx + 1) / scale),
//           fx = fx <= 0 ? 0 : fx - floor(fx) (linear_area_coef).
// An NV12 tap is converted to BGR with cv2's arithmetic (yuv_bgr.cuh) on its own, then
// interpolated.  The coefficients are recomputed per thread from (dx, dy) with unfused IEEE float /
// double operations (the library is built with -fmad=false) -- no tables to upload, nothing to
// keep alive across the asynchronous launch -- and amortised over the frames of the thread's chunk.
//
// One thread per dst pixel in every kernel.  The bilinear kernels take the coefficient rule as a
// template parameter: a word-gather one for BGR frames (3 aligned words per window row, dp2a for
// the horizontal pass, 32 pixels packed into one 96-byte store per warp), one for NV12 frames, and
// a byte-wise one for every other channel count / width.  They are HBM-bound: every source row a
// dst row references is read once (sector-wise), the small frame written once.  The area kernel
// runs the other two INTER_AREA branches with byte loads.
#include <cfloat>
#include <cmath>

#include "bevk_common.cuh"
#include "resize_coef.cuh"
#include "warp_u8c3.cuh"
#include "yuv_bgr.cuh"

namespace {

// word load with a 256-byte L2 prefetch hint: the resize reads (nearly) every byte of the rows it
// touches, so the neighbouring lines are wanted anyway (3 % faster than the plain read-only load)
__device__ __forceinline__ uint32_t ldg_dense(const uint32_t *p)
{
    uint32_t v;
    asm("ld.global.nc.L2::256B.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// ---- any channel count: one thread per dst pixel, byte loads -----------------------------------
template <int C, bool AREA>
__global__ void __launch_bounds__(256) resize_bytes_kernel(const __grid_constant__ BevkResizeParams p)
{
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= p.dst_w || y >= p.dst_h) return;
    int sx, a0, a1, sy, b0, b1;
    bilinear_coef<AREA>(p, x, y, sx, a0, a1, sy, b0, b1);
    const int sx1 = min(sx + 1, p.src_w - 1);
    const int r0 = min(max(sy, 0), p.src_h - 1), r1 = min(max(sy + 1, 0), p.src_h - 1);
    const long long o00 = ((long long)r0 * p.src_w + sx) * C, o01 = ((long long)r0 * p.src_w + sx1) * C;
    const long long o10 = ((long long)r1 * p.src_w + sx) * C, o11 = ((long long)r1 * p.src_w + sx1) * C;
    const long long od = ((long long)y * p.dst_w + x) * C;
    const int f0 = blockIdx.z * p.frames_per_chunk, f1 = min(f0 + p.frames_per_chunk, p.n_frames);
    if constexpr (C == 2 && !AREA) {
        // cv2 sends an exact 2x downscale to INTER_AREA, which for 2 channels rounds the mean of
        // the 2x2 block half to even (for 1, 3, 4 channels it equals the bilinear result).  The
        // window above is then exactly that block.  An upscaling axis never meets this condition.
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
// per 4 pixels) and src_w >= 2.  The 2-pixel window starts inside the image: at the last column
// (sx == src_w - 1) it moves one left and swaps its weights, which relies on a1 == 0 there.  The
// column clamp of both coefficient rules gives exactly that.
template <bool AREA>
__global__ void __launch_bounds__(256) resize_u8c3_kernel(const __grid_constant__ BevkResizeParams p)
{
    const int lane = threadIdx.x, x0 = blockIdx.x * 32;
    const int x = min(x0 + lane, p.dst_w - 1), y = blockIdx.y * 8 + threadIdx.y;
    if (y >= p.dst_h) return;  // a warp is one dst row segment: uniform exit, shuffles stay legal
    int sx, a0, a1, sy, b0, b1;
    bilinear_coef<AREA>(p, x, y, sx, a0, a1, sy, b0, b1);
    const int cs = min(sx, p.src_w - 2);
    const int wa = cs == sx ? a0 : a1, wb = cs == sx ? a1 : a0;
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

// ---- NV12 frames to BGR ------------------------------------------------------------------------
// Layout of frame n: luma rows 0..src_h-1 then chroma rows 0..src_h/2-1 (interleaved U, V bytes),
// each row `pitch` bytes after the previous one, the frame at src + n * src_frame bytes; in-frame
// offsets fit 32 bits.
// One lane per dst pixel, as resize_u8c3_kernel: the coefficients are computed once per frame
// chunk, and the 2-pixel window starts inside the frame (cs = min(sx, src_w - 2), weights swapped
// when it moved).  Every frame gathers two luma rows r0, r1 (2 bytes at cs each; one row twice at
// the top and bottom edges) and the chroma rows r0 / 2, r1 / 2 under them (4 bytes each: the U,V
// pairs of columns cs and cs + 1, one pair twice when cs is even), converts the 4 taps on their
// own, then runs cv2's horizontal pass per channel as one dp2a on the weight pair and its vertical
// pass.  WORDS (pitch, frame stride and src 4-byte aligned): aligned 32-bit words + funnel shifts,
// the second word of a row only when the window straddles it; otherwise byte loads.  PACKED
// (dst_w % 4 == 0): the warp packs 32 pixels into one coalesced 96-byte store, otherwise every
// lane stores its 3 bytes.
// The gather is warp_nv12_kernel's (nv12.cu) with the second luma row at r1 instead of the next
// row.  It is kept separate: moving it into a helper both kernels call changed the register
// allocation and SASS of warp_nv12_kernel's bilinear variants.
template <bool AREA, bool WORDS, bool PACKED, int kBatch>
__global__ void __launch_bounds__(256) resize_nv12_kernel(const __grid_constant__ BevkResizeParams p)
{
    const int lane = threadIdx.x, x0 = blockIdx.x * 32;
    const int x = x0 + lane, y = blockIdx.y * 8 + threadIdx.y;
    if (y >= p.dst_h) return;  // a warp is one dst row segment: uniform exit, shuffles stay legal
    int sx, a0, a1, sy, b0, b1;
    bilinear_coef<AREA>(p, min(x, p.dst_w - 1), y, sx, a0, a1, sy, b0, b1);
    const int cs = min(sx, p.src_w - 2);
    const int wa = cs == sx ? a0 : a1, wb = cs == sx ? a1 : a0;  // sx == src_w - 1 has a1 == 0
    const uint32_t w16 = (uint32_t)wa | ((uint32_t)wb << 16);
    const int r0 = min(max(sy, 0), p.src_h - 1), r1 = min(max(sy + 1, 0), p.src_h - 1);
    const uint32_t pitch = (uint32_t)p.pitch;
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
        const uint8_t *s = p.src + (long long)f * p.src_frame;
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

// ---- INTER_AREA downscales: integer cells (FAST) and general cells ------------------------------
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

// One source row of a frame: the bytes of row y, and for NV12 the chroma row under it.
template <int C, bool NV12> struct Row {
    const uint8_t *l, *c;
    __device__ __forceinline__ Row(const uint8_t *s, const BevkResizeParams &p, int y)
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

// Each thread computes its tap window once per frame chunk and reads its taps with byte loads,
// which serve any alignment and pitch; an NV12 tap is converted to BGR where it is read.
template <int C, bool NV12, bool FAST>
__global__ void __launch_bounds__(256) resize_area_kernel(const __grid_constant__ BevkResizeParams p)
{
    static_assert(!NV12 || C == 3, "NV12 frames convert to BGR");
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    if (x >= p.dst_w || y >= p.dst_h) return;
    const long long od = ((long long)y * p.dst_w + x) * C;
    const int f0 = blockIdx.z * p.frames_per_chunk, f1 = min(f0 + p.frames_per_chunk, p.n_frames);

    if constexpr (FAST) {
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
    } else {
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
    }
}

// ---- launch ------------------------------------------------------------------------------------
const dim3 kBlock(32, 8, 1);

template <bool AREA>
void launch_bilinear(const BevkResizeParams &p, int channels, bool nv12, dim3 grid, cudaStream_t st)
{
    if (nv12) {
        constexpr int kBatch = 2;
        const bool words = ((uintptr_t)p.src % 4) == 0 && (p.pitch % 4) == 0 && (p.src_frame % 4) == 0;
        const bool packed = (p.dst_w % 4) == 0 && ((uintptr_t)p.dst % 4) == 0;
        if (words && packed)
            resize_nv12_kernel<AREA, true, true, kBatch><<<grid, kBlock, 0, st>>>(p);
        else if (words)
            resize_nv12_kernel<AREA, true, false, kBatch><<<grid, kBlock, 0, st>>>(p);
        else if (packed)
            resize_nv12_kernel<AREA, false, true, kBatch><<<grid, kBlock, 0, st>>>(p);
        else
            resize_nv12_kernel<AREA, false, false, kBatch><<<grid, kBlock, 0, st>>>(p);
        return;
    }
    const bool words = channels == 3 && p.src_w >= 2 && (p.src_w % 4) == 0 && (p.dst_w % 4) == 0 &&
                       ((uintptr_t)p.src % 4) == 0 && ((uintptr_t)p.dst % 4) == 0;
    if (words) {
        resize_u8c3_kernel<AREA><<<grid, kBlock, 0, st>>>(p);
        return;
    }
    switch (channels) {
    case 1: resize_bytes_kernel<1, AREA><<<grid, kBlock, 0, st>>>(p); break;
    case 2: resize_bytes_kernel<2, AREA><<<grid, kBlock, 0, st>>>(p); break;
    case 3: resize_bytes_kernel<3, AREA><<<grid, kBlock, 0, st>>>(p); break;
    default: resize_bytes_kernel<4, AREA><<<grid, kBlock, 0, st>>>(p); break;
    }
}

template <bool FAST> void launch_area(const BevkResizeParams &p, int channels, bool nv12, dim3 grid, cudaStream_t st)
{
    if (nv12) {
        resize_area_kernel<3, true, FAST><<<grid, kBlock, 0, st>>>(p);
        return;
    }
    switch (channels) {
    case 1: resize_area_kernel<1, false, FAST><<<grid, kBlock, 0, st>>>(p); break;
    case 2: resize_area_kernel<2, false, FAST><<<grid, kBlock, 0, st>>>(p); break;
    case 3: resize_area_kernel<3, false, FAST><<<grid, kBlock, 0, st>>>(p); break;
    default: resize_area_kernel<4, false, FAST><<<grid, kBlock, 0, st>>>(p); break;
    }
}

// cvRound(scale) within DBL_EPSILON of scale, as cv2's is_area_fast
bool integer_scale(double scale, int &k)
{
    k = (int)std::lround(scale);
    return std::fabs(scale - k) < DBL_EPSILON;
}

}  // namespace

int bevk_launch_resize(const void *src, void *dst, int n_frames, int src_h, int src_w, int channels, int nv12,
                       long long pitch, long long frame_stride, int dst_h, int dst_w, int interpolation,
                       cudaStream_t stream)
{
    BevkResizeParams p;
    dim3 grid;
    const int rc = bevk_plan_resize(src, dst, n_frames, src_h, src_w, channels, pitch, frame_stride, dst_h, dst_w,
                                    p, grid);
    if (rc) return rc;
    // cv2's branch first, then the kernel for the frame layout
    int kx, ky;
    if (interpolation != BEVK_INTER_AREA) {
        launch_bilinear<false>(p, channels, nv12, grid, stream);
    } else if (p.scale_x < 1 || p.scale_y < 1) {
        launch_bilinear<true>(p, channels, nv12, grid, stream);
    } else if (integer_scale(p.scale_x, kx) && integer_scale(p.scale_y, ky)) {
        p.kx = kx;
        p.ky = ky;
        p.inv_area = 1.f / (float)(kx * ky);
        launch_area<true>(p, channels, nv12, grid, stream);
    } else {
        launch_area<false>(p, channels, nv12, grid, stream);
    }
    BEVK_CUDA(cudaGetLastError());
    return BEVK_OK;
}
