// yuv_src.cuh -- the YUV 4:2:0 source formats of the fused warps: how one dst pixel's bilinear or
// nearest window is found, gathered and converted to BGR in a frame of NV12 or I420 bytes.  The
// warps to BGR (nv12.cu) and to YUV 4:2:0 (yuv420.cu) are templated on these structs, so both
// output layouts share one copy of every source's addressing, loads and arithmetic.
//
// A source format S provides the frame-invariant state of one pixel (S::Tap, S::make), the window
// loads of one frame (S::load, S::kWords words) and the pixel's BGR value (S::math), bit-exact
// with cv2.warpPerspective of cv2.cvtColor(frame, COLOR_YUV2BGR_NV12 / _I420): every bilinear tap
// is converted on its own and the four are interpolated with the uint8 x 3 arithmetic of
// warp_u8c3.cuh; a tap outside the frame takes the BGR border colour.  cv2 4.13 converts I420 and
// NV12 with the same arithmetic, so the two formats differ only in where the chroma bytes sit.
//
// Params P: BevkNv12Params or BevkYuvParams (P.w, P.pitch, P.frame_stride).  Frame layout: h luma
// rows then h / 2 rows of chroma, each row P.pitch bytes after the previous one.  NV12 chroma row r
// holds the interleaved U, V pairs of block row r.  I420 chroma follows cv2's packing with a row
// step: U of block row r at row h + r / 2, column (r % 2) * w / 2; V of block row r as U of block
// row r + h / 2.
#pragma once
#include "bevk_common.cuh"
#include "warp_u8c3.cuh"
#include "yuv_bgr.cuh"

namespace {

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

// The clamped 2x2 window of warp_u8c3_direct_kernel: first column / row and the integer weights
// (0..32; nearest: 1 for the tap when it is inside) of its two columns / rows.
template <bool LINEAR>
__device__ __forceinline__ bool clamped_window(const BevkWarpParams &p, const double *M, int x, int y, int &cs,
                                               int &rs, int &wc0, int &wc1, int &wr0, int &wr1)
{
    int X, Y;
    bevk_map_pixel(M, x, y, p.bw0, LINEAR ? 32.0 : 1.0, X, Y);
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
    return act;
}

// dp2a bilinear of warp_u8c3.cuh's lerp_xy with the border folded into the rounding constant:
// wout = the weight of the taps outside the frame (x 64, cv2's scale doubled).
__device__ __forceinline__ uint32_t lerp_border(uint32_t w0, uint32_t w1, uint32_t wout, uint32_t bpx, uint32_t xa,
                                                uint32_t ya, uint32_t xb, uint32_t yb)
{
    const uint32_t t0 = __dp2a_lo(w1, xb, __dp2a_lo(w0, xa, 32768u + byte_of(bpx, 0) * wout));
    const uint32_t t1 = __dp2a_hi(w1, xb, __dp2a_hi(w0, xa, 32768u + byte_of(bpx, 1) * wout));
    const uint32_t t2 = __dp2a_lo(w1, yb, __dp2a_lo(w0, ya, 32768u + byte_of(bpx, 2) * wout));
    return prmt(prmt(t0, t1, 0x4462u), t2, 0x7610u);
}

constexpr uint32_t kInside = 0xffffffffu;  // nearest: "the tap is inside", else the border colour

// The bilinear value of a YUV window: L0, L1 = [Y Y' . .] of window rows 0 / 1, C0, C1 = [U V U' V']
// of the window's left and right column under them.
__device__ __forceinline__ uint32_t yuv_lerp(uint32_t w0, uint32_t w1, uint32_t k, uint32_t bpx, uint32_t L0,
                                             uint32_t L1, uint32_t C0, uint32_t C1)
{
    const uint32_t p00 = yuv_to_bgr(byte_of(L0, 0), byte_of(C0, 0), byte_of(C0, 1));
    const uint32_t p01 = yuv_to_bgr(byte_of(L0, 1), byte_of(C0, 2), byte_of(C0, 3));
    const uint32_t p10 = yuv_to_bgr(byte_of(L1, 0), byte_of(C1, 0), byte_of(C1, 1));
    const uint32_t p11 = yuv_to_bgr(byte_of(L1, 1), byte_of(C1, 2), byte_of(C1, 3));
    // the dp2a operands of lerp_xy: [B0 B0' G0 G0'] and [R0 R0' . .] per window row
    return lerp_border(w0, w1, k, bpx, prmt(p00, p01, 0x5140u), prmt(p00, p01, 0x0062u), prmt(p10, p11, 0x5140u),
                       prmt(p10, p11, 0x0062u));
}

// NV12 frames.  WORDS (src, pitch and frame stride 4-byte aligned): aligned 32-bit words + funnel
// shifts, the second word of a row only when the window straddles it; otherwise byte loads.  The
// window's two luma rows take 2 bytes each, the one or two chroma rows under them 4 bytes each (the
// U, V pairs of the window's one or two chroma columns).
template <bool LINEAR, bool WORDS> struct Nv12Src {
    static constexpr int kWords = LINEAR ? (WORDS ? 8 : 4) : 2;
    struct Tap {
        uint32_t lo;    // luma row rs at column cs
        uint32_t co;    // chroma row rs / 2 at the U of column cs
        uint32_t co_b;  // the chroma row under window row 1
        uint32_t odd;   // cs is odd: the right column uses the next U,V pair
        uint32_t w0, w1, k;
    };
    template <class Prm>
    static __device__ __forceinline__ Tap make(const Prm &P, const double *M, int x, int y, uint32_t bpx)
    {
        int cs, rs, wc0, wc1, wr0, wr1;
        const bool act = clamped_window<LINEAR>(P.w, M, x, y, cs, rs, wc0, wc1, wr0, wr1);
        const uint32_t pitch = (uint32_t)P.pitch;
        Tap t;
        t.lo = (uint32_t)rs * pitch + (uint32_t)cs;
        t.co = ((uint32_t)P.w.src_h + (uint32_t)(rs >> 1)) * pitch + 2u * (uint32_t)(cs >> 1);
        t.co_b = t.co + ((rs & 1) ? pitch : 0u);
        t.odd = cs & 1;
        t.w0 = tap_weight(wc0, wr0) | (tap_weight(wc1, wr0) << 16);
        t.w1 = tap_weight(wc0, wr1) | (tap_weight(wc1, wr1) << 16);
        t.k = LINEAR ? 64u * (uint32_t)(1024 - (wc0 + wc1) * (wr0 + wr1)) : (act ? kInside : bpx);
        return t;
    }
    template <class Prm>
    static __device__ __forceinline__ void load(const Prm &P, const uint8_t *s, const Tap &t, uint32_t (&w)[kWords])
    {
        const uint32_t pitch = (uint32_t)P.pitch;
        auto LD = [](const uint8_t *a) { return ldg_sparse(reinterpret_cast<const uint32_t *>(a)); };
        auto B = [](const uint8_t *a) { return (uint32_t)__ldg(a); };
        if (LINEAR && WORDS) {
            // the second word of a row only when the 2 luma / 4 chroma bytes straddle it
            const bool l_two = (t.lo & 3u) == 3u, c_two = (t.co & 3u) == 2u && t.odd;
            const uint8_t *la = s + (t.lo & ~3u), *ca = s + (t.co & ~3u), *cb = s + (t.co_b & ~3u);
            w[0] = LD(la);
            w[1] = l_two ? LD(la + 4) : 0u;
            w[2] = LD(la + pitch);
            w[3] = l_two ? LD(la + pitch + 4) : 0u;
            w[4] = LD(ca);
            w[5] = c_two ? LD(ca + 4) : 0u;
            w[6] = LD(cb);
            w[7] = c_two ? LD(cb + 4) : 0u;
        } else if (LINEAR) {
            const uint8_t *la = s + t.lo, *ca = s + t.co, *cb = s + t.co_b;
            const uint32_t cn = t.odd ? 2u : 0u;  // offset of the right column's U,V pair
            w[0] = B(la) | (B(la + 1) << 8);
            w[1] = B(la + pitch) | (B(la + pitch + 1) << 8);
            w[2] = B(ca) | (B(ca + 1) << 8) | (B(ca + cn) << 16) | (B(ca + cn + 1) << 24);
            w[3] = B(cb) | (B(cb + 1) << 8) | (B(cb + cn) << 16) | (B(cb + cn + 1) << 24);
        } else if (WORDS) {
            w[0] = LD(s + (t.lo & ~3u));
            w[1] = LD(s + (t.co & ~3u));
        } else {
            w[0] = B(s + t.lo);
            w[1] = B(s + t.co) | (B(s + t.co + 1) << 8);
        }
    }
    static __device__ __forceinline__ uint32_t math(const Tap &t, const uint32_t (&w)[kWords], uint32_t bpx)
    {
        if (!LINEAR) {
            const uint32_t Yw = WORDS ? byte_of(w[0], t.lo & 3u) : w[0];
            const uint32_t Cw = WORDS ? (w[1] >> (8 * (t.co & 2u))) : w[1];
            return t.k == kInside ? yuv_to_bgr(Yw, byte_of(Cw, 0), byte_of(Cw, 1)) : t.k;
        }
        if (!WORDS) return yuv_lerp(t.w0, t.w1, t.k, bpx, w[0], w[1], w[2], w[3]);
        // the left column's U,V pair twice when cs is even (both columns share it)
        const uint32_t csel = t.odd ? 0x3210u : 0x1010u;
        return yuv_lerp(t.w0, t.w1, t.k, bpx, __funnelshift_r(w[0], w[1], 8 * (t.lo & 3u)),
                        __funnelshift_r(w[2], w[3], 8 * (t.lo & 3u)),
                        prmt(__funnelshift_r(w[4], w[5], 8 * (t.co & 3u)), 0u, csel),
                        prmt(__funnelshift_r(w[6], w[7], 8 * (t.co_b & 3u)), 0u, csel));
    }
};

// I420 frames: the luma of Nv12Src; U and V each from their own plane, 1 byte (nearest, or an even
// cs) or 2 bytes (an odd cs: the right column's sample is the next one) per chroma row.  WORDS as
// for Nv12Src; a U or V row segment that straddles a word takes the next word too.
template <bool LINEAR, bool WORDS> struct I420Src {
    static constexpr int kWords = LINEAR ? (WORDS ? 12 : 4) : (WORDS ? 3 : 2);
    struct Tap {
        uint32_t lo;          // luma row rs at column cs
        uint32_t uo, vo;      // U and V of chroma row rs / 2 at column cs / 2
        uint32_t uo_b, vo_b;  // the same under window row 1
        uint32_t odd;         // cs is odd: the right column uses the next U and V samples
        uint32_t w0, w1, k;
    };
    // byte offset of the U sample (r, c) of a frame of P.w.src_h rows: cv2's I420 packing
    template <class Prm> static __device__ __forceinline__ uint32_t u_at(const Prm &P, uint32_t r, uint32_t c)
    {
        return ((uint32_t)P.w.src_h + (r >> 1)) * (uint32_t)P.pitch + (r & 1u) * ((uint32_t)P.w.src_w >> 1) + c;
    }
    template <class Prm>
    static __device__ __forceinline__ Tap make(const Prm &P, const double *M, int x, int y, uint32_t bpx)
    {
        int cs, rs, wc0, wc1, wr0, wr1;
        const bool act = clamped_window<LINEAR>(P.w, M, x, y, cs, rs, wc0, wc1, wr0, wr1);
        const uint32_t r = (uint32_t)rs >> 1, rb = (uint32_t)(rs + 1) >> 1, c = (uint32_t)cs >> 1;
        const uint32_t vr = (uint32_t)P.w.src_h >> 1;  // V of block row r is U of block row r + h / 2
        Tap t;
        t.lo = (uint32_t)rs * (uint32_t)P.pitch + (uint32_t)cs;
        t.uo = u_at(P, r, c);
        t.vo = u_at(P, r + vr, c);
        t.uo_b = LINEAR ? u_at(P, rb, c) : t.uo;
        t.vo_b = LINEAR ? u_at(P, rb + vr, c) : t.vo;
        t.odd = cs & 1;
        t.w0 = tap_weight(wc0, wr0) | (tap_weight(wc1, wr0) << 16);
        t.w1 = tap_weight(wc0, wr1) | (tap_weight(wc1, wr1) << 16);
        t.k = LINEAR ? 64u * (uint32_t)(1024 - (wc0 + wc1) * (wr0 + wr1)) : (act ? kInside : bpx);
        return t;
    }
    template <class Prm>
    static __device__ __forceinline__ void load(const Prm &P, const uint8_t *s, const Tap &t, uint32_t (&w)[kWords])
    {
        const uint32_t pitch = (uint32_t)P.pitch;
        auto LD = [](const uint8_t *a) { return ldg_sparse(reinterpret_cast<const uint32_t *>(a)); };
        auto B = [](const uint8_t *a) { return (uint32_t)__ldg(a); };
        if (LINEAR && WORDS) {
            const bool l_two = (t.lo & 3u) == 3u;
            const uint8_t *la = s + (t.lo & ~3u);
            w[0] = LD(la);
            w[1] = l_two ? LD(la + 4) : 0u;
            w[2] = LD(la + pitch);
            w[3] = l_two ? LD(la + pitch + 4) : 0u;
            const uint32_t co[4] = {t.uo, t.vo, t.uo_b, t.vo_b};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const uint8_t *ca = s + (co[i] & ~3u);
                w[4 + 2 * i] = LD(ca);
                w[5 + 2 * i] = (t.odd && (co[i] & 3u) == 3u) ? LD(ca + 4) : 0u;
            }
        } else if (LINEAR) {
            const uint32_t cn = t.odd;  // offset of the right column's U and V samples
            w[0] = B(s + t.lo) | (B(s + t.lo + 1) << 8);
            w[1] = B(s + t.lo + pitch) | (B(s + t.lo + pitch + 1) << 8);
            w[2] = B(s + t.uo) | (B(s + t.vo) << 8) | (B(s + t.uo + cn) << 16) | (B(s + t.vo + cn) << 24);
            w[3] = B(s + t.uo_b) | (B(s + t.vo_b) << 8) | (B(s + t.uo_b + cn) << 16) | (B(s + t.vo_b + cn) << 24);
        } else if (WORDS) {
            w[0] = LD(s + (t.lo & ~3u));
            w[1] = LD(s + (t.uo & ~3u));
            w[2] = LD(s + (t.vo & ~3u));
        } else {
            w[0] = B(s + t.lo);
            w[1] = B(s + t.uo) | (B(s + t.vo) << 8);
        }
    }
    static __device__ __forceinline__ uint32_t math(const Tap &t, const uint32_t (&w)[kWords], uint32_t bpx)
    {
        if (!LINEAR) {
            const uint32_t Yw = WORDS ? byte_of(w[0], t.lo & 3u) : w[0];
            const uint32_t U = WORDS ? byte_of(w[1], t.uo & 3u) : byte_of(w[1], 0);
            const uint32_t V = WORDS ? byte_of(w[2], t.vo & 3u) : byte_of(w[1], 1);
            return t.k == kInside ? yuv_to_bgr(Yw, U, V) : t.k;
        }
        if (!WORDS) return yuv_lerp(t.w0, t.w1, t.k, bpx, w[0], w[1], w[2], w[3]);
        // [U U' . .] and [V V' . .] of one chroma row -> [U V U' V'] (U V U V when cs is even)
        const uint32_t csel = t.odd ? 0x5140u : 0x4040u;
        const uint32_t U0 = __funnelshift_r(w[4], w[5], 8 * (t.uo & 3u)), V0 = __funnelshift_r(w[6], w[7], 8 * (t.vo & 3u));
        const uint32_t U1 = __funnelshift_r(w[8], w[9], 8 * (t.uo_b & 3u));
        const uint32_t V1 = __funnelshift_r(w[10], w[11], 8 * (t.vo_b & 3u));
        return yuv_lerp(t.w0, t.w1, t.k, bpx, __funnelshift_r(w[0], w[1], 8 * (t.lo & 3u)),
                        __funnelshift_r(w[2], w[3], 8 * (t.lo & 3u)), prmt(U0, V0, csel), prmt(U1, V1, csel));
    }
};

}  // namespace
