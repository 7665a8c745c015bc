// warp_f16c3.cuh -- float16 x 3 pixel-format policy of the staged warp kernel (warp_fast.cu).
//
// cv2.warpPerspective has no float16 path (SURVEY.md 0.4); the contract is
// float16(cv2_float32(float32(src))), i.e. cv2's float32 interpolation on the upcast taps, rounded
// once to half.  cv2's float path (SURVEY.md Appendix A): tx = ax / 32, ty = ay / 32 in fp32,
// w00 = (1-ty)(1-tx), w01 = (1-ty) tx, w10 = ty (1-tx), w11 = ty tx, and
//     dst = ((p00 w00 + p01 w01) + p10 w10) + p11 w11        -- fp32, left to right, never fused.
// A pixel is 6 bytes; a 2-tap window row is 12 bytes starting on any even byte, i.e. up to 4 aligned
// words; 32 pixels are 192 bytes = 48 words.  Out-of-image taps carry weight 0 and a clamped
// address (value * 0 = 0 for every finite neighbour; the direct-gather kernel is the exact path
// for frames that hold Inf / NaN next to the image border).  A pixel with no tap inside the image
// is written as +0, the border value cv2 writes: its sum of zero-weighted negative taps is -0.
#pragma once
#include "bevk_common.cuh"
#include "warp_u8c3.cuh"  // prmt, st_stream

struct PixF16 {
    uint32_t addr;  // byte offset (4-aligned) of the first window word, row 0
    uint32_t sh;    // 0 or 16: the window starts on the low / high half of that word
    uint32_t keep;  // all ones if any tap is inside the image, else 0 (ANDed onto the bilinear result)
    float w00, w01, w10, w11;  // bilinear weights of the window positions; nearest: w00 = 1 or 0
};

struct PxF16C3 {
    static constexpr int kBpp = 6;
    static constexpr int kSegBytes = 192;
    static constexpr int kDtype = BEVK_F16;
    static constexpr int kLinearThreads = 128, kNearestThreads = 256;  // CTA size of the staged kernel (warp_fast.cu)
    static constexpr int kLinearCtas = 4;   // CTAs per SM of the bilinear kernel (bounds its registers)
    static constexpr int kWinWords = 8;     // window words the kernel keeps per pixel
    static constexpr bool kPairs = false;
    using Reg = PixF16;
    struct Out {
        uint32_t x, y;  // halves [c0, c1], [c2, -]
    };
    struct Store {
        uint32_t sel1;  // even lane: its [c0 c1]; odd lane: its [c1 c2]
        bool even;
    };

    template <bool LINEAR>
    static __device__ __forceinline__ Reg make(bool act, uint32_t A, int wc0, int wc1, int wr0, int wr1)
    {
        Reg q;
        q.addr = A & ~3u;
        q.sh = 8 * (A & 3);  // A is even: 0 or 16
        q.keep = act ? 0xffffffffu : 0u;
        if (LINEAR) {
            // wc / wr are 32 - frac, frac or 0: dividing by 32 is exact, so c0 = 1 - tx, c1 = tx ...
            const float c0 = __fmul_rn((float)wc0, 1.0f / 32.0f), c1 = __fmul_rn((float)wc1, 1.0f / 32.0f);
            const float r0 = __fmul_rn((float)wr0, 1.0f / 32.0f), r1 = __fmul_rn((float)wr1, 1.0f / 32.0f);
            q.w00 = __fmul_rn(r0, c0);
            q.w01 = __fmul_rn(r0, c1);
            q.w10 = __fmul_rn(r1, c0);
            q.w11 = __fmul_rn(r1, c1);
        } else {
            q.w00 = act ? 1.0f : 0.0f;
            q.w01 = q.w10 = q.w11 = 0.0f;
        }
        return q;
    }
    template <bool LINEAR> static __device__ __forceinline__ Reg make(bool act, uint32_t A, uint32_t wpk)
    {
        return make<LINEAR>(act, A, (int)(wpk & 0xffu), (int)((wpk >> 8) & 0xffu), (int)((wpk >> 16) & 0xffu),
                            (int)(wpk >> 24));
    }
    // bilinear: 12 window bytes from an even offset span 4 words when the offset is 2 (mod 4);
    // nearest: 6 bytes always fit two words
    template <bool LINEAR> static constexpr int last_word_offset() { return LINEAR ? 12 : 4; }

    template <bool LINEAR, typename LD>
    static __device__ __forceinline__ void load(const Reg &, uint32_t ra, uint32_t rb, uint32_t last_a,
                                                uint32_t last_b, uint32_t (&w)[kWinWords], LD ld)
    {
        w[0] = ld(ra);
        if (LINEAR) {
            w[1] = ld(ra + 4);
            w[2] = ld(ra + 8);
            w[3] = ld(last_a);
            w[4] = ld(rb);
            w[5] = ld(rb + 4);
            w[6] = ld(rb + 8);
            w[7] = ld(last_b);
        } else {
            w[1] = ld(last_a);
        }
    }
    static __device__ __forceinline__ float lo(uint32_t v) { return __half2float(__ushort_as_half((unsigned short)(v & 0xffffu))); }
    static __device__ __forceinline__ float hi(uint32_t v) { return __half2float(__ushort_as_half((unsigned short)(v >> 16))); }
    static __device__ __forceinline__ float blend(const Reg &q, float p00, float p01, float p10, float p11)
    {
        // cv2: ((p00 w00 + p01 w01) + p10 w10) + p11 w11 with every operation rounded.  A tap is a
        // half (11 significant bits) and a weight a product of two 5-bit fractions (10 bits), so
        // every product is exact in float32 and only the additions round: fma(p, w, acc) =
        // round(p w + acc) is bit-identical to add(mul(p, w), acc), at 4 instructions instead of 7.
        float r = __fmaf_rn(p01, q.w01, __fmul_rn(p00, q.w00));
        r = __fmaf_rn(p10, q.w10, r);
        return __fmaf_rn(p11, q.w11, r);
    }
    template <bool LINEAR>
    static __device__ __forceinline__ Out math(const Reg &q, const uint32_t (&w)[kWinWords])
    {
        Out o;
        if (LINEAR) {
            // half-align both rows: a = [t0c0 t0c1] [t0c2 t1c0] [t1c1 t1c2]
            const uint32_t a0 = __funnelshift_r(w[0], w[1], q.sh), a1 = __funnelshift_r(w[1], w[2], q.sh);
            const uint32_t a2 = __funnelshift_r(w[2], w[3], q.sh);
            const uint32_t b0 = __funnelshift_r(w[4], w[5], q.sh), b1 = __funnelshift_r(w[5], w[6], q.sh);
            const uint32_t b2 = __funnelshift_r(w[6], w[7], q.sh);
            const float c0 = blend(q, lo(a0), hi(a1), lo(b0), hi(b1));
            const float c1 = blend(q, hi(a0), lo(a2), hi(b0), lo(b2));
            const float c2 = blend(q, lo(a1), hi(a2), lo(b1), hi(b2));
            const __half2 h01 = __floats2half2_rn(c0, c1);
            o.x = *reinterpret_cast<const uint32_t *>(&h01) & q.keep;
            o.y = (uint32_t)__half_as_ushort(__float2half_rn(c2)) & q.keep;
        } else {
            const uint32_t a0 = __funnelshift_r(w[0], w[1], q.sh);
            const uint32_t a1 = __funnelshift_r(w[1], 0u, q.sh) & 0xffffu;
            const bool in = q.w00 != 0.0f;
            o.x = in ? a0 : 0u;
            o.y = in ? a1 : 0u;
        }
        return o;
    }

    // Lanes 2j, 2j+1 hold pixels 2j, 2j+1 = words 3j..3j+2 of the 192-byte segment:
    //   even lane: word 3j = [c0 c1], word 3j+1 = [c2, c0 of the odd lane];  odd lane: word 3j+2 = [c1 c2].
    static __device__ __forceinline__ Store store_setup(int lane)
    {
        Store s;
        s.even = (lane & 1) == 0;
        s.sel1 = s.even ? 0x3210u : 0x5432u;
        return s;
    }
    static __device__ __forceinline__ uint32_t lane_offset(int lane) { return (3 * (lane >> 1) + 2 * (lane & 1)) * 4; }
    static __device__ __forceinline__ bool lane_stores(int lane, int valid_px) { return (lane & ~1) < valid_px; }
    static __device__ __forceinline__ void store(uint8_t *d, Out v, bool ok, const Store &s, int)
    {
        const uint32_t next = __shfl_down_sync(0xffffffffu, v.x, 1);
        const uint32_t w1 = prmt(v.x, v.y, s.sel1);
        const uint32_t w2 = prmt(v.y, next, 0x5410u);
        if (ok) st_stream(reinterpret_cast<uint32_t *>(d), w1);
        if (ok && s.even) st_stream(reinterpret_cast<uint32_t *>(d + 4), w2);
    }
    static __device__ __forceinline__ void store_zero(uint8_t *d, bool ok, int lane)
    {
        if (ok) st_stream(reinterpret_cast<uint32_t *>(d), 0u);
        if (ok && (lane & 1) == 0) st_stream(reinterpret_cast<uint32_t *>(d + 4), 0u);
    }
};
