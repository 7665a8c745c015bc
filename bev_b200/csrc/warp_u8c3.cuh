// warp_u8c3.cuh -- the per-pixel arithmetic of the uint8 x 3 perspective warp, shared by the staged
// kernel (warp_fast.cu, windows in shared memory) and the direct-gather kernel (warp_generic.cu,
// windows straight from global memory).  Semantics: cv2.warpPerspective 4.13 on BGR frames
// (reference call sites vis_homo.py:89,91), SURVEY.md Appendix A.
#pragma once
#include "bevk_common.cuh"

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    return __byte_perm(a, b, sel);
}
__device__ __forceinline__ void st_stream(uint32_t *p, uint32_t v)
{
    asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// The same streaming store as a compiler intrinsic: no memory clobber, so the gather kernels'
// loads of the NEXT frame may be hoisted above it (their loops live on loads in flight).
__device__ __forceinline__ void st_stream_free(uint32_t *p, uint32_t v) { __stcs(p, v); }

// Read-only word load that asks L2 for a 64-byte fetch instead of the default 128 (measured on
// B200 with a strided probe: a 4-byte ld.global.nc pulls the whole 128-byte line from DRAM, the
// .L2::64B form half of it).  For gathers that use a fraction of every line -- minifying warps.
__device__ __forceinline__ uint32_t ldg_sparse(const uint32_t *p)
{
    uint32_t v;
    asm("ld.global.nc.L2::64B.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// The (matrix, frame-run) group gi that grid z-block z of a direct-gather warp works on.
__device__ __forceinline__ const BevkWarpGroup &find_group(const BevkWarpParams &p, int z, int &gi)
{
    gi = 0;
#pragma unroll 1
    for (int i = 1; i < p.n_groups; ++i)
        if (z >= p.g[i].chunk0) gi = i;
    return p.g[gi];
}

// The dst->src map of this block's group in a device-matrix launch: thread 0 reads the group's
// matrix from the caller's device table when the kernel runs, inverts it with bevk_invert_adj (the
// bits bevk_invert3x3 gives on the host) or takes it as is for WARP_INVERSE_MAP, and shares it
// through sm.  Holds a barrier: every thread of the block calls it, before any thread leaves.
__device__ __forceinline__ const double *dmat_map(const BevkWarpParams &p, double *sm)
{
    if (threadIdx.x == 0 && threadIdx.y == 0) {
        int gi;
        const BevkWarpGroup &g = find_group(p, blockIdx.z, gi);
        double H[9];
#pragma unroll
        for (int i = 0; i < 9; ++i) H[i] = g.d.mat[i];
        if (g.d.invert) {
            bevk_invert_adj(H, sm);
        } else {
#pragma unroll
            for (int i = 0; i < 9; ++i) sm[i] = H[i];
        }
    }
    __syncthreads();
    return sm;
}

// 2-tap window along one axis: first index (clamped into the image) and the weight each of the
// two window positions receives.  Taps outside [0, n) contribute nothing (border value 0).
__device__ __forceinline__ void window(int s, int frac, int n, int &first, int &w0, int &w1)
{
    first = min(max(s, 0), n - 2);
    const int t0 = 32 - frac, t1 = frac;  // weights of taps s and s+1
    w0 = (first == s ? t0 : 0) + (first == s + 1 ? t1 : 0);
    w1 = (first + 1 == s ? t0 : 0) + (first + 1 == s + 1 ? t1 : 0);
}

// Frame-invariant description of one dst pixel.
struct Pix {
    uint32_t addr;   // byte offset (4-aligned) inside a stage of the first window word, row 0
    uint32_t sh;     // 8 * (window start & 3): funnel-shift amount that byte-aligns the window
    uint32_t w0;     // bilinear: the two tap weights of window row 0 as 16-bit halves (dp2a operand)
                     // nearest : 0x00ffffff when the tap is inside the image, else 0
    uint32_t w1;     // the two tap weights of window row 1
};

// cv2's fixed-point weight of one tap, doubled: column weight x row weight (0..32 each, 1/32 px)
// x 64, so that sum(w * p) + 2^15 has the result in byte 2.  32 * 32 * 64 does not fit 16 bits;
// it only occurs when that tap is the pixel's only non-zero one, and 65535 then gives the same
// byte: (65535 p + 32768) >> 16 = p for p <= 255.
__device__ __forceinline__ uint32_t tap_weight(int wc, int wr)
{
    return min((uint32_t)(wc * wr) * 64u, 65535u);
}

// cv2's fixed-point bilinear from gathered taps.  Per window row the channel pairs are gathered
// into xa = [B0 B3 B1 B4], ya = [B2 B5 . .] (row 0) and xb, yb (row 1), B0..B5 being the six bytes
// of the row's two pixels; every channel is then two chained dp2a (row 0, row 1) starting from the
// rounding constant -- no multiplies.  w0 / w1 = the two tap weights of row 0 / 1 as 16-bit halves.
// Result [c0, c1, c2, 0].
__device__ __forceinline__ uint32_t lerp_xy(uint32_t w0, uint32_t w1, uint32_t xa, uint32_t ya, uint32_t xb,
                                            uint32_t yb)
{
    const uint32_t t0 = __dp2a_lo(w1, xb, __dp2a_lo(w0, xa, 32768u));
    const uint32_t t1 = __dp2a_hi(w1, xb, __dp2a_hi(w0, xa, 32768u));
    const uint32_t t2 = __dp2a_lo(w1, yb, __dp2a_lo(w0, ya, 32768u));
    // byte 2 of t is (sum w*p + 2^14) >> 15 in cv2's scale
    return prmt(prmt(t0, t1, 0x4462u), t2, 0x7610u);
}

// One pixel out of its staged window.  f0 / g0 = window bytes 0..3 of row 0 / 1, f1 / g1 = window
// bytes 4.. (already byte-aligned).
__device__ __forceinline__ uint32_t lerp_aligned(const Pix &q, uint32_t f0, uint32_t f1, uint32_t g0,
                                                 uint32_t g1)
{
    return lerp_xy(q.w0, q.w1, prmt(f0, f1, 0x4130u), prmt(f0, f1, 0x0052u), prmt(g0, g1, 0x4130u),
                   prmt(g0, g1, 0x0052u));
}


// ---- the pixel-format policy the staged kernel (warp_fast.cu) is written against ---------------
// uint8 x 3 (BGR video): 3 bytes per pixel; a 2-tap window row is 6 bytes starting on any byte,
// i.e. up to 3 aligned words; 32 pixels are 96 bytes = 24 words.
struct PxU8C3 {
    static constexpr int kBpp = 3;         // bytes per pixel
    static constexpr int kSegBytes = 96;   // bytes of a 32-pixel row segment
    static constexpr int kDtype = BEVK_U8;
    static constexpr int kLinearThreads = 128, kNearestThreads = 256;  // CTA size of the staged kernel (warp_fast.cu)
    static constexpr int kLinearCtas = 6;   // CTAs per SM of the bilinear kernel (bounds its registers)
    static constexpr int kWinWords = 8;     // window words the kernel keeps per pixel
    static constexpr bool kPairs = true;   // the staged kernel's shared-window pair path exists for this format
    using Reg = Pix;
    using Out = uint32_t;                  // [c0, c1, c2, 0]
    struct Store {
        uint32_t sel_pack;  // PRMT selector that packs this lane's word out of (own, next lane's) pixel
    };

    // per-pixel registers from the clamped window: A = byte offset of its first byte inside the
    // stage (or the frame), wc / wr = integer weights (0..32) of the two window columns / rows
    template <bool LINEAR>
    static __device__ __forceinline__ Reg make(bool act, uint32_t A, int wc0, int wc1, int wr0, int wr1)
    {
        Reg q;
        q.addr = A & ~3u;
        q.sh = 8 * (A & 3);
        if (LINEAR) {
            q.w0 = tap_weight(wc0, wr0) | (tap_weight(wc1, wr0) << 16);
            q.w1 = tap_weight(wc0, wr1) | (tap_weight(wc1, wr1) << 16);
        } else {
            q.w0 = act ? 0x00ffffffu : 0u;
            q.w1 = 0;
        }
        return q;
    }
    // the same from the packed integer weights wc0 | wc1 << 8 | wr0 << 16 | wr1 << 24 (0 = inactive)
    template <bool LINEAR> static __device__ __forceinline__ Reg make(bool act, uint32_t A, uint32_t wpk)
    {
        return make<LINEAR>(act, A, (int)(wpk & 0xffu), (int)((wpk >> 8) & 0xffu), (int)((wpk >> 16) & 0xffu),
                            (int)(wpk >> 24));
    }
    // dp2a operands of window rows 0 / 1 from the packed integer weights
    static __device__ __forceinline__ void tap_weights(uint32_t wpk, uint32_t &w0, uint32_t &w1)
    {
        const int wc0 = (int)(wpk & 0xffu), wc1 = (int)((wpk >> 8) & 0xffu);
        const int wr0 = (int)((wpk >> 16) & 0xffu), wr1 = (int)(wpk >> 24);
        w0 = tap_weight(wc0, wr0) | (tap_weight(wc1, wr0) << 16);
        w1 = tap_weight(wc0, wr1) | (tap_weight(wc1, wr1) << 16);
    }
    // window words per row that are always needed / offset of the last one, which only some
    // alignments need (the direct-gather fallback clamps that one into the frame)
    template <bool LINEAR> static constexpr int last_word_offset() { return LINEAR ? 8 : 4; }

    template <bool LINEAR, typename LD>
    static __device__ __forceinline__ void load(const Reg &q, uint32_t ra, uint32_t rb, uint32_t last_a,
                                                uint32_t last_b, uint32_t (&w)[kWinWords], LD ld)
    {
        // ra / rb: address of the first window word in row 0 / 1; last_a / last_b: address of the
        // last word of each row (ra + 8 unless the caller had to clamp it)
        w[0] = ld(ra);
        if (LINEAR) {
            w[1] = ld(ra + 4);
            w[2] = ld(last_a);
            w[3] = ld(rb);
            w[4] = ld(rb + 4);
            w[5] = ld(last_b);
        } else {
            w[1] = ld(last_a);
        }
    }
    template <bool LINEAR>
    static __device__ __forceinline__ Out math(const Reg &q, const uint32_t (&w)[kWinWords])
    {
        if (LINEAR)  // byte-align the window of both rows, then interpolate
            return lerp_aligned(q, __funnelshift_r(w[0], w[1], q.sh), __funnelshift_r(w[1], w[2], q.sh),
                                __funnelshift_r(w[3], w[4], q.sh), __funnelshift_r(w[4], w[5], q.sh));
        return __funnelshift_r(w[0], w[1], q.sh) & q.w0;
    }

    // Lanes 4j..4j+2 write words 3j..3j+2 of a 96-byte segment (32 pixels).
    static __device__ __forceinline__ Store store_setup(int lane)
    {
        const int r4 = lane & 3;
        Store s;
        s.sel_pack = r4 == 0 ? 0x4210u : (r4 == 1 ? 0x5421u : 0x6542u);
        return s;
    }
    static __device__ __forceinline__ uint32_t lane_offset(int lane) { return (3 * (lane >> 2) + (lane & 3)) * 4; }
    // does this lane store for a segment with `valid_px` pixels (a multiple of 4)?
    static __device__ __forceinline__ bool lane_stores(int lane, int valid_px)
    {
        return (lane & 3) < 3 && 4 * (lane >> 2) < valid_px;
    }
    static __device__ __forceinline__ void store(uint8_t *d, Out v, bool ok, const Store &s, int)
    {
        const uint32_t word = prmt(v, __shfl_down_sync(0xffffffffu, v, 1), s.sel_pack);
        if (ok) st_stream(reinterpret_cast<uint32_t *>(d), word);
    }
    static __device__ __forceinline__ void store_zero(uint8_t *d, bool ok, int)
    {
        if (ok) st_stream(reinterpret_cast<uint32_t *>(d), 0u);
    }
};
