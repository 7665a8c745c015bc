// compo.cu -- alpha compositing of BEV frames (sm_100a): the blend of
// bev/tool/compo.py:5-24 (composite_reg_img), the caller of the three warps at compo.py:38,46,47.
//
//     out = uint8(clip(round(fg * (mask / 255) + bg * (1 - mask / 255)), max 255))
//
// The reference evaluates this in numpy float64, element by element, rounding half to even.  With
// k = mask byte the float64 value is within 1e-13 of the rational (fg * k + bg * (255 - k)) / 255,
// whose fractional part is a multiple of 1/255 and therefore never within 1/510 of a tie, so the
// rounded result is exactly
//     (fg * k + bg * (255 - k) + 127) / 255          (integer division)
// for every one of the 2^24 (bg, fg, k) triples (checked exhaustively against the numpy
// expression in tests/test_oracle_compo.py and against the kernel in tests/test_compo_gpu.py).
// The kernels evaluate that with one dot-product instruction per byte and the division as
// ((n + 1) * 0x10101) >> 24, exact for n < 65153.  One pass over the bytes: 3 reads + 1 write per
// output byte, HBM-bound.
// bw_mode (compo.py:13-14): the foreground goes through cv2's BGR -> GRAY -> BGR, i.e.
// gray = (3735 B + 19235 G + 9798 R + 16384) >> 15 (cv2 4.13) replicated into the three channels.
#include "bevk_common.cuh"
#include "warp_u8c3.cuh"
#include <vector>
#include <algorithm>
#include <cstring>

namespace {

// four arbitrary bytes per word (the stand-alone blend)
__device__ __forceinline__ uint32_t blend4(uint32_t bg, uint32_t fg, uint32_t mk)
{
    // mask bytes and their complements as 16-bit lanes: bytes 0, 2 and bytes 1, 3
    const uint32_t k02 = mk & 0x00ff00ffu, k13 = (mk >> 8) & 0x00ff00ffu;
    const uint32_t n02 = k02 ^ 0x00ff00ffu, n13 = k13 ^ 0x00ff00ffu;
    // per byte: (k, 255 - k) . (fg, bg) + 127 + 1, then * 0x10101: the quotient is byte 3
    const uint32_t t0 = __dp2a_lo(prmt(k02, n02, 0x5410u), prmt(fg, bg, 0x0040u), 128u) * 65793u;
    const uint32_t t1 = __dp2a_lo(prmt(k13, n13, 0x5410u), prmt(fg, bg, 0x0051u), 128u) * 65793u;
    const uint32_t t2 = __dp2a_lo(prmt(k02, n02, 0x7632u), prmt(fg, bg, 0x0062u), 128u) * 65793u;
    const uint32_t t3 = __dp2a_lo(prmt(k13, n13, 0x7632u), prmt(fg, bg, 0x0073u), 128u) * 65793u;
    return prmt(prmt(t0, t1, 0x0073u), prmt(t2, t3, 0x0073u), 0x5410u);
}

// one BGR pixel [c0 c1 c2 0] per word (the fused compositor): byte 3 of every operand is zero
__device__ __forceinline__ uint32_t blend_px(uint32_t bg, uint32_t fg, uint32_t mk)
{
    const uint32_t nk = mk ^ 0x00ffffffu;
    const uint32_t t0 = __dp4a(prmt(mk, nk, 0x3340u), prmt(fg, bg, 0x3340u), 128u) * 65793u;
    const uint32_t t1 = __dp4a(prmt(mk, nk, 0x3351u), prmt(fg, bg, 0x3351u), 128u) * 65793u;
    const uint32_t t2 = __dp4a(prmt(mk, nk, 0x3362u), prmt(fg, bg, 0x3362u), 128u) * 65793u;
    return prmt(prmt(t0, t1, 0x0073u), t2, 0x7710u);
}

// cv2.cvtColor(BGR2GRAY) + GRAY2BGR on 4 consecutive BGR pixels held in 3 words
__device__ __forceinline__ void gray3(uint32_t &w0, uint32_t &w1, uint32_t &w2)
{
    uint8_t px[12];
    px[0] = w0; px[1] = w0 >> 8; px[2] = w0 >> 16; px[3] = w0 >> 24;
    px[4] = w1; px[5] = w1 >> 8; px[6] = w1 >> 16; px[7] = w1 >> 24;
    px[8] = w2; px[9] = w2 >> 8; px[10] = w2 >> 16; px[11] = w2 >> 24;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t y = (3735u * px[3 * i] + 19235u * px[3 * i + 1] + 9798u * px[3 * i + 2] + 16384u) >> 15;
        px[3 * i] = px[3 * i + 1] = px[3 * i + 2] = (uint8_t)y;
    }
    w0 = px[0] | (px[1] << 8) | (px[2] << 16) | ((uint32_t)px[3] << 24);
    w1 = px[4] | (px[5] << 8) | (px[6] << 16) | ((uint32_t)px[7] << 24);
    w2 = px[8] | (px[9] << 8) | (px[10] << 16) | ((uint32_t)px[11] << 24);
}

// n12 = number of 12-byte groups (4 BGR pixels), tail_px = pixels after them (< 4); the buffers
// are 4-byte aligned
template <bool BW>
__global__ void __launch_bounds__(256) composite_kernel(const uint32_t *__restrict__ bg,
                                                        const uint32_t *__restrict__ fg,
                                                        const uint32_t *__restrict__ mk,
                                                        uint32_t *__restrict__ out, long long n12,
                                                        int tail_px)
{
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n12;
         i += (long long)gridDim.x * blockDim.x) {
        uint32_t f0 = __ldg(fg + 3 * i), f1 = __ldg(fg + 3 * i + 1), f2 = __ldg(fg + 3 * i + 2);
        if (BW) gray3(f0, f1, f2);
        const uint32_t o0 = blend4(__ldg(bg + 3 * i), f0, __ldg(mk + 3 * i));
        const uint32_t o1 = blend4(__ldg(bg + 3 * i + 1), f1, __ldg(mk + 3 * i + 1));
        const uint32_t o2 = blend4(__ldg(bg + 3 * i + 2), f2, __ldg(mk + 3 * i + 2));
        out[3 * i] = o0;
        out[3 * i + 1] = o1;
        out[3 * i + 2] = o2;
    }
    if (blockIdx.x == 0 && (int)threadIdx.x < tail_px) {  // the last 1..3 pixels, byte by byte
        const long long o = 12 * n12 + 3 * threadIdx.x;
        const uint8_t *b8 = (const uint8_t *)bg + o, *f8 = (const uint8_t *)fg + o, *m8 = (const uint8_t *)mk + o;
        uint32_t f = f8[0] | (f8[1] << 8) | (f8[2] << 16);
        if (BW) {
            const uint32_t y = (3735u * f8[0] + 19235u * f8[1] + 9798u * f8[2] + 16384u) >> 15;
            f = y * 0x010101u;
        }
        const uint32_t r = blend4(b8[0] | (b8[1] << 8) | (b8[2] << 16), f, m8[0] | (m8[1] << 8) | (m8[2] << 16));
        uint8_t *o8 = (uint8_t *)out + o;
        o8[0] = (uint8_t)r;
        o8[1] = (uint8_t)(r >> 8);
        o8[2] = (uint8_t)(r >> 16);
    }
}


// ---- fused BEV compositor ------------------------------------------------------------------------
// composite_bev_img (bev/tool/compo.py:26-50) in ONE pass: per dst pixel the background window is
// gathered through the fixed camera's homography, the foreground and mask windows through the
// rendering camera's, all three are interpolated with cv2's fixed-point bilinear (warp_u8c3.cuh)
// and blended in registers.  Against the unfused route (three warped BEVs written, read back by the
// blend) the output is written once and nothing intermediate touches HBM.  A run of frames that
// shares its homographies keeps the quantised coordinates in registers across the run; a shared
// background frame is interpolated once per run.
constexpr int kCompoGroups = 32;

struct CompoGroup {
    // dst -> src maps of the background / foreground (inverted on the host), or in device-matrix
    // launches (bevk_composite_bev_u8c3_dmat) the group's forward matrices in device memory
    union {
        double Mb[9];
        const double *Hb;
    };
    union {
        double Mf[9];
        const double *Hf;
    };
    int first, count;     // frames first .. first + count - 1
    int chunk0;           // first z-block of the group
    int pad;
};

struct CompoParams {
    const uint8_t *bg, *fg, *mk;
    uint8_t *out;
    int bg_h, bg_w, fg_h, fg_w, dst_h, dst_w;
    uint32_t bg_frame, fg_frame;  // bytes per source frame
    long long dst_frame;
    int bg_shared;                // one background frame for every composite
    int bw0, frames_per_chunk, n_groups;
    CompoGroup g[kCompoGroups];
};

struct Gather {
    Pix q;
    uint32_t off2, row_bytes;
};

__device__ __forceinline__ Gather make_gather(const double *M, int x, int y, int bw0, int src_w,
                                              int src_h, uint32_t frame_bytes)
{
    int X, Y, cs, rs, wc0, wc1, wr0, wr1;
    bevk_map_pixel(M, x, y, bw0, 32.0, X, Y);
    window(bevk_sat16(X >> 5), X & 31, src_w, cs, wc0, wc1);
    window(bevk_sat16(Y >> 5), Y & 31, src_h, rs, wr0, wr1);
    const bool act = (wc0 | wc1) != 0 && (wr0 | wr1) != 0;
    Gather t;
    t.row_bytes = (uint32_t)src_w * 3u;
    const uint32_t A = act ? (uint32_t)rs * t.row_bytes + 3u * (uint32_t)cs : 0u;
    t.q = PxU8C3::make<true>(act, A, act ? wc0 : 0, act ? wc1 : 0, wr0, wr1);
    // the third window word is only used by some alignments: keep its address inside the frame
    t.off2 = min(t.q.addr + 8u, frame_bytes - 4u - t.row_bytes);
    return t;
}

// the six words of a pixel's 2 x 2 window (three aligned words per window row)
__device__ __forceinline__ void gather_load(const Gather &t, const uint8_t *s, uint32_t (&w)[6])
{
    const uint8_t *ra = s + t.q.addr, *rb = ra + t.row_bytes;
    w[0] = __ldg((const uint32_t *)ra);
    w[1] = __ldg((const uint32_t *)(ra + 4));
    w[2] = __ldg((const uint32_t *)(s + t.off2));
    w[3] = __ldg((const uint32_t *)rb);
    w[4] = __ldg((const uint32_t *)(rb + 4));
    w[5] = __ldg((const uint32_t *)(s + t.off2 + t.row_bytes));
}
__device__ __forceinline__ uint32_t gather_math(const Gather &t, const uint32_t (&w)[6])
{
    return lerp_aligned(t.q, __funnelshift_r(w[0], w[1], t.q.sh), __funnelshift_r(w[1], w[2], t.q.sh),
                        __funnelshift_r(w[3], w[4], t.q.sh), __funnelshift_r(w[4], w[5], t.q.sh));
}
__device__ __forceinline__ uint32_t gather_pixel(const Gather &t, const uint8_t *s)
{
    uint32_t w[6];
    gather_load(t, s, w);
    return gather_math(t, w);
}

// The group of this block's z-chunk.  DMAT blocks search with all loads in flight at once: the
// search lies on their critical path, in front of the matrix loads and the barrier (DESIGN 3.13).
// The host-matrix instances keep the serial loop they were tuned and measured with.
template <bool DMAT>
__device__ __forceinline__ const CompoGroup &compo_group(const CompoParams &p)
{
    int gi = 0;
    if constexpr (DMAT) {
        if (p.n_groups > 1) {
#pragma unroll
            for (int i = 1; i < kCompoGroups; ++i)
                if (i < p.n_groups && (int)blockIdx.z >= p.g[i].chunk0) gi = i;
        }
    } else {
#pragma unroll 1
        for (int i = 1; i < p.n_groups; ++i)
            if ((int)blockIdx.z >= p.g[i].chunk0) gi = i;
    }
    return p.g[gi];
}

// DMAT: the group holds device addresses of its forward matrices (CompoGroup::Hb / Hf).  Every
// thread finds the group; threads 0 and 1 of the block each read one of the matrices when the kernel
// runs, invert it with bevk_invert_adj (the bits bevk_invert3x3 gives on the host; a singular matrix
// gives the zero map) and share the map through shared memory behind one barrier, which every
// thread reaches before any thread leaves.
template <int kBatch, bool DMAT>
__global__ void __launch_bounds__(256) composite_bev_kernel(const __grid_constant__ CompoParams p)
{
    const double *dm = nullptr;        // DMAT: the background map, then the foreground map
    const CompoGroup *dg = nullptr;    // DMAT: the block's group
    if constexpr (DMAT) {
        __shared__ double sm[18];
        dg = &compo_group<true>(p);
        const int t = threadIdx.y * 32 + threadIdx.x;
        if (t < 2) {
            const double *H = t ? dg->Hf : dg->Hb;
            double h[9];
#pragma unroll
            for (int i = 0; i < 9; ++i) h[i] = H[i];
            bevk_invert_adj(h, sm + 9 * t);
        }
        __syncthreads();
        dm = sm;
    }
    const int lane = threadIdx.x, x0 = blockIdx.x * 32;
    const int x = x0 + lane, y = blockIdx.y * 8 + threadIdx.y;
    if (y >= p.dst_h) return;  // a warp is one dst row segment: uniform exit
    const CompoGroup &g = DMAT ? *dg : compo_group<false>(p);
    const int f0 = ((int)blockIdx.z - g.chunk0) * p.frames_per_chunk;
    const int f1 = min(f0 + p.frames_per_chunk, g.count);

    const int xc = min(x, p.dst_w - 1);
    const Gather tb = make_gather(DMAT ? dm : g.Mb, xc, y, p.bw0, p.bg_w, p.bg_h, p.bg_frame);
    const Gather tf = make_gather(DMAT ? dm + 9 : g.Mf, xc, y, p.bw0, p.fg_w, p.fg_h, p.fg_frame);

    const int j = lane >> 2, r4 = lane & 3;
    const uint32_t sel_pack = r4 == 0 ? 0x4210u : (r4 == 1 ? 0x5421u : 0x6542u);
    const bool st_ok = r4 < 3 && 4 * j < min(32, p.dst_w - x0);  // dst_w % 4 == 0
    uint8_t *dst = p.out + ((long long)y * p.dst_w + x0) * 3 + (3 * j + r4) * 4;

    // The loop lives on loads in flight (L1 gathers, ~60 % of its stall cycles are scoreboard
    // waits): the windows of kBatch frames are requested before the first one is used.
    uint32_t B = p.bg_shared ? gather_pixel(tb, p.bg) : 0u;
    int f = f0;
    for (; f + kBatch <= f1; f += kBatch) {
        uint32_t wf[kBatch][6], wk[kBatch][6], wb[kBatch][6];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) {
            const long long fr = g.first + f + u;
            gather_load(tf, p.fg + fr * p.fg_frame, wf[u]);
            gather_load(tf, p.mk + fr * p.fg_frame, wk[u]);
            if (!p.bg_shared) gather_load(tb, p.bg + fr * p.bg_frame, wb[u]);
        }
#pragma unroll
        for (int u = 0; u < kBatch; ++u) {
            const long long fr = g.first + f + u;
            if (!p.bg_shared) B = gather_math(tb, wb[u]);
            const uint32_t P = blend_px(B, gather_math(tf, wf[u]), gather_math(tf, wk[u]));
            const uint32_t word = prmt(P, __shfl_down_sync(0xffffffffu, P, 1), sel_pack);
            if (st_ok) st_stream_free(reinterpret_cast<uint32_t *>(dst + fr * p.dst_frame), word);
        }
    }
    for (; f < f1; ++f) {
        const long long fr = g.first + f;
        if (!p.bg_shared) B = gather_pixel(tb, p.bg + fr * p.bg_frame);
        const uint32_t P = blend_px(B, gather_pixel(tf, p.fg + fr * p.fg_frame), gather_pixel(tf, p.mk + fr * p.fg_frame));
        const uint32_t word = prmt(P, __shfl_down_sync(0xffffffffu, P, 1), sel_pack);
        if (st_ok) st_stream_free(reinterpret_cast<uint32_t *>(dst + fr * p.dst_frame), word);
    }
}

}  // namespace

extern "C" int bevk_composite_u8c3(const void *bg, const void *fg, const void *fg_mask, void *out,
                                   int64_t n_pixels, int bw_mode, void *stream)
{
    int rc = bevk_require_device();
    if (rc) return rc;
    if (n_pixels < 0) BEVK_FAIL(BEVK_E_ARG, "bevk_composite_u8c3: n_pixels must be >= 0");
    if (n_pixels == 0) return BEVK_OK;
    if (!bg || !fg || !fg_mask || !out) BEVK_FAIL(BEVK_E_ARG, "bevk_composite_u8c3: null buffer");
    if (((uintptr_t)bg | (uintptr_t)fg | (uintptr_t)fg_mask | (uintptr_t)out) % 4 != 0)
        BEVK_FAIL(BEVK_E_ARG, "bevk_composite_u8c3: buffers must be 4-byte aligned");
    const long long n12 = n_pixels / 4;
    const int tail_px = (int)(n_pixels % 4);
    long long want = (n12 + 255) / 256;
    const long long cap = (long long)bevk_sm_count() * 8;
    want = want < 1 ? 1 : want;
    const int grid = (int)(want < cap ? want : cap);
    cudaStream_t st = (cudaStream_t)stream;
    if (bw_mode)
        composite_kernel<true><<<grid, 256, 0, st>>>((const uint32_t *)bg, (const uint32_t *)fg,
                                                     (const uint32_t *)fg_mask, (uint32_t *)out, n12, tail_px);
    else
        composite_kernel<false><<<grid, 256, 0, st>>>((const uint32_t *)bg, (const uint32_t *)fg,
                                                      (const uint32_t *)fg_mask, (uint32_t *)out, n12, tail_px);
    BEVK_CUDA(cudaGetLastError());
    return BEVK_OK;
}


namespace {

// The fused compositor with host matrices (inverted here) or, dmat, device matrices (read and
// inverted by the kernels when they run).  Both plan runs, groups and frame chunks alike.
int composite_bev(const void *bg, const void *fg, const void *fg_mask, void *out, int n_frames, int n_bg, int bg_h,
                  int bg_w, int fg_h, int fg_w, int dst_h, int dst_w, const double *H_bg, const double *H_fg,
                  int n_mats, bool dmat, void *stream)
{
    if (n_frames < 0) BEVK_FAIL(BEVK_E_ARG, "composite_bev: n_frames must be >= 0");
    if (bg_h < 2 || bg_w < 2 || fg_h < 2 || fg_w < 2 || dst_h <= 0 || dst_w <= 0)
        BEVK_FAIL(BEVK_E_ARG, "composite_bev: sources must be at least 2x2 and the BEV non-empty");
    if (bg_h > 32767 || bg_w > 32767 || fg_h > 32767 || fg_w > 32767 || dst_h > 32767 || dst_w > 32767)
        BEVK_FAIL(BEVK_E_ARG, "composite_bev: sizes above 32767 are not supported (cv2 SHRT_MAX limit)");
    if ((bg_w % 4) != 0 || (fg_w % 4) != 0 || (dst_w % 4) != 0)
        BEVK_FAIL(BEVK_E_ARG, "composite_bev: widths must be multiples of 4 (bg %d, fg %d, bev %d); "
                              "use bevk_warp_perspective + bevk_composite_u8c3 otherwise",
                  bg_w, fg_w, dst_w);
    if (n_bg != 1 && n_bg != n_frames)
        BEVK_FAIL(BEVK_E_ARG, "composite_bev: %d backgrounds for %d frames (need 1 or one each)", n_bg, n_frames);
    if (!H_bg || !H_fg || (n_mats != 1 && n_mats != n_frames))
        BEVK_FAIL(BEVK_E_ARG, "composite_bev: need 1 or n_frames homography pairs, got %d", n_mats);
    int rc = bevk_require_device();
    if (rc) return rc;
    if (n_frames == 0) return BEVK_OK;
    if (!bg || !fg || !fg_mask || !out) BEVK_FAIL(BEVK_E_ARG, "composite_bev: null buffer");
    if (((uintptr_t)bg | (uintptr_t)fg | (uintptr_t)fg_mask | (uintptr_t)out) % 4 != 0)
        BEVK_FAIL(BEVK_E_ARG, "composite_bev: buffers must be 4-byte aligned");

    CompoParams p;
    memset(&p, 0, sizeof(p));
    p.bg = (const uint8_t *)bg;
    p.fg = (const uint8_t *)fg;
    p.mk = (const uint8_t *)fg_mask;
    p.out = (uint8_t *)out;
    p.bg_h = bg_h;
    p.bg_w = bg_w;
    p.fg_h = fg_h;
    p.fg_w = fg_w;
    p.dst_h = dst_h;
    p.dst_w = dst_w;
    p.bg_frame = (uint32_t)bg_h * bg_w * 3u;
    p.fg_frame = (uint32_t)fg_h * fg_w * 3u;
    p.dst_frame = (long long)dst_h * dst_w * 3;
    p.bg_shared = n_bg == 1;
    p.bw0 = bevk_block_width(dst_w, dst_h);

    // runs of frames sharing one homography pair: all of them, or one frame each
    const int n_runs = n_mats == 1 ? 1 : n_frames;
    const long long tiles = (long long)((dst_w + 31) / 32) * ((dst_h + 7) / 8);
    const long long want_blocks = (long long)bevk_sm_count() * 8 * 2;
    cudaStream_t st = (cudaStream_t)stream;
    for (int r0 = 0; r0 < n_runs; r0 += kCompoGroups) {
        const int ng = std::min(kCompoGroups, n_runs - r0);
        const int count = n_mats == 1 ? n_frames : 1;
        int fpc = std::min(count, 64);
        while (fpc > 1 && tiles * ng * ((count + fpc - 1) / fpc) < want_blocks) fpc = (fpc + 1) / 2;
        int z = 0;
        for (int i = 0; i < ng; ++i) {
            CompoGroup &g = p.g[i];
            const size_t k = (size_t)(r0 + i) * 9;
            if (dmat) {
                g.Hb = H_bg + k;
                g.Hf = H_fg + k;
            } else {
                bevk_invert3x3(H_bg + k, g.Mb);  // cv2 inverts a forward matrix
                bevk_invert3x3(H_fg + k, g.Mf);
            }
            g.first = n_mats == 1 ? 0 : r0 + i;
            g.count = count;
            g.chunk0 = z;
            z += (count + fpc - 1) / fpc;
        }
        p.n_groups = ng;
        p.frames_per_chunk = fpc;
        if (z > 65535) BEVK_FAIL(BEVK_E_ARG, "composite_bev: too many frame chunks (%d) for one launch", z);
        dim3 block(32, 8, 1), grid((dst_w + 31) / 32, (dst_h + 7) / 8, z);
        // two frames of windows in flight per thread when runs are long enough to use them; the
        // one-frame build keeps more warps resident for the coordinate-bound camera-per-frame case
        if (dmat)
            fpc >= 2 ? composite_bev_kernel<2, true><<<grid, block, 0, st>>>(p)
                     : composite_bev_kernel<1, true><<<grid, block, 0, st>>>(p);
        else if (fpc >= 2)
            composite_bev_kernel<2, false><<<grid, block, 0, st>>>(p);
        else
            composite_bev_kernel<1, false><<<grid, block, 0, st>>>(p);
        BEVK_CUDA(cudaGetLastError());
    }
    return BEVK_OK;
}

}  // namespace

extern "C" int bevk_composite_bev_u8c3(const void *bg, const void *fg, const void *fg_mask, void *out,
                                       int n_frames, int n_bg, int bg_h, int bg_w, int fg_h, int fg_w,
                                       int dst_h, int dst_w, const double *H_bg, const double *H_fg,
                                       int n_mats, void *stream)
{
    return composite_bev(bg, fg, fg_mask, out, n_frames, n_bg, bg_h, bg_w, fg_h, fg_w, dst_h, dst_w, H_bg, H_fg,
                         n_mats, false, stream);
}

extern "C" int bevk_composite_bev_u8c3_dmat(const void *bg, const void *fg, const void *fg_mask, void *out,
                                            int n_frames, int n_bg, int bg_h, int bg_w, int fg_h, int fg_w,
                                            int dst_h, int dst_w, const double *H_bg, const double *H_fg,
                                            int n_mats, void *stream)
{
    return composite_bev(bg, fg, fg_mask, out, n_frames, n_bg, bg_h, bg_w, fg_h, fg_w, dst_h, dst_w, H_bg, H_fg,
                         n_mats, true, stream);
}
