// warp_generic.cu -- direct-gather perspective warp for every dtype / channel count / border
// value.  It is the catch-all behind bevk_warp_perspective: shapes the staged fast path
// (warp_fast.cu) does not take land here.  One thread owns one dst pixel position, computes its
// quantised source coordinate ONCE (FP64, the expensive part) and then loops over the frames of
// its chunk, so the coordinate cost is amortised over the batch.
//
// Semantics: cv2.warpPerspective 4.13 (reference call sites vis_homo.py:89,91,
// bev/tool/compo.py:38,46,47), restated in SURVEY.md Appendix A.
#include "bevk_common.cuh"
#include "warp_u8c3.cuh"

namespace {

template <typename T> struct Px;
template <> struct Px<uint8_t> {
    static __device__ __forceinline__ float ld(const uint8_t *p) { return (float)__ldg(p); }
};
template <> struct Px<__half> {
    static __device__ __forceinline__ float ld(const __half *p) { return __half2float(__ldg(p)); }
};
template <> struct Px<float> {
    static __device__ __forceinline__ float ld(const float *p) { return __ldg(p); }
};

// Second half of a split launch (BevkWarpParams::hard): is this 32x8 block's staged tile unmarked,
// i.e. already written by the staged kernel?  Block-uniform.
__device__ __forceinline__ bool skip_block(const BevkWarpParams &p, int gi)
{
    return p.hard && !p.hard[gi * p.hard_tiles + (int)(blockIdx.x * 32) / p.hard_tw * p.hard_ty +
                             (int)(blockIdx.y * 8) / p.hard_th];
}

__device__ __forceinline__ uint8_t border_u8(float b)
{
    // cv2: saturate_cast<uchar>(borderValue[c])
    int v = __float2int_rn(b);
    return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// ---- bilinear ---------------------------------------------------------------------------------
template <typename T, int C>
__global__ void __launch_bounds__(256) warp_linear_kernel(const __grid_constant__ BevkWarpParams p)
{
    const int x = blockIdx.x * 32 + threadIdx.x;
    const int y = blockIdx.y * 8 + threadIdx.y;
    if (x >= p.dst_w || y >= p.dst_h) return;
    int gi;
    const BevkWarpGroup &g = find_group(p, blockIdx.z, gi);
    if (skip_block(p, gi)) return;
    const int c_local = blockIdx.z - g.chunk0;
    const int f0 = c_local * p.frames_per_chunk;
    const int f1 = min(f0 + p.frames_per_chunk, g.count);

    int X, Y;
    bevk_map_pixel(g.M, x, y, p.bw0, 32.0, X, Y);
    const int sx = bevk_sat16(X >> 5), sy = bevk_sat16(Y >> 5);
    const int ax = X & 31, ay = Y & 31;
    const bool cx0 = (sx >= 0 && sx < p.src_w), cx1 = (sx + 1 >= 0 && sx + 1 < p.src_w);
    const bool cy0 = (sy >= 0 && sy < p.src_h), cy1 = (sy + 1 >= 0 && sy + 1 < p.src_h);
    const bool in00 = cx0 && cy0, in01 = cx1 && cy0, in10 = cx0 && cy1, in11 = cx1 && cy1;
    // element offsets inside a frame (only dereferenced when the tap is in range)
    const long long o00 = ((long long)sy * p.src_w + sx) * C;
    const long long o01 = o00 + C, o10 = o00 + (long long)p.src_w * C, o11 = o10 + C;
    const long long od = ((long long)y * p.dst_w + x) * C;

    const T *src = (const T *)p.src;
    T *dst = (T *)p.dst;

    if constexpr (sizeof(T) == 1) {
        const int w00 = (32 - ax) * (32 - ay) * 32, w01 = ax * (32 - ay) * 32;
        const int w10 = (32 - ax) * ay * 32, w11 = ax * ay * 32;
        int bconst[C];  // contribution of out-of-range taps (+ rounding), frame invariant
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int bv = border_u8(p.border[c]);
            bconst[c] = 16384 + bv * ((in00 ? 0 : w00) + (in01 ? 0 : w01) + (in10 ? 0 : w10) +
                                      (in11 ? 0 : w11));
        }
        const int v00 = in00 ? w00 : 0, v01 = in01 ? w01 : 0, v10 = in10 ? w10 : 0,
                  v11 = in11 ? w11 : 0;
        for (int f = f0; f < f1; ++f) {
            const long long fr = (long long)(g.first + f * g.stride);
            const uint8_t *s = (const uint8_t *)src + fr * p.src_frame_elems;
            uint8_t *d = (uint8_t *)dst + fr * p.dst_frame_elems + od;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                int acc = bconst[c];
                if (in00) acc += v00 * (int)__ldg(s + o00 + c);
                if (in01) acc += v01 * (int)__ldg(s + o01 + c);
                if (in10) acc += v10 * (int)__ldg(s + o10 + c);
                if (in11) acc += v11 * (int)__ldg(s + o11 + c);
                d[c] = (uint8_t)(acc >> 15);
            }
        }
    } else {
        // cv2's float path: weights in fp32, products summed left to right, never fused
        const float tx = __fmul_rn((float)ax, 1.0f / 32.0f), ty = __fmul_rn((float)ay, 1.0f / 32.0f);
        const float omx = __fsub_rn(1.0f, tx), omy = __fsub_rn(1.0f, ty);
        const float w00 = __fmul_rn(omy, omx), w01 = __fmul_rn(omy, tx);
        const float w10 = __fmul_rn(ty, omx), w11 = __fmul_rn(ty, tx);
        if (!(in00 || in01 || in10 || in11)) {
            // no tap inside: cv2 stores the border value itself, not the weighted sum of four
            // copies of it (which can miss it by an ulp)
            for (int f = f0; f < f1; ++f) {
                const long long fr = (long long)(g.first + f * g.stride);
                T *d = dst + fr * p.dst_frame_elems + od;
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    if constexpr (sizeof(T) == 2)
                        d[c] = __float2half_rn(p.border[c]);
                    else
                        d[c] = p.border[c];
                }
            }
            return;
        }
        for (int f = f0; f < f1; ++f) {
            const long long fr = (long long)(g.first + f * g.stride);
            const T *s = src + fr * p.src_frame_elems;
            T *d = dst + fr * p.dst_frame_elems + od;
#pragma unroll
            for (int c = 0; c < C; ++c) {
                const float bv = p.border[c];
                const float p00 = in00 ? Px<T>::ld(s + o00 + c) : bv;
                const float p01 = in01 ? Px<T>::ld(s + o01 + c) : bv;
                const float p10 = in10 ? Px<T>::ld(s + o10 + c) : bv;
                const float p11 = in11 ? Px<T>::ld(s + o11 + c) : bv;
                float r = __fadd_rn(__fmul_rn(p00, w00), __fmul_rn(p01, w01));
                r = __fadd_rn(r, __fmul_rn(p10, w10));
                r = __fadd_rn(r, __fmul_rn(p11, w11));
                if constexpr (sizeof(T) == 2)
                    d[c] = __float2half_rn(r);
                else
                    d[c] = r;
            }
        }
    }
}

// ---- nearest ----------------------------------------------------------------------------------
template <typename T, int C>
__global__ void __launch_bounds__(256) warp_nearest_kernel(const __grid_constant__ BevkWarpParams p)
{
    const int x = blockIdx.x * 32 + threadIdx.x;
    const int y = blockIdx.y * 8 + threadIdx.y;
    if (x >= p.dst_w || y >= p.dst_h) return;
    int gi;
    const BevkWarpGroup &g = find_group(p, blockIdx.z, gi);
    if (skip_block(p, gi)) return;
    const int c_local = blockIdx.z - g.chunk0;
    const int f0 = c_local * p.frames_per_chunk;
    const int f1 = min(f0 + p.frames_per_chunk, g.count);

    int X, Y;
    bevk_map_pixel(g.M, x, y, p.bw0, 1.0, X, Y);
    const int sx = bevk_sat16(X), sy = bevk_sat16(Y);
    const bool inside = (sx >= 0 && sx < p.src_w && sy >= 0 && sy < p.src_h);
    const long long os = ((long long)sy * p.src_w + sx) * C;
    const long long od = ((long long)y * p.dst_w + x) * C;
    const T *src = (const T *)p.src;
    T *dst = (T *)p.dst;

    T bv[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        if constexpr (sizeof(T) == 1)
            bv[c] = border_u8(p.border[c]);
        else if constexpr (sizeof(T) == 2)
            bv[c] = __float2half_rn(p.border[c]);
        else
            bv[c] = p.border[c];
    }
    for (int f = f0; f < f1; ++f) {
        const long long fr = (long long)(g.first + f * g.stride);
        const T *s = src + fr * p.src_frame_elems + os;
        T *d = dst + fr * p.dst_frame_elems + od;
#pragma unroll
        for (int c = 0; c < C; ++c) d[c] = inside ? __ldg(s + c) : bv[c];
    }
}

// ---- uint8 x 3, zero border: word gathers + the integer arithmetic of the staged kernel ---------
// The BGR-video case without shared-memory staging: every lane owns one dst pixel, reads the two
// 6-byte rows of its 2x2 window as aligned 32-bit words through the read-only L1 path (3 words a
// row instead of 6 byte loads), interpolates with dp4a / dp2a (warp_u8c3.cuh) and the warp packs
// its 32 pixels into 24 words -- one coalesced 96-byte store per warp and frame.  This is the
// kernel for strongly minifying maps (BrnoCompSpeed-sized BEVs of 1080p frames), where a tile's
// source box is mostly untouched pixels and staging it would move more data than the gather.
template <bool LINEAR, int kBatch>
__global__ void __launch_bounds__(256) warp_u8c3_direct_kernel(const __grid_constant__ BevkWarpParams p)
{
    const int lane = threadIdx.x, x0 = blockIdx.x * 32;
    const int x = x0 + lane, y = blockIdx.y * 8 + threadIdx.y;
    if (y >= p.dst_h) return;  // a warp is one dst row segment: uniform exit, shuffles stay legal
    int gi;
    const BevkWarpGroup &g = find_group(p, blockIdx.z, gi);
    if (skip_block(p, gi)) return;  // split launch: only the tiles the staged kernel marked
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
    const uint32_t row_bytes = (uint32_t)p.src_w * 3u;
    const uint32_t A = act ? (uint32_t)rs * row_bytes + 3u * (uint32_t)cs : 0u;
    const uint32_t last_word = (uint32_t)p.src_frame_elems - 4u;
    const Pix q = PxU8C3::make<LINEAR>(act, A, act ? wc0 : 0, act ? wc1 : 0, wr0, wr1);
    // third (nearest: second) window word, clamped into the frame where unused
    const uint32_t off2 = LINEAR ? min(q.addr + 8u, last_word - row_bytes) : min(q.addr + 4u, last_word);
    // lanes 4j..4j+2 write words 3j..3j+2 of the warp's 96-byte segment
    const int j = lane >> 2, r4 = lane & 3;
    const uint32_t sel_pack = r4 == 0 ? 0x4210u : (r4 == 1 ? 0x5421u : 0x6542u);
    const bool st_ok = r4 < 3 && 4 * j < min(32, p.dst_w - x0);  // dst_w % 4 == 0
    const uint8_t *src = (const uint8_t *)p.src;
    uint8_t *dst = (uint8_t *)p.dst + ((long long)y * p.dst_w + x0) * 3 + (3 * j + r4) * 4;

    // The loop lives on loads in flight: the windows of kBatch frames are requested before the
    // first one is interpolated (explicitly -- left to itself the compiler keeps one frame's worth).
    constexpr int kWords = LINEAR ? 6 : 2;
    // 64-byte L2 fetches: this kernel serves the minifying maps, which use a fraction of each line
    auto LD = [](const uint32_t *a) { return ldg_sparse(a); };
    auto load = [&](int f, uint32_t(&w)[kWords]) {
        const uint8_t *s = src + (long long)(g.first + f * g.stride) * p.src_frame_elems;
        if (LINEAR) {
            const uint8_t *ra = s + q.addr, *rb = ra + row_bytes;
            w[0] = LD((const uint32_t *)ra);
            w[1] = LD((const uint32_t *)(ra + 4));
            w[2] = LD((const uint32_t *)(s + off2));
            w[3] = LD((const uint32_t *)rb);
            w[4] = LD((const uint32_t *)(rb + 4));
            w[5] = LD((const uint32_t *)(s + off2 + row_bytes));
        } else {
            w[0] = LD((const uint32_t *)(s + q.addr));
            w[1] = LD((const uint32_t *)(s + off2));
        }
    };
    auto finish = [&](int f, const uint32_t(&w)[kWords]) {
        uint32_t P;
        if (LINEAR)
            P = lerp_aligned(q, __funnelshift_r(w[0], w[1], q.sh), __funnelshift_r(w[1], w[2], q.sh),
                             __funnelshift_r(w[3], w[4], q.sh), __funnelshift_r(w[4], w[5], q.sh));
        else
            P = __funnelshift_r(w[0], w[1], q.sh) & q.w0;
        const uint32_t word = prmt(P, __shfl_down_sync(0xffffffffu, P, 1), sel_pack);
        const long long fr = (long long)(g.first + f * g.stride);
        if (st_ok) st_stream_free(reinterpret_cast<uint32_t *>(dst + fr * p.dst_frame_elems), word);
    };
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

// returns true if it launched
bool launch_u8c3_direct(const BevkWarpParams &p, int linear, cudaStream_t stream)
{
    if (p.border[0] != 0.f || p.border[1] != 0.f || p.border[2] != 0.f) return false;
    // rows of a multiple of 4 bytes: both rows of a window then share one word alignment
    if (p.src_w < 2 || p.src_h < 2 || (p.src_w % 4) != 0 || (p.dst_w % 4) != 0) return false;
    if (((uintptr_t)p.src % 4) != 0 || ((uintptr_t)p.dst % 4) != 0) return false;
    if ((p.src_frame_elems % 4) != 0 || (p.dst_frame_elems % 4) != 0) return false;
    if (p.src_frame_elems > 0xffffffffLL) return false;
    dim3 block(32, 8, 1);
    dim3 grid((p.dst_w + 31) / 32, (p.dst_h + 7) / 8, p.total_chunks);
    if (linear)
        warp_u8c3_direct_kernel<true, 2><<<grid, block, 0, stream>>>(p);
    else
        warp_u8c3_direct_kernel<false, 4><<<grid, block, 0, stream>>>(p);
    return true;
}

template <typename T, int C>
int launch_tc(const BevkWarpParams &p, int linear, cudaStream_t stream)
{
    dim3 block(32, 8, 1);
    dim3 grid((p.dst_w + 31) / 32, (p.dst_h + 7) / 8, p.total_chunks);
    if (linear)
        warp_linear_kernel<T, C><<<grid, block, 0, stream>>>(p);
    else
        warp_nearest_kernel<T, C><<<grid, block, 0, stream>>>(p);
    BEVK_CUDA(cudaGetLastError());
    return BEVK_OK;
}

template <typename T>
int launch_t(const BevkWarpParams &p, int channels, int linear, cudaStream_t stream)
{
    switch (channels) {
    case 1: return launch_tc<T, 1>(p, linear, stream);
    case 2: return launch_tc<T, 2>(p, linear, stream);
    case 3: return launch_tc<T, 3>(p, linear, stream);
    case 4: return launch_tc<T, 4>(p, linear, stream);
    }
    BEVK_FAIL(BEVK_E_ARG, "channels must be 1..4, got %d", channels);
}

}  // namespace

int bevk_plan_generic_chunks(BevkWarpParams &p, int channels)
{
    (void)channels;
    // Frames per chunk: large enough to amortise the FP64 coordinate set-up, small enough that the
    // grid covers every SM with at least 2 waves of blocks -- and, as long as a chunk keeps 8
    // frames, with 12 waves (24 for BEVs of fewer tiles than two waves): few, long blocks leave a
    // costly last wave, and when a whole BEV is less than a wave the blocks in flight span several
    // chunks, i.e. many frames at once (cfg 4: 6.2 ms at 64 frames per chunk, 5.3 ms at 8).
    const long long tiles = (long long)((p.dst_w + 31) / 32) * ((p.dst_h + 7) / 8);
    const long long wave = (long long)bevk_sm_count() * 8;
    int max_count = 0;
    for (int i = 0; i < p.n_groups; ++i) max_count = max_count > p.g[i].count ? max_count : p.g[i].count;
    auto blocks_at = [&](int fpc) {
        long long blocks = 0;
        for (int i = 0; i < p.n_groups; ++i) blocks += tiles * ((p.g[i].count + fpc - 1) / fpc);
        return blocks;
    };
    int fpc = max_count < 64 ? max_count : 64;
    while (fpc > 1 && blocks_at(fpc) < 2 * wave) fpc = (fpc + 1) / 2;
    const long long want = (tiles < 2 * wave ? 24 : 12) * wave;
    while (fpc >= 12 && blocks_at(fpc) < want) fpc = (fpc + 1) / 2;
    fpc = fpc < 1 ? 1 : fpc;
    p.frames_per_chunk = fpc;
    int z = 0;
    for (int i = 0; i < p.n_groups; ++i) {
        p.g[i].chunk0 = z;
        z += (p.g[i].count + fpc - 1) / fpc;
    }
    p.total_chunks = z;
    if (z > 65535) BEVK_FAIL(BEVK_E_ARG, "warp: too many frame chunks (%d) for one launch", z);
    return BEVK_OK;
}

int bevk_launch_warp_generic(const BevkWarpParams &p, int channels, int dtype, int linear,
                             cudaStream_t stream)
{
    if (dtype == BEVK_U8 && channels == 3 && launch_u8c3_direct(p, linear, stream)) {
        BEVK_CUDA(cudaGetLastError());
        return BEVK_OK;
    }
    switch (dtype) {
    case BEVK_U8: return launch_t<uint8_t>(p, channels, linear, stream);
    case BEVK_F16: return launch_t<__half>(p, channels, linear, stream);
    case BEVK_F32: return launch_t<float>(p, channels, linear, stream);
    }
    BEVK_FAIL(BEVK_E_ARG, "warp dtype must be BEVK_U8/F16/F32, got %d", dtype);
}

// ---- touched-pixel accounting -----------------------------------------------------------------
namespace {
__global__ void footprint_mark_kernel(uint8_t *mask, int src_h, int src_w, int dst_h, int dst_w,
                                      BevkWarpGroup g, int bw0, int linear, int *rows)
{
    const int x = blockIdx.x * 32 + threadIdx.x;
    const int y = blockIdx.y * 8 + threadIdx.y;
    if (x >= dst_w || y >= dst_h) return;
    int X, Y;
    bevk_map_pixel(g.M, x, y, bw0, linear ? 32.0 : 1.0, X, Y);
    const int sx = bevk_sat16(linear ? (X >> 5) : X), sy = bevk_sat16(linear ? (Y >> 5) : Y);
    const int nt = linear ? 2 : 1;
    for (int j = 0; j < nt; ++j)
        for (int i = 0; i < nt; ++i) {
            const int u = sx + i, v = sy + j;
            if (u >= 0 && u < src_w && v >= 0 && v < src_h) {
                mask[(size_t)v * src_w + u] = 1;
                atomicMin(&rows[0], v);
                atomicMax(&rows[1], v);
            }
        }
}
__global__ void footprint_count_kernel(const uint8_t *mask, size_t n, unsigned long long *count)
{
    unsigned long long local = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n;
         i += (size_t)gridDim.x * blockDim.x)
        local += mask[i];
    for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(count, local);
}
}  // namespace

extern "C" int64_t bevk_warp_touched_pixels(int src_h, int src_w, int dst_h, int dst_w,
                                            const double M[9], int flags, int *row_range)
{
    int rc = bevk_require_device();
    if (rc) return rc;
    if (!M || src_h <= 0 || src_w <= 0 || dst_h <= 0 || dst_w <= 0)
        BEVK_FAIL(BEVK_E_ARG, "bevk_warp_touched_pixels: bad sizes / null matrix");
    const int interp = flags & 7;
    if (interp != BEVK_INTER_NEAREST && interp != BEVK_INTER_LINEAR)
        BEVK_FAIL(BEVK_E_ARG, "unsupported interpolation flag %d", interp);
    BevkWarpGroup g = {};
    if (flags & BEVK_WARP_INVERSE_MAP)
        for (int i = 0; i < 9; ++i) g.M[i] = M[i];
    else
        bevk_invert3x3(M, g.M);
    uint8_t *mask = nullptr;
    int *rows = nullptr;
    unsigned long long *count = nullptr;
    const size_t n = (size_t)src_h * src_w;
    BEVK_CUDA(cudaMalloc(&mask, n));
    BEVK_CUDA(cudaMalloc(&rows, 2 * sizeof(int)));
    BEVK_CUDA(cudaMalloc(&count, sizeof(unsigned long long)));
    const int init_rows[2] = {src_h, -1};
    cudaMemset(mask, 0, n);
    cudaMemset(count, 0, sizeof(unsigned long long));
    cudaMemcpy(rows, init_rows, sizeof(init_rows), cudaMemcpyHostToDevice);
    dim3 block(32, 8), grid((dst_w + 31) / 32, (dst_h + 7) / 8);
    footprint_mark_kernel<<<grid, block>>>(mask, src_h, src_w, dst_h, dst_w, g,
                                           bevk_block_width(dst_w, dst_h),
                                           interp == BEVK_INTER_LINEAR, rows);
    footprint_count_kernel<<<296, 256>>>(mask, n, count);
    unsigned long long h_count = 0;
    int h_rows[2] = {0, 0};
    cudaError_t e = cudaMemcpy(&h_count, count, sizeof(h_count), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(h_rows, rows, sizeof(h_rows), cudaMemcpyDeviceToHost);
    cudaFree(mask);
    cudaFree(rows);
    cudaFree(count);
    if (e != cudaSuccess) BEVK_FAIL(BEVK_E_CUDA, "footprint kernels failed: %s", cudaGetErrorString(e));
    if (row_range) {
        row_range[0] = h_rows[0];
        row_range[1] = h_rows[1];
    }
    return (int64_t)h_count;
}
