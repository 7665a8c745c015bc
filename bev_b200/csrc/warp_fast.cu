// warp_fast.cu -- staged perspective warp for 3-channel frames (the BASELINE hot path:
// cv2.warpPerspective on BGR video frames, reference vis_homo.py:85-91), sm_100a.
//
// The kernel is written against a pixel-format policy PX (warp_u8c3.cuh: uint8 x 3,
// warp_f16c3.cuh: float16 x 3, warp_formats.cuh: uint8 x 1, uint8 x 4, float32 x 3) that owns the
// per-pixel registers, the window loads, the interpolation and the store packing.
//
// Work item = (chunk of frames, homography group, dst tile).  A persistent CTA of 4 or 8 warps (a
// constant of the pixel-format policy) pulls items from a counter in the launch's scratch; a tile
// is 128 dst pixels per warp, 4 per thread, as 128xN, 64x2N or 32x4N (picked per launch on the
// host, pick_tile_shape):
//
//   1. set-up, once per item: the exact FP64 coordinate pipeline of cv2 (bevk_map_pixel_xb) gives
//      each pixel its 2x2 source window, and frame-invariant registers are derived from it -- the
//      shared-memory offset of the window, a funnel-shift amount that byte-aligns it and the tap
//      weights laid out as the policy's operands.  Out-of-image taps get weight 0 and a clamped
//      address, so the frame loop has no border branches.  A block reduction yields the tile's
//      source bounding box.  (uint8 bilinear: the tile's first chunk publishes positions, weights
//      and box in the scratch, the other chunks re-read them.)
//   2. frame loop: the bounding box of the next frames is fetched by the TMA unit as 2-D tensor
//      boxes (cp.async.bulk.tensor.2d, at most 3 requests per frame and tile, completion on an
//      mbarrier) into a 2-, 4- or 8-deep shared-memory ring of up to 8 frames per stage while the
//      warps interpolate the current frames out of shared memory.  The producer role rotates over
//      the warps; the warp whose turn it is issues a whole stage in one pass (one lane per frame
//      and box); full[] / empty[] mbarriers are the only synchronisation in the loop, and all but
//      one stage of the ring are in flight.  The box shape is picked per tile from a menu of 224
//      tensor maps over the source batch viewed as a [frames*rows][row_bytes/4] uint32 (or /8
//      uint64) matrix: widths 64..2048 B, heights 1..32 rows.  A first version issued one
//      cp.async.bulk per source row: the TMA unit retired only one such ~300-byte request per ~70
//      cycles per SM, which capped the kernel at 33 % of the HBM roofline (profiles/r01_fast_v1_*).
//   3. stores: the policy packs the lanes' pixels into words (one shuffle + PRMT for uint8) and
//      writes fully coalesced row segments with streaming stores.
//
// Tiles whose box does not stage (too wide / tall for the menu, larger than half the ring): a few
// of them fall back, inside the kernel, to aligned 32-bit global loads with the same arithmetic;
// when the host predicts 2-35 % of the tiles the launch is SPLIT -- the kernel only marks them in
// BevkWarpParams::hard and the direct-gather kernel (warp_generic.cu) follows on the stream over
// the marked tiles; above that the whole launch goes to the direct-gather kernel.
//
// HBM traffic per frame is the touched source footprint (bounding boxes overlap by a row /
// column and are partly re-served by L2: tiles are walked column-major so that neighbours run
// concurrently, and the frame chunks keep the CTAs within a few dozen frames of each other) plus
// the output, about 1.2x the algorithmic bytes of SURVEY.md 8d.  What bounds the kernel is
// instruction issue (75 % of the slots, 0.31 of its 0.38 ms on cfg 2), see DESIGN.md 3.1.
#include "bevk_common.cuh"
#include "warp_u8c3.cuh"
#include "warp_f16c3.cuh"
#include "warp_formats.cuh"

#include <cuda.h>  // CUtensorMap + enums only; the encoder is fetched through the runtime
#include <mutex>
#include <string.h>

namespace {

// CTA size is a property of the kernel (pixel format x interpolation, see cta_threads below): 4 warps
// (tiles of 512 pixels, 6 CTAs per SM for the 80-register kernels) or 8 warps (1024 pixels, 3 CTAs).
// Both hold the same registers and ring bytes per SM; twice as many independent CTAs hide each
// other's item boundaries (barrier skew, set-up, first TMA round trip) better where the boxes are
// narrow -- uint8 x 3 bilinear: cfg 2 0.421 -> 0.411 ms, cfg 5 0.453 -> 0.436 ms, float16 0.90 ->
// 0.86 ms -- while 4-byte pixels (0.465 -> 0.509 ms) and nearest (+2 %) do better with the taller tile.
template <typename PX, bool LINEAR> constexpr int cta_threads()
{
    return LINEAR ? PX::kLinearThreads : PX::kNearestThreads;
}
// Tile shapes.  A CTA always owns 1024 dst pixels, 4 per thread; SEGS = 32-pixel segments per tile
// row: 4 -> 128x8 (warp w owns tile row w), 2 -> 64x16 (rows 2w, 2w+1), 1 -> 32x32 (rows 4w..4w+3).
// Narrower tiles bound the width of the source box where the map minifies horizontally.
__host__ __device__ constexpr int tile_w(int segs) { return 32 * segs; }
__host__ __device__ constexpr int tile_h(int segs, int warps) { return warps * (4 / segs); }
// Tensor-map menu: one map per box shape.
//   narrow boxes: 12 widths (64..512 B in steps of 64, 640..1024 B in steps of 128) x 16 heights
//                 (1..8, 10..16 in steps of 2, 20..32 in steps of 4), uint32 elements;
//   wide boxes  :  4 widths (1280..2048 B in steps of 256) x 8 heights (4..32 in steps of 4),
//                 uint64 elements (a box row holds at most 256 elements).
// A tile's bounding box is fetched with one box whenever it has at most 32 rows (taller ones take
// up to kMaxBoxes).
constexpr int kNarrowW = 12, kNarrowH = 16, kWideW = 4, kWideH = 8;
constexpr int kMapCount = kNarrowW * kNarrowH + kWideW * kWideH;
constexpr int kMaxBoxWidth = 2048, kMaxBoxHeight = 32;
constexpr int kMaxBoxes = 3;
constexpr int kMaxStageFrames = 8;              // frames that share one ring stage / mbarrier phase
constexpr int kBarBytes = 256;                  // 28 mbarriers: ring depths 2, 4 and 8
constexpr int kPrefetchAhead = 2;               // depth-2 rings: L2 prefetch runs this many stages ahead
constexpr int kTailSlack = 64;                  // window words may run a few bytes past a stage

__host__ __device__ constexpr int map_width(int wi)
{
    return wi < 8 ? 64 * (wi + 1) : (wi < 12 ? 512 + 128 * (wi - 7) : 1024 + 256 * (wi - 11));
}
__host__ __device__ constexpr bool map_is_wide(int wi) { return wi >= kNarrowW; }
// heights of the narrow menu; the wide menu has 4 * (hi + 1)
__host__ __device__ constexpr int map_height(int hi)
{
    return hi < 8 ? hi + 1 : (hi < 12 ? 10 + 2 * (hi - 8) : 20 + 4 * (hi - 12));
}
// smallest menu entry that covers `bytes` / `rows`
__host__ __device__ __forceinline__ int map_width_index(int bytes)
{
    return bytes <= 512 ? (bytes + 63) / 64 - 1
                        : (bytes <= 1024 ? 7 + (bytes - 512 + 127) / 128 : 11 + (bytes - 1024 + 255) / 256);
}
__host__ __device__ __forceinline__ int map_height_index(int rows)
{
    return rows <= 8 ? rows - 1 : (rows <= 16 ? 8 + (rows - 9) / 2 : 12 + (rows - 17) / 4);
}
// box height the menu offers for `rows` (<= kMaxBoxHeight) at width index wi, and its map index
__host__ __device__ __forceinline__ int box_height(int wi, int rows)
{
    return map_is_wide(wi) ? (rows + 3) / 4 * 4 : map_height(map_height_index(rows));
}
__host__ __device__ __forceinline__ int box_map_index(int wi, int rows)
{
    return map_is_wide(wi) ? kNarrowW * kNarrowH + (wi - kNarrowW) * kWideH + (rows + 3) / 4 - 1
                           : wi * kNarrowH + map_height_index(rows);
}

struct WarpFastMaps {
    CUtensorMap m[kMapCount];
};

// Frame chunks of one launch.  Chunk k of a group with `count` frames covers frames
// [count * cum[k] >> 16, count * cum[k + 1] >> 16): the chunks shrink towards the end of the item
// list, so that the CTAs, which pull items from a shared counter, finish almost together.
constexpr int kMaxChunks = 12;
struct ChunkPlan {
    int n_chunks;
    uint32_t cum[kMaxChunks + 1];  // cum[0] = 0, cum[n_chunks] = 65536
};

// Per-launch scratch (stream-ordered allocation, see bevk_launch_warp_fast): the item counter and,
// when a tile is worked on in several frame chunks, the set-up of every (group, tile) -- computed
// by the CTA that runs the tile's first chunk, published through `ready`, re-used by the others.
constexpr int kRecWords = 8;   // per thread: 4 pixels x (window position, packed weights)
constexpr int kHdrInts = 8;    // per tile : source bounding box, "any pixel inside" flag
struct WarpScratch {
    int *next_item;   // zeroed
    int *ready;       // [groups * tiles], zeroed; NULL: every item computes its own set-up
    int *hdr;         // [groups * tiles][kHdrInts]
    uint32_t *rec;    // [groups * tiles][kRecWords][kThreads]
    uint32_t recip_per_chunk, recip_tiles, recip_tiles_y;  // ceil(2^32 / d) for the item decode
};

// ---- PTX wrappers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t"
        "}" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// 2-D tensor box global -> shared, completion counted in bytes on an mbarrier (the TMA path)
__device__ __forceinline__ void tma_box_g2s(uint32_t dst, const CUtensorMap *map, int x, int y,
                                            uint32_t bar)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
        " [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(x), "r"(y)
        : "memory");
}
// the same box, global -> L2 only (no shared memory, no completion)
__device__ __forceinline__ void tma_box_prefetch(const CUtensorMap *map, int x, int y)
{
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(
                     reinterpret_cast<uint64_t>(map)),
                 "r"(x), "r"(y)
                 : "memory");
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ int ld_acquire(const int *p)
{
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int *p, int v)
{
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// Stops the compiler from re-deriving a loop-invariant value inside the frame loop.
__device__ __forceinline__ void keep(uint32_t &v) { asm volatile("" : "+r"(v)); }
__device__ __forceinline__ void keep(int &v) { asm volatile("" : "+r"(v)); }

// What the producing warp needs to fetch the frames' bounding boxes.
struct BoxPlan {
    int n_boxes;
    int x;                  // first column, in elements of the map (TMA wants 16-byte aligned box rows)
    int y0;                 // first source row of the box
    uint32_t bytes;         // sum of the box sizes (the mbarrier's transaction count per frame)
    int frame0, frame_step; // source frame of the item's frame i = frame0 + i * frame_step
    int src_h;
    int n_frames, fps;      // frames of the item / per ring stage
    int slog;               // log2 of the ring depth in use
    uint32_t ring, full0;   // shared-memory addresses: ring, first barrier of the set in use
    uint32_t stride, frame_bytes, pitch;  // bytes per stage / staged frame / staged row
    int map_idx[kMaxBoxes];
    int row[kMaxBoxes];     // row offset of each box inside the stage
};

// A decoded work item (thread 0 decodes the next one while the CTA works on the current one).
struct ItemDesc {
    int item;                 // >= total_items: no more work
    int gi, tile_x, tile_y;   // homography group, tile position
    int f0, n_frames;         // frames [f0, f0 + n_frames) of the group's run
    int first, stride;        // the run: frame index = first + f * stride
    int chunk;                // frame chunk; chunk 0 computes (and publishes) the tile's set-up
    int ready;                // chunk > 0: the tile's set-up was already published when the item was decoded
};

// The consumers' loop state (kept small so that the frame loop fits its register budget); the
// producing warp reads what it needs from the BoxPlan in shared memory.
struct LoopCtx {
    uint32_t ring, full0;          // shared-memory addresses of the ring / first barrier of the set
    uint32_t stride;               // bytes per stage (fps frames)
    uint32_t frame_bytes;          // bytes per staged frame
    uint32_t pitch;                // bytes per staged row
    int fps;                       // frames per stage
    int n_frames;
    int slog;                      // ring depth 2^slog stages
    int ahead;                     // stages in flight ahead of the one being consumed
    const WarpFastMaps *maps;
    const BoxPlan *plan;           // in shared memory
};

// One warp pulls the stage that starts at frame i0 of the item towards the SM: lane l issues box
// (l % n_boxes) of the stage's frame (l / n_boxes), so all requests of a stage (at most
// kMaxStageFrames * kMaxBoxes = 24) leave in one pass.  TO_SMEM starts the copies into the stage's
// ring slot (`use` is the running count of stages this CTA has pushed through the barrier set);
// otherwise the boxes are only prefetched into L2 so that the later copy does not wait on HBM
// (used by depth-2 rings, whose copies run just one stage ahead).  Deliberately not inlined: it
// runs in one warp per stage and must not cost the frame loop registers.
template <bool TO_SMEM>
__device__ __noinline__ void produce(const BoxPlan *plan, const WarpFastMaps *maps, int i0,
                                     uint32_t use, int lane)
{
    const BoxPlan &pl = *plan;
    const int nf = min(pl.fps, pl.n_frames - i0);
    const int nb = pl.n_boxes;
    const int f = nb == 1 ? lane : (nb == 2 ? lane >> 1 : (lane * 11) >> 5);  // lane / 3 for lane < 32
    const int b = lane - f * nb;
    const bool mine = f < nf;
    const int row = pl.row[mine ? b : 0];
    const CUtensorMap *map = &maps->m[pl.map_idx[mine ? b : 0]];
    const int y = (pl.frame0 + (i0 + f) * pl.frame_step) * pl.src_h + pl.y0 + row;
    if (TO_SMEM) {
        const uint32_t slot = use & ((1u << pl.slog) - 1u);
        const uint32_t fb = pl.full0 + 8 * slot;
        // k-th fill of a slot waits for the (k-1)-th release; the first passes at once
        mbar_wait(fb + (8u << pl.slog), ((use >> pl.slog) & 1u) ^ 1u);
        if (lane == 0) mbar_expect_tx(fb, pl.bytes * nf);
        __syncwarp();
        if (mine)
            tma_box_g2s(pl.ring + slot * pl.stride + f * pl.frame_bytes + row * pl.pitch, map, pl.x, y, fb);
    } else if (mine) {
        tma_box_prefetch(map, pl.x, y);
    }
}

// Keep the ring (and, for depth-2 rings, the L2 prefetch window) full.  `done` = frames of the
// item consumed up to and including the current stage.  The producer role rotates over the warps
// so that no warp is slower than the others -- a fixed producer warp paces the whole CTA, because
// every warp waits on the stages it issues.  (It is in effect the fastest warps that produce: the
// refill of a slot waits for the slowest warp to release it.  Handing the refill to the warp that
// releases a slot last was tried: 7 % slower, it loads the warp that is already behind.)
template <int WARPS>
__device__ __forceinline__ void feed(const LoopCtx &c, int done, uint32_t use, int lane, int warp)
{
    const int turn = ((int)use - warp) & (WARPS - 1);
    const int i_load = done + (c.ahead - 1) * c.fps;  // first frame of the stage `ahead` stages on
    if (turn == 0 && i_load < c.n_frames) produce<true>(c.plan, c.maps, i_load, use + c.ahead, lane);
    if (c.slog == 1 && turn == WARPS / 2 && i_load + kPrefetchAhead * c.fps < c.n_frames)
        produce<false>(c.plan, c.maps, i_load + kPrefetchAhead * c.fps, 0, lane);
}

// The frame loop of a staged item: ring of 2^slog stages of c.fps frames each, c.ahead of them in
// flight ahead of the stage being consumed, the rest slack between the warps.  body(sa, d)
// interpolates the thread's pixels of ONE frame staged at shared address sa into d.  A warp hands
// a slot back once it is through the stage's last frame (testing for the last frame inside the
// body, to release a little earlier, costs more than it gains: the frame loop is one straight
// block this way).  Returns the advanced stage counter.
// started() is run by thread 0 once the first copies of the item are on their way (the decode of
// the CTA's next item: thread-0 work that would otherwise delay every item's first bytes).
template <int WARPS, typename BODY, typename STARTED>
__device__ __forceinline__ uint32_t stage_loop(const LoopCtx &c, uint32_t use, uint8_t *d,
                                               const uint32_t d_step, const int tid, BODY body, STARTED started)
{
    const uint32_t smask = (1u << c.slog) - 1u;
    const int lane = tid & 31, warp = tid >> 5;
    if (warp == 0) {
        for (int s = 0; s < c.ahead && s * c.fps < c.n_frames; ++s)
            produce<true>(c.plan, c.maps, s * c.fps, use + s, lane);
        for (int s = c.ahead; c.slog == 1 && s < c.ahead + kPrefetchAhead && s * c.fps < c.n_frames; ++s)
            produce<false>(c.plan, c.maps, s * c.fps, 0, lane);
        if (tid == 0) started();
    }
    int done = 0;
#pragma unroll 1
    while (done < c.n_frames) {
        const uint32_t slot = use & smask;
        const uint32_t fb = c.full0 + 8 * slot;
        mbar_wait(fb, (use >> c.slog) & 1u);
        uint32_t sa = c.ring + slot * c.stride;  // first frame of the stage
        int nf = min(c.fps, c.n_frames - done);
        done += nf;
#pragma unroll 1
        for (; nf > 0; --nf, sa += c.frame_bytes, d += d_step) body(sa, d);
        __syncwarp();
        if (lane == 0) mbar_arrive(fb + (8u << c.slog));
        feed<WARPS>(c, done, use, lane, warp);
        ++use;
    }
    return use;
}

// ---- which dst pixels a thread owns ---------------------------------------------------------------
// A warp owns two adjacent dst rows x 64 columns (SEGS >= 2) or four rows x 32 columns (SEGS == 1);
// thread pixel k = 2 j + i is row i of vertical PAIR j: the two pixels of a pair are vertical
// neighbours, so wherever the map magnifies vertically their 2x2 source windows overlap and the
// pair path below loads the window rows once for both.
// (PAIRS = the kernel has the pair path, i.e. uint8 x 3 bilinear.)  Kernels without it keep each
// warp on ONE dst row where the tile is wide enough -- 4 / 2 / 1 segments of 32 pixels in a row --
// so that a warp writes the longest contiguous run the tile offers.
template <int SEGS, bool PAIRS> __device__ __forceinline__ int warp_px_x(int warp)
{
    if (!PAIRS) return 0;
    return SEGS >= 2 ? 64 * (warp % (SEGS >= 2 ? SEGS / 2 : 1)) : 0;
}
template <int SEGS, bool PAIRS> __device__ __forceinline__ int warp_px_y(int warp)
{
    if (!PAIRS) return warp * (4 / SEGS);
    return SEGS >= 2 ? 2 * (warp / (SEGS >= 2 ? SEGS / 2 : 1)) : 4 * warp;
}
template <int SEGS, bool PAIRS> __device__ __forceinline__ constexpr int px_seg(int k)
{
    return PAIRS ? (SEGS >= 2 ? (k >> 1) : 0) : k % SEGS;
}
template <int SEGS, bool PAIRS> __device__ __forceinline__ constexpr int px_row(int k)
{
    return PAIRS ? (SEGS >= 2 ? (k & 1) : k) : k / SEGS;
}

// Frame-invariant registers of a vertical pixel pair that shares its window loads (uint8 x 3,
// bilinear).  `first` is the pixel whose window starts on the pair's first source row; the second
// one's starts on the same row (2-row variant) or one row below (3-row variant).  Columns: the
// pair's 12-byte span per row starts at the smaller of the two window columns, a pixel's window
// starts 0 or 3 bytes into it.
struct PairReg {
    uint32_t addr;         // byte offset (4-aligned) inside a staged frame of the span, first row
    uint32_t sh;           // funnel-shift amount that byte-aligns the span: 8 * (start & 3)
    uint32_t sel_f, sel_s; // PRMT selector of the first / second pixel: window at span byte 0 or 3
    uint32_t sel_y;        // PRMT selector that gathers the third channel's taps of both pixels
    uint32_t wf0, wf1;     // dp2a tap weights of the first pixel, its window rows 0 / 1
    uint32_t ws0, ws1;     // ... of the second pixel
};

// One staged row of a pair's span, byte-aligned: g0 = span bytes 0..3, g1 = 4..7, and the pool
// (u, w2) that holds the third-channel taps b2, b5 (u = [b2 . . b5]) and b8 (byte `start & 3` of
// the raw word w2).  A window at span byte 0 / 3 is gathered as
//   xa = prmt(g0, g1, 0x4130 / 0x7463) = [b0 b3 b1 b4] / [b3 b6 b4 b7]   (channels 0, 1: two taps each)
//   y  = prmt(u, w2, sel_y)            = [c2 taps of the first pixel | c2 taps of the second]
struct PairRow {
    uint32_t g0, g1, u, w2;
};
__device__ __forceinline__ PairRow pair_row(uint32_t a, uint32_t sh)
{
    const uint32_t w0 = lds32(a), w1 = lds32(a + 4);
    PairRow r;
    r.w2 = lds32(a + 8);
    r.g0 = __funnelshift_r(w0, w1, sh);
    r.g1 = __funnelshift_r(w1, r.w2, sh);
    r.u = prmt(r.g0, r.g1, 0x5002u);
    return r;
}
// sel_y for window offsets df, ds (0 or 1 pixel into the span) and span start byte o = start & 3
__device__ __forceinline__ uint32_t pair_sel_y(bool df, bool ds, uint32_t o)
{
    const uint32_t f = df ? (3u | ((4u + o) << 4)) : (0u | (3u << 4));
    const uint32_t s2 = ds ? (3u | ((4u + o) << 4)) : (0u | (3u << 4));
    return f | (s2 << 8);
}
// cv2's fixed-point bilinear of the pair's two pixels: rows (a0, a1) hold the first pixel's window,
// (b0, b1) the second's (the same two rows in the 2-row variant).  ya* / yb* = the y gathers of
// those rows.  Results [c0 c1 c2 0].
__device__ __forceinline__ void pair_lerp(const PairReg &q, const PairRow &a0, const PairRow &a1,
                                          const PairRow &b0, const PairRow &b1, uint32_t ya0, uint32_t ya1,
                                          uint32_t yb0, uint32_t yb1, uint32_t &pf, uint32_t &ps)
{
    const uint32_t rnd = 32768u;
    {
        const uint32_t x0 = prmt(a0.g0, a0.g1, q.sel_f), x1 = prmt(a1.g0, a1.g1, q.sel_f);
        const uint32_t t0 = __dp2a_lo(q.wf1, x1, __dp2a_lo(q.wf0, x0, rnd));
        const uint32_t t1 = __dp2a_hi(q.wf1, x1, __dp2a_hi(q.wf0, x0, rnd));
        const uint32_t t2 = __dp2a_lo(q.wf1, ya1, __dp2a_lo(q.wf0, ya0, rnd));
        pf = prmt(prmt(t0, t1, 0x4462u), t2, 0x7610u);
    }
    {
        const uint32_t x0 = prmt(b0.g0, b0.g1, q.sel_s), x1 = prmt(b1.g0, b1.g1, q.sel_s);
        const uint32_t t0 = __dp2a_lo(q.ws1, x1, __dp2a_lo(q.ws0, x0, rnd));
        const uint32_t t1 = __dp2a_hi(q.ws1, x1, __dp2a_hi(q.ws0, x0, rnd));
        const uint32_t t2 = __dp2a_hi(q.ws1, yb1, __dp2a_hi(q.ws0, yb0, rnd));
        ps = prmt(prmt(t0, t1, 0x4462u), t2, 0x7610u);
    }
}

// MINB = CTAs per SM the register allocation is bounded for (4 -> 64 registers, 3 -> 80);
// SEGS = tile shape (see tile_w / tile_h).
template <typename PX, bool LINEAR, int MINB, int SEGS>
__global__ void __launch_bounds__((cta_threads<PX, LINEAR>()), MINB)
warp_fast_kernel(const __grid_constant__ BevkWarpParams p,
                      const __grid_constant__ WarpFastMaps maps,
                      const __grid_constant__ ChunkPlan plan, const int tiles_x, const int tiles_y,
                      const int total_items, const int ring_bytes, const WarpScratch sc)
{
    constexpr int kThreads = cta_threads<PX, LINEAR>(), kWarps = kThreads / 32;
    extern __shared__ __align__(128) uint8_t smem[];
    // three barrier sets, one per ring depth S = 2, 4, 8: full[S] then empty[S], at byte
    // offsets 0, 32 and 96.  Each set keeps its own running stage counter (s_use) across items,
    // so barrier phases never need a reset when consecutive items use different depths.
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + ring_bytes);
    __shared__ int s_box[4];
    __shared__ int s_any;
    __shared__ uint32_t s_use[3];
    __shared__ ItemDesc s_item[2];  // current / next work item, decoded by thread 0
    __shared__ double s_M[BEVK_MAX_GROUPS][9];
    __shared__ BoxPlan s_plan;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t ring = smem_u32(smem);
    const uint32_t bar0 = smem_u32(bars);
    if (tid == 0) {
        for (int sl = 1; sl <= 3; ++sl) {
            const int S = 1 << sl, base = 16 * S - 32;
            for (int i = 0; i < S; ++i) {
                mbar_init(bar0 + base + 8 * i, 1);                // full: the producer's expect_tx
                mbar_init(bar0 + base + 8 * (S + i), kWarps);     // empty: one arrival per warp
            }
            s_use[sl - 1] = 0;
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }

    const int n_tiles = tiles_x * tiles_y;
    const uint8_t *src = (const uint8_t *)p.src;
    uint8_t *dst = (uint8_t *)p.dst;
    constexpr int kBpp = PX::kBpp;
    constexpr bool kPairMap = LINEAR && PX::kPairs;  // which dst pixels a thread owns (see warp_px_x)
    const int src_row_bytes = p.src_w * kBpp;
    const long long src_frame_bytes = (long long)src_row_bytes * p.src_h;
    const long long dst_frame_bytes = (long long)p.dst_w * p.dst_h * kBpp;

    // Items are (chunk, group, tile) with the chunk index slowest: long chunks first.  Every item
    // is pulled from *sc.next_item -- also a CTA's first one, so that a CTA which has not started
    // yet never holds a tile's first chunk while others wait for its set-up.  Thread 0 decodes an
    // item (integer divisions, parameter reads) one item ahead of its use.
    const int per_chunk = p.n_groups * n_tiles;
    // n / d for n < 2^31 with the host's reciprocal ceil(2^32 / d): one multiply and a fix-up
    // instead of an integer division (the decode runs on one thread, every cycle of it delays warp 0)
    auto fast_div = [](int n, int d, uint32_t recip) {
        uint32_t q = __umulhi((uint32_t)n, recip);
        if (q * (uint32_t)d > (uint32_t)n) --q;          // ceil() made the quotient one too large
        if ((q + 1u) * (uint32_t)d <= (uint32_t)n) ++q;  // d == 1: the reciprocal saturates at 2^32 - 1
        return (int)q;
    };
    auto decode = [&](int item, ItemDesc &o) {
        o.item = item;
        if (item >= total_items) return;
        const int chunk = fast_div(item, per_chunk, sc.recip_per_chunk), rem = item - chunk * per_chunk;
        const int gi = fast_div(rem, n_tiles, sc.recip_tiles), tile = rem - gi * n_tiles;
        // column-major walk: concurrently running CTAs cover whole tile columns, i.e. both the
        // magnified far field (store-heavy) and the minified near field (load-heavy)
        o.gi = gi;
        o.tile_x = fast_div(tile, tiles_y, sc.recip_tiles_y);
        o.tile_y = tile - o.tile_x * tiles_y;
        const int count = p.g[gi].count;
        o.f0 = (int)(((unsigned long long)count * plan.cum[chunk]) >> 16);
        o.n_frames = (int)(((unsigned long long)count * plan.cum[chunk + 1]) >> 16) - o.f0;
        o.first = p.g[gi].first;
        o.stride = p.g[gi].stride;
        o.chunk = chunk;
        // one item ahead of its use: by then the first chunk's CTA has nearly always published
        o.ready = (sc.ready != nullptr && chunk > 0)
                      ? ld_acquire(sc.ready + (gi * n_tiles + o.tile_x * tiles_y + o.tile_y))
                      : 1;
    };
    for (int i = tid; i < p.n_groups * 9; i += kThreads) s_M[i / 9][i % 9] = p.g[i / 9].M[i % 9];
    if (tid == 0) {
        decode(atomicAdd(sc.next_item, 1), s_item[0]);
        s_box[0] = s_box[2] = 1 << 30;
        s_box[1] = s_box[3] = -1;
        s_any = 0;
    }
    __syncthreads();
    const bool bw0_pow2 = (p.bw0 & (p.bw0 - 1)) == 0;
    const uint32_t row_bytes = (uint32_t)p.dst_w * (uint32_t)kBpp;

    int par = 0;
#pragma unroll 1
    while (true) {
        const int item = s_item[par].item;
        if (item >= total_items) break;
        const int gi = s_item[par].gi, tile_x = s_item[par].tile_x, tile_y = s_item[par].tile_y;
        const int f0 = s_item[par].f0, n_frames = s_item[par].n_frames;
        const int g_first = s_item[par].first, g_stride = s_item[par].stride;
        const int chunk = s_item[par].chunk;
        const bool published = s_item[par].ready != 0;
        // the index of the CTA's NEXT item: requested now, needed only once this item's first
        // copies are in flight (next_item_decode below), so the atomic's round trip costs nothing
        int next_raw = 0;
        if (tid == 0) next_raw = atomicAdd(sc.next_item, 1);
        const int x0 = tile_x * tile_w(SEGS) + warp_px_x<SEGS, kPairMap>(warp);
        const int y0 = tile_y * tile_h(SEGS, kWarps) + warp_px_y<SEGS, kPairMap>(warp);
        const int tile_id = gi * n_tiles + tile_x * tiles_y + tile_y;
        par ^= 1;

        // ---- 1. set-up: window position and tap weights of the thread's four pixels, the tile's
        //         source bounding box -- computed by the tile's first chunk, re-read by the others
        int cs[4], rs[4];
        uint32_t wpk[4];  // wc0 | wc1 << 8 | wr0 << 16 | wr1 << 24 (0..32 each); 0 = pixel inactive
        int bx0, bx1, by0, by1;
        bool any;
        if (sc.ready == nullptr || chunk == 0) {
            bx0 = by0 = 1 << 30;
            bx1 = by1 = -1;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int x = x0 + lane + 32 * px_seg<SEGS, kPairMap>(k), y = y0 + px_row<SEGS, kPairMap>(k);
                const bool in_dst = (x < p.dst_w) && (y < p.dst_h);
                int X, Y, wc0, wc1, wr0, wr1;
                const int xc = min(x, p.dst_w - 1);
                const int xb = bw0_pow2 ? (xc & ~(p.bw0 - 1)) : (xc / p.bw0) * p.bw0;
                bevk_map_pixel_xb(s_M[gi], xb, xc - xb, min(y, p.dst_h - 1), LINEAR ? 32.0 : 1.0, X, Y);
                if (LINEAR) {
                    const int sx = bevk_sat16(X >> 5), sy = bevk_sat16(Y >> 5);
                    window(sx, X & 31, p.src_w, cs[k], wc0, wc1);
                    window(sy, Y & 31, p.src_h, rs[k], wr0, wr1);
                } else {
                    const int sx = bevk_sat16(X), sy = bevk_sat16(Y);
                    const bool in = sx >= 0 && sx < p.src_w && sy >= 0 && sy < p.src_h;
                    cs[k] = min(max(sx, 0), p.src_w - 1);
                    rs[k] = min(max(sy, 0), p.src_h - 1);
                    wc0 = wr0 = in ? 1 : 0;
                    wc1 = wr1 = 0;
                }
                const bool active = in_dst && (wc0 | wc1) != 0 && (wr0 | wr1) != 0;
                wpk[k] = active ? (uint32_t)(wc0 | (wc1 << 8) | (wr0 << 16) | (wr1 << 24)) : 0u;
                if (active) {
                    bx0 = min(bx0, cs[k]);
                    bx1 = max(bx1, cs[k] + (LINEAR ? 1 : 0));
                    by0 = min(by0, rs[k]);
                    by1 = max(by1, rs[k] + (LINEAR ? 1 : 0));
                }
            }
            bx0 = __reduce_min_sync(0xffffffffu, bx0);
            bx1 = __reduce_max_sync(0xffffffffu, bx1);
            by0 = __reduce_min_sync(0xffffffffu, by0);
            by1 = __reduce_max_sync(0xffffffffu, by1);
            if (lane == 0 && bx1 >= 0) {
                atomicMin(&s_box[0], bx0);
                atomicMax(&s_box[1], bx1);
                atomicMin(&s_box[2], by0);
                atomicMax(&s_box[3], by1);
                s_any = 1;
            }
            __syncthreads();
            any = s_any != 0;
            bx0 = s_box[0];
            bx1 = s_box[1];
            by0 = s_box[2];
            by1 = s_box[3];
            if (sc.ready != nullptr) {
                uint32_t *rec = sc.rec + (size_t)tile_id * (kRecWords * kThreads) + tid;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    __stcg(rec + (2 * k) * kThreads, (uint32_t)cs[k] | ((uint32_t)rs[k] << 16));
                    __stcg(rec + (2 * k + 1) * kThreads, wpk[k]);
                }
                if (tid == 0) {
                    int4 *h = reinterpret_cast<int4 *>(sc.hdr + (size_t)tile_id * kHdrInts);
                    __stcg(h, make_int4(bx0, bx1, by0, by1));
                    __stcg(h + 1, make_int4(any ? 1 : 0, 0, 0, 0));
                }
                __threadfence();  // ordered before the release store that follows the next barrier
            }
        } else {
            if (!published) {  // rare: wait for the CTA that runs the tile's first chunk
                if (tid == 0) {
                    const int *flag = sc.ready + tile_id;
                    while (ld_acquire(flag) == 0) __nanosleep(100);
                }
            }
            __syncthreads();
            const int4 *h = reinterpret_cast<const int4 *>(sc.hdr + (size_t)tile_id * kHdrInts);
            const int4 hb = __ldcg(h), hf = __ldcg(h + 1);
            bx0 = hb.x;
            bx1 = hb.y;
            by0 = hb.z;
            by1 = hb.w;
            any = hf.x != 0;
            const uint32_t *rec = sc.rec + (size_t)tile_id * (kRecWords * kThreads) + tid;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t pos = __ldcg(rec + (2 * k) * kThreads);
                cs[k] = (int)(pos & 0xffffu);
                rs[k] = (int)(pos >> 16);
                wpk[k] = __ldcg(rec + (2 * k + 1) * kThreads);
            }
        }

        // staged geometry: 16-byte aligned first column, box shapes from the tensor-map menu
        const int a0 = (kBpp * bx0) & ~15;
        const int need_w = ((kBpp * (bx1 + 1) + 15) & ~15) - a0;
        const int wi = map_width_index(need_w);
        const int pitch = map_width(wi);
        const int nrows = by1 - by0 + 1;
        bool staged = any && need_w <= kMaxBoxWidth && nrows <= kMaxBoxes * kMaxBoxHeight;
        // rows the boxes cover: at most kMaxBoxes boxes, each the smallest menu height that fits
        int box_rows = 0;
        if (staged)
            for (int rem = nrows; rem > 0;) {
                const int h = box_height(wi, min(rem, kMaxBoxHeight));
                box_rows += h;
                rem -= h;
            }
        const uint32_t frame_bytes = ((uint32_t)(box_rows * pitch) + 127u) & ~127u;
        staged = staged && 2 * frame_bytes <= (uint32_t)ring_bytes;
        // nearest reads one pixel per dst pixel: where the map minifies, most of the box would be
        // staged for nothing (and fetched from HBM for nothing) -- gather those tiles directly
        if (!LINEAR && frame_bytes > 3u * 1024u * (uint32_t)kBpp) staged = false;
        // frames per stage: as many as still leave a ring of 4 stages
        const int fps = 4 * kMaxStageFrames * frame_bytes <= (uint32_t)ring_bytes ? kMaxStageFrames
                        : 4 * 4 * frame_bytes <= (uint32_t)ring_bytes ? 4
                        : 8 * frame_bytes <= (uint32_t)ring_bytes ? 2 : 1;
        const int stage_stride = fps * (int)frame_bytes;
        const int slog = (8 * stage_stride <= ring_bytes) ? 3 : (4 * stage_stride <= ring_bytes ? 2 : 1);
        const uint32_t full0 = bar0 + 16 * (1 << slog) - 32;  // the set's empty[] follow its full[]
        if (tid == 0) {
            if (staged) {
                int rem = nrows, row = 0, nb = 0;
                while (rem > 0) {
                    const int r = min(rem, kMaxBoxHeight);
                    s_plan.map_idx[nb] = box_map_index(wi, r);
                    s_plan.row[nb] = row;
                    row += box_height(wi, r);
                    rem -= box_height(wi, r);
                    ++nb;
                }
                s_plan.n_boxes = nb;
                s_plan.x = map_is_wide(wi) ? a0 >> 3 : a0 >> 2;  // in elements of the map
                s_plan.y0 = by0;
                s_plan.bytes = (uint32_t)(box_rows * pitch);
                s_plan.frame0 = g_first + f0 * g_stride;
                s_plan.frame_step = g_stride;
                s_plan.src_h = p.src_h;
                s_plan.n_frames = n_frames;
                s_plan.fps = fps;
                s_plan.slog = slog;
                s_plan.ring = ring;
                s_plan.full0 = full0;
                s_plan.stride = stage_stride;
                s_plan.frame_bytes = frame_bytes;
                s_plan.pitch = pitch;
            }
        }
        __syncthreads();  // s_plan visible to the producer lanes; every thread has read s_box
        if (tid == 0) {
            // the tile's set-up is in global memory (every thread fenced its part before the barrier)
            if (sc.ready != nullptr && chunk == 0) st_release(sc.ready + tile_id, 1);
            // re-arm the box for the next item (its first atomics come after this item's last barrier)
            s_box[0] = s_box[2] = 1 << 30;
            s_box[1] = s_box[3] = -1;
            s_any = 0;
        }
        // thread 0, once this item's first copies are issued (or at once where nothing is staged)
        auto next_item_decode = [&]() { decode(next_raw, s_item[par]); };

        // ---- store geometry ---------------------------------------------------------------------
        // which words of a 32-pixel row segment this lane writes is the pixel format's business
        const typename PX::Store st = PX::store_setup(lane);
        bool seg_ok[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            // pixels left in this 32-pixel segment: a multiple of 4 (dst_w % 4 == 0)
            const int valid_px = min(32, p.dst_w - (x0 + 32 * px_seg<SEGS, kPairMap>(k)));
            seg_ok[k] = (y0 + px_row<SEGS, kPairMap>(k) < p.dst_h) && PX::lane_stores(lane, valid_px);
        }
        // where pixel k's segment goes, from the thread's pointer into dst row y0 (dd) and the one
        // into row y0 + 1 (dd1): compile-time segment offsets, one runtime row step
        auto seg_ptr = [row_bytes](uint8_t *dd, uint8_t *dd1, int k) -> uint8_t * {
            const int row = px_row<SEGS, kPairMap>(k), seg = px_seg<SEGS, kPairMap>(k);
            return (row & 1 ? dd1 : dd) + (row >> 1) * 2 * (size_t)row_bytes + PX::kSegBytes * seg;
        };
        uint32_t d_step = (uint32_t)g_stride * (uint32_t)dst_frame_bytes;  // < 2^32 (host check)
        keep(d_step);
        uint8_t *d = dst + (long long)(g_first + f0 * g_stride) * dst_frame_bytes +
                     ((long long)y0 * p.dst_w + x0) * kBpp + PX::lane_offset(lane);

        if ((!any || !staged) && tid == 0) next_item_decode();
        if (!any) {
            // whole tile maps outside the source: constant border (0) for every frame
#pragma unroll 1
            for (int i = 0; i < n_frames; ++i, d += d_step)
#pragma unroll
                for (int k = 0; k < 4; ++k) PX::store_zero(seg_ptr(d, d + row_bytes, k), seg_ok[k], lane);
        } else if (staged) {
            LoopCtx c;
            c.ring = ring;
            c.full0 = full0;
            c.stride = stage_stride;
            c.frame_bytes = frame_bytes;
            c.pitch = pitch;
            c.fps = fps;
            c.n_frames = n_frames;
            c.slog = slog;
            // stages in flight ahead of the one being consumed: all but one.  With a whole warp issuing
            // a stage in one pass the producer's detour is short, and every kernel does best this way
            // (against half the ring: float16 cfg 5 0.792 -> 0.749 ms, uint8 x 4 0.441 -> 0.430 ms,
            // nearest 0.316 -> 0.310 ms); the whole ring in flight is worse again for the 4-warp kernels.
            // Two-slot rings refill the slot that was just released (the producing warp waits for the
            // other warps' release), so that the copy of stage n + 2 runs under stage n + 1 -- with one
            // stage ahead the copy only started when the frame before it was done (cfg 5 0.424 -> 0.393
            // ms, cfg 2 0.391 -> 0.382 ms).  Only those rings prefetch into L2, kPrefetchAhead stages
            // further on (feed).
            c.ahead = slog == 1 ? 2 : (1 << slog) - 1;
            c.maps = &maps;
            c.plan = &s_plan;
            keep(c.ring);
            keep(c.full0);
            keep(c.slog);  // else the stage loop re-derives the ring depth from ring_bytes in every stage
            // every thread tracks the counter in a register; thread 0 publishes it for the next item
            uint32_t use = s_use[slog - 1];

            // Pair path (uint8 x 3 bilinear): can every vertical pair of this warp share its
            // window loads?  Needs windows at most one column apart and the same row step --
            // 0 (both on the same two rows), +1 or -1 (the second / first pixel of the pair one
            // row below) -- across the warp, so that the choice of window rows is warp-uniform.
            int var = 3;
            if constexpr (LINEAR && PX::kPairs) {
                bool ok0 = true, ok1 = true, ok2 = true;
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    const int a = 2 * j, b = a + 1;
                    const bool aa = wpk[a] != 0, ab = wpk[b] != 0;
                    if (aa && ab) {
                        const int dr = rs[b] - rs[a], dc = cs[b] - cs[a];
                        const bool near = dc >= -1 && dc <= 1;
                        ok0 = ok0 && near && dr == 0;
                        ok1 = ok1 && near && dr == 1;
                        ok2 = ok2 && near && dr == -1;
                    } else if (aa || ab) {
                        // one active pixel: it can take either role as long as the pair's rows
                        // stay inside the staged box
                        const int r = aa ? rs[a] : rs[b];
                        ok1 = ok1 && (aa ? r + 2 <= by1 : r - 1 >= by0);
                        ok2 = ok2 && (ab ? r + 2 <= by1 : r - 1 >= by0);
                    } else {
                        ok1 = ok1 && by1 - by0 >= 2;
                        ok2 = ok2 && by1 - by0 >= 2;
                    }
                }
                var = __all_sync(0xffffffffu, ok0) ? 0
                      : (__all_sync(0xffffffffu, ok1) ? 1 : (__all_sync(0xffffffffu, ok2) ? 2 : 3));
            }
            if constexpr (LINEAR && PX::kPairs) if (var != 3) {
                PairReg pr[2];
                uint32_t ok = 0;  // store predicates as a bit mask: bit 2 j = first, 2 j + 1 = second pixel of pair j
                const bool sw = var == 2;  // the pair's first pixel is the one in the lower dst row
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                    // first / second pixel of the pair (explicit selects: no dynamically indexed arrays)
                    const int rs_f = sw ? rs[2 * j + 1] : rs[2 * j], rs_s = sw ? rs[2 * j] : rs[2 * j + 1];
                    const int cs_f = sw ? cs[2 * j + 1] : cs[2 * j], cs_s = sw ? cs[2 * j] : cs[2 * j + 1];
                    const uint32_t wp_f = sw ? wpk[2 * j + 1] : wpk[2 * j], wp_s = sw ? wpk[2 * j] : wpk[2 * j + 1];
                    const bool af = wp_f != 0, as = wp_s != 0;
                    const int step = var ? 1 : 0;
                    const int rf = af ? rs_f : (as ? rs_s - step : by0);
                    const int cf = af ? cs_f : (as ? cs_s : bx0), cn = as ? cs_s : cf;
                    const int c0 = min(cf, cn);
                    const uint32_t A = (uint32_t)((rf - by0) * pitch + kBpp * c0 - a0);
                    pr[j].addr = A & ~3u;
                    pr[j].sh = 8 * (A & 3);
                    pr[j].sel_f = cf != c0 ? 0x7463u : 0x4130u;
                    pr[j].sel_s = cn != c0 ? 0x7463u : 0x4130u;
                    pr[j].sel_y = pair_sel_y(cf != c0, cn != c0, A & 3);
                    PxU8C3::tap_weights(wp_f, pr[j].wf0, pr[j].wf1);
                    PxU8C3::tap_weights(wp_s, pr[j].ws0, pr[j].ws1);
                    keep(pr[j].addr);
                    keep(pr[j].sh);
                    keep(pr[j].sel_y);
                    keep(pr[j].sel_f);
                    keep(pr[j].sel_s);
                    ok |= ((sw ? seg_ok[2 * j + 1] : seg_ok[2 * j]) ? 1u : 0u) << (2 * j);
                    ok |= ((sw ? seg_ok[2 * j] : seg_ok[2 * j + 1]) ? 2u : 0u) << (2 * j);
                }
                keep(ok);
                const long long d_second = sw ? -(long long)row_bytes : (long long)row_bytes;
                uint8_t *d_first = sw ? d + row_bytes : d;
                if (var == 0) {
                    use = stage_loop<kWarps>(c, use, d_first, d_step, tid, [&](uint32_t sa, uint8_t *dd) {
                        const uint32_t sb = sa + c.pitch;
                        uint32_t P[4];
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const PairRow r0 = pair_row(pr[j].addr + sa, pr[j].sh);
                            const PairRow r1 = pair_row(pr[j].addr + sb, pr[j].sh);
                            const uint32_t y0 = prmt(r0.u, r0.w2, pr[j].sel_y), y1 = prmt(r1.u, r1.w2, pr[j].sel_y);
                            pair_lerp(pr[j], r0, r1, r0, r1, y0, y1, y0, y1, P[2 * j], P[2 * j + 1]);
                        }
                        // dd points into the first pixels' dst row, the second pixels' is one row on / back
                        uint8_t *ds = dd + d_second;
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            PX::store(seg_ptr(dd, dd, 2 * j), P[2 * j], (ok >> (2 * j)) & 1u, st, lane);
                            PX::store(seg_ptr(ds, ds, 2 * j), P[2 * j + 1], (ok >> (2 * j + 1)) & 1u, st, lane);
                        }
                    }, next_item_decode);
                } else {
                    use = stage_loop<kWarps>(c, use, d_first, d_step, tid, [&](uint32_t sa, uint8_t *dd) {
                        const uint32_t sb = sa + c.pitch, sc2 = sb + c.pitch;
                        uint32_t P[4];
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            const PairRow r0 = pair_row(pr[j].addr + sa, pr[j].sh);
                            const PairRow r1 = pair_row(pr[j].addr + sb, pr[j].sh);
                            const PairRow r2 = pair_row(pr[j].addr + sc2, pr[j].sh);
                            const uint32_t y0 = prmt(r0.u, r0.w2, pr[j].sel_y), y1 = prmt(r1.u, r1.w2, pr[j].sel_y);
                            const uint32_t y2 = prmt(r2.u, r2.w2, pr[j].sel_y);
                            pair_lerp(pr[j], r0, r1, r1, r2, y0, y1, y1, y2, P[2 * j], P[2 * j + 1]);
                        }
                        // dd points into the first pixels' dst row, the second pixels' is one row on / back
                        uint8_t *ds = dd + d_second;
#pragma unroll
                        for (int j = 0; j < 2; ++j) {
                            PX::store(seg_ptr(dd, dd, 2 * j), P[2 * j], (ok >> (2 * j)) & 1u, st, lane);
                            PX::store(seg_ptr(ds, ds, 2 * j), P[2 * j + 1], (ok >> (2 * j + 1)) & 1u, st, lane);
                        }
                    }, next_item_decode);
                }
            }
            if (var == 3) {
                constexpr uint32_t kLast = PX::template last_word_offset<LINEAR>();
                typename PX::Reg px[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const bool act = wpk[k] != 0;
                    const int A = act ? (rs[k] - by0) * pitch + kBpp * cs[k] - a0 : 0;
                    px[k] = PX::template make<LINEAR>(act, (uint32_t)A, wpk[k]);
                    keep(px[k].addr);
                    keep(px[k].sh);
                }
                use = stage_loop<kWarps>(c, use, d, d_step, tid, [&](uint32_t sa, uint8_t *dd) {
                    const uint32_t sb = sa + c.pitch;  // row 1 of the windows
                    typename PX::Out P[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        uint32_t w[PX::kWinWords];
                        const uint32_t a = px[k].addr + sa, b = px[k].addr + sb;
                        PX::template load<LINEAR>(px[k], a, b, a + kLast, b + kLast, w,
                                                  [](uint32_t ad) { return lds32(ad); });
                        P[k] = PX::template math<LINEAR>(px[k], w);
                    }
                    // pack the lanes' pixels into words and store coalesced row segments
#pragma unroll
                    for (int k = 0; k < 4; ++k) PX::store(seg_ptr(dd, dd + row_bytes, k), P[k], seg_ok[k], st, lane);
                }, next_item_decode);
            }
            __syncthreads();  // every warp has read s_use and left the ring
            if (tid == 0) s_use[slog - 1] = use;
            continue;
        } else if (p.hard) {
            // split launch: leave the tile to the direct-gather kernel that follows on the stream
            if (tid == 0) p.hard[tile_id] = 1;
        } else {
            // bounding box too large for the ring (strong minification) or too wide / tall for the
            // tensor-map menu: the same arithmetic on aligned 32-bit loads straight from global
            // memory (L1-cached, read-only path).  Frames are 16-byte aligned (src is, and a frame
            // is a multiple of 16 bytes), so the window words are addressed like the staged ones.
            constexpr uint32_t kLast = PX::template last_word_offset<LINEAR>();
            typename PX::Reg px[4];
            uint32_t last[4];  // last window word; clamped into the frame where it is not needed
            const uint32_t last_word = (uint32_t)src_frame_bytes - 4u;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const bool act = wpk[k] != 0;
                const uint32_t A = act ? (uint32_t)rs[k] * (uint32_t)src_row_bytes + (uint32_t)kBpp * (uint32_t)cs[k] : 0u;
                px[k] = PX::template make<LINEAR>(act, A, wpk[k]);
                // bilinear reads row 1 of the window at +src_row_bytes: clamp so that also that
                // read stays inside the frame (the alignments that need the word never clamp)
                last[k] = min(px[k].addr + kLast, last_word - (LINEAR ? (uint32_t)src_row_bytes : 0u));
            }
            const uint8_t *s = src + (long long)(g_first + f0 * g_stride) * src_frame_bytes;
            const long long s_step = (long long)g_stride * src_frame_bytes;
#pragma unroll 1
            for (int i = 0; i < n_frames; ++i, d += d_step, s += s_step) {
                typename PX::Out P[4];
                // all window words of the frame are requested before the first is used: this loop
                // lives on loads in flight
                uint32_t w[4][PX::kWinWords];
#pragma unroll
                for (int k = 0; k < 4; ++k)  // "addresses" are byte offsets inside the frame here
                    PX::template load<LINEAR>(px[k], px[k].addr, px[k].addr + src_row_bytes, last[k],
                                              last[k] + src_row_bytes, w[k],
                                              [s](uint32_t off) { return ldg_sparse((const uint32_t *)(s + off)); });
#pragma unroll
                for (int k = 0; k < 4; ++k) P[k] = PX::template math<LINEAR>(px[k], w[k]);
#pragma unroll
                for (int k = 0; k < 4; ++k) PX::store(seg_ptr(d, d + row_bytes, k), P[k], seg_ok[k], st, lane);
            }
        }
        __syncthreads();  // the next item's descriptor (s_item) is complete and visible
    }
}

// ---- host side: tensor-map menu ---------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *,
                                  const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct MapCacheEntry {
    const void *base = nullptr;
    int row_bytes = 0;
    long long rows = 0;
    unsigned long long stamp = 0;
    WarpFastMaps maps;
};
constexpr int kMapCacheSize = 8;
MapCacheEntry g_map_cache[kMapCacheSize];
unsigned long long g_map_stamp = 0;
std::mutex g_map_mutex;
EncodeTiledFn g_encode = nullptr;

// The batch viewed as a [rows][row_bytes / 4] uint32 matrix: one tensor map per box shape.
int get_maps(const void *base, int row_bytes, long long rows, WarpFastMaps &out)
{
    std::lock_guard<std::mutex> lock(g_map_mutex);
    if (!g_encode) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        BEVK_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !fn)
            BEVK_FAIL(BEVK_E_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
        g_encode = (EncodeTiledFn)fn;
    }
    MapCacheEntry *victim = &g_map_cache[0];
    for (int i = 0; i < kMapCacheSize; ++i) {
        MapCacheEntry &e = g_map_cache[i];
        if (e.base == base && e.row_bytes == row_bytes && e.rows == rows) {
            e.stamp = ++g_map_stamp;
            out = e.maps;
            return BEVK_OK;
        }
        if (e.stamp < victim->stamp) victim = &e;
    }
    const cuuint64_t gstride[1] = {(cuuint64_t)row_bytes};
    const cuuint32_t estride[2] = {1, 1};
    // every box row starts 16-byte aligned in global memory, which the TMA unit requires (a
    // start on another byte raises an illegal-instruction fault -- tried for a 2-byte shifted
    // second copy); 4-byte elements give boxes up to 1024 B wide, 8-byte elements up to 2048 B
    for (int wi = 0; wi < kNarrowW + kWideW; ++wi) {
        const bool wide = map_is_wide(wi);
        const int es = wide ? 8 : 4;
        const cuuint64_t gdim[2] = {(cuuint64_t)(row_bytes / es), (cuuint64_t)rows};
        for (int hi = 0; hi < (wide ? kWideH : kNarrowH); ++hi) {
            const int h = wide ? 4 * (hi + 1) : map_height(hi);
            const cuuint32_t box[2] = {(cuuint32_t)(map_width(wi) / es), (cuuint32_t)h};
            CUresult r = g_encode(&victim->maps.m[box_map_index(wi, h)],
                                  wide ? CU_TENSOR_MAP_DATA_TYPE_UINT64 : CU_TENSOR_MAP_DATA_TYPE_UINT32,
                                  2, const_cast<void *>(base), gdim, gstride, box, estride,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) {
                victim->base = nullptr;
                BEVK_FAIL(BEVK_E_CUDA, "cuTensorMapEncodeTiled failed (code %d) for a %ux%u box",
                          (int)r, box[0] * es, box[1]);
            }
        }
    }
    victim->base = base;
    victim->row_bytes = row_bytes;
    victim->rows = rows;
    victim->stamp = ++g_map_stamp;
    out = victim->maps;
    return BEVK_OK;
}

struct KernelConfig {
    bool ready = false;
    int ctas_per_sm = 0;
    int ring_bytes = 0;
};
// CTAs per SM the register allocation of a kernel is bounded for: PX::kLinearCtas for the bilinear
// kernels (a 64-register build spills in the frame loop and is slower); nearest kernels fit 64
// registers without spilling (4 CTAs of 8 warps) and gain 5 % from the fourth CTA.
template <typename PX, bool LINEAR> constexpr int min_ctas()
{
    return LINEAR ? PX::kLinearCtas : 4 * (256 / cta_threads<PX, LINEAR>());
}
// Everything that belongs to one device: the kernels' shared-memory opt-in and ring size
// (cudaFuncSetAttribute is per device), the SM count, the memory-pool set-up.  Guarded by g_map_mutex.
constexpr int kMaxDevices = 64;
struct DeviceState {
    KernelConfig cfg[5][2][3];  // [pixel format, see format_index][linear][tile shape: SEGS 4, 2, 1]
    int sm_count = 0;
    bool pool_ready = false;
};
DeviceState g_dev[kMaxDevices];
inline int segs_index(int segs) { return segs == 4 ? 0 : (segs == 2 ? 1 : 2); }

// Pixel formats the staged kernel is instantiated for.
inline int format_index(int dtype, int channels)
{
    if (dtype == BEVK_U8) return channels == 3 ? 0 : (channels == 1 ? 2 : (channels == 4 ? 3 : -1));
    if (dtype == BEVK_F16) return channels == 3 ? 1 : -1;
    if (dtype == BEVK_F32) return channels == 3 ? 4 : -1;
    return -1;
}
template <typename F> auto with_format(int fmt, F f)
{
    switch (fmt) {
    case 1: return f(PxF16C3());
    case 2: return f(PxU8C1());
    case 3: return f(PxU8C4());
    case 4: return f(PxF32C3());
    default: return f(PxU8C3());
    }
}
inline int format_bpp(int fmt)
{
    return with_format(fmt, [](auto px) { return (int)decltype(px)::kBpp; });
}

template <typename PX, bool LINEAR, int SEGS> int configure(KernelConfig &cfg)
{
    constexpr int kMinCtas = min_ctas<PX, LINEAR>();
    constexpr int kThreads = cta_threads<PX, LINEAR>();
    auto kern = warp_fast_kernel<PX, LINEAR, kMinCtas, SEGS>;
    // how many CTAs the register file allows, then split the shared memory evenly between them
    BEVK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 * 1024));
    int by_regs = 0;
    BEVK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&by_regs, kern, kThreads, 16 * 1024));
    if (by_regs < 1) BEVK_FAIL(BEVK_E_CUDA, "staged warp kernel does not fit an SM");
    by_regs = by_regs > kMinCtas ? kMinCtas : by_regs;
    int dev = 0, smem_sm = 0;
    BEVK_CUDA(cudaGetDevice(&dev));
    BEVK_CUDA(cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev));
    // per CTA: 1 KB reserved by the driver + static shared memory
    cudaFuncAttributes attr;
    BEVK_CUDA(cudaFuncGetAttributes(&attr, kern));
    int ring = smem_sm / by_regs - 1024 - (int)attr.sharedSizeBytes - kBarBytes - kTailSlack;
    ring &= ~127;
    if (ring > 200 * 1024) ring = 200 * 1024;
    BEVK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   ring + kBarBytes + kTailSlack));
    cfg.ctas_per_sm = by_regs;
    cfg.ring_bytes = ring;
    cfg.ready = true;
    return BEVK_OK;
}

template <typename PX, bool LINEAR> int configure_segs(int segs, KernelConfig &cfg)
{
    return segs == 4 ? configure<PX, LINEAR, 4>(cfg)
                     : (segs == 2 ? configure<PX, LINEAR, 2>(cfg) : configure<PX, LINEAR, 1>(cfg));
}
template <typename PX> int configure_any(int linear, int segs, KernelConfig &cfg)
{
    return linear ? configure_segs<PX, true>(segs, cfg) : configure_segs<PX, false>(segs, cfg);
}

template <typename PX, bool LINEAR, int SEGS>
void launch(int grid, int smem, cudaStream_t stream, const BevkWarpParams &p, const WarpFastMaps &maps,
            const ChunkPlan &plan, int tiles_x, int tiles_y, int items, int ring_bytes, const WarpScratch &sc)
{
    warp_fast_kernel<PX, LINEAR, min_ctas<PX, LINEAR>(), SEGS><<<grid, cta_threads<PX, LINEAR>(), smem, stream>>>(
        p, maps, plan, tiles_x, tiles_y, items, ring_bytes, sc);
}
template <typename PX>
void launch_any(int linear, int segs, int grid, int smem, cudaStream_t stream, const BevkWarpParams &p,
                const WarpFastMaps &maps, const ChunkPlan &plan, int tiles_x, int tiles_y, int items,
                int ring_bytes, const WarpScratch &sc)
{
#define BEVK_LAUNCH(LIN, SEGS) \
    launch<PX, LIN, SEGS>(grid, smem, stream, p, maps, plan, tiles_x, tiles_y, items, ring_bytes, sc)
    if (linear) {
        if (segs == 4) BEVK_LAUNCH(true, 4);
        else if (segs == 2) BEVK_LAUNCH(true, 2);
        else BEVK_LAUNCH(true, 1);
    } else {
        if (segs == 4) BEVK_LAUNCH(false, 4);
        else if (segs == 2) BEVK_LAUNCH(false, 2);
        else BEVK_LAUNCH(false, 1);
    }
#undef BEVK_LAUNCH
}

// ---- host side: which tile shape stages --------------------------------------------------------
// Fraction of the (sampled) tiles of one shape whose source box cannot be staged: wider than the
// widest tensor box, taller than kMaxBoxes boxes, or larger than half the ring.  The box of a tile
// is spanned by its four corner pixels (a projective map is monotone along lines as long as w
// keeps its sign); tiles where w changes sign are left out of the estimate (the kernel copes).
double unstaged_fraction(const BevkWarpParams &p, int linear, int bpp, int segs, int warps, int ring_bytes)
{
    const int tw = tile_w(segs), th = tile_h(segs, warps);
    const int tiles_x = (p.dst_w + tw - 1) / tw, tiles_y = (p.dst_h + th - 1) / th;
    // up to 16 x 32 evenly spaced tiles, first and last row / column included
    const int nsx = tiles_x < 16 ? tiles_x : 16, nsy = tiles_y < 32 ? tiles_y : 32;
    const double scale = linear ? 32.0 : 1.0;
    long long active = 0, bad = 0;
    for (int gi = 0; gi < p.n_groups; ++gi) {
        const double *M = p.g[gi].M;
        for (int iy = 0; iy < nsy; ++iy)
            for (int ix = 0; ix < nsx; ++ix) {
                const int ty = nsy > 1 ? (int)((long long)iy * (tiles_y - 1) / (nsy - 1)) : 0;
                const int tx = nsx > 1 ? (int)((long long)ix * (tiles_x - 1) / (nsx - 1)) : 0;
                const int x0 = tx * tw, y0 = ty * th;
                const int x1 = (x0 + tw < p.dst_w ? x0 + tw : p.dst_w) - 1;
                const int y1 = (y0 + th < p.dst_h ? y0 + th : p.dst_h) - 1;
                const int cx[4] = {x0, x1, x0, x1}, cy[4] = {y0, y0, y1, y1};
                int lo_x = 1 << 30, hi_x = -(1 << 30), lo_y = 1 << 30, hi_y = -(1 << 30), pos = 0, neg = 0;
                for (int c = 0; c < 4; ++c) {
                    const double w = M[6] * cx[c] + M[7] * cy[c] + M[8];
                    pos += w > 0;
                    neg += w < 0;
                    int X, Y;
                    bevk_map_pixel(M, cx[c], cy[c], p.bw0, scale, X, Y);
                    const int sx = bevk_sat16(linear ? (X >> 5) : X), sy = bevk_sat16(linear ? (Y >> 5) : Y);
                    lo_x = sx < lo_x ? sx : lo_x;
                    hi_x = sx > hi_x ? sx : hi_x;
                    lo_y = sy < lo_y ? sy : lo_y;
                    hi_y = sy > hi_y ? sy : hi_y;
                }
                hi_x += linear;
                hi_y += linear;
                if (hi_x < 0 || hi_y < 0 || lo_x >= p.src_w || lo_y >= p.src_h) continue;  // border only
                if (pos != 4 && neg != 4) continue;  // horizon inside the tile: corners say nothing
                ++active;
                lo_x = lo_x < 0 ? 0 : lo_x;
                lo_y = lo_y < 0 ? 0 : lo_y;
                hi_x = hi_x > p.src_w - 1 ? p.src_w - 1 : hi_x;
                hi_y = hi_y > p.src_h - 1 ? p.src_h - 1 : hi_y;
                const int a0 = (bpp * lo_x) & ~15;
                const int need_w = ((bpp * (hi_x + 1) + 15) & ~15) - a0 + 16;  // one chunk of margin
                const int rows = hi_y - lo_y + 1 + 1;
                const int pitch = need_w <= kMaxBoxWidth ? map_width(map_width_index(need_w)) : need_w;
                if (need_w > kMaxBoxWidth || rows > kMaxBoxes * kMaxBoxHeight ||
                    2LL * pitch * (rows + 3) > ring_bytes)
                    ++bad;
            }
    }
    return active ? (double)bad / (double)active : 0.0;
}

struct ModeKey {
    double M[BEVK_MAX_GROUPS][9];
    int n_groups, src_h, src_w, dst_h, dst_w, linear, bpp, warps;
};
struct ModeEntry {
    ModeKey key;
    int segs;  // 4, 2, 1, or 0: leave it to the direct-gather kernel
    int best;  // the shape with the fewest unstaged tiles (what a forced launch uses)
    bool split;
    unsigned long long stamp = 0;
    bool valid = false;
};
// Above this fraction of unstaged tiles the whole launch goes to the direct-gather kernel; between
// kNegligible and this the launch is split (staged kernel + direct kernel over the marked tiles).
constexpr double kMaxSplit = 0.35;
constexpr int kModeCacheSize = 8;
ModeEntry g_mode_cache[kModeCacheSize];
unsigned long long g_mode_stamp = 0;

// Largest tile shape whose boxes all stage; 0 if even the best shape leaves more than
// kMaxUnstaged of the tiles to the in-kernel fallback (strong minification: the boxes are mostly
// untouched pixels, the direct-gather kernel moves less data).
// *split is set when the chosen shape still leaves a noticeable fraction of the tiles unstaged:
// those tiles are cheaper in a second, direct-gather launch than in the staged kernel's fallback.
int pick_tile_shape(const BevkWarpParams &p, int linear, int bpp, int warps, int ring_bytes, bool force, bool *split)
{
    // nearest reads one tap per pixel, so its in-kernel fallback costs little: keep wide tiles
    const double kNegligible = linear ? 0.002 : 0.05;
    ModeKey key;
    memset(&key, 0, sizeof(key));
    for (int i = 0; i < p.n_groups; ++i) memcpy(key.M[i], p.g[i].M, sizeof(key.M[i]));
    key.n_groups = p.n_groups;
    key.src_h = p.src_h;
    key.src_w = p.src_w;
    key.dst_h = p.dst_h;
    key.dst_w = p.dst_w;
    key.linear = linear;
    key.bpp = bpp;
    key.warps = warps;
    std::lock_guard<std::mutex> lock(g_map_mutex);
    ModeEntry *victim = &g_mode_cache[0];  // an empty entry (stamp 0), else the least recently used
    for (int i = 0; i < kModeCacheSize; ++i) {
        ModeEntry &e = g_mode_cache[i];
        if (e.valid && memcmp(&e.key, &key, sizeof(key)) == 0) {
            e.stamp = ++g_mode_stamp;
            *split = e.split && e.segs != 0;
            return (e.segs == 0 && force) ? e.best : e.segs;
        }
        if (e.stamp < victim->stamp) victim = &e;
    }
    // the widest shape that stages (nearly) everything; else the shape that stages most
    int best = 0;
    double best_frac = 2.0;
    static const int shapes[3] = {4, 2, 1};
    for (int si = 0; si < 3; ++si) {
        const double f = unstaged_fraction(p, linear, bpp, shapes[si], warps, ring_bytes);
        if (f < best_frac - 1e-9) {
            best_frac = f;
            best = shapes[si];
        }
        if (f <= kNegligible) break;
    }
    const int segs = best_frac <= kMaxSplit ? best : 0;
    victim->key = key;
    victim->segs = segs;
    victim->best = best ? best : 1;
    // up to ~2 % the in-kernel fallback is as fast as a second launch (measured on the cfg-4 cameras)
    victim->split = best_frac > (kNegligible > 0.02 ? kNegligible : 0.02);
    victim->stamp = ++g_mode_stamp;
    victim->valid = true;
    *split = victim->split && segs != 0;
    return (segs == 0 && force) ? victim->best : segs;
}

}  // namespace

int bevk_launch_warp_fast(const BevkWarpParams &p_in, int channels, int dtype, int linear, int force,
                          cudaStream_t stream)
{
    // qualification: a pixel format the kernel is instantiated for, zero border, rows the tensor
    // maps / word stores can address, per-frame dst pointer steps that fit 32 bits
    const int fmt = format_index(dtype, channels);
    if (fmt < 0) return 0;
    const int bpp = format_bpp(fmt);
    const int threads = with_format(fmt, [&](auto px) {
        using PX = decltype(px);
        return linear ? cta_threads<PX, true>() : cta_threads<PX, false>();
    });
    const int warps = threads / 32;
    for (int c = 0; c < channels; ++c)
        if (p_in.border[c] != 0.f) return 0;
    if (p_in.src_w < 2 || p_in.src_h < 2) return 0;
    if ((p_in.src_w * bpp) % 16 != 0 || (p_in.dst_w % 4) != 0) return 0;
    if (((uintptr_t)p_in.src % 16) != 0 || ((uintptr_t)p_in.dst % 4) != 0) return 0;

    BevkWarpParams p = p_in;
    int n_src_frames = 0, max_count = 0;
    for (int i = 0; i < p.n_groups; ++i)
        if ((long long)p.g[i].stride * p.dst_frame_elems * (bpp / channels) > 0xffffffffLL || p.g[i].stride < 1)
            return 0;
    for (int i = 0; i < p.n_groups; ++i) {
        const int last = p.g[i].first + (p.g[i].count - 1) * p.g[i].stride;
        n_src_frames = n_src_frames > last + 1 ? n_src_frames : last + 1;
        max_count = max_count > p.g[i].count ? max_count : p.g[i].count;
    }
    // The staged kernel pays an FP64 set-up per (tile, chunk); with fewer than kMinFrames frames
    // per homography the direct-gather kernel is faster (measured: 27 vs 39 us for one 1080p frame)
    constexpr int kMinFrames = 4;
    if (!force && max_count < kMinFrames) return 0;
    const long long rows = (long long)n_src_frames * p.src_h;
    if (rows > 0x7fffffffLL) return 0;  // TMA coordinates are int32

    // per-device state: shared-memory opt-in + ring size of the kernels, SM count, memory pool
    int dev = 0;
    BEVK_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kMaxDevices) return 0;
    DeviceState &ds = g_dev[dev];
    KernelConfig cfg0, cfg;
    {
        std::lock_guard<std::mutex> lock(g_map_mutex);
        if (!ds.sm_count) BEVK_CUDA(cudaDeviceGetAttribute(&ds.sm_count, cudaDevAttrMultiProcessorCount, dev));
        if (!ds.pool_ready) {
            // scratch comes from the device's default stream-ordered pool: keep what it has grown to
            cudaMemPool_t pool;
            BEVK_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
            unsigned long long keep_all = ~0ull;
            BEVK_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep_all));
            ds.pool_ready = true;
        }
        // tile shape: every shape's kernel has the same ring size, so configure the widest first
        KernelConfig &c0 = ds.cfg[fmt][linear ? 1 : 0][0];
        if (!c0.ready) {
            int rc = with_format(fmt, [&](auto px) { return configure_any<decltype(px)>(linear, 4, c0); });
            if (rc) return rc;
        }
        cfg0 = c0;
    }
    bool split = false;
    const int segs = pick_tile_shape(p, linear, bpp, warps, cfg0.ring_bytes, force != 0, &split);
    if (segs == 0) return 0;
    {
        std::lock_guard<std::mutex> lock(g_map_mutex);
        KernelConfig &c = ds.cfg[fmt][linear ? 1 : 0][segs_index(segs)];
        if (!c.ready) {
            int rc = with_format(fmt, [&](auto px) { return configure_any<decltype(px)>(linear, segs, c); });
            if (rc) return rc;
        }
        cfg = c;
    }

    WarpFastMaps maps;
    int rc = get_maps(p.src, p.src_w * bpp, rows, maps);
    if (rc) return rc;

    const int tiles_x = (p.dst_w + tile_w(segs) - 1) / tile_w(segs);
    const int tiles_y = (p.dst_h + tile_h(segs, warps) - 1) / tile_h(segs, warps);
    const long long n_tiles = (long long)tiles_x * tiles_y;
    const int ctas = ds.sm_count * cfg.ctas_per_sm;

    // Frame chunks.  The CTAs pull (tile, chunk) items from a shared counter, so the LAST items
    // should be short: with enough frames the chunk lengths decay (5/16, 4/16, 3/16, 1/8, then
    // ever smaller).  The FP64 set-up of a tile is computed by its first chunk and re-read by the
    // others (WarpScratch).  Short batches get fewer, equal chunks, just enough for ~3 items per CTA.
    ChunkPlan plan;
    memset(&plan, 0, sizeof(plan));
    const long long tile_groups = n_tiles * p.n_groups;
    if (max_count >= 128 && tile_groups * 5 >= 2LL * ctas) {
        static const uint32_t cum[8] = {0, 20480, 36864, 49152, 57344, 61952, 64512, 65536};
        plan.n_chunks = 7;
        memcpy(plan.cum, cum, sizeof(cum));
    } else {
        int k = (int)((3LL * ctas + tile_groups - 1) / tile_groups);
        k = k < 1 ? 1 : k;
        k = k > kMaxChunks ? kMaxChunks : k;
        k = k > (max_count + 7) / 8 ? (max_count + 7) / 8 : k;  // at least ~8 frames per chunk
        k = k < 1 ? 1 : k;
        plan.n_chunks = k;
        for (int i = 0; i <= k; ++i) plan.cum[i] = (uint32_t)(65536LL * i / k);
    }
    const long long items = tile_groups * plan.n_chunks;
    if (items > 0x7fffffffLL) return 0;
    const int grid = (int)(items < ctas ? items : ctas);

    // Per-launch scratch, allocated and freed in stream order (launches on other streams or from
    // other threads get their own): [item counter | split flags | set-up ready flags] zeroed, then
    // the tiles' set-up headers and records.
    // Sharing a tile's set-up between its frame chunks pays where the set-up is expensive relative to
    // the per-frame work and the issue slots are the scarce resource: uint8 x 3 bilinear (cfg 2: 0.444 ->
    // 0.428 ms) and uint8 x 1 bilinear (0.277 -> 0.256 ms).  The other kernels have issue slots to spare
    // and gain nothing (float16, uint8 x 4, float32) or lose a little to the extra round trips
    // (nearest 0.326 -> 0.331 ms), so they recompute.
    const bool share_setup = (fmt == 0 || fmt == 2) && linear && plan.n_chunks > 1 &&
                             tile_groups * kRecWords * threads * 4 <= (512LL << 20);
    const size_t off_hard = 256;
    const size_t off_ready = off_hard + (((size_t)(split ? tile_groups : 0) + 255) & ~(size_t)255);
    const size_t off_hdr = off_ready + (((size_t)(share_setup ? tile_groups * 4 : 0) + 255) & ~(size_t)255);
    const size_t off_rec = off_hdr + (share_setup ? (size_t)tile_groups * kHdrInts * 4 : 0);
    const size_t total = off_rec + (share_setup ? (size_t)tile_groups * kRecWords * threads * 4 : 0);
    unsigned char *scratch = nullptr;
    BEVK_CUDA(cudaMallocAsync((void **)&scratch, total, stream));
    cudaError_t e = cudaMemsetAsync(scratch, 0, off_hdr, stream);
    WarpScratch sc;
    sc.next_item = (int *)scratch;
    sc.ready = share_setup ? (int *)(scratch + off_ready) : nullptr;
    sc.hdr = share_setup ? (int *)(scratch + off_hdr) : nullptr;
    sc.rec = share_setup ? (uint32_t *)(scratch + off_rec) : nullptr;
    auto recip = [](long long d) { return d <= 1 ? 0xffffffffu : (uint32_t)(((1ULL << 32) + d - 1) / d); };
    sc.recip_per_chunk = recip(tile_groups);
    sc.recip_tiles = recip(n_tiles);
    sc.recip_tiles_y = recip(tiles_y);
    if (split) {
        // one byte per (group, tile): the staged kernel marks the tiles it leaves to the second launch
        p.hard = scratch + off_hard;
        p.hard_tw = tile_w(segs);
        p.hard_th = tile_h(segs, warps);
        p.hard_ty = tiles_y;
        p.hard_tiles = (int)n_tiles;
    }

    int rc2 = 0;
    if (e == cudaSuccess) {
        const int smem = cfg.ring_bytes + kBarBytes + kTailSlack;
        with_format(fmt, [&](auto px) {
            launch_any<decltype(px)>(linear, segs, grid, smem, stream, p, maps, plan, tiles_x, tiles_y, (int)items,
                                     cfg.ring_bytes, sc);
            return 0;
        });
        e = cudaGetLastError();
        if (e == cudaSuccess && split) {
            // the tiles the staged kernel marked, through the direct-gather kernel (same stream)
            rc2 = bevk_plan_generic_chunks(p, channels);
            if (!rc2) rc2 = bevk_launch_warp_generic(p, channels, dtype, linear, false, stream);
        }
    }
    const cudaError_t ef = cudaFreeAsync(scratch, stream);  // stream-ordered: after the kernels above
    if (e != cudaSuccess) {
        bevk_set_error("staged warp launch failed: %s", cudaGetErrorString(e));
        return BEVK_E_CUDA;
    }
    if (rc2) return rc2;
    BEVK_CUDA(ef);
    return 1;
}
