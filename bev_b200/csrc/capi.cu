// capi.cu -- extern "C" surface of libbev_b200.so: argument checking, host-side planning
// (matrix inversion, frame runs, chunking) and the pipelined host-buffer entry point.
// See include/bev_b200.h for the contract of every function.
#include "bevk_common.cuh"

#include <algorithm>
#include <math.h>
#include <mutex>
#include <string.h>
#include <vector>

// ----------------------------------------------------------------------------- errors / device
static thread_local char g_err[512] = "";

void bevk_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// Per-device probe results (a process may drive several B200s: one state per device ordinal).
constexpr int kMaxDevices = 64;
struct DeviceProbe {
    int state = 0;  // 0 unknown, 1 ok, -1 unusable
    int sm_count = 0, cc_major = 0, cc_minor = 0;
};
static DeviceProbe g_probe[kMaxDevices];
static int g_no_device = 0;  // 1: the runtime reports no CUDA device at all
static std::mutex g_dev_mutex;

static DeviceProbe *current_probe()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) {
        cudaGetLastError();
        return nullptr;
    }
    return &g_probe[dev];
}

int bevk_require_device(void)
{
    std::lock_guard<std::mutex> lock(g_dev_mutex);
    DeviceProbe *pr = nullptr;
    if (!g_no_device) {
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess || n == 0) {
            g_no_device = 1;
            cudaGetLastError();
        } else {
            pr = current_probe();
        }
    }
    if (pr && pr->state == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) {
            pr->sm_count = prop.multiProcessorCount;
            pr->cc_major = prop.major;
            pr->cc_minor = prop.minor;
            pr->state = (prop.major == 10) ? 1 : -1;
        } else {
            cudaGetLastError();
            pr->state = -1;
        }
    }
    if (!pr || pr->state < 0) {
        bevk_set_error("libbev_b200 needs an sm_100 (B200) CUDA device; found %s (cc %d.%d). "
                       "There is no CPU fallback.",
                       pr && pr->sm_count ? "an unsupported GPU" : "no usable GPU", pr ? pr->cc_major : 0,
                       pr ? pr->cc_minor : 0);
        return BEVK_E_NOGPU;
    }
    return BEVK_OK;
}

int bevk_sm_count(void)
{
    std::lock_guard<std::mutex> lock(g_dev_mutex);
    DeviceProbe *pr = current_probe();
    return (pr && pr->sm_count > 0) ? pr->sm_count : 148;
}

static thread_local int g_warp_path = 0;  // default kernel family of the calling thread (testing aid)

extern "C" {

int bevk_version(void) { return BEVK_VERSION; }
const char *bevk_last_error(void) { return g_err; }

int bevk_device_info(int *sm_count, int *cc_major, int *cc_minor)
{
    int rc = bevk_require_device();
    std::lock_guard<std::mutex> lock(g_dev_mutex);
    DeviceProbe *pr = current_probe();
    if (sm_count) *sm_count = pr ? pr->sm_count : 0;
    if (cc_major) *cc_major = pr ? pr->cc_major : 0;
    if (cc_minor) *cc_minor = pr ? pr->cc_minor : 0;
    return rc;
}

// Adjugate inverse evaluated in the order cv2.invert uses for 3x3 double matrices (host code in
// this file is compiled with -ffp-contract=off, so no product-difference is fused).
int bevk_invert3x3(const double H[9], double M[9])
{
    const double a00 = H[0], a01 = H[1], a02 = H[2];
    const double a10 = H[3], a11 = H[4], a12 = H[5];
    const double a20 = H[6], a21 = H[7], a22 = H[8];
    double d = a00 * (a11 * a22 - a12 * a21) - a01 * (a10 * a22 - a12 * a20) +
               a02 * (a10 * a21 - a11 * a20);
    if (d == 0.0) {
        for (int i = 0; i < 9; ++i) M[i] = 0.0;
        return 0;
    }
    d = 1.0 / d;
    double t[9];
    t[0] = (a11 * a22 - a12 * a21) * d;
    t[1] = (a02 * a21 - a01 * a22) * d;
    t[2] = (a01 * a12 - a02 * a11) * d;
    t[3] = (a12 * a20 - a10 * a22) * d;
    t[4] = (a00 * a22 - a02 * a20) * d;
    t[5] = (a02 * a10 - a00 * a12) * d;
    t[6] = (a10 * a21 - a11 * a20) * d;
    t[7] = (a01 * a20 - a00 * a21) * d;
    t[8] = (a00 * a11 - a01 * a10) * d;
    for (int i = 0; i < 9; ++i) M[i] = t[i];
    return 1;
}

int bevk_warp_set_path(int path)
{
    if (path < 0 || path > 2) BEVK_FAIL(BEVK_E_ARG, "bevk_warp_set_path: path must be 0, 1 or 2");
    g_warp_path = path;
    return BEVK_OK;
}

}  // extern "C"

// ----------------------------------------------------------------------------- warp planning
namespace {

struct WarpArgs {
    int n_frames, src_h, src_w, dst_h, dst_w, channels, dtype, linear;
    size_t elem_size;
    float border[4];
};

// The frame sizes every warp and resize takes: 1..32767.
int check_sizes(const char *what, int src_h, int src_w, int dst_h, int dst_w)
{
    if (src_h <= 0 || src_w <= 0 || dst_h <= 0 || dst_w <= 0)
        BEVK_FAIL(BEVK_E_ARG, "%s: image sizes must be positive (src %dx%d, dst %dx%d)", what, src_w, src_h,
                  dst_w, dst_h);
    if (src_h > 32767 || src_w > 32767 || dst_h > 32767 || dst_w > 32767)
        BEVK_FAIL(BEVK_E_ARG, "%s: sizes above 32767 are not supported (cv2 SHRT_MAX limit)", what);
    return BEVK_OK;
}

int check_warp_args(const void *src, void *dst, int n_frames, int src_h, int src_w, int dst_h,
                    int dst_w, int channels, int dtype, const double *M, int n_mats,
                    const int32_t *mat_index, int flags, int border_mode,
                    const double *border_value, WarpArgs &a)
{
    if (n_frames < 0) BEVK_FAIL(BEVK_E_ARG, "warp: n_frames must be >= 0");
    int rc = check_sizes("warp", src_h, src_w, dst_h, dst_w);
    if (rc) return rc;
    if (channels < 1 || channels > 4) BEVK_FAIL(BEVK_E_ARG, "warp: channels must be 1..4, got %d", channels);
    if (dtype != BEVK_U8 && dtype != BEVK_F16 && dtype != BEVK_F32)
        BEVK_FAIL(BEVK_E_ARG, "warp: dtype must be uint8, float16 or float32 (code %d)", dtype);
    const int interp = flags & ~BEVK_WARP_INVERSE_MAP;
    if (interp != BEVK_INTER_NEAREST && interp != BEVK_INTER_LINEAR)
        BEVK_FAIL(BEVK_E_ARG, "warp: only INTER_NEAREST and INTER_LINEAR are implemented (flags %d)", flags);
    if (border_mode != BEVK_BORDER_CONSTANT)
        BEVK_FAIL(BEVK_E_ARG, "warp: only BORDER_CONSTANT is implemented (borderMode %d)", border_mode);
    if (!M || n_mats < 1) BEVK_FAIL(BEVK_E_ARG, "warp: at least one 3x3 matrix is required");
    if (!mat_index && n_mats != 1 && n_mats != n_frames)
        BEVK_FAIL(BEVK_E_ARG, "warp: %d matrices for %d frames needs a mat_index", n_mats, n_frames);
    if (mat_index)
        for (int i = 0; i < n_frames; ++i)
            if (mat_index[i] < 0 || mat_index[i] >= n_mats)
                BEVK_FAIL(BEVK_E_ARG, "warp: mat_index[%d] = %d out of range [0, %d)", i,
                          mat_index[i], n_mats);
    if (n_frames > 0 && (!src || !dst)) BEVK_FAIL(BEVK_E_ARG, "warp: null src / dst");
    a.n_frames = n_frames;
    a.src_h = src_h;
    a.src_w = src_w;
    a.dst_h = dst_h;
    a.dst_w = dst_w;
    a.channels = channels;
    a.dtype = dtype;
    a.linear = interp == BEVK_INTER_LINEAR;
    a.elem_size = dtype == BEVK_U8 ? 1 : (dtype == BEVK_F16 ? 2 : 4);
    for (int c = 0; c < 4; ++c) a.border[c] = border_value ? (float)border_value[c] : 0.0f;
    return BEVK_OK;
}

// dst->src maps of all matrices (cv2 inverts a forward matrix; WARP_INVERSE_MAP uses it as is)
void effective_maps(const double *M, int n_mats, int flags, std::vector<double> &maps)
{
    maps.resize((size_t)n_mats * 9);
    for (int k = 0; k < n_mats; ++k) {
        if (flags & BEVK_WARP_INVERSE_MAP)
            memcpy(&maps[(size_t)k * 9], M + (size_t)k * 9, 9 * sizeof(double));
        else
            bevk_invert3x3(M + (size_t)k * 9, &maps[(size_t)k * 9]);
    }
}

// Split the frames of every matrix into arithmetic runs (first, count, stride).
void build_groups(int n_frames, int n_mats, const int32_t *mat_index, const std::vector<double> &maps,
                  std::vector<BevkWarpGroup> &groups)
{
    auto push = [&](int k, int first, int count, int stride) {
        BevkWarpGroup g;
        memcpy(g.M, &maps[(size_t)k * 9], 9 * sizeof(double));
        g.first = first;
        g.count = count;
        g.stride = stride;
        g.chunk0 = 0;
        groups.push_back(g);
    };
    if (!mat_index) {
        if (n_mats == 1)
            push(0, 0, n_frames, 1);
        else
            for (int i = 0; i < n_frames; ++i) push(i, i, 1, 1);
        return;
    }
    std::vector<std::vector<int>> per(n_mats);
    for (int i = 0; i < n_frames; ++i) per[mat_index[i]].push_back(i);
    for (int k = 0; k < n_mats; ++k) {
        const std::vector<int> &f = per[k];
        size_t i = 0;
        while (i < f.size()) {
            if (i + 1 == f.size()) {
                push(k, f[i], 1, 1);
                break;
            }
            const int stride = f[i + 1] - f[i];
            size_t j = i + 1;
            while (j + 1 < f.size() && f[j + 1] - f[j] == stride) ++j;
            push(k, f[i], (int)(j - i + 1), stride);
            i = j + 1;
        }
    }
}

// Fill p from a and walk the groups in launches of up to BEVK_MAX_GROUPS: launch() plans and
// launches the groups p holds.
template <typename Launch>
int launch_warp_groups(BevkWarpParams &p, const void *src, void *dst, const WarpArgs &a,
                       const std::vector<BevkWarpGroup> &groups, Launch launch)
{
    memset(&p, 0, sizeof(p));
    p.src = src;
    p.dst = dst;
    p.src_h = a.src_h;
    p.src_w = a.src_w;
    p.dst_h = a.dst_h;
    p.dst_w = a.dst_w;
    p.src_frame_elems = (long long)a.src_h * a.src_w * a.channels;
    p.dst_frame_elems = (long long)a.dst_h * a.dst_w * a.channels;
    p.bw0 = bevk_block_width(a.dst_w, a.dst_h);
    for (int c = 0; c < 4; ++c) p.border[c] = a.border[c];

    for (size_t g0 = 0; g0 < groups.size(); g0 += BEVK_MAX_GROUPS) {
        const int ng = (int)std::min<size_t>(BEVK_MAX_GROUPS, groups.size() - g0);
        p.n_groups = ng;
        for (int i = 0; i < ng; ++i) p.g[i] = groups[g0 + i];
        const int rc = launch();
        if (rc) return rc;
    }
    return BEVK_OK;
}

// The BGR warp: the staged kernel where it qualifies (path 0 or 2), else the direct-gather kernels.
int run_warp_device(const void *src, void *dst, const WarpArgs &a,
                    const std::vector<BevkWarpGroup> &groups, int path, cudaStream_t stream)
{
    BevkWarpParams p;
    return launch_warp_groups(p, src, dst, a, groups, [&]() -> int {
        if (path != 1) {
            const int launched = bevk_launch_warp_fast(p, a.channels, a.dtype, a.linear, path == 2, stream);
            if (launched < 0) return launched;
            if (launched) return BEVK_OK;
            if (path == 2) BEVK_FAIL(BEVK_E_ARG, "warp: shape does not qualify for the staged fast path");
        }
        const int rc = bevk_plan_generic_chunks(p, a.channels);
        if (rc) return rc;
        return bevk_launch_warp_generic(p, a.channels, a.dtype, a.linear, stream);
    });
}

// Source rows referenced by one dst->src map.  A projective map restricted to a line is monotone
// wherever w keeps its sign, so the extreme rows of the dst rectangle are reached on its border:
// evaluate the exact quantised coordinate along the four edges.  If w changes sign inside the
// rectangle (horizon crossing) fall back to the whole frame.
void referenced_rows(const double *Mk, const WarpArgs &a, int &r0, int &r1)
{
    const double cx[4] = {0.0, (double)(a.dst_w - 1), 0.0, (double)(a.dst_w - 1)};
    const double cy[4] = {0.0, 0.0, (double)(a.dst_h - 1), (double)(a.dst_h - 1)};
    int pos = 0, neg = 0;
    for (int i = 0; i < 4; ++i) {
        const double w = Mk[6] * cx[i] + Mk[7] * cy[i] + Mk[8];
        if (w > 0) ++pos;
        else if (w < 0) ++neg;
    }
    if (pos != 4 && neg != 4) {
        r0 = 0;
        r1 = a.src_h - 1;
        return;
    }
    const int bw0 = bevk_block_width(a.dst_w, a.dst_h);
    const double scale = a.linear ? 32.0 : 1.0;
    int lo = 1 << 30, hi = -(1 << 30);
    auto visit = [&](int x, int y) {
        int X, Y;
        bevk_map_pixel(Mk, x, y, bw0, scale, X, Y);
        const int sy = bevk_sat16(a.linear ? (Y >> 5) : Y);
        lo = std::min(lo, sy);
        hi = std::max(hi, sy + (a.linear ? 1 : 0));
    };
    for (int x = 0; x < a.dst_w; ++x) {
        visit(x, 0);
        visit(x, a.dst_h - 1);
    }
    for (int y = 0; y < a.dst_h; ++y) {
        visit(0, y);
        visit(a.dst_w - 1, y);
    }
    r0 = std::max(0, lo - 1);
    r1 = std::min(a.src_h - 1, hi + 1);
    if (r1 < r0) {  // nothing in range: upload one row so sizes stay positive
        r0 = 0;
        r1 = 0;
    }
}

void referenced_rows_union(const std::vector<double> &maps, int n_mats, const WarpArgs &a, int &r0,
                           int &r1)
{
    r0 = a.src_h;
    r1 = -1;
    for (int k = 0; k < n_mats; ++k) {
        int k0, k1;
        referenced_rows(&maps[(size_t)k * 9], a, k0, k1);
        r0 = std::min(r0, k0);
        r1 = std::max(r1, k1);
    }
}

// grow-only device workspace of the host-buffer entry point, one per device: kHostSlots chunks in
// flight, each with its own stream and device buffers.  A workspace is only ever touched under its
// own mutex and is never freed because another device is being used.
constexpr int kHostSlots = 3;
struct HostWorkspace {
    std::mutex mu;
    void *d_src[kHostSlots] = {};
    void *d_dst[kHostSlots] = {};
    size_t src_cap = 0, dst_cap = 0;
    cudaStream_t stream[kHostSlots] = {};
    bool ready = false;
};
HostWorkspace g_ws[kMaxDevices];

// A byte range of every source frame that the host pipeline uploads.
struct HostBand {
    size_t offset, bytes;
};

// The pipelined host-buffer warp of the n_frames > 0 frames of a: frames of src_frame_bytes, of which
// only `bands` are uploaded, to frames of dst_frame_bytes.  Chunks of frames go through the device
// workspace, kHostSlots at a time, so that the copies and kernels of neighbouring chunks overlap.
// run(d_src, d_dst, args, groups, stream) enqueues the kernels of one chunk; maps are the dst->src
// maps of all n_mats matrices.
template <typename Run>
int host_pipeline(const void *src, void *dst, const WarpArgs &a, const std::vector<double> &maps, int n_mats,
                  const int32_t *mat_index, size_t src_frame_bytes, size_t dst_frame_bytes,
                  const std::vector<HostBand> &bands, Run run)
{
    const int n_frames = a.n_frames;
    int chunk = (int)std::max<size_t>(1, (size_t)(64u << 20) / std::max(src_frame_bytes, dst_frame_bytes));
    chunk = std::min(chunk, std::max(1, (n_frames + 3) / 4));
    chunk = std::min(chunk, n_frames);

    int dev = 0;
    BEVK_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= kMaxDevices) BEVK_FAIL(BEVK_E_ARG, "warp: device ordinal %d is not supported", dev);
    HostWorkspace &ws = g_ws[dev];
    std::lock_guard<std::mutex> lock(ws.mu);  // concurrent host calls on one device take turns
    if (!ws.ready) {
        for (int i = 0; i < kHostSlots; ++i)
            BEVK_CUDA(cudaStreamCreateWithFlags(&ws.stream[i], cudaStreamNonBlocking));
        ws.ready = true;
    }
    if (ws.src_cap < src_frame_bytes * chunk) {
        for (int i = 0; i < kHostSlots; ++i) {
            // the previous call synchronised every slot stream before it returned: nothing is in flight
            if (ws.d_src[i]) cudaFree(ws.d_src[i]);
            ws.d_src[i] = nullptr;
        }
        ws.src_cap = 0;
        for (int i = 0; i < kHostSlots; ++i) BEVK_CUDA(cudaMalloc(&ws.d_src[i], src_frame_bytes * chunk));
        ws.src_cap = src_frame_bytes * chunk;
    }
    if (ws.dst_cap < dst_frame_bytes * chunk) {
        for (int i = 0; i < kHostSlots; ++i) {
            if (ws.d_dst[i]) cudaFree(ws.d_dst[i]);
            ws.d_dst[i] = nullptr;
        }
        ws.dst_cap = 0;
        for (int i = 0; i < kHostSlots; ++i) BEVK_CUDA(cudaMalloc(&ws.d_dst[i], dst_frame_bytes * chunk));
        ws.dst_cap = dst_frame_bytes * chunk;
    }

    // From the first enqueue on, every exit -- also an error exit -- first waits for the slot
    // streams: copies in flight still read / write the caller's host buffers.
    auto drain = [&ws]() {
        for (int i = 0; i < kHostSlots; ++i) cudaStreamSynchronize(ws.stream[i]);
    };
#define BEVK_CUDA_DRAIN(expr)                                                                       \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            drain();                                                                                \
            bevk_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return BEVK_E_CUDA;                                                                     \
        }                                                                                           \
    } while (0)

    int slot = 0;
    for (int f0 = 0; f0 < n_frames; f0 += chunk, slot = (slot + 1) % kHostSlots) {
        const int nf = std::min(chunk, n_frames - f0);
        cudaStream_t st = ws.stream[slot];
        // frames are "rows" of a 2-D copy: pitch = whole frame, width = the band
        for (const HostBand &b : bands)
            BEVK_CUDA_DRAIN(cudaMemcpy2DAsync((char *)ws.d_src[slot] + b.offset, src_frame_bytes,
                                              (const char *)src + (size_t)f0 * src_frame_bytes + b.offset,
                                              src_frame_bytes, b.bytes, nf, cudaMemcpyHostToDevice, st));
        std::vector<BevkWarpGroup> groups;
        std::vector<int32_t> idx;
        const int32_t *idx_ptr = nullptr;
        std::vector<double> chunk_maps;
        const std::vector<double> *use_maps = &maps;
        int use_n_mats = n_mats;
        if (mat_index) {
            idx.assign(mat_index + f0, mat_index + f0 + nf);
            idx_ptr = idx.data();
        } else if (n_mats != 1) {  // one matrix per frame: this chunk's slice
            chunk_maps.assign(maps.begin() + (size_t)f0 * 9, maps.begin() + (size_t)(f0 + nf) * 9);
            use_maps = &chunk_maps;
            use_n_mats = nf;
        }
        build_groups(nf, use_n_mats, idx_ptr, *use_maps, groups);
        WarpArgs ac = a;
        ac.n_frames = nf;
        const int rc = run(ws.d_src[slot], ws.d_dst[slot], ac, groups, st);
        if (rc) {
            drain();
            return rc;
        }
        BEVK_CUDA_DRAIN(cudaMemcpyAsync((char *)dst + (size_t)f0 * dst_frame_bytes, ws.d_dst[slot],
                                        dst_frame_bytes * nf, cudaMemcpyDeviceToHost, st));
    }
    for (int i = 0; i < kHostSlots; ++i) BEVK_CUDA_DRAIN(cudaStreamSynchronize(ws.stream[i]));
    return BEVK_OK;
#undef BEVK_CUDA_DRAIN
}

}  // namespace

extern "C" {

int bevk_warp_perspective(const void *src, void *dst, int n_frames, int src_h, int src_w,
                          int dst_h, int dst_w, int channels, int dtype, const double *M,
                          int n_mats, const int32_t *mat_index, int flags, int border_mode,
                          const double *border_value, void *stream)
{
    return bevk_warp_perspective_path(src, dst, n_frames, src_h, src_w, dst_h, dst_w, channels, dtype, M,
                                      n_mats, mat_index, flags, border_mode, border_value, -1, stream);
}

int bevk_warp_perspective_path(const void *src, void *dst, int n_frames, int src_h, int src_w,
                               int dst_h, int dst_w, int channels, int dtype, const double *M,
                               int n_mats, const int32_t *mat_index, int flags, int border_mode,
                               const double *border_value, int path, void *stream)
{
    if (path < -1 || path > 2) BEVK_FAIL(BEVK_E_ARG, "warp: path must be -1 (thread default), 0, 1 or 2");
    if (path < 0) path = g_warp_path;
    WarpArgs a;
    int rc = check_warp_args(src, dst, n_frames, src_h, src_w, dst_h, dst_w, channels, dtype, M,
                             n_mats, mat_index, flags, border_mode, border_value, a);
    if (rc) return rc;
    rc = bevk_require_device();
    if (rc) return rc;
    if (n_frames == 0) return BEVK_OK;
    std::vector<double> maps;
    effective_maps(M, n_mats, flags, maps);
    std::vector<BevkWarpGroup> groups;
    build_groups(n_frames, n_mats, mat_index, maps, groups);
    return run_warp_device(src, dst, a, groups, path, (cudaStream_t)stream);
}

}  // extern "C"

namespace {
// The NV12 frame rules of the NV12 entry points: even sizes, rows at least a luma row apart.
int check_nv12_layout(const char *what, int n_frames, int h, int w, int pitch, int64_t frame_stride)
{
    if (n_frames < 0) BEVK_FAIL(BEVK_E_ARG, "%s: n_frames must be >= 0", what);
    if (h <= 0 || w <= 0 || (h % 2) != 0 || (w % 2) != 0)
        BEVK_FAIL(BEVK_E_ARG, "%s: NV12 frames need an even, positive width and height (got %dx%d)", what, w, h);
    if (pitch < w) BEVK_FAIL(BEVK_E_ARG, "%s: pitch %d is smaller than the width %d", what, pitch, w);
    if (frame_stride < 0) BEVK_FAIL(BEVK_E_ARG, "%s: negative frame stride", what);
    return BEVK_OK;
}

// check_nv12_layout for the fused kernels, which address a frame with 32-bit byte offsets
int check_nv12_layout32(const char *what, int n_frames, int h, int w, int pitch, int64_t frame_stride)
{
    int rc = check_nv12_layout(what, n_frames, h, w, pitch, frame_stride);
    if (rc) return rc;
    if ((int64_t)pitch * (h / 2 * 3) > 0xffffffffLL)
        BEVK_FAIL(BEVK_E_ARG, "%s: a frame of pitch %d and %d rows spans 4 GB or more", what, pitch, h / 2 * 3);
    return BEVK_OK;
}

// The resize entry points after their frame-format checks: n_frames >= 0 frames of `channels`
// uint8 channels, or NV12 frames (nv12, channels 3) converted to BGR; rows `pitch` and frames
// `frame_stride` bytes apart.
int resize_frames(const char *what, const void *src, void *dst, int n_frames, int src_h, int src_w, int channels,
                  int nv12, long long pitch, long long frame_stride, int dst_h, int dst_w, int interpolation,
                  void *stream)
{
    if (interpolation != BEVK_INTER_LINEAR && interpolation != BEVK_INTER_AREA)
        BEVK_FAIL(BEVK_E_ARG, "%s: only INTER_LINEAR (cv2.resize's default) and INTER_AREA are implemented, got %d",
                  what, interpolation);
    int rc = check_sizes(what, src_h, src_w, dst_h, dst_w);
    if (rc) return rc;
    if (n_frames > 0 && (!src || !dst)) BEVK_FAIL(BEVK_E_ARG, "%s: null src / dst", what);
    rc = bevk_require_device();
    if (rc) return rc;
    if (n_frames == 0) return BEVK_OK;
    return bevk_launch_resize(src, dst, n_frames, src_h, src_w, channels, nv12, pitch, frame_stride, dst_h, dst_w,
                              interpolation, (cudaStream_t)stream);
}
// The YUV 4:2:0 destinations (I420 or NV12 frames of h x w): even sizes, rows at least w bytes
// apart, in-frame offsets below 4 GB.
int check_yuv420_dst(const char *what, int n_frames, int h, int w, int layout, int pitch, int64_t frame_stride)
{
    if (layout != BEVK_YUV_I420 && layout != BEVK_YUV_NV12)
        BEVK_FAIL(BEVK_E_ARG, "%s: layout must be BEVK_YUV_I420 (0) or BEVK_YUV_NV12 (1), got %d", what, layout);
    if (h <= 0 || w <= 0 || (h % 2) != 0 || (w % 2) != 0)
        BEVK_FAIL(BEVK_E_ARG, "%s: YUV 4:2:0 frames need an even, positive width and height (got %dx%d)", what, w, h);
    return check_nv12_layout32(what, n_frames, h, w, pitch, frame_stride);
}

// The fused warps to YUV 4:2:0 of these groups on device buffers: BGR (src_format BEVK_BGR,
// contiguous frames), NV12 or I420 frames, rows `pitch` and frames `frame_stride` bytes apart.
int run_warp_yuv420(const void *src, void *dst, const WarpArgs &a, const std::vector<BevkWarpGroup> &groups,
                    int src_format, long long pitch, long long frame_stride, int layout, int dst_pitch,
                    int64_t dst_frame_stride, cudaStream_t stream)
{
    BevkYuvParams P;
    memset(&P, 0, sizeof(P));
    P.pitch = (int)pitch;
    P.frame_stride = frame_stride;
    P.dst_pitch = dst_pitch;
    P.dst_frame_stride = dst_frame_stride;
    return launch_warp_groups(P.w, src, dst, a, groups, [&]() {
        // a thread owns a 2x2 dst block: plan the frame chunks over the grid of blocks
        P.w.dst_w /= 2;
        P.w.dst_h /= 2;
        const int rc = bevk_plan_generic_chunks(P.w, 3);
        P.w.dst_w *= 2;
        P.w.dst_h *= 2;
        if (rc) return rc;
        return bevk_launch_warp_yuv420(P, src_format, layout == BEVK_YUV_NV12, a.linear, stream);
    });
}

// The NV12 or I420 (src_format) to BGR warp of these groups on device buffers.
int run_warp_yuv_bgr(const void *src, void *dst, const WarpArgs &a, const std::vector<BevkWarpGroup> &groups,
                     int src_format, int pitch, int64_t frame_stride, cudaStream_t stream)
{
    BevkNv12Params P;
    memset(&P, 0, sizeof(P));
    P.pitch = pitch;
    P.frame_stride = frame_stride;
    return launch_warp_groups(P.w, src, dst, a, groups, [&]() {
        const int rc = bevk_plan_generic_chunks(P.w, 3);
        if (rc) return rc;
        return bevk_launch_warp_nv12(P, src_format, a.linear, stream);
    });
}

// The fused warps to YUV 4:2:0 after their source-layout checks: BGR (src_format BEVK_BGR,
// contiguous frames) or NV12 frames, rows `pitch` and frames `frame_stride` bytes apart.
int warp_yuv420(const char *what, const void *src, void *dst, int n_frames, int src_h, int src_w, int src_format,
                long long pitch, long long frame_stride, int dst_h, int dst_w, int layout, int dst_pitch,
                int64_t dst_frame_stride, const double *M, int n_mats, const int32_t *mat_index, int flags,
                int border_mode, const double *border_value, void *stream)
{
    int rc = check_yuv420_dst(what, n_frames, dst_h, dst_w, layout, dst_pitch, dst_frame_stride);
    if (rc) return rc;
    WarpArgs a;
    rc = check_warp_args(src, dst, n_frames, src_h, src_w, dst_h, dst_w, 3, BEVK_U8, M, n_mats, mat_index, flags,
                         border_mode, border_value, a);
    if (rc) return rc;
    rc = bevk_require_device();
    if (rc) return rc;
    if (n_frames == 0) return BEVK_OK;
    std::vector<double> maps;
    effective_maps(M, n_mats, flags, maps);
    std::vector<BevkWarpGroup> groups;
    build_groups(n_frames, n_mats, mat_index, maps, groups);
    return run_warp_yuv420(src, dst, a, groups, src_format, pitch, frame_stride, layout, dst_pitch, dst_frame_stride,
                           (cudaStream_t)stream);
}
}  // namespace

extern "C" {

int bevk_nv12_to_bgr(const void *src, void *dst, int n_frames, int h, int w, int pitch,
                     int64_t frame_stride, void *stream)
{
    int rc = check_nv12_layout("nv12_to_bgr", n_frames, h, w, pitch, frame_stride);
    if (rc) return rc;
    if (n_frames > 0 && (!src || !dst)) BEVK_FAIL(BEVK_E_ARG, "nv12_to_bgr: null src / dst");
    rc = bevk_require_device();
    if (rc) return rc;
    if (n_frames == 0) return BEVK_OK;
    return bevk_launch_nv12_to_bgr(src, dst, n_frames, h, w, pitch, frame_stride, (cudaStream_t)stream);
}

int bevk_warp_perspective_nv12(const void *src, void *dst, int n_frames, int src_h, int src_w,
                               int pitch, int64_t frame_stride, int dst_h, int dst_w,
                               const double *M, int n_mats, const int32_t *mat_index, int flags,
                               int border_mode, const double *border_value, void *stream)
{
    int rc = check_nv12_layout32("warp_nv12", n_frames, src_h, src_w, pitch, frame_stride);
    if (rc) return rc;
    WarpArgs a;
    rc = check_warp_args(src, dst, n_frames, src_h, src_w, dst_h, dst_w, 3, BEVK_U8, M, n_mats, mat_index,
                         flags, border_mode, border_value, a);
    if (rc) return rc;
    rc = bevk_require_device();
    if (rc) return rc;
    if (n_frames == 0) return BEVK_OK;
    std::vector<double> maps;
    effective_maps(M, n_mats, flags, maps);
    std::vector<BevkWarpGroup> groups;
    build_groups(n_frames, n_mats, mat_index, maps, groups);
    return run_warp_yuv_bgr(src, dst, a, groups, BEVK_YUV_NV12, pitch, frame_stride, (cudaStream_t)stream);
}

int bevk_bgr_to_yuv420(const void *src, void *dst, int n_frames, int h, int w, int layout, int dst_pitch,
                       int64_t dst_frame_stride, void *stream)
{
    int rc = check_yuv420_dst("bgr_to_yuv420", n_frames, h, w, layout, dst_pitch, dst_frame_stride);
    if (rc) return rc;
    if (w > 32767 || h > 32767) BEVK_FAIL(BEVK_E_ARG, "bgr_to_yuv420: sizes above 32767 are not supported");
    if (n_frames > 0 && (!src || !dst)) BEVK_FAIL(BEVK_E_ARG, "bgr_to_yuv420: null src / dst");
    rc = bevk_require_device();
    if (rc) return rc;
    if (n_frames == 0) return BEVK_OK;
    return bevk_launch_bgr_to_yuv420(src, dst, n_frames, h, w, layout == BEVK_YUV_NV12, dst_pitch, dst_frame_stride,
                                     (cudaStream_t)stream);
}

int bevk_warp_perspective_yuv420(const void *src, void *dst, int n_frames, int src_h, int src_w, int dst_h,
                                 int dst_w, int layout, int dst_pitch, int64_t dst_frame_stride, const double *M,
                                 int n_mats, const int32_t *mat_index, int flags, int border_mode,
                                 const double *border_value, void *stream)
{
    return warp_yuv420("warp_yuv420", src, dst, n_frames, src_h, src_w, BEVK_BGR, 3LL * src_w,
                       3LL * src_w * src_h, dst_h, dst_w, layout, dst_pitch, dst_frame_stride, M, n_mats, mat_index,
                       flags, border_mode, border_value, stream);
}

int bevk_warp_perspective_nv12_yuv420(const void *src, void *dst, int n_frames, int src_h, int src_w, int pitch,
                                      int64_t frame_stride, int dst_h, int dst_w, int layout, int dst_pitch,
                                      int64_t dst_frame_stride, const double *M, int n_mats,
                                      const int32_t *mat_index, int flags, int border_mode,
                                      const double *border_value, void *stream)
{
    const int rc = check_nv12_layout32("warp_nv12_yuv420", n_frames, src_h, src_w, pitch, frame_stride);
    if (rc) return rc;
    return warp_yuv420("warp_nv12_yuv420", src, dst, n_frames, src_h, src_w, BEVK_YUV_NV12, pitch, frame_stride,
                       dst_h, dst_w, layout, dst_pitch, dst_frame_stride, M, n_mats, mat_index, flags, border_mode,
                       border_value, stream);
}

int bevk_resize(const void *src, void *dst, int n_frames, int src_h, int src_w, int dst_h, int dst_w, int channels,
                int dtype, int interpolation, void *stream)
{
    if (n_frames < 0) BEVK_FAIL(BEVK_E_ARG, "resize: n_frames must be >= 0");
    if (channels < 1 || channels > 4) BEVK_FAIL(BEVK_E_ARG, "resize: channels must be 1..4, got %d", channels);
    if (dtype != BEVK_U8) BEVK_FAIL(BEVK_E_ARG, "resize: only uint8 frames are implemented (dtype code %d)", dtype);
    return resize_frames("resize", src, dst, n_frames, src_h, src_w, channels, 0, (long long)src_w * channels,
                         (long long)src_h * src_w * channels, dst_h, dst_w, interpolation, stream);
}

int bevk_resize_nv12(const void *src, void *dst, int n_frames, int src_h, int src_w, int pitch,
                     int64_t frame_stride, int dst_h, int dst_w, void *stream)
{
    return bevk_resize_nv12_interp(src, dst, n_frames, src_h, src_w, pitch, frame_stride, dst_h, dst_w,
                                   BEVK_INTER_LINEAR, stream);
}

int bevk_resize_nv12_interp(const void *src, void *dst, int n_frames, int src_h, int src_w, int pitch,
                            int64_t frame_stride, int dst_h, int dst_w, int interpolation, void *stream)
{
    const int rc = check_nv12_layout32("resize_nv12", n_frames, src_h, src_w, pitch, frame_stride);
    if (rc) return rc;
    return resize_frames("resize_nv12", src, dst, n_frames, src_h, src_w, 3, 1, pitch, frame_stride, dst_h, dst_w,
                         interpolation, stream);
}

int bevk_warp_host_rows(int src_h, int src_w, int dst_h, int dst_w, const double *M, int n_mats,
                        int flags, int rows[2])
{
    if (!M || !rows || n_mats < 1 || src_h <= 0 || src_w <= 0 || dst_h <= 0 || dst_w <= 0)
        BEVK_FAIL(BEVK_E_ARG, "bevk_warp_host_rows: bad arguments");
    WarpArgs a = {};
    a.src_h = src_h;
    a.src_w = src_w;
    a.dst_h = dst_h;
    a.dst_w = dst_w;
    a.linear = (flags & 7) == BEVK_INTER_LINEAR;
    std::vector<double> maps;
    effective_maps(M, n_mats, flags, maps);
    referenced_rows_union(maps, n_mats, a, rows[0], rows[1]);
    return BEVK_OK;
}

int bevk_warp_perspective_host(const void *src, void *dst, int n_frames, int src_h, int src_w,
                               int dst_h, int dst_w, int channels, int dtype, const double *M,
                               int n_mats, const int32_t *mat_index, int flags, int border_mode,
                               const double *border_value)
{
    WarpArgs a;
    int rc = check_warp_args(src, dst, n_frames, src_h, src_w, dst_h, dst_w, channels, dtype, M,
                             n_mats, mat_index, flags, border_mode, border_value, a);
    if (rc) return rc;
    rc = bevk_require_device();
    if (rc) return rc;
    if (n_frames == 0) return BEVK_OK;
    std::vector<double> maps;
    effective_maps(M, n_mats, flags, maps);

    // union of the source rows any matrix references: only those are uploaded
    int r0, r1;
    referenced_rows_union(maps, n_mats, a, r0, r1);
    const size_t row_bytes = (size_t)a.src_w * a.channels * a.elem_size;
    const size_t dst_frame_bytes = (size_t)a.dst_w * a.dst_h * a.channels * a.elem_size;
    return host_pipeline(src, dst, a, maps, n_mats, mat_index, row_bytes * a.src_h, dst_frame_bytes,
                         {{r0 * row_bytes, row_bytes * (size_t)(r1 - r0 + 1)}},
                         [](const void *s, void *d, const WarpArgs &ac, const std::vector<BevkWarpGroup> &groups,
                            cudaStream_t st) { return run_warp_device(s, d, ac, groups, g_warp_path, st); });
}

int bevk_warp_perspective_video_host(const void *src, int src_format, void *dst, int dst_format, int n_frames,
                                     int src_h, int src_w, int dst_h, int dst_w, const double *M, int n_mats,
                                     const int32_t *mat_index, int flags, int border_mode,
                                     const double *border_value)
{
    const char *what = "warp_video_host";
    auto known = [](int f) { return f == BEVK_BGR || f == BEVK_YUV_I420 || f == BEVK_YUV_NV12; };
    if (!known(src_format) || !known(dst_format))
        BEVK_FAIL(BEVK_E_ARG, "%s: formats must be BEVK_YUV_I420 (0), BEVK_YUV_NV12 (1) or BEVK_BGR (2), got src %d, "
                  "dst %d", what, src_format, dst_format);
    const bool yuv_src = src_format != BEVK_BGR, yuv_dst = dst_format != BEVK_BGR;
    int rc;
    if (yuv_src) {
        rc = check_nv12_layout32(what, n_frames, src_h, src_w, src_w, (int64_t)src_w * src_h / 2 * 3);
        if (rc) return rc;
    }
    if (yuv_dst) {
        rc = check_yuv420_dst(what, n_frames, dst_h, dst_w, dst_format, dst_w, (int64_t)dst_w * dst_h / 2 * 3);
        if (rc) return rc;
    }
    WarpArgs a;
    rc = check_warp_args(src, dst, n_frames, src_h, src_w, dst_h, dst_w, 3, BEVK_U8, M, n_mats, mat_index, flags,
                         border_mode, border_value, a);
    if (rc) return rc;
    rc = bevk_require_device();
    if (rc) return rc;
    if (n_frames == 0) return BEVK_OK;
    std::vector<double> maps;
    effective_maps(M, n_mats, flags, maps);

    // the referenced luma (BGR) row band [r0, r1] and, for YUV, the chroma rows under it
    int r0, r1;
    referenced_rows_union(maps, n_mats, a, r0, r1);
    const size_t h = (size_t)src_h, w = (size_t)src_w, rows = (size_t)(r1 - r0 + 1);
    size_t src_frame_bytes;
    std::vector<HostBand> bands;
    if (!yuv_src) {
        src_frame_bytes = 3 * w * h;
        bands.push_back({3 * w * r0, 3 * w * rows});
    } else {
        src_frame_bytes = w * h / 2 * 3;
        bands.push_back({w * r0, w * rows});
        const size_t c0 = (size_t)(r0 / 2), nc = (size_t)(r1 / 2) - c0 + 1;
        if (src_format == BEVK_YUV_NV12) {
            bands.push_back({w * (h + c0), w * nc});
        } else {  // the U plane, then the V plane: (h / 2) x (w / 2) each, contiguous
            const size_t cw = w / 2;
            bands.push_back({w * h + cw * c0, cw * nc});
            bands.push_back({w * h + cw * (h / 2 + c0), cw * nc});
        }
    }
    const size_t dst_frame_bytes = (size_t)dst_w * dst_h * (yuv_dst ? 1 : 2) * 3 / 2;
    const long long pitch = yuv_src ? src_w : 3LL * src_w;
    return host_pipeline(src, dst, a, maps, n_mats, mat_index, src_frame_bytes, dst_frame_bytes, bands,
                         [&](const void *s, void *d, const WarpArgs &ac, const std::vector<BevkWarpGroup> &groups,
                             cudaStream_t st) -> int {
                             if (yuv_dst)
                                 return run_warp_yuv420(s, d, ac, groups, src_format, pitch, src_frame_bytes,
                                                        dst_format, dst_w, dst_frame_bytes, st);
                             if (yuv_src)
                                 return run_warp_yuv_bgr(s, d, ac, groups, src_format, src_w, src_frame_bytes, st);
                             return run_warp_device(s, d, ac, groups, g_warp_path, st);
                         });
}

}  // extern "C"
