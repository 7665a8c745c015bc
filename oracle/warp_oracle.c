/*
 * oracle/warp_oracle.c -- TEST INFRASTRUCTURE ONLY.
 *
 * CPU restatement of the perspective warp the reference performs at
 *   /root/reference/vis_homo.py:89,91 and /root/reference/bev/tool/compo.py:38,46,47
 * (cv2.warpPerspective with default flags). The arithmetic lives in third-party
 * OpenCV, un-vendored and un-pinned by the reference; the version it resolves to in
 * this image is opencv-python-headless 4.13.0.92. This file restates that library's
 * observable behaviour (SURVEY.md Appendix A) and is pinned bit-for-bit against the
 * live cv2 build by tests/test_oracle_warp.py and against the fixtures under tests/golden/.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load this. The product path (bev_b200/) never does.
 *
 * Build: see oracle/Makefile (gcc -O2 -ffp-contract=off: coordinate math must stay
 * unfused IEEE double).
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define BEVO_INTER_NEAREST 0
#define BEVO_INTER_LINEAR 1
#define BEVO_WARP_INVERSE_MAP 16

#define BEVO_U8 0
#define BEVO_F32 2

/* 3x3 inverse exactly as cv2.invert evaluates it for a 3x3 double matrix:
 * determinant by first-row cofactor expansion, d = 1/det, every adjugate entry
 * (a*b - c*d) * d. Returns 0 when det == 0 (cv2 then yields the zero matrix). */
int bevo_invert3x3(const double *H, double *M)
{
    const double a00 = H[0], a01 = H[1], a02 = H[2];
    const double a10 = H[3], a11 = H[4], a12 = H[5];
    const double a20 = H[6], a21 = H[7], a22 = H[8];
    double d = a00 * (a11 * a22 - a12 * a21) - a01 * (a10 * a22 - a12 * a20) +
               a02 * (a10 * a21 - a11 * a20);
    if (d == 0.0) {
        memset(M, 0, 9 * sizeof(double));
        return 0;
    }
    d = 1.0 / d;
    M[0] = (a11 * a22 - a12 * a21) * d;
    M[1] = (a02 * a21 - a01 * a22) * d;
    M[2] = (a01 * a12 - a02 * a11) * d;
    M[3] = (a12 * a20 - a10 * a22) * d;
    M[4] = (a00 * a22 - a02 * a20) * d;
    M[5] = (a02 * a10 - a00 * a12) * d;
    M[6] = (a10 * a21 - a11 * a20) * d;
    M[7] = (a01 * a20 - a00 * a21) * d;
    M[8] = (a00 * a11 - a01 * a10) * d;
    return 1;
}

static inline int sat_int(double v)
{
    /* clamp to the int32 range, then round half to even (default FP environment) */
    if (v < -2147483648.0) v = -2147483648.0;
    if (v > 2147483647.0) v = 2147483647.0;
    return (int)lrint(v);
}

static inline int sat16(int v)
{
    return v < -32768 ? -32768 : (v > 32767 ? 32767 : v);
}

/* Quantised source coordinate of dst pixel (x, y) under the dst->src map M.
 * scale is 32 for bilinear (1/32 px sub-pixel grid) or 1 for nearest.
 * The column is split into a block base xb (blocks of bw0 columns) and an in-block
 * offset x1, and the products are summed in exactly this order -- exact-tie pixels
 * flip otherwise (SURVEY.md Appendix A note 2). */
static inline void map_pixel(const double *M, int x, int y, int bw0, double scale, int *X, int *Y)
{
    const int xb = (x / bw0) * bw0;
    const int x1 = x - xb;
    const double X0 = (M[0] * xb + M[1] * y) + M[2];
    const double Y0 = (M[3] * xb + M[4] * y) + M[5];
    const double W0 = (M[6] * xb + M[7] * y) + M[8];
    double w = W0 + M[6] * x1;
    w = (w != 0.0) ? scale / w : 0.0;
    *X = sat_int((X0 + M[0] * x1) * w);
    *Y = sat_int((Y0 + M[3] * x1) * w);
}

static inline int block_width(int dst_w, int dst_h)
{
    int bh0 = dst_h < 16 ? dst_h : 16;
    int bw0 = 1024 / bh0;
    if (bw0 > dst_w) bw0 = dst_w;
    return bw0;
}

/* dst->src map from the user matrix and flags (cv2 inverts unless WARP_INVERSE_MAP). */
static void effective_map(const double *H, int flags, double *M)
{
    if (flags & BEVO_WARP_INVERSE_MAP)
        memcpy(M, H, 9 * sizeof(double));
    else
        bevo_invert3x3(H, M);
}

/*
 * One frame. src: [src_h][src_w][ch] contiguous, dst: [dst_h][dst_w][ch] contiguous.
 * dtype BEVO_U8 or BEVO_F32. border: per-channel constant (BORDER_CONSTANT only).
 * Returns 0 on success, <0 on bad arguments.
 */
int bevo_warp_perspective(const void *src_, int src_h, int src_w, int ch, int dtype, void *dst_,
                          int dst_h, int dst_w, const double *H, int flags, const double *border)
{
    if (!src_ || !dst_ || !H || ch < 1 || ch > 4 || dst_h <= 0 || dst_w <= 0 || src_h <= 0 ||
        src_w <= 0)
        return -1;
    const int interp = flags & 7;
    if (interp != BEVO_INTER_NEAREST && interp != BEVO_INTER_LINEAR) return -2;
    if (dtype != BEVO_U8 && dtype != BEVO_F32) return -3;

    double M[9];
    effective_map(H, flags, M);
    const int bw0 = block_width(dst_w, dst_h);
    const double zero4[4] = {0, 0, 0, 0};
    if (!border) border = zero4;

    for (int y = 0; y < dst_h; ++y) {
        for (int x = 0; x < dst_w; ++x) {
            int X, Y;
            if (interp == BEVO_INTER_NEAREST) {
                map_pixel(M, x, y, bw0, 1.0, &X, &Y);
                const int sx = sat16(X), sy = sat16(Y);
                const int inside = (sx >= 0 && sx < src_w && sy >= 0 && sy < src_h);
                for (int c = 0; c < ch; ++c) {
                    const size_t di = ((size_t)y * dst_w + x) * ch + c;
                    const size_t si = ((size_t)sy * src_w + sx) * ch + c;
                    if (dtype == BEVO_U8) {
                        uint8_t bv = (uint8_t)(border[c] < 0 ? 0 : (border[c] > 255 ? 255 : lrint(border[c])));
                        ((uint8_t *)dst_)[di] = inside ? ((const uint8_t *)src_)[si] : bv;
                    } else {
                        ((float *)dst_)[di] = inside ? ((const float *)src_)[si] : (float)border[c];
                    }
                }
                continue;
            }
            map_pixel(M, x, y, bw0, 32.0, &X, &Y);
            const int sx = sat16(X >> 5), sy = sat16(Y >> 5); /* arithmetic shift */
            const int ax = X & 31, ay = Y & 31;
            const int in00 = (sx >= 0 && sx < src_w && sy >= 0 && sy < src_h);
            const int in01 = (sx + 1 >= 0 && sx + 1 < src_w && sy >= 0 && sy < src_h);
            const int in10 = (sx >= 0 && sx < src_w && sy + 1 >= 0 && sy + 1 < src_h);
            const int in11 = (sx + 1 >= 0 && sx + 1 < src_w && sy + 1 >= 0 && sy + 1 < src_h);
            const size_t b00 = ((size_t)((long)sy * src_w + sx)) * ch;
            const size_t b01 = b00 + ch;
            const size_t b10 = b00 + (size_t)src_w * ch;
            const size_t b11 = b10 + ch;
            if (dtype == BEVO_U8) {
                const int w00 = (32 - ax) * (32 - ay) * 32, w01 = ax * (32 - ay) * 32;
                const int w10 = (32 - ax) * ay * 32, w11 = ax * ay * 32;
                const uint8_t *s = (const uint8_t *)src_;
                uint8_t *d = (uint8_t *)dst_ + ((size_t)y * dst_w + x) * ch;
                for (int c = 0; c < ch; ++c) {
                    const int bv = (int)(border[c] < 0 ? 0 : (border[c] > 255 ? 255 : lrint(border[c])));
                    const int p00 = in00 ? s[b00 + c] : bv, p01 = in01 ? s[b01 + c] : bv;
                    const int p10 = in10 ? s[b10 + c] : bv, p11 = in11 ? s[b11 + c] : bv;
                    const int v = (w00 * p00 + w01 * p01 + w10 * p10 + w11 * p11 + 16384) >> 15;
                    d[c] = (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v));
                }
            } else if (!(in00 || in01 || in10 || in11)) {
                /* no tap inside: cv2 stores the border value itself, not the weighted sum of four
                 * copies of it (which can miss it by an ulp) */
                float *d = (float *)dst_ + ((size_t)y * dst_w + x) * ch;
                for (int c = 0; c < ch; ++c) d[c] = (float)border[c];
            } else {
                const float tx = (float)ax * (1.0f / 32.0f), ty = (float)ay * (1.0f / 32.0f);
                const float w00 = (1.0f - ty) * (1.0f - tx), w01 = (1.0f - ty) * tx;
                const float w10 = ty * (1.0f - tx), w11 = ty * tx;
                const float *s = (const float *)src_;
                float *d = (float *)dst_ + ((size_t)y * dst_w + x) * ch;
                for (int c = 0; c < ch; ++c) {
                    const float bv = (float)border[c];
                    const float p00 = in00 ? s[b00 + c] : bv, p01 = in01 ? s[b01 + c] : bv;
                    const float p10 = in10 ? s[b10 + c] : bv, p11 = in11 ? s[b11 + c] : bv;
                    d[c] = ((p00 * w00 + p01 * w01) + p10 * w10) + p11 * w11;
                }
            }
        }
    }
    return 0;
}

/* Batch of n frames sharing one matrix (serial; callers thread over frames from Python --
 * ctypes releases the GIL -- because this image's gcc has no libgomp). */
int bevo_warp_perspective_batch(const void *src, int n, int src_h, int src_w, int ch, int dtype,
                                void *dst, int dst_h, int dst_w, const double *H, int flags,
                                const double *border)
{
    const size_t es = dtype == BEVO_U8 ? 1 : 4;
    const size_t sfs = (size_t)src_h * src_w * ch * es, dfs = (size_t)dst_h * dst_w * ch * es;
    int rc = 0;
    for (int i = 0; i < n; ++i) {
        int r = bevo_warp_perspective((const char *)src + i * sfs, src_h, src_w, ch, dtype,
                                      (char *)dst + i * dfs, dst_h, dst_w, H, flags, border);
        if (r) rc = r;
    }
    return rc;
}

/*
 * Roofline accounting (SURVEY.md 8d): T = number of distinct in-bounds source pixels that any
 * tap of the coordinate map references (4 taps bilinear, 1 nearest). Also returns through
 * row_range[2] the min / max source row touched (used by the host-buffer entry point tests).
 * Returns T, or <0 on error.
 */
long bevo_touched_pixels(int src_h, int src_w, int dst_h, int dst_w, const double *H, int flags,
                         int *row_range)
{
    const int interp = flags & 7;
    if (interp != BEVO_INTER_NEAREST && interp != BEVO_INTER_LINEAR) return -2;
    double M[9];
    effective_map(H, flags, M);
    const int bw0 = block_width(dst_w, dst_h);
    uint8_t *mark = (uint8_t *)calloc((size_t)src_h * src_w, 1);
    if (!mark) return -4;
    int rmin = src_h, rmax = -1;
    for (int y = 0; y < dst_h; ++y)
        for (int x = 0; x < dst_w; ++x) {
            int X, Y;
            map_pixel(M, x, y, bw0, interp == BEVO_INTER_LINEAR ? 32.0 : 1.0, &X, &Y);
            int sx, sy, nt;
            if (interp == BEVO_INTER_LINEAR) {
                sx = sat16(X >> 5);
                sy = sat16(Y >> 5);
                nt = 2;
            } else {
                sx = sat16(X);
                sy = sat16(Y);
                nt = 1;
            }
            for (int j = 0; j < nt; ++j)
                for (int i = 0; i < nt; ++i) {
                    const int u = sx + i, v = sy + j;
                    if (u >= 0 && u < src_w && v >= 0 && v < src_h) {
                        mark[(size_t)v * src_w + u] = 1;
                        if (v < rmin) rmin = v;
                        if (v > rmax) rmax = v;
                    }
                }
        }
    long T = 0;
    for (size_t i = 0; i < (size_t)src_h * src_w; ++i) T += mark[i];
    free(mark);
    if (row_range) {
        row_range[0] = rmin;
        row_range[1] = rmax;
    }
    return T;
}
