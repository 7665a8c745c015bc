/*
 * bev_b200.h -- C ABI of libbev_b200.so: the B200 (sm_100a) hot path of minghanz/bev.
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes (no torch / numpy types),
 * returns 0 on success or a negative BEVK_E_* code, and leaves a human-readable message for
 * bevk_last_error() (thread-local).  Device-pointer entry points enqueue on `stream`
 * (a cudaStream_t passed as void*; NULL = the legacy default stream) and return without
 * synchronising.  `*_host` entry points take HOST buffers, move the data themselves (pipelined
 * H2D / kernel / D2H on internal streams) and return when the result is in the host buffer.
 *
 * Each function cites the reference interface it replaces (paths relative to the reference
 * checkout of minghanz/bev).  The arithmetic contract (bit-exact vs cv2 4.13 for uint8/float32,
 * 1e-5 relative vs the reference's float64 numpy path for projections) is stated in DESIGN.md.
 */
#ifndef BEV_B200_H
#define BEV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BEVK_VERSION 100

/* flags: same numeric values as cv2.INTER_NEAREST / INTER_LINEAR / WARP_INVERSE_MAP */
#define BEVK_INTER_NEAREST 0
#define BEVK_INTER_LINEAR 1
/* resize only: cv2.INTER_AREA */
#define BEVK_INTER_AREA 3
#define BEVK_WARP_INVERSE_MAP 16
/* border_mode: cv2.BORDER_CONSTANT (the only mode any reference call site uses) */
#define BEVK_BORDER_CONSTANT 0

/* element types */
#define BEVK_U8 0
#define BEVK_F16 1
#define BEVK_F32 2
#define BEVK_F64 3

/* coordinate conventions of bev/rbox_torch.py:12-22 */
#define BEVK_MODE_BEV 0   /* yaw 0 = +v, yaw = atan2(u, v); w along u, h along v */
#define BEVK_MODE_WORLD 1 /* yaw 0 = +x, yaw = atan2(y, x); h along x, w along y */

/* error codes */
#define BEVK_OK 0
#define BEVK_E_ARG (-1)     /* bad argument (message says which) */
#define BEVK_E_CUDA (-2)    /* CUDA runtime error */
#define BEVK_E_NOGPU (-3)   /* no sm_100 device / driver */
#define BEVK_E_AFFINE (-4)  /* H is not affine / not a similarity where the reference asserts it */

int bevk_version(void);
const char *bevk_last_error(void);
/* Fills SM count and compute capability of the current device; BEVK_E_NOGPU without one. */
int bevk_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* Host helper: 3x3 adjugate inverse, bit-equal to cv2.invert (which cv2.warpPerspective applies
 * to a forward matrix).  Returns 1, or 0 when det == 0 (M is then all zeros, as in cv2). */
int bevk_invert3x3(const double H[9], double M[9]);

/*
 * Batched perspective warp.  Replaces the per-frame loop around
 *     cv2.warpPerspective(img, H_bev_img, (bspec.u_size, bspec.v_size))
 * at vis_homo.py:85-91 and the three warps of bev/tool/compo.py:38,46,47.
 *
 *   src  [n_frames][src_h][src_w][channels]  contiguous, interleaved channels (cv2 HWC layout)
 *   dst  [n_frames][dst_h][dst_w][channels]  contiguous, same dtype
 *   dtype      BEVK_U8 | BEVK_F16 | BEVK_F32;  channels 1..4
 *   M          HOST pointer to n_mats row-major 3x3 float64 matrices, with cv2 meaning:
 *              forward src->dst unless flags has BEVK_WARP_INVERSE_MAP
 *   mat_index  HOST int32[n_frames] -> matrix of each frame, or NULL: n_mats == 1 (one matrix for
 *              all frames) or n_mats == n_frames (frame i uses matrix i)
 *   flags      BEVK_INTER_NEAREST | BEVK_INTER_LINEAR, optionally | BEVK_WARP_INVERSE_MAP
 *   border_value  HOST double[4] per-channel constant, or NULL for 0
 */
int bevk_warp_perspective(const void *src, void *dst, int n_frames, int src_h, int src_w,
                          int dst_h, int dst_w, int channels, int dtype, const double *M,
                          int n_mats, const int32_t *mat_index, int flags, int border_mode,
                          const double *border_value, void *stream);

/* Same contract with HOST src / dst buffers (pinned or pageable).  Only the source rows the
 * homographies reference are uploaded; copies and kernels overlap chunk by chunk. */
int bevk_warp_perspective_host(const void *src, void *dst, int n_frames, int src_h, int src_w,
                               int dst_h, int dst_w, int channels, int dtype, const double *M,
                               int n_mats, const int32_t *mat_index, int flags, int border_mode,
                               const double *border_value);

/* The source-row band [rows[0], rows[1]] that bevk_warp_perspective_host uploads for these matrices
 * (the union of the rows their maps can reference; the whole frame if a map crosses the horizon).
 * Host-only, no GPU needed. */
int bevk_warp_host_rows(int src_h, int src_w, int dst_h, int dst_w, const double *M, int n_mats,
                        int flags, int rows[2]);

/* bevk_warp_perspective with the kernel family chosen per call: path 0 = automatic, 1 = the
 * direct-gather kernels, 2 = the staged (TMA) kernel (BEVK_E_ARG if the shape does not qualify),
 * -1 = the calling thread's default (bevk_warp_set_path).  Same reference interface as
 * bevk_warp_perspective (vis_homo.py:85-91); the extra argument exists for tests and benchmarks
 * that compare the kernel families. */
int bevk_warp_perspective_path(const void *src, void *dst, int n_frames, int src_h, int src_w,
                               int dst_h, int dst_w, int channels, int dtype, const double *M,
                               int n_mats, const int32_t *mat_index, int flags, int border_mode,
                               const double *border_value, int path, void *stream);

/* Default kernel family of the CALLING THREAD for bevk_warp_perspective / _host (0 automatic --
 * the initial value --, 1 direct-gather, 2 staged).  Thread-local: it never affects other
 * threads' calls.  Testing / benchmarking aid. */
int bevk_warp_set_path(int path);

/*
 * NV12 frames, as a GPU video decoder hands them out, to BGR: cv2.cvtColor(f, COLOR_YUV2BGR_NV12)
 * (cv2 4.13: BT.601 limited range, chroma shared by each 2x2 luma block) on a batch, byte-identical.
 * Serves the decode half of "decode -> warp without a host round trip" (SURVEY.md 8f rank 4) for
 * the frame loop of vis_homo.py:85-91, whose frames are BGR.
 *   src  device buffer; frame n starts at src + n * frame_stride bytes and holds h luma rows then
 *        h / 2 rows of interleaved U, V bytes, each row `pitch` bytes after the previous one
 *        (pitch >= w; a contiguous (n, h * 3 / 2, w) buffer has pitch = w, frame_stride = w * h * 3 / 2)
 *   dst  [n_frames][h][w][3] contiguous uint8 BGR
 *   h, w even and positive.
 */
int bevk_nv12_to_bgr(const void *src, void *dst, int n_frames, int h, int w, int pitch,
                     int64_t frame_stride, void *stream);

/*
 * Perspective warp of NV12 frames straight to BGR: dst[i] is byte-identical to
 *     cv2.warpPerspective(cv2.cvtColor(src[i], COLOR_YUV2BGR_NV12), M[k], (dst_w, dst_h), flags,
 *                         BORDER_CONSTANT, border_value)
 * in one pass, without the BGR copy of the frames.  Replaces the warp of vis_homo.py:85-91 for
 * frames decoded on the GPU (SURVEY.md 8f rank 4).  src layout, pitch and frame_stride as for
 * bevk_nv12_to_bgr with src_h x src_w luma pixels (both even); dst [n_frames][dst_h][dst_w][3]
 * uint8.  M, n_mats, mat_index, flags, border_mode and border_value mean what they mean for
 * bevk_warp_perspective (border_value: B, G, R).  A frame must span less than 4 GB
 * (pitch * src_h * 3 / 2 < 2^32).
 */
int bevk_warp_perspective_nv12(const void *src, void *dst, int n_frames, int src_h, int src_w,
                               int pitch, int64_t frame_stride, int dst_h, int dst_w,
                               const double *M, int n_mats, const int32_t *mat_index, int flags,
                               int border_mode, const double *border_value, void *stream);

/*
 * Roofline accounting helper (SURVEY.md 8d): number of distinct in-bounds source pixels that the
 * coordinate map of one matrix references (4 taps bilinear / 1 tap nearest), computed on the
 * device with the same coordinate code as the warp.  row_range (HOST int[2], may be NULL)
 * receives the first / last referenced source row.  Synchronous.  Returns the count or <0.
 */
int64_t bevk_warp_touched_pixels(int src_h, int src_w, int dst_h, int dst_w, const double M[9],
                                 int flags, int *row_range);

/*
 * Batched cv2.resize(img, (dst_w, dst_h), interpolation=...) on uint8 frames: replaces the
 * per-frame call at vis_homo.py:90 (the small-frame path; its result feeds the warp at
 * vis_homo.py:91 through the homography of Calib.scale(align_corners=False), bev/calib.py:142-198).
 * src [n_frames][src_h][src_w][channels], dst [n_frames][dst_h][dst_w][channels], device buffers,
 * channels 1..4, dtype BEVK_U8, interpolation BEVK_INTER_LINEAR (cv2's default) or BEVK_INTER_AREA
 * (what OpenCV recommends for downscaling).  Bit-identical to OpenCV 4.13.
 */
int bevk_resize(const void *src, void *dst, int n_frames, int src_h, int src_w, int dst_h,
                int dst_w, int channels, int dtype, int interpolation, void *stream);

/*
 * Batched cv2.resize of NV12 frames straight to small BGR frames: dst[i] is byte-identical to
 *     cv2.resize(cv2.cvtColor(src[i], COLOR_YUV2BGR_NV12), (dst_w, dst_h))
 * with the default INTER_LINEAR, in one pass, without the BGR copy of the frames.  Replaces the
 * small-frame copy at vis_homo.py:90 for frames decoded on the GPU (SURVEY.md 8f rank 4).  src
 * layout, pitch and frame_stride as for bevk_nv12_to_bgr with src_h x src_w luma pixels (both
 * even); dst [n_frames][dst_h][dst_w][3] contiguous uint8 BGR.  All sizes 1..32767; a frame must
 * span less than 4 GB (pitch * src_h * 3 / 2 < 2^32).
 */
int bevk_resize_nv12(const void *src, void *dst, int n_frames, int src_h, int src_w, int pitch,
                     int64_t frame_stride, int dst_h, int dst_w, void *stream);

/*
 * bevk_resize_nv12 with a choice of interpolation: BEVK_INTER_LINEAR, or BEVK_INTER_AREA for
 *     cv2.resize(cv2.cvtColor(src[i], COLOR_YUV2BGR_NV12), (dst_w, dst_h), interpolation=INTER_AREA).
 * bevk_resize_nv12 is this function with BEVK_INTER_LINEAR.  Same layouts and limits.
 */
int bevk_resize_nv12_interp(const void *src, void *dst, int n_frames, int src_h, int src_w, int pitch,
                            int64_t frame_stride, int dst_h, int dst_w, int interpolation, void *stream);

/*
 * Alpha compositing of uint8 BGR frames, the blend behind the three warps of
 * bev/tool/compo.py:38,46,47 -- replaces composite_reg_img (bev/tool/compo.py:5-24):
 *     out = uint8(min(round_half_even(fg * (mask / 255) + bg * (1 - mask / 255)), 255))
 * evaluated like the reference's numpy float64 expression (bit-identical).  bg, fg, fg_mask and
 * out are device buffers of n_pixels x 3 bytes (any batch of same-sized frames, flattened;
 * 4-byte aligned).  bw_mode != 0 first turns fg grey the way
 * cv2.cvtColor(BGR2GRAY) -> GRAY2BGR does (compo.py:13-14).
 */
int bevk_composite_u8c3(const void *bg, const void *fg, const void *fg_mask, void *out,
                        int64_t n_pixels, int bw_mode, void *stream);

/*
 * Fused BEV compositor: replaces composite_bev_img (bev/tool/compo.py:26-50) -- the three
 * cv2.warpPerspective calls at compo.py:38,46,47 and the blend at :49 -- in one pass:
 *     out[i] = blend(warp(bg[i or 0], H_bg[k]), warp(fg[i], H_fg[k]), warp(fg_mask[i], H_fg[k]))
 * with k = 0 (n_mats == 1, one camera pair for the batch) or k = i (n_mats == n_frames).  Warps are
 * bilinear, border 0, to a dst_w x dst_h BEV; H_bg / H_fg are HOST float64 [n_mats][9] FORWARD
 * (image -> BEV) matrices exactly as the reference hands them to cv2.  bg is n_bg (1 or n_frames)
 * frames of bg_h x bg_w x 3 bytes, fg and fg_mask n_frames frames of fg_h x fg_w x 3, out n_frames
 * BEVs; device buffers, 4-byte aligned.  Results are bit-identical to the three-warp route.
 * Widths (bg_w, fg_w, dst_w) must be multiples of 4; other shapes take bevk_warp_perspective +
 * bevk_composite_u8c3 (BEVK_E_ARG says so).
 */
int bevk_composite_bev_u8c3(const void *bg, const void *fg, const void *fg_mask, void *out,
                            int n_frames, int n_bg, int bg_h, int bg_w, int fg_h, int fg_w,
                            int dst_h, int dst_w, const double *H_bg, const double *H_fg,
                            int n_mats, void *stream);

/*
 * Homogeneous point projection with divide.  Replaces rbox.pts_world_bev (bev/rbox.py:136-151)
 * and the cv2.perspectiveTransform call sites (bev/visualizer/rbox_vis.py:54,61,74).
 *   pts/out [n][dim], dim 2 (w = 1 implied, 2 columns out) or 3 (homogeneous in, 3 columns out,
 *   last column 1);  dtype BEVK_F32 | BEVK_F64;  H HOST 3x3 float64.
 */
int bevk_pts_project(const void *pts, void *out, int64_t n, int dim, int dtype, const double H[9],
                     void *stream);

/*
 * xywh-yaw boxes [n][5] -> 4 corners [n][8] (tl, bl, br, tr).  Replaces rbox_torch.xywhr2xyxy
 * (bev/rbox_torch.py:52-99, external_aa=False).  With H != NULL the corners are also pushed
 * through the homography (with divide) in the same pass -- the fused chain of
 * bev/visualizer/rbox_vis.py:38-55 -- so each box is read once and written once.
 */
int bevk_xywhr2xyxy(const void *xywhr, void *xy8, int64_t n, int mode, int dtype, const double *H,
                    void *stream);

/*
 * 4 corners [n][8] -> xywh-yaw [n][5].  Replaces rbox.xy82xywhr (bev/rbox.py:50-63).  With
 * H != NULL the corners are first projected through H (the "and back" leg of configs[2]).
 */
int bevk_xy82xywhr(const void *xy8, void *xywhr, int64_t n, int mode, int dtype, const double *H,
                   void *stream);

/*
 * Similarity transform of xywh-yaw boxes between BEV and world.  Replaces
 * rbox_torch.rbox_world_bev (bev/rbox_torch.py:123-168; numpy twin bev/rbox.py:173-219).
 * H is normalised by H[8]; returns BEVK_E_AFFINE when |H20|+|H21| >= 1e-5 or the two axis scales
 * differ by >= 1e-5 (the reference's asserts).  src_mode = coordinate system of the input.
 */
int bevk_rbox_world_bev(const void *xywhr_in, void *xywhr_out, int64_t n, int src_mode, int dtype,
                        const double H[9], void *stream);

/*
 * 7-dof boxes with a projected height tail (x, y, w, h, yaw, du, dv).  Replaces
 * rbox.rboxtt_world_bev (bev/rbox.py:258-288): the first five columns go through
 * bevk_rbox_world_bev, the tail through the linear part of the same (affine) H.
 */
int bevk_rboxtt_world_bev(const void *rboxtt_in, void *rboxtt_out, int64_t n, int src_mode, int dtype,
                          const double H[9], void *stream);
/*
 * World boxes with height (x, y, w, h, yaw, z, t) -> ground boxes with a height tail
 * (x', y', w, h, yaw, du, dv): the box foot (x, y, z) and its top (x, y, z + t) are projected into
 * the camera K [R|t] (depth clipped at 1e-2) and back onto the ground plane through
 * inv(K [r1 r2 t]).  Replaces rbox.rbox_zt2tt_world (bev/rbox.py:228-256).
 * K: HOST 3x3 float64, Rt: HOST 3x4 float64 (row-major [R|t]).
 */
int bevk_rbox_zt2tt_world(const void *rboxzt, void *rboxtt, int64_t n, int dtype, const double K[9],
                          const double Rt[12], void *stream);

/* Heading segments [n][4] = [x, y, x + h*dx, y + h*dy].  rbox_torch.xywhr2xyvec (:101-112). */
int bevk_xywhr2xyvec(const void *xywhr, void *xyvec, int64_t n, int mode, int dtype, void *stream);
/* Yaw angles through a similarity: yaw2v(src) -> H[:2,:2] . v -> v2yaw(other system).
 * rbox.angle_world_bev (bev/rbox.py:162-171); H is used as given (not normalised), like there. */
int bevk_angle_world_bev(const void *yaw_in, void *yaw_out, int64_t n, int src_mode, int dtype,
                         const double H[9], void *stream);
/* Lengths through a similarity: dist * sqrt(H00^2 + H10^2).  rbox.dist_world_bev
 * (bev/rbox.py:153-160); BEVK_E_AFFINE when the two column norms differ by >= 1e-5 (its assert). */
int bevk_dist_world_bev(const void *dist_in, void *dist_out, int64_t n, int dtype, const double H[9],
                        void *stream);
/* Heading segments from corners.  rbox_torch.xy82xyvec (:114-121). */
int bevk_xy82xyvec(const void *xy8, void *xyvec, int64_t n, int dtype, void *stream);
/* v [n][2] -> yaw [n].  rbox_torch.v2yaw (:24-31). */
int bevk_v2yaw(const void *v, void *yaw, int64_t n, int mode, int dtype, void *stream);
/* yaw [n] -> unit vector [n][2].  rbox_torch.yaw2v (:33-40). */
int bevk_yaw2v(const void *yaw, void *v, int64_t n, int mode, int dtype, void *stream);
/* yaw [n] -> rotation [n][2][2].  rbox_torch.yaw2mat (:42-50). */
int bevk_yaw2mat(const void *yaw, void *mat, int64_t n, int mode, int dtype, void *stream);

/* HOST-buffer forms of the two configs[2] legs (float32): upload, project, download. */
int bevk_xywhr2xyxy_host(const float *xywhr, float *xy8, int64_t n, int mode, const double *H);
int bevk_xy82xywhr_host(const float *xy8, float *xywhr, int64_t n, int mode, const double *H);

/*
 * Rotated-box IoU matrix: replaces d3d.box.box2d_iou(boxes1, boxes2, method="rbox") as called by
 * iou_batch_rbox (bev/tracker/rbox_tracker.py:87-92; association step :383-405).
 *   boxes1 [n] rows of stride1 elements, boxes2 [m] rows of stride2 elements (stride >= 5, so
 *   detections carrying a score column need no copy); the first five are [x, y, w, h, r]:
 *   centre, side w along (cos r, sin r), side h along (-sin r, cos r).  yaw_offset is added to
 *   every r (the reference passes r + pi/2).  out [n][m], IoU = |A n B| / (|A| + |B| - |A n B|).
 *   dtype BEVK_F32 | BEVK_F64 (boxes and out); device buffers.
 */
int bevk_rbox_iou_matrix(const void *boxes1, int64_t n, int stride1, const void *boxes2, int64_t m,
                         int stride2, void *out, int dtype, double yaw_offset, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BEV_B200_H */
