"""torch.ops.bev_cuda on the GPU beyond eager calls: the operators added for the remaining device entry
points give the bytes of their ctypes twins, every operator passes torch.library.opcheck, the frame
loop, the compositor and the tracker chain compile with torch.compile(fullgraph=True), and captured
CUDA graphs replay new frames to the eager bytes."""
import math

import numpy as np
import pytest
import torch

from bev_b200 import _native, homo, rbox_torch, torch_ops
from tests import util
from tests.test_torch_ops_meta import ERRORS

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ops = torch.ops.bev_cuda
F64 = torch.float64
S4 = np.diag([0.25, 0.25, 1.0])
H1080 = util.h_canon()               # 1920x1080 -> 1024^2
H270 = S4 @ H1080 @ np.linalg.inv(S4)  # 480x270 -> 256^2
SMALL = (852, 480)
HSIM = np.array([[0.0, -0.125, 45.0], [-0.125, 0.0, 27.0], [0.0, 0.0, 1.0]])
H270_T, HSIM_T = torch.from_numpy(H270), torch.from_numpy(HSIM)
H_FG = torch.from_numpy(np.stack([H270 @ np.diag([1.0 + 0.05 * i, 1.0, 1.0]) for i in range(3)]))
H_BG = torch.from_numpy(np.stack([H270] * 3))


@pytest.fixture(scope="module", autouse=True)
def _ops():
    torch_ops.load()


def _u8(seed, *shape):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(0, 256, shape, dtype=torch.uint8, device=DEV, generator=g)


def _boxes(seed, n, dtype=torch.float32, extra=0):
    """(n, 5 + extra) boxes [x, y, w, h, yaw, ...] on a 1024^2 BEV"""
    rng = np.random.default_rng(seed)
    b = np.stack([rng.uniform(0, 1024, n), rng.uniform(0, 1024, n), rng.uniform(4, 40, n), rng.uniform(8, 120, n),
                  rng.uniform(-np.pi, np.pi, n)] + [rng.uniform(0, 1, n) for _ in range(extra)], 1)
    return torch.from_numpy(b).to(DEV, dtype)


def _small_h(H, ssize, small):
    """the small frame's map: Calib.scale(align_corners=False) of the frame's calibration"""
    fx, fy = ssize[0] / small[0], ssize[1] / small[1]
    return H @ np.array([[fx, 0.0, 0.5 * fx - 0.5], [0.0, fy, 0.5 * fy - 0.5], [0.0, 0.0, 1.0]])


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float64))


def _equal(a, b):
    if isinstance(a, torch.Tensor):
        return torch.equal(a, b)
    return len(a) == len(b) and all(_equal(x, y) for x, y in zip(a, b))


# ---- the new operators against their ctypes twins ------------------------------------------------

def test_resize_matches_ctypes_route():
    t = _u8(1, 3, 1080, 1920, 3)
    for interp in (1, 3):
        assert torch.equal(ops.resize(t, 852, 480, interp), homo.resize(t, SMALL, interpolation=interp))
    assert torch.equal(ops.resize(t[1], 852, 480), homo.resize(t[1], SMALL))
    for shape in ((270, 479), (2, 270, 479, 1), (2, 270, 479, 4)):
        f = _u8(2, *shape)
        assert torch.equal(ops.resize(f, 213, 120), homo.resize(f, (213, 120))), shape


def test_warp_perspective_nv12_yuv420_matches_ctypes_route():
    base = _u8(3, 5, 405, 512)
    surface = base[:, :, :480]  # pitched decoder surface: 270 luma rows, pitch 512
    Ms = np.stack([np.linalg.inv(H270), np.linalg.inv(H270) @ np.diag([1.0, 0.9, 1.0])])
    idx = torch.tensor([1, 0, 0, 1, 1], dtype=torch.int32)
    for layout, name in ((0, "i420"), (1, "nv12")):
        for flags in (1, 0, 17):
            out = ops.warp_perspective_nv12_yuv420(surface, _t(Ms), 256, 256, layout, flags, 0, 0.0, idx)
            ref = homo.warp_perspective_nv12_yuv420(surface, Ms, (256, 256), layout=name, flags=flags,
                                                    mat_index=idx.numpy())
            assert torch.equal(out, ref), (name, flags)
        one = ops.warp_perspective_nv12_yuv420(surface[2], _t(H270), 256, 256, layout)
        assert tuple(one.shape) == (384, 256)
        assert torch.equal(one, homo.warp_perspective_nv12_yuv420(surface[2], H270, (256, 256), layout=name))


def test_compositor_operators_match_ctypes_route():
    bg, fg, mask = _u8(4, 2, 270, 480, 3), _u8(5, 2, 270, 480, 3), _u8(6, 2, 270, 480, 3)
    for bw in (0, 1):
        assert torch.equal(ops.composite(bg, fg, mask, bw), _native.composite_u8c3(bg, fg, mask, bw_mode=bw))
    fg3, mask3 = _u8(7, 3, 270, 480, 3), _u8(8, 3, 270, 480, 3)
    H_bg, H_fg = np.stack([H270] * 3), H_FG.numpy()  # one background camera, a rendering camera per frame
    out = ops.composite_bev(bg[:1], fg3, mask3, _t(H_bg), H_FG, 256, 128)
    assert torch.equal(out, _native.composite_bev_u8c3(bg[:1], fg3, mask3, H_bg, H_fg, (256, 128)))
    one = ops.composite_bev(bg[0], fg3[1], mask3[1], H270_T, H_FG[1], 256, 128)
    assert tuple(one.shape) == (128, 256, 3)
    assert torch.equal(one, _native.composite_bev_u8c3(bg[0], fg3[1:2], mask3[1:2], H270, H_fg[1], (256, 128))[0])


def test_box_operators_match_ctypes_route():
    for dtype in (torch.float32, torch.float64):
        dets, trks = _boxes(10, 300, dtype, extra=1), _boxes(11, 77, dtype, extra=2)
        iou = ops.rbox_iou_matrix(dets, trks, math.pi / 2)
        assert tuple(iou.shape) == (300, 77) and torch.equal(iou, rbox_torch.iou_batch_rbox(dets, trks))
        # a view of the first five columns is read in place, through its row stride
        assert torch.equal(ops.rbox_iou_matrix(dets[:, :5], trks[:, :5]), rbox_torch.box2d_iou(dets, trks))
        b = _boxes(12, 1001, dtype)
        assert torch.equal(ops.rbox_heading(b, 0), rbox_torch.xywhr2xyvec(b, "bev"))
        xy8 = rbox_torch.xywhr2xyxy(b, "world")
        assert torch.equal(ops.corners_heading(xy8), rbox_torch.xy82xyvec(xy8))
        assert torch.equal(ops.angle_similarity(b[:, 4], HSIM_T, 1), rbox_torch.angle_world_bev(b[:, 4], HSIM, "world"))
        d = b[:, 2:4]
        assert torch.equal(ops.dist_similarity(d, HSIM_T), rbox_torch.dist_world_bev(d, HSIM))
        v = b[:, :2] - 512.0
        for mode, name in ((0, "bev"), (1, "world")):
            assert torch.equal(ops.v2yaw(v, mode), rbox_torch.v2yaw(v, name))
            assert torch.equal(ops.yaw2v(b[:, 4], mode), rbox_torch.yaw2v(b[:, 4], name))
            assert torch.equal(ops.yaw2mat(b[:, 4], mode), rbox_torch.yaw2mat(b[:, 4], name))
    K7 = util.load_npz("rbox7_kat.npz")
    zt = torch.from_numpy(K7["zt"].astype(np.float32)).to(DEV)
    tt = ops.rbox_zt2tt_world(zt, _t(K7["K"]), _t(K7["Rt"]))
    assert torch.equal(tt, rbox_torch.rbox_zt2tt_world(zt, K7["K"], K7["Rt"]))
    assert torch.equal(ops.rboxtt_similarity(tt, _t(K7["H"]), 1), rbox_torch.rboxtt_world_bev(tt, K7["H"], "world"))
    with pytest.raises(RuntimeError, match="AssertionError"):  # a non-affine H, where the reference asserts
        ops.rboxtt_similarity(tt, _t(H1080), 1)


@pytest.mark.parametrize("op, make, msg", ERRORS, ids=["%s-%d" % (e[0], i) for i, e in enumerate(ERRORS)])
def test_shape_errors_on_cuda_as_on_meta(op, make, msg):
    for dev in ("meta", DEV):
        with pytest.raises(RuntimeError, match=msg):
            getattr(ops, op)(*make(dev))


# ---- opcheck ------------------------------------------------------------------------------------

def _opcheck_samples():
    f = _u8(20, 2, 64, 96, 3)
    nv12 = _u8(21, 2, 96, 128)[:, :, :96]
    M, idx = _t(np.stack([S4 @ H270, S4 @ H270 @ np.diag([1.0, 0.95, 1.0])])), torch.tensor([1, 0], dtype=torch.int32)
    b, K7 = _boxes(22, 33), util.load_npz("rbox7_kat.npz")
    zt = torch.from_numpy(K7["zt"].astype(np.float32)).to(DEV)
    return {
        "warp_perspective": (f, M, 48, 32, 1, 0, 0.0, idx),
        "resize": (f, 40, 24, 3),
        "nv12_to_bgr": (nv12,),
        "warp_perspective_nv12": (nv12, M, 48, 32, 1, 0, 0.0, idx),
        "resize_nv12": (nv12, 40, 24),
        "bgr_to_yuv420": (f, 1),
        "warp_perspective_yuv420": (f, M, 48, 32, 0, 1, 0, 0.0, idx),
        "warp_perspective_nv12_yuv420": (nv12, M, 48, 32, 1, 1, 0, 0.0, idx),
        "composite": (f, _u8(23, 2, 64, 96, 3), _u8(24, 2, 64, 96, 3), 1),
        "composite_bev": (f[:1], _u8(25, 2, 64, 96, 3), _u8(26, 2, 64, 96, 3), M.flip(0), M, 48, 32),
        "project_points": (b[:, :2].contiguous(), _t(H1080)),
        "rbox_corners_project": (b, _t(H1080), 0),
        "corners_to_rbox": (rbox_torch.xywhr2xyxy(b, "bev"), None, 0),
        "rbox_similarity": (b, HSIM_T, 1),
        "rboxtt_similarity": (zt, _t(K7["H"]), 1),
        "rbox_zt2tt_world": (zt, _t(K7["K"]), _t(K7["Rt"])),
        "rbox_heading": (b, 1),
        "corners_heading": (rbox_torch.xywhr2xyxy(b, "bev"),),
        "angle_similarity": (b[:, 4].contiguous(), HSIM_T, 0),
        "dist_similarity": (b[:, 2:4].contiguous(), HSIM_T),
        "v2yaw": (b[:, :2].contiguous(), 0),
        "yaw2v": (b[:, 4].contiguous(), 1),
        "yaw2mat": (b[:, 4].contiguous(), 0),
        "rbox_iou_matrix": (b, _boxes(27, 9, extra=1), 0.5),
    }


def test_opcheck_every_operator():
    samples = _opcheck_samples()
    assert set(samples) == set(torch_ops.OPS)
    for name, args in samples.items():
        torch.library.opcheck(getattr(ops, name).default, args)


# ---- torch.compile ------------------------------------------------------------------------------

HT, HST = _t(H1080), _t(_small_h(H1080, (1920, 1080), SMALL))


def bgr_frame_loop(frames):
    """vis_homo.py:85-111: the BEV, the small frame, its BEV, and both BEVs as I420 for an encoder"""
    bev = ops.warp_perspective(frames, HT, 1024, 1024)
    small = ops.resize(frames, *SMALL)
    bev_small = ops.warp_perspective(small, HST, 1024, 1024)
    return bev, small, bev_small, ops.bgr_to_yuv420(bev), ops.bgr_to_yuv420(bev_small)


def nv12_frame_loop(frames):
    """the same from GPU decoder frames: the encoder's BEV straight from NV12"""
    bev = ops.warp_perspective_nv12(frames, HT, 1024, 1024)
    small = ops.resize_nv12(frames, *SMALL)
    bev_small = ops.warp_perspective(small, HST, 1024, 1024)
    return bev, small, bev_small, ops.warp_perspective_nv12_yuv420(frames, HT, 1024, 1024), ops.bgr_to_yuv420(bev_small)


def test_compile_frame_loops_with_dynamic_batch():
    for chain, shape in ((bgr_frame_loop, (1080, 1920, 3)), (nv12_frame_loop, (1620, 1920))):
        compiled = torch.compile(chain, fullgraph=True, dynamic=True)
        for seed, n in ((30, 2), (31, 3)):
            frames = _u8(seed, n, *shape)
            out = compiled(frames)
            assert out[0].shape[0] == n and _equal(out, chain(frames)), (chain.__name__, n)


def test_compile_compositor_and_tracker_chain():
    def compo(bg, fg, mask):
        return ops.composite_bev(bg, fg, mask, H_BG, H_FG, 256, 128)

    bg, fg, mask = _u8(40, 1, 270, 480, 3), _u8(41, 3, 270, 480, 3), _u8(42, 3, 270, 480, 3)
    assert torch.equal(torch.compile(compo, fullgraph=True)(bg, fg, mask), compo(bg, fg, mask))

    H_img_bev = _t(np.linalg.inv(H1080))

    def tracker(world_dets, trks):
        bev = ops.rbox_similarity(world_dets, HSIM_T, 1)
        return ops.rbox_iou_matrix(bev, trks, math.pi / 2), ops.rbox_corners_project(bev, H_img_bev, 0)

    dets = _boxes(43, 200)
    trks = ops.rbox_similarity(_boxes(44, 50), HSIM_T, 1)
    assert _equal(torch.compile(tracker, fullgraph=True)(dets, trks), tracker(dets, trks))


# ---- CUDA-graph capture -------------------------------------------------------------------------

def _check_capture(fn, static, fresh):
    """Capture fn(*static) once, refill the static inputs with `fresh`, replay: the same bytes as an
    eager fn(*fresh)."""
    fn(*static)  # eager first: kernel set-up, map caches
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn(*static)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn(*static)
    for s, f in zip(static, fresh):
        s.copy_(f)
    graph.replay()
    torch.cuda.synchronize()
    ref = fn(*fresh)
    assert _equal(out, ref)
    return graph


@pytest.mark.parametrize("path", ["fast", "auto"], ids=["staged", "direct_gather"])
def test_capture_cfg1_warp(path):
    """cfg 1: one 1080p frame -> 1024^2.  The staged kernel (forced: a single frame goes to the
    direct-gather kernel by default) takes its scratch with cudaMallocAsync on the capturing stream."""
    _native.set_warp_path(path)
    try:
        _check_capture(lambda f: ops.warp_perspective(f, HT, 1024, 1024), [_u8(50, 1, 1080, 1920, 3)],
                       [_u8(51, 1, 1080, 1920, 3)])
    finally:
        _native.set_warp_path("auto")


def test_capture_matrix_table_of_several_launches():
    """40 frames over 20 matrices in an irregular order: more (matrix, frame-run) groups than one
    launch takes, through the staged kernel and the direct-gather kernel in one graph"""
    Ms = _t(np.stack([np.linalg.inv(H270) @ np.diag([1.0, 1.0 + 0.01 * k, 1.0]) for k in range(20)]))
    idx = torch.from_numpy(np.random.default_rng(52).permutation(np.arange(40) % 20).astype(np.int32))

    def fn(f):
        _native.set_warp_path("fast")
        staged = ops.warp_perspective(f, Ms, 256, 256, 17, 0, 0.0, idx)
        _native.set_warp_path("generic")
        direct = ops.warp_perspective(f, Ms, 256, 256, 17, 0, 0.0, idx)
        _native.set_warp_path("auto")
        return staged, direct

    try:
        _check_capture(fn, [_u8(53, 40, 270, 480, 3)], [_u8(54, 40, 270, 480, 3)])
    finally:
        _native.set_warp_path("auto")


def test_capture_nv12_and_yuv_operators():
    base, base_new = _u8(60, 3, 405, 512), _u8(61, 3, 405, 512)
    Ms = _t(np.stack([H270, H270 @ np.diag([0.9, 1.0, 1.0])]))
    idx = torch.tensor([0, 1, 0], dtype=torch.int32)

    def fn(surface, bgr):
        nv12 = surface[:, :, :480]  # pitched
        return (ops.nv12_to_bgr(nv12), ops.warp_perspective_nv12(nv12, Ms, 256, 256, mat_index=idx),
                ops.resize_nv12(nv12, 213, 120), ops.resize_nv12(nv12, 120, 68, 3),
                ops.warp_perspective_nv12_yuv420(nv12, Ms, 256, 256, 1, mat_index=idx),
                ops.bgr_to_yuv420(bgr), ops.warp_perspective_yuv420(bgr, Ms, 256, 256, 0, mat_index=idx),
                ops.resize(bgr, 213, 120))

    _check_capture(fn, [base, _u8(62, 3, 270, 480, 3)], [base_new, _u8(63, 3, 270, 480, 3)])


def test_capture_compositor():
    def fn(bg, fg, mask):
        bev = ops.composite_bev(bg, fg, mask, H_BG, H_FG, 256, 128)
        return bev, ops.composite(bev, bev.flip(0).contiguous(), bev, 1)

    _check_capture(fn, [_u8(70, 1, 270, 480, 3), _u8(71, 3, 270, 480, 3), _u8(72, 3, 270, 480, 3)],
                   [_u8(73, 1, 270, 480, 3), _u8(74, 3, 270, 480, 3), _u8(75, 3, 270, 480, 3)])


def test_capture_box_operators():
    K7 = util.load_npz("rbox7_kat.npz")
    K, Rt, H7 = _t(K7["K"]), _t(K7["Rt"]), _t(K7["H"])
    zt = torch.from_numpy(K7["zt"].astype(np.float32)).to(DEV)

    def fn(b, z):
        xy8 = ops.rbox_corners_project(b, None, 0)
        tt = ops.rbox_zt2tt_world(z, K, Rt)
        return (ops.project_points(b[:, :2].contiguous(), HT), xy8, ops.corners_to_rbox(xy8, HT, 0),
                ops.rbox_similarity(b, HSIM_T, 1), tt, ops.rboxtt_similarity(tt, H7, 1), ops.rbox_heading(b, 1),
                ops.corners_heading(xy8), ops.angle_similarity(b[:, 4].contiguous(), HSIM_T, 0),
                ops.dist_similarity(b[:, 2:4].contiguous(), HSIM_T), ops.v2yaw(b[:, :2].contiguous(), 1),
                ops.yaw2v(b[:, 4].contiguous(), 0), ops.yaw2mat(b[:, 4].contiguous(), 1),
                ops.rbox_iou_matrix(b, b, math.pi / 2))

    _check_capture(fn, [_boxes(80, 500), zt.clone()], [_boxes(81, 500), zt.flip(0).contiguous()])


def test_cuda_mat_index_during_capture_raises():
    f, nv12 = _u8(90, 4, 64, 96, 3), _u8(91, 4, 96, 96)
    Ms = _t(np.stack([S4 @ H270, S4 @ H270 @ np.diag([1.0, 0.9, 1.0])]))
    idx = torch.tensor([0, 1, 1, 0], dtype=torch.int32, device=DEV)
    calls = [lambda: ops.warp_perspective(f, Ms, 64, 64, mat_index=idx),
             lambda: ops.warp_perspective_nv12(nv12, Ms, 64, 64, mat_index=idx),
             lambda: ops.warp_perspective_yuv420(f, Ms, 64, 64, mat_index=idx),
             lambda: ops.warp_perspective_nv12_yuv420(nv12, Ms, 64, 64, mat_index=idx)]
    for call in calls:
        eager = call()  # outside capture a CUDA mat_index keeps working
        assert torch.equal(eager, call())
        graph = torch.cuda.CUDAGraph()
        with pytest.raises(RuntimeError, match="Pass mat_index as a CPU int32 tensor"):
            with torch.cuda.graph(graph):
                call()
        del graph
    torch.cuda.synchronize()
