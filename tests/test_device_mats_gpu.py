"""GPU: the warps with homographies in CUDA tensors (the bevk_*_dmat entry points, the _native.*_dmat
functions and the four warp operators given a CUDA M).  Every result is held bit for bit to the same
call with the matrices on the host, to live cv2, across launches of several matrix groups, in stream
order, inside a captured CUDA graph that replays new matrices, and under torch.compile."""
import numpy as np
import pytest
import torch

from bev_b200 import _native, torch_ops
from oracle import yuv420_oracle as yo
from tests import cv2_cases as cc
from tests import util
from tests.test_cv2_parity_gpu import WARP_SEED, check_frame, cv2_refs, cv2_warp, nv12_batch, warp_batches

cv2 = pytest.importorskip("cv2")

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ops = torch.ops.bev_cuda
POISON = 0xA5
S4 = np.diag([0.25, 0.25, 1.0])
H1080 = util.h_canon()                 # 1920x1080 -> 1024^2
H270 = S4 @ H1080 @ np.linalg.inv(S4)  # 480x270 -> 256^2
SMALL = (852, 480)


@pytest.fixture(scope="module", autouse=True)
def _ops():
    torch_ops.load()


def _u8(seed, *shape):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(0, 256, shape, dtype=torch.uint8, device=DEV, generator=g)


def _frames(seed, n, h, w, c, dtype):
    g = torch.Generator(device=DEV).manual_seed(seed)
    if dtype == torch.uint8:
        return torch.randint(0, 256, (n, h, w, c), dtype=dtype, device=DEV, generator=g)
    return (torch.rand((n, h, w, c), device=DEV, generator=g) * 300 - 20).to(dtype)


def _dev(M):
    return torch.from_numpy(np.ascontiguousarray(M, np.float64)).to(DEV)


def _host(M):
    return torch.from_numpy(np.ascontiguousarray(M, np.float64))


def _poison(shape, dtype=torch.uint8):
    t = torch.empty(shape, dtype=dtype, device=DEV)
    if dtype == torch.uint8:
        return t.fill_(POISON)
    return t.fill_(float("nan"))


def _same(a, b):
    """bitwise equality (NaN-safe for float frames)"""
    a, b = a.contiguous(), b.contiguous()
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a.view(torch.uint8), b.view(torch.uint8))


def _table(flags, k=3):
    """k forward 480x270 -> 256x192 maps (the matrices of WARP_INVERSE_MAP calls: their inverses)"""
    Hs = [np.diag([1.0, 0.75, 1.0]) @ H270 @ np.diag([1.0 + 0.03 * i, 1.0 - 0.02 * i, 1.0]) for i in range(k)]
    Hs[-1] = np.array([[1.0, 0.0, -6.5], [0.0, 1.0, 3.0], [0.0, 0.0, 1.0]]) @ Hs[-1]
    return np.stack([np.linalg.inv(H) if flags & 16 else H for H in Hs])


FLAGS = (0, 1, 16, 17)
BORDERS = ((0.0,), (7.0, 200.0, 33.0, 90.0))


# ---- 1. the same bytes as host matrices -----------------------------------------------------------

@pytest.mark.parametrize("flags", FLAGS)
@pytest.mark.parametrize("dtype", [torch.uint8, torch.float16, torch.float32], ids=["u8", "f16", "f32"])
def test_warp_perspective_equals_host_matrices(flags, dtype):
    Ms = _table(flags)
    idx = np.array([2, 0, 0, 1, 2], np.int32)
    for c in (1, 2, 3, 4):
        src = _frames(100 + c, 5, 270, 480, c, dtype)
        for border in BORDERS:
            kw = dict(flags=flags, borderValue=border, mat_index=idx)
            out = _native.warp_perspective_dmat(src, _dev(Ms), (256, 192), dst=_poison((5, 192, 256, c), dtype), **kw)
            for path in ("generic", "auto"):
                ref = _native.warp_perspective(src, Ms, (256, 192), path=path, **kw)
                assert _same(out, ref), (flags, dtype, c, border, path)
            # one matrix for all frames, unbatched frames, the operator
            one = _native.warp_perspective_dmat(src[0], _dev(Ms[1]), (256, 192), **dict(kw, mat_index=None))
            assert _same(one, _native.warp_perspective(src[0], Ms[1], (256, 192), path="auto",
                                                       **dict(kw, mat_index=None)))
            b = border[0]
            op = ops.warp_perspective(src, _dev(Ms), 256, 192, flags, 0, b, torch.from_numpy(idx))
            assert _same(op, ops.warp_perspective(src, _host(Ms), 256, 192, flags, 0, b, torch.from_numpy(idx)))


def _nv12_surface(seed, n, h, w, pad):
    """pitched NV12 frames: a (n, h*3/2, w + pad) surface seen as (n, h*3/2, w)"""
    return _u8(seed, n, h * 3 // 2, w + pad)[:, :, :w]


@pytest.mark.parametrize("flags", FLAGS)
def test_video_warps_equal_host_matrices(flags):
    Ms = _table(flags)
    idx = np.array([1, 2, 0, 1], np.int32)
    bgr = _u8(200, 4, 270, 480, 3)
    for pad in (0, 36):
        nv12 = _nv12_surface(201 + pad, 4, 270, 480, pad)
        for border in ((0.0, 0.0, 0.0), (7.0, 200.0, 33.0)):
            kw = dict(flags=flags, borderValue=border, mat_index=idx)
            out = _native.warp_perspective_nv12_dmat(nv12, _dev(Ms), (256, 192), dst=_poison((4, 192, 256, 3)), **kw)
            assert _same(out, _native.warp_perspective_nv12(nv12, Ms, (256, 192), **kw)), (flags, pad, border)
            for layout in ("i420", "nv12"):
                for src, fn, twin in ((bgr, _native.warp_perspective_yuv420_dmat, _native.warp_perspective_yuv420),
                                      (nv12, _native.warp_perspective_nv12_yuv420_dmat,
                                       _native.warp_perspective_nv12_yuv420)):
                    # a destination with padded rows: the padding stays untouched
                    big = _poison((4, 288, 256 + 20))
                    out = fn(src, _dev(Ms), (256, 192), layout, dst=big[:, :, :256], **kw)
                    ref = twin(src, Ms, (256, 192), layout, **kw)
                    assert _same(out, ref), (fn.__name__, layout, flags, pad, border)
                    assert bool((big[:, :, 256:] == POISON).all()), (fn.__name__, "row padding written")
            b = border[0]
            I = torch.from_numpy(idx)
            for name, s, extra in (("warp_perspective_nv12", nv12, ()), ("warp_perspective_yuv420", bgr, (1,)),
                                   ("warp_perspective_nv12_yuv420", nv12, (0,))):
                op = getattr(ops, name)
                a = op(s, _dev(Ms), 256, 192, *extra, flags, 0, b, I)
                assert _same(a, op(s, _host(Ms), 256, 192, *extra, flags, 0, b, I)), (name, flags, pad, b)


def test_float32_cuda_matrices_are_converted():
    """The operators convert a non-float64 CUDA M on the stream, as they convert a CPU one."""
    src, nv12 = _u8(210, 3, 270, 480, 3), _nv12_surface(211, 3, 270, 480, 16)
    M32 = torch.from_numpy(_table(1).astype(np.float32))
    I = torch.tensor([0, 2, 1], dtype=torch.int32)
    assert _same(ops.warp_perspective(src, M32.to(DEV), 256, 192, mat_index=I),
                 ops.warp_perspective(src, M32, 256, 192, mat_index=I))
    assert _same(ops.warp_perspective_nv12(nv12, M32.to(DEV), 256, 192, mat_index=I),
                 ops.warp_perspective_nv12(nv12, M32, 256, 192, mat_index=I))


def test_python_validation():
    src = _u8(220, 2, 64, 64, 3)
    with pytest.raises(TypeError, match="CUDA tensor"):
        _native.warp_perspective_dmat(src, np.eye(3), (32, 32))
    with pytest.raises(TypeError, match="CUDA tensor"):
        _native.warp_perspective_dmat(src, torch.eye(3, dtype=torch.float64), (32, 32))
    with pytest.raises(TypeError, match="float64"):
        _native.warp_perspective_dmat(src, torch.eye(3, device=DEV), (32, 32))
    with pytest.raises(ValueError, match="3x3"):
        _native.warp_perspective_dmat(src, torch.eye(4, dtype=torch.float64, device=DEV), (32, 32))
    with pytest.raises(ValueError, match="mat_index"):
        _native.warp_perspective_dmat(src, _dev(np.stack([np.eye(3)] * 3)), (32, 32))
    with pytest.raises(_native.NativeError, match="out of range"):
        _native.warp_perspective_dmat(src, _dev(np.stack([np.eye(3)] * 2)), (32, 32), mat_index=[0, 2])


# ---- 2. against live cv2 ------------------------------------------------------------------------

def test_warp_perspective_dmat_vs_cv2():
    """tests/cv2_cases.py's warp cases (singular and zero maps, horizons inside the output, saturating
    coordinates ...), with the float nearest 1/4-channel deviation test_cv2_parity_gpu.py documents"""
    ran = 0
    for case, dt, frames, Ms, idx in warp_batches():
        out = _native.warp_perspective_dmat(torch.from_numpy(frames).to(DEV), _dev(Ms if Ms.shape[0] > 1 else Ms[0]),
                                            case["dsize"], flags=case["flags"], borderValue=case["border"],
                                            mat_index=idx).cpu().numpy()
        for i, (ref, H) in enumerate(cv2_refs(frames, Ms, idx, case, dt)):
            check_frame(out[i], ref, frames[i], H, case, dt, "device matrices, frame %d" % i)
        ran += 1
    assert ran > 400


TIES = [np.diag([2.0, 2.0, 1.0]), np.diag([0.5, 0.5, 1.0]), np.diag([4.0, 2.0, 1.0]), np.zeros((3, 3)),
        np.array([[1.0, 2.0, 3.0], [2.0, 4.0, 6.0], [0.0, 0.0, 1.0]]),  # singular
        np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.05, -1.5]])]  # horizon inside the output


@pytest.mark.parametrize("flags", FLAGS)
def test_exact_ties_and_degenerate_maps_vs_cv2(flags):
    frames = _u8(230, 1, 61, 97, 3)
    f = frames[0].cpu().numpy()
    nv12 = _u8(231, 1, 96, 128)
    nv12_bgr = cv2.cvtColor(nv12[0].cpu().numpy(), cv2.COLOR_YUV2BGR_NV12)
    for H in TIES:
        for border in ((0.0, 0.0, 0.0), (9.0, 99.0, 199.0)):
            b4 = list(border) + [0.0]
            ref = cv2.warpPerspective(f, H, (80, 64), flags=flags, borderMode=cv2.BORDER_CONSTANT, borderValue=b4)
            out = _native.warp_perspective_dmat(frames, _dev(H), (80, 64), flags=flags, borderValue=border)
            assert np.array_equal(out[0].cpu().numpy(), ref), (H.tolist(), flags, border)
            ref = cv2.warpPerspective(nv12_bgr, H, (80, 64), flags=flags, borderMode=cv2.BORDER_CONSTANT,
                                      borderValue=b4)
            out = _native.warp_perspective_nv12_dmat(nv12, _dev(H), (80, 64), flags=flags, borderValue=border)
            assert np.array_equal(out[0].cpu().numpy(), ref), ("nv12", H.tolist(), flags, border)
            out = _native.warp_perspective_nv12_yuv420_dmat(nv12, _dev(H), (80, 64), "i420", flags=flags,
                                                            borderValue=border)
            assert np.array_equal(out[0].cpu().numpy(), cv2.cvtColor(ref, cv2.COLOR_BGR2YUV_I420)), ("yuv", H.tolist())


def test_video_warps_dmat_vs_cv2():
    for case in cc.warp_cases(WARP_SEED, 160, dtypes=("uint8",)):
        n = 3
        dw, dh = (v + v % 2 for v in case["dsize"])
        case = dict(case, channels=3, dsize=(dw, dh), bw0=cc.block_width(dw, dh))
        border = (list(case["border"]) + [0.0, 0.0])[:3]
        nv12, nv12_bgr = nv12_batch(case, n)
        nv12_t = torch.from_numpy(nv12).to(DEV)
        Hd = _dev(case["H"])
        out = _native.warp_perspective_nv12_dmat(nv12_t, Hd, (dw, dh), flags=case["flags"],
                                                 borderValue=border).cpu().numpy()
        bgr = cc.warp_src(case, n)
        yuv = _native.warp_perspective_yuv420_dmat(torch.from_numpy(bgr).to(DEV), Hd, (dw, dh), "nv12",
                                                   flags=case["flags"], borderValue=border).cpu().numpy()
        for i in range(n):
            ref = cv2_warp(nv12_bgr[i], case["H"], case, border)
            assert util.bits_equal(out[i], ref), "nv12: %s" % cc.describe(case)
            ref = yo.i420_to_nv12(cv2.cvtColor(cv2_warp(bgr[i], case["H"], case, border), cv2.COLOR_BGR2YUV_I420))
            assert util.bits_equal(yuv[i], ref), "bgr -> nv12: %s" % cc.describe(case)


# ---- 3. matrix tables of several launches -------------------------------------------------------

def _batching_cases():
    rng = np.random.default_rng(300)
    yield "17 groups", 34, 17, rng.permutation(np.arange(34) % 17).astype(np.int32)
    yield "33 groups, 7 unused matrices", 66, 40, rng.permutation(np.arange(66) % 33).astype(np.int32)
    yield "runs with stride, one-frame runs", 41, 20, np.array([(i * 7) % 20 if i % 3 else i % 5 for i in range(41)],
                                                              np.int32)
    yield "per-frame table", 33, 33, None


@pytest.mark.parametrize("flags", [1, 16])
def test_matrix_tables_of_several_launches(flags):
    for what, n, k, idx in _batching_cases():
        Ms = np.stack([np.diag([1.0, 0.75, 1.0]) @ H270 @ np.diag([1.0, 1.0 + 0.004 * j, 1.0]) for j in range(k)])
        if flags & 16:
            Ms = np.linalg.inv(Ms)
        Md = _dev(Ms)
        bgr = _u8(310, n, 270, 480, 3)
        nv12 = _nv12_surface(311, n, 270, 480, 32)
        kw = dict(flags=flags, mat_index=idx)
        out = _native.warp_perspective_dmat(bgr, Md, (256, 192), dst=_poison((n, 192, 256, 3)), **kw)
        assert _same(out, _native.warp_perspective(bgr, Ms, (256, 192), path="auto", **kw)), what
        # a frame checked against a call of its own
        j = n // 2
        one = _native.warp_perspective(bgr[j], Ms[j if idx is None else idx[j]], (256, 192), flags=flags)
        assert _same(out[j], one), what
        out = _native.warp_perspective_nv12_dmat(nv12, Md, (256, 192), dst=_poison((n, 192, 256, 3)), **kw)
        assert _same(out, _native.warp_perspective_nv12(nv12, Ms, (256, 192), **kw)), what
        for src, fn, twin in ((bgr, _native.warp_perspective_yuv420_dmat, _native.warp_perspective_yuv420),
                              (nv12, _native.warp_perspective_nv12_yuv420_dmat, _native.warp_perspective_nv12_yuv420)):
            out = fn(src, Md, (256, 192), "nv12", dst=_poison((n, 288, 256)), **kw)
            assert _same(out, twin(src, Ms, (256, 192), "nv12", **kw)), (what, fn.__name__)


# ---- 4. stream order ----------------------------------------------------------------------------

def test_matrices_are_read_in_stream_order():
    """M.copy_(new) enqueued behind a long kernel, then the warps, with no host sync: they use new."""
    old, new = _table(1)[0], _table(1)[2]
    bgr, nv12 = _u8(400, 2, 270, 480, 3), _nv12_surface(401, 2, 270, 480, 0)
    refs = [_native.warp_perspective(bgr, new, (256, 192)), _native.warp_perspective_nv12(nv12, new, (256, 192)),
            _native.warp_perspective_yuv420(bgr, new, (256, 192)),
            _native.warp_perspective_nv12_yuv420(nv12, new, (256, 192))]
    new_d = _dev(new)
    for trial in range(2):
        M = _dev(old)
        torch.cuda.synchronize()
        torch.cuda._sleep(200_000_000)  # a long kernel ahead of the copy
        M.copy_(new_d)
        if trial == 0:
            outs = [_native.warp_perspective_dmat(bgr, M, (256, 192)),
                    _native.warp_perspective_nv12_dmat(nv12, M, (256, 192)),
                    _native.warp_perspective_yuv420_dmat(bgr, M, (256, 192)),
                    _native.warp_perspective_nv12_yuv420_dmat(nv12, M, (256, 192))]
        else:
            outs = [ops.warp_perspective(bgr, M, 256, 192), ops.warp_perspective_nv12(nv12, M, 256, 192),
                    ops.warp_perspective_yuv420(bgr, M, 256, 192), ops.warp_perspective_nv12_yuv420(nv12, M, 256, 192)]
        assert not torch.cuda.current_stream().query(), "the host waited for the stream"
        torch.cuda.synchronize()
        for o, r in zip(outs, refs):
            assert _same(o, r), trial


# ---- 5. CUDA-graph capture ----------------------------------------------------------------------

def _pitch_roll(H, pitch, roll):
    """a homography changed on the GPU: H composed with a small rotation of the image plane about
    the frame centre and a vertical shift (per-frame pitch / roll compensation)"""
    c, s = torch.cos(roll), torch.sin(roll)
    zero, one = torch.zeros_like(c), torch.ones_like(c)
    T = torch.stack([torch.stack([c, -s, 960 * (1 - c) + 540 * s]),
                     torch.stack([s, c, 540 * (1 - c) - 960 * s + pitch]),
                     torch.stack([zero, zero, one])])
    return H @ T


def test_capture_cfg1_loop_replays_new_homographies():
    """cfg 1: one 1080p frame -> its BEV, its 852x480 copy and that copy's BEV.  Captured once with
    CUDA H and Hs, replayed with three homography pairs made on the GPU and three frames: each
    replay equals eager calls with the pair on the host."""
    fx, fy = 1920 / SMALL[0], 1080 / SMALL[1]
    Sc = np.array([[fx, 0.0, 0.5 * fx - 0.5], [0.0, fy, 0.5 * fy - 0.5], [0.0, 0.0, 1.0]])
    H0, Sc_d = _dev(H1080), _dev(Sc)
    H, Hs = H0.clone(), (H0 @ Sc_d).contiguous()
    frame = _u8(500, 1, 1080, 1920, 3)

    def loop(f):
        bev = ops.warp_perspective(f, H, 1024, 1024)
        small = ops.resize(f, *SMALL)
        return bev, small, ops.warp_perspective(small, Hs, 1024, 1024)

    loop(frame)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        loop(frame)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = loop(frame)
    for k in range(3):
        Hk = _pitch_roll(H0, torch.tensor(4.0 * (k + 1), dtype=torch.float64, device=DEV),
                         torch.tensor(0.01 * (k - 1), dtype=torch.float64, device=DEV))
        H.copy_(Hk)
        Hs.copy_(Hk @ Sc_d)
        frame.copy_(_u8(501 + k, 1, 1080, 1920, 3))
        graph.replay()
        torch.cuda.synchronize()
        Hh, Hsh = H.cpu(), Hs.cpu()
        ref_bev = ops.warp_perspective(frame, Hh, 1024, 1024)
        ref_small = ops.resize(frame, *SMALL)
        assert _same(out[0], ref_bev), k
        assert _same(out[1], ref_small), k
        assert _same(out[2], ops.warp_perspective(ref_small, Hsh, 1024, 1024)), k
        assert not _same(out[0], ops.warp_perspective(frame, _host(H1080), 1024, 1024)), "replayed the old H"


def test_capture_video_warps_replay_new_homographies():
    Ms = _dev(_table(1))
    I = torch.tensor([2, 0, 1], dtype=torch.int32)
    surface, bgr = _u8(510, 3, 405, 512), _u8(511, 3, 270, 480, 3)

    def fn():
        nv12 = surface[:, :, :480]
        return (ops.warp_perspective_nv12(nv12, Ms, 256, 192, mat_index=I),
                ops.warp_perspective_yuv420(bgr, Ms, 256, 192, 1, mat_index=I),
                ops.warp_perspective_nv12_yuv420(nv12, Ms, 256, 192, 0, mat_index=I))

    fn()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    Ms.copy_(_dev(_table(1)[::-1]))
    surface.copy_(_u8(512, 3, 405, 512))
    graph.replay()
    torch.cuda.synchronize()
    host = _host(_table(1)[::-1])
    nv12 = surface[:, :, :480]
    ref = (ops.warp_perspective_nv12(nv12, host, 256, 192, mat_index=I),
           ops.warp_perspective_yuv420(bgr, host, 256, 192, 1, mat_index=I),
           ops.warp_perspective_nv12_yuv420(nv12, host, 256, 192, 0, mat_index=I))
    for a, b in zip(out, ref):
        assert _same(a, b)


# ---- 6. torch.compile ---------------------------------------------------------------------------

def bgr_loop(frames, H, Hs):
    bev = ops.warp_perspective(frames, H, 1024, 1024)
    small = ops.resize(frames, *SMALL)
    bev_small = ops.warp_perspective(small, Hs, 1024, 1024)
    return bev, small, bev_small, ops.warp_perspective_yuv420(frames, H, 1024, 1024)


def nv12_loop(frames, H, Hs):
    bev = ops.warp_perspective_nv12(frames, H, 1024, 1024)
    small = ops.resize_nv12(frames, *SMALL)
    bev_small = ops.warp_perspective(small, Hs, 1024, 1024)
    return bev, small, bev_small, ops.warp_perspective_nv12_yuv420(frames, H, 1024, 1024)


def test_compile_frame_loops_with_cuda_matrices():
    H, Hs = _dev(H1080), _dev(H1080 @ np.diag([2.25, 2.25, 1.0]))
    for loop, shape in ((bgr_loop, (1080, 1920, 3)), (nv12_loop, (1620, 1920))):
        compiled = torch.compile(loop, fullgraph=True, dynamic=True)
        for seed, n in ((600, 2), (601, 3)):
            frames = _u8(seed, n, *shape)
            out = compiled(frames, H, Hs)
            ref = loop(frames, H.cpu(), Hs.cpu())
            assert out[0].shape[0] == n and all(_same(a, b) for a, b in zip(out, ref)), (loop.__name__, n)


# ---- 7. opcheck ---------------------------------------------------------------------------------

def test_opcheck_warps_with_cuda_matrices():
    f = _u8(700, 2, 64, 96, 3)
    nv12 = _u8(701, 2, 96, 128)[:, :, :96]
    M = _dev(np.stack([S4 @ H270, S4 @ H270 @ np.diag([1.0, 0.95, 1.0])]))
    idx = torch.tensor([1, 0], dtype=torch.int32)
    for M_ in (M, M.float(), M[0]):
        i = idx if M_.dim() == 3 else None
        samples = {
            "warp_perspective": (f, M_, 48, 32, 1, 0, 0.0, i),
            "warp_perspective_nv12": (nv12, M_, 48, 32, 0, 0, 5.0, i),
            "warp_perspective_yuv420": (f, M_, 48, 32, 0, 17, 0, 0.0, i),
            "warp_perspective_nv12_yuv420": (nv12, M_, 48, 32, 1, 1, 0, 0.0, i),
        }
        for name, args in samples.items():
            torch.library.opcheck(getattr(ops, name).default, args)
