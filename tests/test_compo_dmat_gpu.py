"""GPU: the fused BEV compositor with homographies in CUDA tensors (bevk_composite_bev_u8c3_dmat,
_native.composite_bev_u8c3_dmat, the composite_bev operator and compo.composite_bev_batch given CUDA
matrices).  Every result is held bit for bit to the same call with the matrices on the host and to
live cv2 (three cv2.warpPerspective calls and the reference's float64 blend), across launches of
several groups, in stream order, inside a captured CUDA graph that replays new camera poses, and
under torch.compile."""
import numpy as np
import pytest
import torch

from bev_b200 import _native, compo, torch_ops
from oracle import compo_oracle as co
from tests import util
from tests.test_compo_gpu import _quad_h

cv2 = pytest.importorskip("cv2")

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ops = torch.ops.bev_cuda
POISON = 0xA5
S4 = np.diag([0.25, 0.25, 1.0])
H270 = S4 @ util.h_canon() @ np.linalg.inv(S4)  # 480x270 -> 256^2


@pytest.fixture(scope="module", autouse=True)
def _ops():
    torch_ops.load()


def _u8(seed, *shape):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.randint(0, 256, shape, dtype=torch.uint8, device=DEV, generator=g)


def _mask(seed, n, h, w):
    """3-channel masks with opaque, transparent and partial regions"""
    m = _u8(seed, n, h, w, 1).repeat(1, 1, 1, 3)
    m[:, : h // 3] = 255
    m[:, h // 3: h // 2] = 0
    return m


def _dev(M):
    return torch.from_numpy(np.ascontiguousarray(M, np.float64)).to(DEV)


def _poison(shape):
    return torch.full(shape, POISON, dtype=torch.uint8, device=DEV)


def _cv2_chain(B, F, M, Hb, Hf, dsize):
    """compo.py:36-49 with live cv2: three warps and the reference's float64 blend per frame"""
    B, F, M = (t.cpu().numpy() for t in (B, F, M))
    Hb, Hf = np.asarray(Hb, np.float64).reshape(-1, 3, 3), np.asarray(Hf, np.float64).reshape(-1, 3, 3)
    out = []
    for i in range(F.shape[0]):
        b, hb, hf = B[i % B.shape[0]], Hb[i % Hb.shape[0]], Hf[i % Hf.shape[0]]
        out.append(co.composite_reg_img(cv2.warpPerspective(b, hb, dsize), cv2.warpPerspective(F[i], hf, dsize),
                                        cv2.warpPerspective(M[i], hf, dsize)))
    return np.stack(out)


def _check_all_routes(B, F, M, Hb, Hf, dsize, what, cv2_ref=True):
    """The device-matrix ctypes call, operator and composite_bev_batch equal the host-matrix call and,
    with cv2_ref, live cv2"""
    n = F.shape[0]
    w, h = dsize
    ref = _native.composite_bev_u8c3(B, F, M, Hb, Hf, dsize)
    out = _native.composite_bev_u8c3_dmat(B, F, M, _dev(Hb), _dev(Hf), dsize, out=_poison((n, h, w, 3)))
    assert torch.equal(out, ref), what
    assert torch.equal(ops.composite_bev(B, F, M, _dev(Hb), _dev(Hf), w, h), ref), what
    assert torch.equal(compo.composite_bev_batch(B, F, M, _dev(Hb), _dev(Hf), dsize), ref), what
    if cv2_ref:
        assert np.array_equal(out.cpu().numpy(), _cv2_chain(B, F, M, Hb, Hf, dsize)), what
    return out


# ---- 1. the same bytes as host matrices, and as live cv2 -----------------------------------------

@pytest.mark.parametrize("n_bg", ["1", "N"])
@pytest.mark.parametrize("pairs", ["shared", "per-frame"])
def test_equals_host_matrices_and_cv2(n_bg, pairs):
    rng = np.random.default_rng(11 + (n_bg == "N") + 2 * (pairs == "per-frame"))
    n, dsize = 5, (96, 72)
    B = _u8(20, 1 if n_bg == "1" else n, 60, 88, 3)
    F, M = _u8(21, n, 64, 48, 3), _mask(22, n, 64, 48)
    k = 1 if pairs == "shared" else n
    Hb = np.stack([_quad_h(rng, (88, 60), dsize, 0.3) for _ in range(k)])
    Hf = np.stack([_quad_h(rng, (48, 64), dsize, 0.3) for _ in range(k)])
    _check_all_routes(B, F, M, Hb, Hf, dsize, (n_bg, pairs))
    # unbatched 3x3 matrices and one frame through the operator
    one = ops.composite_bev(B[0], F[1], M[1], _dev(Hb[0]), _dev(Hf[0]), *dsize)
    assert torch.equal(one, _native.composite_bev_u8c3(B[:1], F[1:2], M[1:2], Hb[0], Hf[0], dsize)[0])


def test_full_size_renders():
    """1080p renders over a 1080p background into a 1024^2 BEV, with a pair per frame"""
    rng = np.random.default_rng(13)
    n = 3
    B, F, M = _u8(30, 1, 1080, 1920, 3), _u8(31, n, 1080, 1920, 3), _mask(32, n, 1080, 1920)
    Hb = np.repeat(util.h_canon()[None], n, 0)
    Hf = np.stack([_quad_h(rng, (1920, 1080), (1024, 1024), 0.15) for _ in range(n)])
    _check_all_routes(B, F, M, Hb, Hf, (1024, 1024), "1080p", cv2_ref=False)
    assert np.array_equal(_native.composite_bev_u8c3_dmat(B, F[:1], M[:1], _dev(Hb[0]), _dev(Hf[0]), (1024, 1024))
                          .cpu().numpy(), _cv2_chain(B, F[:1], M[:1], Hb[0], Hf[0], (1024, 1024)))


def test_float32_cuda_matrices_are_converted():
    """The ctypes call and the operator convert non-float64 CUDA matrices on the stream, as the
    operator converts CPU ones"""
    rng = np.random.default_rng(14)
    B, F, M = _u8(40, 2, 60, 88, 3), _u8(41, 2, 64, 48, 3), _mask(42, 2, 64, 48)
    Hb = np.stack([_quad_h(rng, (88, 60), (96, 72), 0.3) for _ in range(2)]).astype(np.float32)
    Hf = np.stack([_quad_h(rng, (48, 64), (96, 72), 0.3) for _ in range(2)]).astype(np.float32)
    ref = ops.composite_bev(B, F, M, torch.from_numpy(Hb), torch.from_numpy(Hf), 96, 72)
    Hbd, Hfd = torch.from_numpy(Hb).to(DEV), torch.from_numpy(Hf).to(DEV)
    assert torch.equal(ops.composite_bev(B, F, M, Hbd, Hfd, 96, 72), ref)
    assert torch.equal(_native.composite_bev_u8c3_dmat(B, F, M, Hbd, Hfd, (96, 72)), ref)


# ---- 2. matrix tables of several launches ---------------------------------------------------------

@pytest.mark.parametrize("n", [33, 65])
def test_per_frame_pairs_over_several_launches(n):
    """A launch carries 32 groups: 33 and 65 per-frame pairs take two and three launches"""
    rng = np.random.default_rng(n)
    dsize = (48, 32)
    B, F, M = _u8(50 + n, n, 32, 44, 3), _u8(51 + n, n, 24, 36, 3), _mask(52 + n, n, 24, 36)
    Hb = np.stack([_quad_h(rng, (44, 32), dsize, 0.3) for _ in range(n)])
    Hf = np.stack([_quad_h(rng, (36, 24), dsize, 0.3) for _ in range(n)])
    _check_all_routes(B, F, M, Hb, Hf, dsize, n)
    _check_all_routes(B[:1], F, M, Hb, Hf, dsize, (n, "one background"))


# ---- 3. exact ties and degenerate maps ------------------------------------------------------------

TIES = [np.diag([2.0, 2.0, 1.0]), np.diag([0.5, 0.5, 1.0]), np.diag([4.0, 2.0, 1.0]),
        np.array([[1.0, 0.0, -6.5], [0.0, 1.0, 3.0], [0.0, 0.0, 1.0]]),
        np.zeros((3, 3)),                                                   # singular: the zero map
        np.array([[1.0, 2.0, 3.0], [2.0, 4.0, 6.0], [0.0, 0.0, 1.0]]),      # singular
        np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.05, -1.5]])]  # horizon inside the output


def test_exact_ties_and_singular_maps():
    B, F, M = _u8(60, 1, 61, 96, 3), _u8(61, 1, 58, 100, 3), _mask(62, 1, 58, 100)
    for i, Hb in enumerate(TIES):
        for Hf in (TIES[(i + 2) % len(TIES)], np.diag([0.5, 0.5, 1.0])):
            _check_all_routes(B, F, M, Hb, Hf, (80, 64), (Hb.tolist(), Hf.tolist()))
    # a per-frame table whose singular pair sits between regular ones
    Bn, Fn, Mn = _u8(63, 3, 61, 96, 3), _u8(64, 3, 58, 100, 3), _mask(65, 3, 58, 100)
    Hs = np.stack([TIES[0], TIES[5], TIES[1]])
    _check_all_routes(Bn, Fn, Mn, Hs, Hs[::-1], (80, 64), "table with a singular pair")


# ---- 4. widths that are not multiples of 4: the unfused route -------------------------------------

@pytest.mark.parametrize("n_bg, pairs", [(1, 1), (1, 3), (3, 3)])
def test_unfused_route_with_cuda_matrices(n_bg, pairs):
    rng = np.random.default_rng(70 + n_bg + pairs)
    dsize = (37, 22)
    B, F, M = _u8(70, n_bg, 30, 41, 3), _u8(71, 3, 30, 41, 3), _mask(72, 3, 30, 41)
    Hb = np.stack([_quad_h(rng, (41, 30), dsize, 0.2) for _ in range(pairs)])
    Hf = np.stack([_quad_h(rng, (41, 30), dsize, 0.2) for _ in range(pairs)])
    out = compo.composite_bev_batch(B, F, M, _dev(Hb), _dev(Hf), dsize)
    assert torch.equal(out, compo.composite_bev_batch(B, F, M, Hb, Hf, dsize))
    assert np.array_equal(out.cpu().numpy(), _cv2_chain(B, F, M, Hb, Hf, dsize))
    with pytest.raises(_native.NativeError, match="multiples of 4"):
        compo.composite_bev_batch(B, F, M, _dev(Hb), _dev(Hf), dsize, fused=True)


@pytest.mark.parametrize("n_bg, pairs", [(1, 1), (1, 4), (4, 4)])
def test_fused_and_unfused_routes_agree(n_bg, pairs):
    rng = np.random.default_rng(80 + n_bg + pairs)
    dsize = (128, 96)
    B, F, M = _u8(80, n_bg, 90, 160, 3), _u8(81, 4, 72, 128, 3), _mask(82, 4, 72, 128)
    Hb = _dev(np.stack([_quad_h(rng, (160, 90), dsize, 0.2) for _ in range(pairs)]))
    Hf = _dev(np.stack([_quad_h(rng, (128, 72), dsize, 0.2) for _ in range(pairs)]))
    fused = compo.composite_bev_batch(B, F, M, Hb, Hf, dsize, fused=True)
    assert torch.equal(fused, compo.composite_bev_batch(B, F, M, Hb, Hf, dsize, fused=False))
    assert torch.equal(fused, compo.composite_bev_batch(B, F, M, Hb.cpu().numpy(), Hf.cpu().numpy(), dsize))


def test_argument_validation():
    B, F, M = _u8(90, 1, 8, 8, 3), _u8(91, 2, 8, 8, 3), _u8(92, 2, 8, 8, 3)
    Hd, Hh = torch.eye(3, dtype=torch.float64, device=DEV), torch.eye(3, dtype=torch.float64)
    with pytest.raises(TypeError, match="CUDA tensor"):
        _native.composite_bev_u8c3_dmat(B, F, M, np.eye(3), np.eye(3), (8, 8))
    with pytest.raises(TypeError, match="CUDA tensor"):
        _native.composite_bev_u8c3_dmat(B, F, M, Hd, Hh, (8, 8))
    with pytest.raises(ValueError, match="3x3"):
        _native.composite_bev_u8c3_dmat(B, F, M, torch.eye(4, dtype=torch.float64, device=DEV), Hd, (8, 8))
    with pytest.raises(ValueError, match="homography pairs"):
        _native.composite_bev_u8c3_dmat(B, F, M, Hd.expand(3, 3, 3), Hd.expand(3, 3, 3), (8, 8))
    with pytest.raises(TypeError, match="CUDA tensor"):  # one CUDA and one host matrix: no silent copy
        compo.composite_bev_batch(B, F, M, np.eye(3), Hd, (8, 8))
    with pytest.raises(TypeError, match="CUDA tensor"):
        compo.composite_bev_batch(B, F, M, Hd, Hh, (7, 8))
    for a, b in ((Hd, Hh), (Hh, Hd)):
        with pytest.raises(RuntimeError, match="both homographies on the host or both"):
            ops.composite_bev(B, F, M, a, b, 8, 8)


# ---- 5. stream order ------------------------------------------------------------------------------

def test_matrices_are_read_in_stream_order():
    """H_fg.copy_(new) enqueued behind a long kernel, then the compositor, with no host sync: it uses new"""
    rng = np.random.default_rng(95)
    dsize = (96, 72)
    B, F, M = _u8(95, 1, 60, 88, 3), _u8(96, 3, 64, 48, 3), _mask(97, 3, 64, 48)
    Hb = _quad_h(rng, (88, 60), dsize, 0.3)
    old, new = _quad_h(rng, (48, 64), dsize, 0.3), _quad_h(rng, (48, 64), dsize, 0.3)
    ref = _native.composite_bev_u8c3(B, F, M, Hb, new, dsize)
    Hbd, new_d = _dev(Hb), _dev(new)
    for trial in range(3):
        Hf = _dev(old)
        torch.cuda.synchronize()
        torch.cuda._sleep(200_000_000)  # a long kernel ahead of the copy
        Hf.copy_(new_d)
        if trial == 0:
            out = _native.composite_bev_u8c3_dmat(B, F, M, Hbd, Hf, dsize)
        elif trial == 1:
            out = ops.composite_bev(B, F, M, Hbd, Hf, *dsize)
        else:
            out = compo.composite_bev_batch(B, F, M, Hbd, Hf, dsize)
        assert not torch.cuda.current_stream().query(), "the host waited for the stream"
        torch.cuda.synchronize()
        assert torch.equal(out, ref), trial


# ---- 6. CUDA-graph capture ------------------------------------------------------------------------

def _render_pose(yaw, tilt, height):
    """H_img2bev of a rendering camera made on the GPU: H_world2bev @ inv(K [r1 r2 t]) for a camera
    above the ground plane looking down, turned by yaw and tilted by tilt (radians)"""
    f64 = dict(dtype=torch.float64, device=DEV)
    K = torch.tensor([[400.0, 0.0, 239.5], [0.0, 400.0, 134.5], [0.0, 0.0, 1.0]], **f64)
    W2B = torch.tensor([[12.8, 0.0, 128.0], [0.0, -12.8, 128.0], [0.0, 0.0, 1.0]], **f64)
    c, s = torch.cos(yaw), torch.sin(yaw)
    ct, st = torch.cos(tilt), torch.sin(tilt)
    zero, one = torch.zeros_like(c), torch.ones_like(c)
    Rz = torch.stack([torch.stack([c, -s, zero]), torch.stack([s, c, zero]), torch.stack([zero, zero, one])])
    Rx = torch.stack([torch.stack([one, zero, zero]), torch.stack([zero, ct, -st]), torch.stack([zero, st, ct])])
    R = Rx @ torch.diag(torch.tensor([1.0, -1.0, -1.0], **f64)) @ Rz
    C = torch.stack([zero, zero, height])
    t = -(R @ C)
    H_world2img = K @ torch.stack([R[:, 0], R[:, 1], t], 1)
    return W2B @ torch.linalg.inv(H_world2img)


def test_graph_replays_new_camera_poses():
    """One composite_bev captured with CUDA H_bg / H_fg, replayed with three rendering-camera poses
    made in torch and three new renders: each replay equals the eager call, with host and with
    device matrices"""
    bg, fg, mask = _u8(100, 270, 480, 3), _u8(101, 2, 270, 480, 3), _mask(102, 2, 270, 480)
    Hb = _dev(np.stack([H270, np.diag([1.0, 0.9, 1.0]) @ H270]))
    f64 = dict(dtype=torch.float64, device=DEV)
    Hf = _render_pose(torch.tensor(0.0, **f64), torch.tensor(0.0, **f64), torch.tensor(10.0, **f64))
    Hf = Hf.expand(2, 3, 3).contiguous()

    def fn():
        return ops.composite_bev(bg, fg, mask, Hb, Hf, 256, 256)

    fn()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn()
    first = None
    for k in range(3):
        for i in range(2):
            Hf[i].copy_(_render_pose(torch.tensor(0.2 * k + 0.1 * i, **f64), torch.tensor(0.05 * (k - 1), **f64),
                                     torch.tensor(9.0 + k, **f64)))
        fg.copy_(_u8(103 + k, 2, 270, 480, 3))
        graph.replay()
        torch.cuda.synchronize()
        Hh = Hf.cpu()
        assert torch.equal(out, ops.composite_bev(bg, fg, mask, Hb.cpu(), Hh, 256, 256)), k
        assert torch.equal(out, fn()), k
        if first is None:
            first = (out.clone(), Hh)
        else:
            assert not torch.equal(out[0], first[0][0]) and not torch.equal(Hh, first[1]), "replayed the old pose"


# ---- 7. torch.compile and opcheck -----------------------------------------------------------------

def composite_loop(bg, fg, mask, Hb, Hf):
    return ops.composite_bev(bg, fg, mask, Hb, Hf, 256, 128)


def test_compile_with_cuda_matrices():
    compiled = torch.compile(composite_loop, fullgraph=True, dynamic=True)
    bg = _u8(110, 270, 480, 3)
    Hb = _dev(np.diag([1.0, 0.5, 1.0]) @ H270)
    for seed, n in ((111, 2), (112, 3)):
        fg, mask = _u8(seed, n, 270, 480, 3), _mask(seed + 10, n, 270, 480)
        Hf = _dev(np.stack([np.diag([1.0, 0.5 + 0.01 * i, 1.0]) @ H270 for i in range(n)]))
        out = compiled(bg, fg, mask, Hb.expand(n, 3, 3), Hf)
        ref = composite_loop(bg, fg, mask, Hb.expand(n, 3, 3).cpu(), Hf.cpu())
        assert out.shape[0] == n and torch.equal(out, ref), n


def test_opcheck_with_cuda_matrices():
    f, m, b = _u8(120, 2, 64, 96, 3), _mask(121, 2, 64, 96), _u8(122, 64, 96, 3)
    M = _dev(np.stack([S4 @ H270, S4 @ H270 @ np.diag([1.0, 0.95, 1.0])]))
    for Hb, Hf in ((M, M.flip(0)), (M.float(), M), (M[0], M[1])):
        torch.library.opcheck(ops.composite_bev.default, (b, f, m, Hb, Hf, 48, 32))
