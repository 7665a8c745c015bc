"""torch.ops.bev_cuda without a GPU: every operator's Meta kernel (the same C++ function as its CUDA
kernel, returning after the shape checks) gives the documented output shape and dtype, carries a
symbolic batch dimension through FakeTensor without a guard, raises shape errors, and CPU frames still
fail in the dispatcher."""
import pytest
import torch
from torch._dynamo.source import ConstantSource
from torch._subclasses.fake_tensor import FakeTensorMode
from torch.fx.experimental.symbolic_shapes import DimDynamic, ShapeEnv

from bev_b200 import torch_ops

U8, F32, F64 = torch.uint8, torch.float32, torch.float64


@pytest.fixture(scope="module", autouse=True)
def _ops():
    torch_ops.load()


def _cases(n, dev):
    """name -> (args, expected shape, expected dtype) for a batch of n (None: one unbatched frame; the
    box operators always take rows).  Frames and boxes on `dev`; matrices are host float64."""
    def t(*shape, dtype=U8):
        return torch.empty(shape, dtype=dtype, device=dev)

    def B(*shape):
        return shape if n is None else (n,) + shape

    M, K, Rt = torch.eye(3, dtype=F64), torch.eye(3, dtype=F64), torch.zeros((3, 4), dtype=F64)
    rows = 7 if n is None else n
    return {
        "warp_perspective": ((t(*B(270, 480, 3)), M, 256, 128), B(128, 256, 3), U8),
        "resize": ((t(*B(1080, 1920, 3)), 852, 480), B(480, 852, 3), U8),
        "nv12_to_bgr": ((t(*B(1620, 1920)),), B(1080, 1920, 3), U8),
        "warp_perspective_nv12": ((t(*B(1620, 1920)), M, 256, 128), B(128, 256, 3), U8),
        "resize_nv12": ((t(*B(1620, 1920)), 852, 480, 3), B(480, 852, 3), U8),
        "bgr_to_yuv420": ((t(*B(1080, 1920, 3)), 1), B(1620, 1920), U8),
        "warp_perspective_yuv420": ((t(*B(270, 480, 3)), M, 256, 128), B(192, 256), U8),
        "warp_perspective_nv12_yuv420": ((t(*B(1620, 1920)), M, 256, 128, 1), B(192, 256), U8),
        "composite": ((t(*B(64, 96, 3)), t(*B(64, 96, 3)), t(*B(64, 96, 3)), 1), B(64, 96, 3), U8),
        "composite_bev": ((t(270, 480, 3), t(*B(270, 480, 3)), t(*B(270, 480, 3)), M, M, 256, 128),
                          B(128, 256, 3), U8),
        "project_points": ((t(rows, 3, dtype=F32), M), (rows, 3), F32),
        "rbox_corners_project": ((t(rows, 5, dtype=F64), None, 0), (rows, 8), F64),
        "corners_to_rbox": ((t(rows, 8, dtype=F32), M, 1), (rows, 5), F32),
        "rbox_similarity": ((t(rows, 5, dtype=F32), M, 1), (rows, 5), F32),
        "rboxtt_similarity": ((t(rows, 7, dtype=F32), M, 1), (rows, 7), F32),
        "rbox_zt2tt_world": ((t(rows, 7, dtype=F32), K, Rt), (rows, 7), F32),
        "rbox_heading": ((t(rows, 5, dtype=F32), 0), (rows, 4), F32),
        "corners_heading": ((t(rows, 8, dtype=F64),), (rows, 4), F64),
        "angle_similarity": ((t(rows, 2, dtype=F32), M, 0), (rows * 2,), F32),
        "dist_similarity": ((t(rows, 2, dtype=F32), M), (rows, 2), F32),
        "v2yaw": ((t(rows, 2, dtype=F32), 1), (rows,), F32),
        "yaw2v": ((t(rows, dtype=F32), 1), (rows, 2), F32),
        "yaw2mat": ((t(rows, dtype=F64), 0), (rows, 2, 2), F64),
        "rbox_iou_matrix": ((t(rows, 6, dtype=F32)[:, :5], t(11, 5, dtype=F32), 1.5), (rows, 11), F32),
    }


def test_registered_operators_are_the_documented_list():
    registered = {name.split("::")[1] for name in torch._C._dispatch_get_all_op_names()
                  if name.startswith("bev_cuda::")}
    assert registered == set(torch_ops.OPS)
    assert set(_cases(3, "meta")) == set(torch_ops.OPS)
    for name in torch_ops.OPS:
        assert name in torch_ops.__doc__, name


@pytest.mark.parametrize("n", [3, None], ids=["batched", "unbatched"])
def test_meta_shapes(n):
    for name, (args, shape, dtype) in _cases(n, "meta").items():
        out = getattr(torch.ops.bev_cuda, name)(*args)
        assert out.device.type == "meta" and tuple(out.shape) == shape and out.dtype == dtype, name
        assert out.is_contiguous(), name


def test_meta_pitched_nv12_and_mat_index():
    surface = torch.empty((4, 1620, 2048), dtype=U8, device="meta")[:, :, :1920]  # padded decoder rows
    M = torch.eye(3, dtype=F64).expand(2, 3, 3)
    idx = torch.tensor([0, 1, 1, 0], dtype=torch.int32)
    ops = torch.ops.bev_cuda
    assert ops.nv12_to_bgr(surface).shape == (4, 1080, 1920, 3)
    assert ops.warp_perspective_nv12(surface, M, 256, 128, mat_index=idx).shape == (4, 128, 256, 3)
    assert ops.warp_perspective_nv12_yuv420(surface, M, 256, 128, mat_index=idx).shape == (4, 192, 256)
    assert ops.resize_nv12(surface[1], 852, 480).shape == (480, 852, 3)
    assert ops.warp_perspective(torch.empty((4, 8, 8, 1), dtype=torch.float16, device="meta"), M, 4, 2,
                                mat_index=idx).shape == (4, 2, 4, 1)
    assert ops.resize(torch.empty((2, 9, 7, 4), dtype=U8, device="meta"), 3, 5).shape == (2, 5, 3, 4)
    assert ops.warp_perspective(torch.empty((9, 7), dtype=U8, device="meta"), M[0], 3, 5).shape == (5, 3)


def test_symbolic_batch_passes_every_operator_without_a_guard():
    env = ShapeEnv()
    mode = FakeTensorMode(shape_env=env)
    src = ConstantSource("n_frames")
    n = env.create_symintnode(env.create_symbol(5, source=src, dynamic_dim=DimDynamic.DYNAMIC), hint=5, source=src)
    with mode:
        cases = _cases(n, "cuda")
        guards = len(env.guards)
        for name, (args, shape, dtype) in cases.items():
            out = getattr(torch.ops.bev_cuda, name)(*args)
            assert out.device.type == "cuda" and out.dtype == dtype, name
            assert len(out.shape) == len(shape) and all(a == b for a, b in zip(out.shape, shape)), name
            assert isinstance(out.shape[0], torch.SymInt), name
        assert env.guards[guards:] == []  # nothing was specialised on the batch size


def test_fake_tensor_outputs_follow_the_frames_device():
    with FakeTensorMode():
        for name, (args, shape, dtype) in _cases(3, "cuda").items():
            out = getattr(torch.ops.bev_cuda, name)(*args)
            assert out.device == torch.device("cuda", 0) and tuple(out.shape) == shape, name


ERRORS = [  # (operator, args on `dev`, message)
    ("warp_perspective", lambda d: (torch.empty((2, 3, 4, 5, 3), dtype=U8, device=d), torch.eye(3, dtype=F64),
                                    4, 4), "src must be"),
    ("warp_perspective", lambda d: (torch.empty((2, 4, 4, 3), dtype=U8, device=d), torch.zeros(8, dtype=F64), 4, 4),
     "multiple of 9"),
    ("warp_perspective", lambda d: (torch.empty((2, 4, 4, 3), dtype=U8, device=d), torch.eye(3, dtype=F64), 4, 4,
                                    1, 0, 0.0, torch.zeros(3, dtype=torch.int32)), "mat_index has 3 entries for 2"),
    ("resize", lambda d: (torch.empty((2, 4, 4, 5), dtype=U8, device=d), 2, 2), "1 to 4 channels"),
    ("resize", lambda d: (torch.empty((4, 4, 3), dtype=F32, device=d), 2, 2), "uint8"),
    ("nv12_to_bgr", lambda d: (torch.empty((7, 8), dtype=U8, device=d),), "H\\*3/2 rows"),
    ("resize_nv12", lambda d: (torch.empty((6, 7), dtype=U8, device=d), 2, 2), "even width"),
    ("warp_perspective_nv12", lambda d: (torch.empty((12, 16), dtype=U8, device=d)[:, ::2],
                                         torch.eye(3, dtype=F64), 4, 4), "inner stride 1"),
    ("bgr_to_yuv420", lambda d: (torch.empty((5, 4, 3), dtype=U8, device=d),), "even width and height"),
    ("warp_perspective_yuv420", lambda d: (torch.empty((4, 4, 3), dtype=U8, device=d), torch.eye(3, dtype=F64),
                                           5, 4), "even width and height"),
    ("warp_perspective_nv12_yuv420", lambda d: (torch.empty((6, 4), dtype=U8, device=d), torch.eye(3, dtype=F64),
                                                5, 6, 0), "even width and height"),
    ("composite", lambda d: (torch.empty((4, 4, 3), dtype=U8, device=d), torch.empty((4, 4, 3), dtype=U8, device=d),
                             torch.empty((4, 5, 3), dtype=U8, device=d)), "share one shape"),
    ("composite_bev", lambda d: (torch.empty((3, 8, 8, 3), dtype=U8, device=d),
                                 torch.empty((2, 8, 8, 3), dtype=U8, device=d),
                                 torch.empty((2, 8, 8, 3), dtype=U8, device=d), torch.eye(3, dtype=F64),
                                 torch.eye(3, dtype=F64), 8, 8), "need 1 or one each"),
    ("rbox_iou_matrix", lambda d: (torch.empty((3, 4), device=d), torch.empty((3, 5), device=d)), "\\(N, >=5\\)"),
    ("rbox_corners_project", lambda d: (torch.empty((3, 5), dtype=U8, device=d), None, 0), "not boxes"),
    ("rbox_similarity", lambda d: (torch.empty((3, 5), device=d), torch.eye(2, dtype=F64), 0), "must be 3x3"),
    ("rbox_zt2tt_world", lambda d: (torch.empty((3, 7), device=d), torch.eye(3, dtype=F64),
                                    torch.eye(3, dtype=F64)), "Rt must be 3x4"),
    ("v2yaw", lambda d: (torch.empty((3, 3), device=d), 0), "expects shape \\(N, 2\\)"),
]


@pytest.mark.parametrize("op, make, msg", ERRORS, ids=["%s-%d" % (e[0], i) for i, e in enumerate(ERRORS)])
def test_shape_errors_on_meta(op, make, msg):
    with pytest.raises(RuntimeError, match=msg):
        getattr(torch.ops.bev_cuda, op)(*make("meta"))


def test_cpu_frames_still_fail_in_the_dispatcher():
    for name, (args, _, _) in _cases(2, "cpu").items():
        with pytest.raises(NotImplementedError):
            getattr(torch.ops.bev_cuda, name)(*args)
    with FakeTensorMode():
        for name, (args, _, _) in _cases(2, "cpu").items():
            with pytest.raises(NotImplementedError):
                getattr(torch.ops.bev_cuda, name)(*args)
