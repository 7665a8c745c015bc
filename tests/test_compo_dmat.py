"""CPU: the device-matrix compositor (bevk_composite_bev_u8c3_dmat) rejects bad arguments with BEVK_E_ARG
before it looks for a device, as its host-matrix twin does, and composite_bev's Meta / FakeTensor
kernel gives the output shape when the homographies live on a device."""
import ctypes

import numpy as np
import pytest
import torch
from torch._dynamo.source import ConstantSource
from torch._subclasses.fake_tensor import FakeTensorMode
from torch.fx.experimental.symbolic_shapes import DimDynamic, ShapeEnv

from bev_b200 import _native, torch_ops

ARG, NOGPU = -1, -3
ENTRIES = ("bevk_composite_bev_u8c3_dmat", "bevk_composite_bev_u8c3")
_buf = ctypes.create_string_buffer(4096)
_mats = np.zeros((4, 9), np.float64)  # stands in for a device table: a rejected call never reads it


@pytest.fixture(scope="module", autouse=True)
def _ops():
    torch_ops.load()


def _call(entry, n=2, n_bg=1, bg_h=8, bg_w=8, fg_h=8, fg_w=8, dh=4, dw=4, Hb=True, Hf=True, n_mats=1):
    """One call of the compositor entry point; returns (rc, error message)."""
    lib = _native.lib()
    m = _mats.ctypes.data_as(ctypes.POINTER(ctypes.c_double))
    rc = getattr(lib, entry)(_buf, _buf, _buf, _buf, n, n_bg, bg_h, bg_w, fg_h, fg_w, dh, dw, m if Hb else None,
                             m if Hf else None, n_mats, None)
    return rc, lib.bevk_last_error().decode()


CASES = [
    (dict(Hb=False), "homography pairs"),
    (dict(Hf=False), "homography pairs"),
    (dict(Hb=False, Hf=False), "homography pairs"),
    (dict(n_mats=0), "homography pairs"),
    (dict(n_mats=3), "homography pairs"),
    (dict(n=3, n_mats=2), "homography pairs"),
    (dict(n_bg=0), "backgrounds"),
    (dict(n_bg=3), "backgrounds"),
    (dict(n=4, n_bg=2, n_mats=4), "backgrounds"),
    (dict(bg_w=6), "multiples of 4"),
    (dict(fg_w=10), "multiples of 4"),
    (dict(dw=5), "multiples of 4"),
    (dict(bg_h=40000), "32767"),
    (dict(fg_w=32768), "32767"),
    (dict(dh=32768), "32767"),
    (dict(fg_h=1), "at least 2x2"),
    (dict(dw=0), "at least 2x2"),
    (dict(n=-1), "n_frames"),
]


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("kw, msg", CASES, ids=[str(i) for i in range(len(CASES))])
def test_c_argument_errors(entry, kw, msg):
    """BEVK_E_ARG with a message, before any device probe: also on a machine without a GPU.  The
    host-matrix twin gives the same answer to every case."""
    rc, err = _call(entry, **kw)
    assert rc == ARG, (entry, kw, rc, err)
    assert msg in err, (entry, kw, err)


@pytest.mark.parametrize("entry", ENTRIES)
def test_good_arguments_reach_the_device_probe(entry):
    """Arguments that pass return BEVK_OK (0 frames: nothing to do) or, without an sm_100 device,
    BEVK_E_NOGPU: the checks above are the only ones made on the host.  Only empty batches: the
    buffers here are host memory, which a launch on a GPU machine must never be given."""
    for kw in (dict(n=0, n_bg=0, n_mats=0), dict(n=0)):
        rc, err = _call(entry, **kw)
        assert rc in (0, NOGPU), (entry, kw, err)


def test_dmat_entry_point_is_bound():
    assert _native.SIGNATURES["bevk_composite_bev_u8c3_dmat"] == _native.SIGNATURES["bevk_composite_bev_u8c3"]


def _frames(n, dev):
    t = lambda *s: torch.empty(s, dtype=torch.uint8, device=dev)  # noqa: E731
    return t(270, 480, 3), t(n, 270, 480, 3), t(n, 270, 480, 3)


@pytest.mark.parametrize("k", [1, 3])
def test_meta_shapes_with_meta_matrices(k):
    bg, fg, mask = _frames(3, "meta")
    for H in (torch.empty((k, 3, 3), dtype=torch.float64, device="meta"),
              torch.empty((k * 9,), dtype=torch.float32, device="meta")):
        out = torch.ops.bev_cuda.composite_bev(bg, fg, mask, H, H, 256, 128)
        assert out.device.type == "meta" and tuple(out.shape) == (3, 128, 256, 3) and out.dtype == torch.uint8
    one = torch.ops.bev_cuda.composite_bev(bg, fg[0], mask[0], H[:9], H[:9], 256, 128)
    assert tuple(one.shape) == (128, 256, 3)
    other = torch.empty((k + 1, 3, 3), dtype=torch.float64, device="meta")
    with pytest.raises(RuntimeError, match="as many matrices"):
        torch.ops.bev_cuda.composite_bev(bg, fg, mask, H, other, 256, 128)


def test_fake_cuda_matrices_with_a_symbolic_batch():
    """torch.compile's view: CUDA frames and CUDA matrices of a symbolic batch, no guard on it."""
    env = ShapeEnv()
    src = ConstantSource("n_frames")
    n = env.create_symintnode(env.create_symbol(5, source=src, dynamic_dim=DimDynamic.DYNAMIC), hint=5, source=src)
    with FakeTensorMode(shape_env=env):
        bg, fg, mask = _frames(n, "cuda")
        H = torch.empty((n, 3, 3), dtype=torch.float64, device="cuda")
        guards = len(env.guards)
        out = torch.ops.bev_cuda.composite_bev(bg, fg, mask, H, H, 256, 128)
        assert out.device == torch.device("cuda", 0) and isinstance(out.shape[0], torch.SymInt)
        assert tuple(out.shape[1:]) == (128, 256, 3)
        assert env.guards[guards:] == []
