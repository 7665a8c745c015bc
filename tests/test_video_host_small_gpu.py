"""GPU: the one-pass host video call with small frames (bevk_warp_perspective_video_host_small) for
every pair of BGR, I420 and NV12 frame formats, INTER_LINEAR and INTER_AREA small frames, bit for bit
against cv2's own chains: decode -> warpPerspective -> encode for the BEV, decode -> resize ->
warpPerspective -> encode for the small leg.  The device workspace is filled with frames of another
seed before the checked calls, so a row that the upload misses shows up as wrong bytes."""
import cv2
import numpy as np
import pytest
import torch

from bev_b200 import homo
from oracle import yuv420_oracle as yo
from tests import util
from tests.test_video_host_gpu import BV, FORMATS, PAIRS, cv2_chain, frames, quad_map

pytestmark = pytest.mark.gpu

INTERPS = {"linear": cv2.INTER_LINEAR, "area": cv2.INTER_AREA}


def to_bgr(f, fmt):
    return {"bgr": lambda: f, "i420": lambda: cv2.cvtColor(f, cv2.COLOR_YUV2BGR_I420),
            "nv12": lambda: cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)}[fmt]()


def small_map(M, ssize, small_size):
    """The forward map of the small frames: M after scaling small-frame pixels up to the frame."""
    S = np.diag([ssize[0] / small_size[0], ssize[1] / small_size[1], 1.0])
    return M @ S


def poison(sfmt, dfmt, n, ssize, dsize, small_size, interp, seed):
    """The same shapes through the shared device workspace with frames of another seed."""
    H = np.eye(3)
    homo.warp_perspective_video_host_small(frames(sfmt, n, ssize[1], ssize[0], seed + 1000), H, H, dsize,
                                           small_size, sfmt, dfmt, interpolation=interp)


def check(outs, f, sfmt, dfmt, Ms, Ms_small, idx, dsize, small_size, flags, interp, bv, what):
    bev, small, bev_small = outs
    for i in range(len(f)):
        k = i if idx is None and len(Ms) > 1 else (0 if idx is None else idx[i])
        ref_small = cv2.resize(to_bgr(f[i], sfmt), small_size, interpolation=interp)
        refs = (("bev", bev[i], cv2_chain(f[i], sfmt, dfmt, Ms[k], dsize, flags, bv)),
                ("small", small[i], ref_small),
                ("bev_small", bev_small[i], cv2_chain(ref_small, "bgr", dfmt, Ms_small[k], dsize, flags, bv)))
        for name, out, ref in refs:
            assert out.shape == ref.shape and out.dtype == np.uint8, (what, name, out.shape, ref.shape)
            if not np.array_equal(out, ref):
                bad = np.argwhere(out != ref)
                pytest.fail("%s: %s of frame %d differs from cv2 at %d positions, first %s"
                            % (what, name, i, len(bad), bad[0]))


@pytest.mark.parametrize("ssize,dsize,small_size", [((480, 270), (256, 192), (212, 120)),
                                                    ((482, 272), (130, 98), (141, 77))], ids=["w4", "w2"])
@pytest.mark.parametrize("interp", list(INTERPS), ids=list(INTERPS))
@pytest.mark.parametrize("flags", [0, 1])
@pytest.mark.parametrize("sfmt,dfmt", PAIRS, ids=["%s-%s" % p for p in PAIRS])
def test_every_pair_vs_cv2(sfmt, dfmt, flags, interp, ssize, dsize, small_size):
    """All nine pairs, nearest and bilinear warps, both resizes, source widths with W % 4 == 0 (word
    gathers) and == 2 (byte gathers); 141-pixel small frames have an odd width."""
    rng = np.random.default_rng([ssize[0], flags, FORMATS.index(sfmt), FORMATS.index(dfmt), INTERPS[interp]])
    n = 3
    f = frames(sfmt, n, ssize[1], ssize[0], rng.integers(1 << 30))
    H = quad_map(rng, ssize, dsize, (40, ssize[1] - 30))
    Hs = small_map(H, ssize, small_size)
    poison(sfmt, dfmt, n, ssize, dsize, small_size, INTERPS[interp], 1)
    outs = homo.warp_perspective_video_host_small(f, H, Hs, dsize, small_size, sfmt, dfmt, flags=flags,
                                                  interpolation=INTERPS[interp], borderValue=BV)
    check(outs, f, sfmt, dfmt, H[None], Hs[None], None, dsize, small_size, flags, INTERPS[interp], BV,
          "%s -> %s flags %d %s" % (sfmt, dfmt, flags, interp))
    one = homo.warp_perspective_video_host_small(f[1], H, Hs, dsize, small_size, sfmt, dfmt, flags=flags,
                                                 interpolation=INTERPS[interp], borderValue=BV)
    for a, b in zip(one, outs):  # an unbatched frame
        assert np.array_equal(a, b[1])


@pytest.mark.parametrize("small_size", [(240, 135), (160, 90), (960, 540), (97, 55), (1, 1), (33, 200)])
@pytest.mark.parametrize("sfmt", FORMATS)
@pytest.mark.parametrize("ssize", [(480, 270), (482, 272)], ids=["w4", "w2"])
def test_resize_branches(ssize, sfmt, small_size):
    """cv2's INTER_AREA branches from 480 x 270 frames -- exact 2x and 3x integer cells, an upscale,
    non-integer cells, 1-pixel frames, one axis up and one down -- and INTER_LINEAR on the same sizes;
    from 482-wide frames too, so that word and byte gathers each meet packed and unpacked stores."""
    dsize, n = (64, 48), 3
    rng = np.random.default_rng([ssize[0], small_size[0], FORMATS.index(sfmt)])
    f = frames(sfmt, n, ssize[1], ssize[0], rng.integers(1 << 30))
    H = quad_map(rng, ssize, dsize, (30, 250))
    Hs = small_map(H, ssize, small_size)
    for name, interp in INTERPS.items():
        poison(sfmt, "bgr", n, ssize, dsize, small_size, interp, 2)
        outs = homo.warp_perspective_video_host_small(f, H, Hs, dsize, small_size, sfmt, "bgr", interpolation=interp)
        check(outs, f, sfmt, "bgr", H[None], Hs[None], None, dsize, small_size, 1, interp, 0,
              "%s %s %s" % (sfmt, small_size, name))


@pytest.mark.parametrize("sfmt,dfmt", [("i420", "i420"), ("bgr", "bgr"), ("nv12", "i420"), ("bgr", "nv12")])
def test_chunks_cameras_and_per_frame_matrices(sfmt, dfmt):
    """9 full-HD frames go up in 3 chunks; three cameras picked by mat_index, and one matrix per frame."""
    ssize, dsize, small_size, n = (1920, 1080), (256, 192), (852, 480), 9
    rng = np.random.default_rng([FORMATS.index(sfmt), FORMATS.index(dfmt)])
    f = frames(sfmt, n, ssize[1], ssize[0], rng.integers(1 << 30))
    mats = np.stack([quad_map(rng, ssize, dsize, (100 + 150 * k, 600 + 200 * k)) for k in range(n)])
    mats_small = np.stack([small_map(M, ssize, small_size) for M in mats])
    idx = np.array([2, 0, 1, 1, 0, 2, 2, 1, 0], np.int32)
    for what, Ms, Mss, ix in (("mat_index", mats[:3], mats_small[:3], idx), ("per-frame", mats, mats_small, None)):
        for interp in INTERPS.values():
            poison(sfmt, dfmt, n, ssize, dsize, small_size, interp, 3)
            kw = {} if ix is None else {"mat_index": ix}
            outs = homo.warp_perspective_video_host_small(f, Ms, Mss, dsize, small_size, sfmt, dfmt,
                                                          interpolation=interp, **kw)
            check(outs, f, sfmt, dfmt, Ms, Mss, ix, dsize, small_size, 1, interp, 0,
                  "%s -> %s %s interp %d" % (sfmt, dfmt, what, interp))
            bev = homo.warp_perspective_video_host(f, Ms, dsize, sfmt, dfmt, **kw)
            assert np.array_equal(outs[0], bev), what


def _cfg4_camera0():
    from bev_b200.bev import BEVWorldSpec
    from bev_b200.calib import Calib
    cam = util.load_json("cfg4_cams.json")[0]
    calib = Calib(vp1=np.array(cam["vp1"]), vp2=np.array(cam["vp2"]), height=cam["height"],
                  u_size=1920, v_size=1080)
    bspec = BEVWorldSpec(**{k: v for k, v in cam["bspec"].items() if v is not None and k not in ("x_max", "y_max")})
    return calib, bspec


@pytest.mark.parametrize("interp", list(INTERPS), ids=list(INTERPS))
@pytest.mark.parametrize("flags", [0, 1])
def test_equals_the_device_routes(flags, interp):
    """The calib helper's three images equal the device twins on the uploaded frames:
    warp_img_to_bev_video_host for the BEV, warp_small_img_to_bev / warp_small_nv12_img_to_bev for
    the small leg; an I420 frame gives the bytes of its NV12 relayout."""
    calib, bspec = _cfg4_camera0()
    n = 6
    i420 = frames("i420", n, 1080, 1920, 21 + flags)
    src = {"bgr": frames("bgr", n, 1080, 1920, 23 + flags), "i420": i420,
           "nv12": np.stack([yo.i420_to_nv12(x) for x in i420])}
    it = INTERPS[interp]
    got = {}
    for sfmt in FORMATS:
        got[sfmt] = homo.warp_img_and_small_to_bev_video_host(src[sfmt], calib, bspec, 852, 480, sfmt, "bgr",
                                                              flags=flags, interpolation=it)
        bev = homo.warp_img_to_bev_video_host(src[sfmt], calib, bspec, sfmt, "bgr", flags=flags)
        assert np.array_equal(got[sfmt][0], bev), sfmt
    t = torch.from_numpy(src["bgr"]).cuda()
    small, bev_small = homo.warp_small_img_to_bev(t, calib, bspec, 852, 480, flags=flags, interpolation=it)
    assert np.array_equal(got["bgr"][1], small.cpu().numpy()) and np.array_equal(got["bgr"][2], bev_small.cpu().numpy())
    t = torch.from_numpy(src["nv12"]).cuda()
    small, bev_small = homo.warp_small_nv12_img_to_bev(t, calib, bspec, 852, 480, flags=flags, interpolation=it)
    assert np.array_equal(got["nv12"][1], small.cpu().numpy())
    assert np.array_equal(got["nv12"][2], bev_small.cpu().numpy())
    for a, b in zip(got["i420"], got["nv12"]):
        assert np.array_equal(a, b)
    # the YUV BEVs of the same call are the encoder's frames of these BGR BEVs
    yuv = homo.warp_img_and_small_to_bev_video_host(i420, calib, bspec, 852, 480, "i420", "i420", flags=flags,
                                                    interpolation=it)
    for k in (0, 2):
        for i in (0, n - 1):
            assert np.array_equal(yuv[k][i], cv2.cvtColor(got["i420"][k][i], cv2.COLOR_BGR2YUV_I420)), (k, i)
    assert np.array_equal(yuv[1], got["i420"][1])


def test_pinned_pageable_and_empty():
    """Pinned CPU tensors in and out (the fast route) and pageable numpy arrays give the same bytes;
    0 frames return empty batches."""
    ssize, dsize, small_size, n = (1920, 1080), (512, 512), (852, 480), 5
    H = homo.homo_from_pts(np.array([[700, 420], [1220, 420], [1900, 1060], [20, 1060]], np.float64),
                           np.array([[0, 0], [512, 0], [512, 512], [0, 512]], np.float64))
    Hs = small_map(H, ssize, small_size)
    for sfmt, dfmt in (("i420", "i420"), ("nv12", "bgr"), ("bgr", "nv12")):
        f = frames(sfmt, n, ssize[1], ssize[0], 7)
        pageable = homo.warp_perspective_video_host_small(f, H, Hs, dsize, small_size, sfmt, dfmt)
        src = torch.from_numpy(f).pin_memory()
        outs = tuple(torch.empty(p.shape, dtype=torch.uint8).pin_memory() for p in pageable)
        got = homo.warp_perspective_video_host_small(src, H, Hs, dsize, small_size, sfmt, dfmt, dst=outs[0],
                                                     small=outs[1], dst_small=outs[2])
        assert all(g is o for g, o in zip(got, outs))
        for o, p in zip(outs, pageable):
            assert np.array_equal(o.numpy(), p)
        check(tuple(p[[0, n - 1]] for p in pageable), f[[0, n - 1]], sfmt, dfmt, H[None], Hs[None], None, dsize,
              small_size, 1, cv2.INTER_LINEAR, 0, "%s -> %s" % (sfmt, dfmt))
        empty = homo.warp_perspective_video_host_small(f[:0], H, Hs, dsize, small_size, sfmt, dfmt)
        assert [e.shape for e in empty] == [(0,) + p.shape[1:] for p in pageable]


def test_device_buffers_are_refused():
    """Frames or outputs on the GPU are refused, with the name of the function that takes host buffers."""
    H = np.eye(3)
    f = np.zeros((12, 8), np.uint8)
    call = homo.warp_perspective_video_host_small
    with pytest.raises(ValueError, match="src is on cuda.*warp_perspective_video_host_small takes host buffers"):
        call(torch.from_numpy(f).cuda(), H, H, (4, 4), (4, 2), "i420", "i420")
    for name, shape in (("dst", (6, 4)), ("small", (2, 4, 3)), ("dst_small", (6, 4))):
        out = torch.zeros(shape, dtype=torch.uint8, device="cuda")
        with pytest.raises(ValueError, match="%s is on cuda.*warp_perspective_video_host_small takes" % name):
            call(f, H, H, (4, 4), (4, 2), "i420", "i420", **{name: out})
