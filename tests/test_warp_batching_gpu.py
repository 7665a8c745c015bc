"""Warp batches whose matrix tables need more than one launch, on every warp entry point.

The host code of every warp splits the frames of each matrix into arithmetic runs (``build_groups``
in csrc/capi.cu) and hands them to the kernels in launches of BEVK_MAX_GROUPS = 16 runs.  Each
launch plans on its own: frame chunks, whether the staged kernel runs (``kMinFrames`` = 4 frames in
its longest run), tile shape, split, TMA map and scratch.  The host-buffer entry point also cuts
the batch into upload chunks and slices ``mat_index`` or the per-frame matrices for each.

The cases below reach 1 to 3 launches with regular, irregular and permuted camera orders, unused
matrices and per-frame tables.  ``launch_structure`` restates ``build_groups`` in Python and the CPU
test holds every case to the launch structure it was written for, so the GPU cases cannot drift
back into a single launch.  The GPU tests compare every frame, bit for bit, with the oracle of its
own matrix and with a single-frame call of the same entry point (one run, one launch).  Outputs go
to buffers filled with a poison byte first, so a frame no launch writes cannot pass by holding an
earlier result.
"""
import functools

import numpy as np
import pytest
import torch

from bev_b200 import _native, homo
from oracle import nv12_oracle as no
from oracle import warp_oracle as wo
from oracle import yuv420_oracle as yo
from tests import util

DEV = "cuda:0"
SEED = 20261021
MAX_GROUPS = 16  # BEVK_MAX_GROUPS (csrc/bevk_common.cuh)
MIN_FRAMES = 4   # kMinFrames of bevk_launch_warp_fast (csrc/warp_fast.cu)
SRC_H, SRC_W = 270, 480
DSIZE = (256, 256)  # (w, h): a width that is a multiple of 4, so the staged kernel qualifies
PATHS = ("generic", "auto", "fast")
FLAGS = (0, 1, 16, 17)
LAYOUTS = ("i420", "nv12")
POISON = 0xA5


# ---- the launch structure (reference only: the library does not use it) -------------------------

def build_groups(n, n_mats, idx):
    """(matrix, first, count, stride) runs in the order csrc/capi.cu's build_groups makes them."""
    if idx is None:
        return [(0, 0, n, 1)] if n_mats == 1 else [(i, i, 1, 1) for i in range(n)]
    per = [[] for _ in range(n_mats)]
    for i, k in enumerate(idx):
        per[int(k)].append(i)
    groups = []
    for k, f in enumerate(per):
        i = 0
        while i < len(f):
            if i + 1 == len(f):
                groups.append((k, f[i], 1, 1))
                break
            stride, j = f[i + 1] - f[i], i + 1
            while j + 1 < len(f) and f[j + 1] - f[j] == stride:
                j += 1
            groups.append((k, f[i], j - i + 1, stride))
            i = j + 1
    return groups


def launch_structure(n, n_mats, idx):
    """[(groups, longest run)] of each launch."""
    g = build_groups(n, n_mats, idx)
    return [(len(g[i:i + MAX_GROUPS]), max(r[2] for r in g[i:i + MAX_GROUPS])) for i in range(0, len(g), MAX_GROUPS)]


# ---- the cases ----------------------------------------------------------------------------------

def _arrival_order(seed, n=40, cams=8, swaps=4):
    """Cameras in turn, with `swaps` frames of cameras 1..6 exchanged (decoder arrival jitter):
    cameras 0 and 7 keep runs of 5, the others break into irregular runs."""
    rng = np.random.default_rng(seed)
    idx = np.arange(n) % cams
    for _ in range(swaps):
        a, b = rng.choice(np.flatnonzero((idx > 0) & (idx < cams - 1)), 2, replace=False)
        idx[a], idx[b] = idx[b], idx[a]
    return idx.astype(np.int32)


def _cases():
    ar = np.arange
    tail = np.r_[ar(64) % 16, [16, 17, 18, 19]]
    perm = np.random.default_rng([SEED, 1]).permutation(96)
    cases = [
        # name, frames, matrices, mat_index (None: one matrix per frame), launches [(groups, longest run)]
        ("i%24", 96, 24, ar(96) % 24, [(16, 4), (8, 4)]),
        ("i%16_then_4_singles", 68, 20, tail, [(16, 4), (4, 1)]),
        ("i%17", 68, 17, ar(68) % 17, [(16, 4), (1, 4)]),
        ("per_frame_33", 33, 33, None, [(16, 1), (16, 1), (1, 1)]),
        ("random_camera_of_8", 64, 8, np.random.default_rng(1).integers(0, 8, 64), [(16, 3), (16, 3), (1, 2)]),
        ("exactly_16", 64, 16, ar(64) % 16, [(16, 4)]),
        ("exactly_32", 128, 32, ar(128) % 32, [(16, 4), (16, 4)]),
        ("odd_half_of_40", 80, 40, 2 * (ar(80) % 20) + 1, [(16, 4), (4, 4)]),
        ("all_to_5_of_8", 24, 8, np.full(24, 5), [(1, 24)]),
        ("reversed_index_33", 33, 33, ar(33)[::-1], [(16, 1), (16, 1), (1, 1)]),
        ("i%24_permuted", 96, 24, (ar(96) % 24)[perm], [(16, 2), (16, 3), (16, 2)]),
    ]
    out = []
    for i, (name, n, k, idx, launches) in enumerate(cases):
        out.append({"name": name, "n": n, "mats": k, "idx": None if idx is None else np.asarray(idx, np.int32),
                    "launches": launches, "seed": [SEED, 0 if name.startswith("i%24") else 100 + i],
                    "perm": perm if name == "i%24_permuted" else None})
    return out


CASES = _cases()
BY_NAME = {c["name"]: c for c in CASES}
WITH_INDEX = [c for c in CASES if c["idx"] is not None]
UNPERMUTED = [c for c in CASES if c["perm"] is None]

CAMS_1080P = {"name": "cfg4_cameras_1080p", "n": 40, "mats": 8, "idx": _arrival_order([SEED, 13]),
              "launches": [(16, 5), (2, 5)]}


def describe(case):
    return "; ".join("%s=%s" % (k, case[k].tolist() if isinstance(case[k], np.ndarray) else case[k])
                     for k in ("name", "n", "mats", "idx", "launches", "seed") if k in case)


def ids(cases):
    return [c["name"] for c in cases]


# ---- CPU: the cases reach the launch structures they exist for ----------------------------------

def test_cases_reach_their_launch_structure():
    for case in CASES + [CAMS_1080P]:
        got = launch_structure(case["n"], case["mats"], case["idx"])
        assert got == case["launches"], "%s reaches %s" % (describe(case), got)
        if case["idx"] is not None:
            assert len(case["idx"]) == case["n"] and 0 <= case["idx"].min() and case["idx"].max() < case["mats"]
        else:
            assert case["mats"] == case["n"]


def test_case_list_covers_the_launch_edges():
    groups = {c["name"]: build_groups(c["n"], c["mats"], c["idx"]) for c in CASES + [CAMS_1080P]}
    counts = {len(g) for g in groups.values()}
    for n_groups in (MAX_GROUPS, MAX_GROUPS + 1, 2 * MAX_GROUPS, 2 * MAX_GROUPS + 1):
        assert n_groups in counts, "no case with %d groups" % n_groups
    launches = [c["launches"] for c in CASES + [CAMS_1080P]]
    assert any(len(L) == 1 and L[0][0] == MAX_GROUPS for L in launches), "no single full launch"
    assert any(len(L) >= 3 for L in launches), "no case of three launches"
    assert any(any(a[1] >= MIN_FRAMES > b[1] for a, b in zip(L, L[1:])) for L in launches), \
        "no staged launch followed by a direct-gather one"
    assert sum(len(L) >= 2 and all(c >= MIN_FRAMES for _, c in L) for L in launches) >= 2, \
        "fewer than two cases that run the staged kernel in every launch"
    runs = [r for g in groups.values() for r in g]
    assert any(r[3] > 1 and r[2] > 1 for r in runs), "no run with stride > 1"
    assert any(r[2] == 1 for r in runs), "no run of one frame"
    assert any(sum(r[0] == k for r in g) >= 2 for g in groups.values() for k in {r[0] for r in g}), \
        "no matrix with two or more runs"
    assert any(c["idx"] is not None and len(set(c["idx"].tolist())) < c["mats"] for c in CASES), "no unused matrix"
    assert any(c["idx"] is None and c["mats"] > 1 for c in CASES), "no per-frame table without an index"
    assert any(c["perm"] is not None for c in CASES), "no permuted frame order"


# ---- inputs and references ----------------------------------------------------------------------

def quad_maps(rng, k, src_rows=(0, SRC_H - 1)):
    """k distinct forward homographies taking jittered quads of the source rows src_rows to the BEV."""
    r0, r1 = src_rows
    quad = np.array([[0, r0], [SRC_W - 1, r0], [SRC_W - 1, r1], [0, r1]], np.float64)
    d = np.array([[0, 0], [DSIZE[0] - 1, 0], [DSIZE[0] - 1, DSIZE[1] - 1], [0, DSIZE[1] - 1]], np.float64)
    jitter = min(30.0, (r1 - r0) / 16.0)
    return np.stack([homo.homo_from_pts_numpy(quad + rng.normal(size=(4, 2)) * jitter, d) for _ in range(k)])


@functools.lru_cache(maxsize=None)
def table(name):
    if name == CAMS_1080P["name"]:
        cams = util.load_json("cfg4_cams.json")
        return np.stack([np.diag([1024.0 / c["bspec"]["u_size"], 1024.0 / c["bspec"]["v_size"], 1.0])
                         @ np.array(c["H_bev_img"]) for c in cams])
    case = BY_NAME[name]
    return quad_maps(np.random.default_rng(case["seed"] + [1]), case["mats"])


def mats(name, flags):
    """The case's table as the call takes it: forward, or dst->src maps with WARP_INVERSE_MAP."""
    Hs = table(name)
    return np.linalg.inv(Hs) if flags & 16 else Hs


def frame_matrix(case, i):
    return case["idx"][i] if case["idx"] is not None else i


def _permuted(case, a):
    return a[case["perm"]] if case["perm"] is not None else a


@functools.lru_cache(maxsize=4)
def frames(name, fmt="u8c3"):
    case = BY_NAME[name]
    rng = np.random.default_rng(case["seed"] + [2, sum(map(ord, fmt))])
    n = case["n"]
    if fmt.startswith("u8"):
        f = rng.integers(0, 256, (n, SRC_H, SRC_W, int(fmt[-1])), dtype=np.uint8)
    else:
        f = rng.uniform(-100, 100, (n, SRC_H, SRC_W, 3)).astype(np.float32 if fmt == "f32c3" else np.float16)
    return _permuted(case, f)


@functools.lru_cache(maxsize=4)
def nv12_frames(name):
    case = BY_NAME[name]
    rng = np.random.default_rng(case["seed"] + [3])
    return _permuted(case, rng.integers(0, 256, (case["n"], SRC_H * 3 // 2, SRC_W), dtype=np.uint8))


@functools.lru_cache(maxsize=16)
def oracle_bgr(name, flags, fmt="u8c3", nv12=False, border=0):
    """Every frame warped by the oracle with its own matrix: (n, h, w, c)."""
    case = BY_NAME[name]
    Ms = mats(name, flags)
    out = []
    for i in range(case["n"]):
        f = no.nv12_to_bgr(nv12_frames(name)[i]) if nv12 else frames(name, fmt)[i]
        out.append(wo.warp_perspective(f, Ms[frame_matrix(case, i)], DSIZE, flags=flags, borderValue=border))
    return np.stack(out)


def oracle_yuv(name, flags, layout, nv12=False):
    return np.stack([yo.convert(b, layout) for b in oracle_bgr(name, flags, nv12=nv12)])


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def poisoned(shape, dtype):
    """A contiguous device tensor whose bytes are all POISON."""
    n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    return torch.full((n,), POISON, dtype=torch.uint8, device=DEV).view(dtype).view(shape)


def poison_allocator(nbytes):
    """Leave a freed block of nbytes poison bytes in the caching allocator, so that the next
    allocation of that size (an operator's output) starts out poisoned."""
    torch.full((nbytes,), POISON, dtype=torch.uint8, device=DEV)


def laid_out(f, pitch, gap_rows):
    """NV12 frames (N, H*3/2, W) as a decoder surface: rows `pitch` bytes apart, `gap_rows` unused rows
    after each frame."""
    n, rows, w = f.shape
    buf = torch.full((n * (rows + gap_rows) * pitch + pitch,), POISON, dtype=torch.uint8, device=DEV)
    view = buf.as_strided((n, rows, w), ((rows + gap_rows) * pitch, pitch, 1))
    view.copy_(cu(f))
    return view


def surface(n, h, w, pitch, gap_rows):
    """An encoder surface for n YUV 4:2:0 frames of h x w filled with POISON: the (N, H*3/2, W) view
    and a mask of the bytes outside it."""
    rows = h * 3 // 2
    buf = torch.full((n * (rows + gap_rows) * pitch,), POISON, dtype=torch.uint8, device=DEV)
    view = buf.as_strided((n, rows, w), ((rows + gap_rows) * pitch, pitch, 1))
    mask = torch.ones_like(buf, dtype=torch.bool)
    mask.as_strided((n, rows, w), ((rows + gap_rows) * pitch, pitch, 1)).fill_(False)
    return buf, view, mask


def assert_frames(out, ref, what, case):
    """Every frame of out (device or host) equals ref bit for bit; names the first frame that does not."""
    out = out.cpu().numpy() if isinstance(out, torch.Tensor) else out
    assert out.shape == ref.shape and out.dtype == ref.dtype, (what, out.shape, ref.shape, describe(case))
    if out.tobytes() != ref.tobytes():
        bad = [i for i in range(ref.shape[0]) if out[i].tobytes() != ref[i].tobytes()]
        pytest.fail("%s: %d of %d frames differ (first %s, matrix %d); %s"
                    % (what, len(bad), ref.shape[0], bad[:8], frame_matrix(case, bad[0]), describe(case)))


def assert_singles(out, single, what, case):
    """out equals the stack of the single-frame calls single(i) (one run, one launch each)."""
    ones = torch.stack([single(i) for i in range(case["n"])])
    if not torch.equal(out, ones):
        bad = [i for i in range(case["n"]) if not torch.equal(out[i], ones[i])]
        pytest.fail("%s differs from single-frame calls at frames %s; %s" % (what, bad[:8], describe(case)))


# ---- BGR frames ---------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=ids(CASES))
def test_warp_perspective_batches(case):
    """uint8 x 3 on every path, both interpolations, with and without WARP_INVERSE_MAP, and a
    non-zero border (which keeps the staged kernel out)."""
    name, n = case["name"], case["n"]
    t = cu(frames(name))
    for flags in FLAGS:
        Ms = mats(name, flags)
        ref = oracle_bgr(name, flags)
        for path in PATHS:
            dst = poisoned((n,) + DSIZE[::-1] + (3,), torch.uint8)
            out = homo.warp_perspective(t, Ms, DSIZE, dst=dst, flags=flags, mat_index=case["idx"], path=path)
            what = "warp_perspective %s path, flags %d" % (path, flags)
            assert_frames(out, ref, what, case)
            assert_singles(out, lambda i: homo.warp_perspective(t[i], Ms[frame_matrix(case, i)], DSIZE, flags=flags,
                                                                path=path), what, case)
    bv = (3, 50, 250)
    ref = oracle_bgr(name, 1, border=bv)
    for path in ("generic", "auto"):
        dst = poisoned((n,) + DSIZE[::-1] + (3,), torch.uint8)
        out = homo.warp_perspective(t, mats(name, 1), DSIZE, dst=dst, flags=1, borderValue=bv,
                                    mat_index=case["idx"], path=path)
        assert_frames(out, ref, "warp_perspective %s path, border %s" % (path, bv), case)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["u8c1", "u8c4", "f16c3", "f32c3"])
@pytest.mark.parametrize("name", ["i%24", "i%16_then_4_singles"])
def test_staged_pixel_formats(name, fmt):
    """The other pixel formats of the staged kernel: float16 against float16(oracle(float32))."""
    case = BY_NAME[name]
    f = frames(name, fmt)
    t = cu(f)
    for flags in FLAGS:
        Ms = mats(name, flags)
        src = f.astype(np.float32) if fmt == "f16c3" else f
        ref = np.stack([wo.warp_perspective(src[i], Ms[frame_matrix(case, i)], DSIZE, flags=flags)
                        for i in range(case["n"])]).astype(f.dtype)
        for path in PATHS:
            dst = poisoned((case["n"],) + DSIZE[::-1] + (f.shape[3],), t.dtype)
            out = homo.warp_perspective(t, Ms, DSIZE, dst=dst, flags=flags, mat_index=case["idx"], path=path)
            assert_frames(out, ref, "%s warp_perspective %s path, flags %d" % (fmt, path, flags), case)


# ---- NV12 frames --------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=ids(CASES))
def test_warp_perspective_nv12_batches(case):
    """Contiguous frames and a pitched, gapped decoder surface."""
    name, n = case["name"], case["n"]
    f = nv12_frames(name)
    for layout, v in (("contiguous", cu(f)), ("pitch 512, gap 3", laid_out(f, 512, 3))):
        for flags in FLAGS:
            Ms = mats(name, flags)
            dst = poisoned((n,) + DSIZE[::-1] + (3,), torch.uint8)
            out = homo.warp_perspective_nv12(v, Ms, DSIZE, dst=dst, flags=flags, mat_index=case["idx"])
            what = "warp_perspective_nv12, %s, flags %d" % (layout, flags)
            assert_frames(out, oracle_bgr(name, flags, nv12=True), what, case)
            assert_singles(out, lambda i: homo.warp_perspective_nv12(v[i], Ms[frame_matrix(case, i)], DSIZE,
                                                                     flags=flags), what, case)


# ---- YUV 4:2:0 BEVs -----------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=ids(CASES))
def test_warp_to_yuv420_batches(case):
    """BGR and NV12 sources, I420 and NV12 output, and once into pitched surfaces whose padding must
    stay as it was."""
    name, n = case["name"], case["n"]
    t, v = cu(frames(name)), cu(nv12_frames(name))
    shape = (n, DSIZE[1] * 3 // 2, DSIZE[0])
    routes = (("warp_perspective_yuv420", t, homo.warp_perspective_yuv420, False),
              ("warp_perspective_nv12_yuv420", v, homo.warp_perspective_nv12_yuv420, True))
    for what, src, fn, nv12 in routes:
        for layout in LAYOUTS:
            for flags in FLAGS:
                Ms = mats(name, flags)
                out = fn(src, Ms, DSIZE, layout, dst=poisoned(shape, torch.uint8), flags=flags,
                         mat_index=case["idx"])
                w = "%s, %s, flags %d" % (what, layout, flags)
                assert_frames(out, oracle_yuv(name, flags, layout, nv12), w, case)
                assert_singles(out, lambda i: fn(src[i], Ms[frame_matrix(case, i)], DSIZE, layout, flags=flags), w,
                               case)
        buf, view, pad = surface(n, DSIZE[1], DSIZE[0], 288, 2)
        assert fn(src, mats(name, 1), DSIZE, "nv12", dst=view, flags=1, mat_index=case["idx"]) is view
        assert_frames(view, oracle_yuv(name, 1, "nv12", nv12), what + " into a pitched surface", case)
        assert bool((buf[pad] == POISON).all()), "%s wrote padding bytes; %s" % (what, describe(case))


# ---- the torch operators ------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", WITH_INDEX, ids=ids(WITH_INDEX))
def test_torch_operators_match_ctypes_route(case):
    from bev_b200 import torch_ops
    torch_ops.load()
    name, n = case["name"], case["n"]
    t, v = cu(frames(name)), cu(nv12_frames(name))
    idx = torch.from_numpy(case["idx"])
    w, h = DSIZE
    for flags in (0, 1, 17):
        Ms = mats(name, flags)
        Mt = torch.from_numpy(Ms)
        poison_allocator(n * h * w * 3)
        out = torch.ops.bev_cuda.warp_perspective(t, Mt, w, h, flags, 0, 0.0, idx)
        assert torch.equal(out, homo.warp_perspective(t, Ms, DSIZE, flags=flags, mat_index=case["idx"])), \
            "warp_perspective operator, flags %d; %s" % (flags, describe(case))
        poison_allocator(n * h * w * 3)
        out = torch.ops.bev_cuda.warp_perspective_nv12(v, Mt, w, h, flags, 0, 0.0, idx)
        assert torch.equal(out, homo.warp_perspective_nv12(v, Ms, DSIZE, flags=flags, mat_index=case["idx"])), \
            "warp_perspective_nv12 operator, flags %d; %s" % (flags, describe(case))
        for code, layout in enumerate(LAYOUTS):
            poison_allocator(n * h * w * 3 // 2)
            out = torch.ops.bev_cuda.warp_perspective_yuv420(t, Mt, w, h, code, flags, 0, 0.0, idx)
            ref = homo.warp_perspective_yuv420(t, Ms, DSIZE, layout, flags=flags, mat_index=case["idx"])
            assert torch.equal(out, ref), "warp_perspective_yuv420 operator, %s, flags %d; %s" % (
                layout, flags, describe(case))
    torch.cuda.synchronize()


# ---- permuting the frames permutes the output ---------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", UNPERMUTED, ids=ids(UNPERMUTED))
def test_permuting_frames_and_index_permutes_the_output(case):
    """Whatever runs, launches and kernels each order goes through, frame i of a permuted batch is
    frame perm[i] of the batch."""
    name, n = case["name"], case["n"]
    perm = np.random.default_rng(case["seed"] + [4]).permutation(n)
    pt = torch.from_numpy(perm).to(DEV)
    t, v = cu(frames(name)), cu(nv12_frames(name))
    for flags in (1, 16):
        Ms = mats(name, flags)
        if case["idx"] is None:  # one matrix per frame: the table moves with the frames
            kw, kw_p = {}, {}
            Ms_p = Ms[perm]
        else:
            kw, kw_p = {"mat_index": case["idx"]}, {"mat_index": case["idx"][perm]}
            Ms_p = Ms
        for path in PATHS:
            out = homo.warp_perspective(t, Ms, DSIZE, flags=flags, path=path, **kw)
            out_p = homo.warp_perspective(t[pt], Ms_p, DSIZE, flags=flags, path=path, **kw_p)
            assert torch.equal(out_p, out[pt]), "warp_perspective %s path, flags %d; %s" % (path, flags,
                                                                                           describe(case))
        out = homo.warp_perspective_nv12_yuv420(v, Ms, DSIZE, "nv12", flags=flags, **kw)
        out_p = homo.warp_perspective_nv12_yuv420(v[pt], Ms_p, DSIZE, "nv12", flags=flags, **kw_p)
        assert torch.equal(out_p, out[pt]), "warp_perspective_nv12_yuv420, flags %d; %s" % (flags, describe(case))


# ---- 1080p frames of the eight cfg-4 cameras ----------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, 1])
def test_cfg4_cameras_in_arrival_order(flags):
    """40 1080p frames of the eight cfg-4 cameras, all stretched to one 1024^2 BEV, in an irregular
    camera order: two launches, both staged in "auto", where most cameras' tiles split between the
    staged and the direct-gather kernel.  Every frame equals a single-frame call; one frame per
    camera equals the oracle."""
    case = CAMS_1080P
    Hs, idx = table(case["name"]), case["idx"]
    f = np.random.default_rng([SEED, 5]).integers(0, 256, (case["n"], 1080, 1920, 3), dtype=np.uint8)
    t = cu(f)
    firsts = [int(np.flatnonzero(idx == k)[0]) for k in range(case["mats"])]
    refs = {i: wo.warp_perspective(f[i], Hs[idx[i]], (1024, 1024), flags=flags) for i in firsts}
    for path in PATHS:
        out = homo.warp_perspective(t, Hs, (1024, 1024), dst=poisoned((case["n"], 1024, 1024, 3), torch.uint8),
                                    flags=flags, mat_index=idx, path=path)
        what = "%s path, flags %d" % (path, flags)
        assert_singles(out, lambda i: homo.warp_perspective(t[i], Hs[idx[i]], (1024, 1024), flags=flags,
                                                            path=path), what, case)
        for i, ref in refs.items():
            assert util.bits_equal(out[i].cpu().numpy(), ref), "%s, frame %d (camera %d) != oracle; %s" % (
                what, i, idx[i], describe(case))


# ---- the host-buffer entry point ----------------------------------------------------------------

def _poison_host_workspace(n):
    """Fill the host entry point's device buffers with frames of one value: a horizon-crossing map
    uploads whole frames.  A later call that reads a row it did not upload then reads that value."""
    M = np.array([[1.0, 0.2, -3.0], [0.1, 1.1, -2.0], [0.0, 0.03, -0.5]])  # w changes sign inside the BEV
    assert _native.warp_host_rows((SRC_W, SRC_H), DSIZE, M, 16) == (0, SRC_H - 1)
    const = np.full((n, SRC_H, SRC_W, 3), 0x5A, np.uint8)
    _native.warp_perspective_host(const, M, DSIZE, flags=16)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [41, 64])
def test_host_entry_point_chunks(n):
    """Upload chunks (11 frames of 41, 16 of 64) that cut through the runs of mat_index and through a
    table of per-frame matrices.  The matrices look at two row bands, the top and the bottom of the
    source: only the union of the bands is uploaded, and it must hold every row each matrix reads."""
    rng = np.random.default_rng([SEED, 6, n])
    f = rng.integers(0, 256, (n, SRC_H, SRC_W, 3), dtype=np.uint8)
    top, bottom = quad_maps(rng, 3, (20, 100)), quad_maps(rng, 3, (160, 230))
    band = np.stack([top[0], bottom[0], top[1], bottom[1], top[2], bottom[2]])  # matrix 0 sees the top band only
    per_frame = np.stack([(top if i % 2 else bottom)[i % 3] for i in range(n)])
    case = {"name": "host_%d" % n, "n": n, "seed": [SEED, 6, n]}
    for flags in (1, 16):
        tables = (("mat_index i %% 3 over top/bottom bands", band, (np.arange(n) % 3) * 2 + (np.arange(n) // 7) % 2),
                  ("per-frame matrices", per_frame, None))
        for what, Hs, idx in tables:
            Ms = np.linalg.inv(Hs) if flags & 16 else Hs
            r0, r1 = _native.warp_host_rows((SRC_W, SRC_H), DSIZE, Ms, flags)
            assert 0 < r0 and r1 < SRC_H - 1, (what, r0, r1)  # a partial upload
            _poison_host_workspace(64)
            dst = np.full((n,) + DSIZE[::-1] + (3,), POISON, np.uint8)
            kw = {} if idx is None else {"mat_index": idx.astype(np.int32)}
            out = _native.warp_perspective_host(f, Ms, DSIZE, dst=dst, flags=flags, **kw)
            ref = np.stack([wo.warp_perspective(f[i], Ms[i if idx is None else idx[i]], DSIZE, flags=flags)
                            for i in range(n)])
            case["idx"] = idx
            assert_frames(out, ref, "warp_perspective_host, %s, flags %d" % (what, flags), case)
