#!/usr/bin/env python
"""tools/kbench.py -- kernel-only timing of the warp workloads (development aid, not the bench).

    python tools/kbench.py [--steps K] [--path auto|generic|fast] [workload ...]

Prints: workload, ms per launch (CUDA events), Mpix/s, fraction of the measured HBM peak
(algorithmic bytes of SURVEY.md 8d)."""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from bev_b200 import _native, homo  # noqa: E402
from oracle import yuv420_oracle  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--path", default="auto")
    ap.add_argument("--check", action="store_true", help="compare frame 0 and the last frame with the oracle")
    ap.add_argument("--lib", default=None, help="a variant library built by tools/ab_build.sh (A/B runs)")
    ap.add_argument("workloads", nargs="*")
    args = ap.parse_args()
    wls = args.workloads or ["cfg2_1080p_to_bev1024_u8c3_bilinear_x256", "cfg2_nearest",
                             "cfg5_4k_to_bev2048_u8c3_x64", "cfg5_inv_bev2048_to_4k_u8c3_x64"]
    if args.lib:
        _native.LIB_PATH = os.path.abspath(args.lib)
    _native.set_warp_path(args.path)
    peak, _ = bench.measured_peak()
    dev = torch.device("cuda", 0)
    for wl in wls:
        n, ssize, dsize, ch, dtype, flags, hscale, inverse = bench.WORKLOADS[wl]
        H = bench.h_canon(hscale)
        if inverse:
            H = np.linalg.inv(H)
        tdtype = {"uint8": torch.uint8, "float16": torch.float16, "float32": torch.float32}[dtype]
        es = {"uint8": 1, "float16": 2, "float32": 4}[dtype]
        g = torch.Generator(device=dev).manual_seed(1234)
        frames = torch.randint(0, 256, (n, ssize[1], ssize[0], ch), dtype=torch.uint8, device=dev, generator=g)
        if tdtype != torch.uint8:
            frames = (frames.to(torch.float32) / 255.0).to(tdtype)
        out = torch.empty((n, dsize[1], dsize[0], ch), dtype=tdtype, device=dev)
        T, _, _ = _native.warp_touched_pixels(ssize, dsize, H, flags)
        algo = (T + dsize[0] * dsize[1]) * ch * es * n
        for _ in range(3):
            homo.warp_perspective(frames, H, dsize, dst=out, flags=flags)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            homo.warp_perspective(frames, H, dsize, dst=out, flags=flags)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        msg = "%s %.4f ms %.0f Mpix/s frac %.4f" % (wl, ms, n * dsize[0] * dsize[1] / ms / 1e3,
                                                   algo / (ms * 1e-3) / 1e9 / peak)
        if args.check:
            from oracle import warp_oracle as wo
            bad = 0
            for i in (0, n - 1):
                src = frames[i].cpu().numpy()
                if tdtype == torch.float16:
                    ref = wo.warp_perspective(src, H, dsize, flags=flags)
                else:
                    ref = wo.warp_perspective(src, H, dsize, flags=flags)
                bad += int(np.count_nonzero(out[i].cpu().numpy() != ref))
            msg += " mismatches %d" % bad
        print(msg, flush=True)
        del frames, out
        torch.cuda.empty_cache()




def cfg4(n_frames=1000, steps=3):
    """BASELINE configs[3] on one GPU: 8 BrnoCompSpeed-shaped cameras x n_frames 1080p frames, one
    homography and one BEV size per camera (tests/golden/cfg4_cams.json)."""
    import json
    cams = json.load(open(os.path.join(ROOT, "tests", "golden", "cfg4_cams.json")))
    peak, _ = bench.measured_peak()
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1234)
    frames = torch.randint(0, 256, (n_frames, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    tot_ms, tot_px, tot_bytes = 0.0, 0, 0
    for c in cams:
        H = np.array(c["H_bev_img"])
        dsize = (int(c["bspec"]["u_size"]), int(c["bspec"]["v_size"]))
        out = torch.empty((n_frames, dsize[1], dsize[0], 3), dtype=torch.uint8, device=dev)
        T, _, _ = _native.warp_touched_pixels((1920, 1080), dsize, H, 1)
        algo = (T + dsize[0] * dsize[1]) * 3 * n_frames
        homo.warp_perspective(frames, H, dsize, dst=out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            homo.warp_perspective(frames, H, dsize, dst=out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        print("cfg4 cam %s bev %dx%d: %.3f ms %.0f Mpix/s frac %.3f" % (
            c.get("id", "?"), dsize[0], dsize[1], ms, n_frames * dsize[0] * dsize[1] / ms / 1e3,
            algo / (ms * 1e-3) / 1e9 / peak), flush=True)
        tot_ms += ms
        tot_px += n_frames * dsize[0] * dsize[1]
        tot_bytes += algo
        del out
    print("cfg4 total: %.3f ms %.0f Mpix/s frac %.3f" % (tot_ms, tot_px / tot_ms / 1e3,
                                                         tot_bytes / (tot_ms * 1e-3) / 1e9 / peak))


def compo_bench(n=64, steps=10):
    """BEV compositing (SURVEY 8f rank 1): n 1080p renders + masks over ONE 1080p background into
    1024^2 BEVs, fused kernel against three warps + blend.  Algorithmic bytes: touched pixels of
    the background once, of render and mask per frame, plus the composite written once."""
    from bev_b200 import compo
    dev = torch.device("cuda", 0)
    peak, _ = bench.measured_peak()
    g = torch.Generator(device=dev).manual_seed(1234)
    ssize, dsize = (1920, 1080), (1024, 1024)
    B = torch.randint(0, 256, (1, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    F = torch.randint(0, 256, (n, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    M = torch.randint(0, 256, (n, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    H = bench.h_canon(1)
    T, _, _ = _native.warp_touched_pixels(ssize, dsize, H, 1)
    D = dsize[0] * dsize[1]
    algo = 3 * (T + n * (2 * T + D))
    for per_frame in (False, True):
        Hb = np.repeat(H[None], n, 0) if per_frame else H
        for fused in (True, False):
            for _ in range(2):
                out = compo.composite_bev_batch(B, F, M, Hb, Hb, dsize, fused=fused)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                out = compo.composite_bev_batch(B, F, M, Hb, Hb, dsize, fused=fused)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            print("compo x%d %s %s: %.3f ms %.0f Mpix/s frac %.3f" % (
                n, "camera per frame" if per_frame else "shared cameras", "fused" if fused else "3 warps + blend",
                ms, n * D / ms / 1e3, algo / (ms * 1e-3) / 1e9 / peak))
            del out


def resize_bench(n=256, steps=10):
    """cv2.resize of the reference's small-frame path (vis_homo.py:90): n 1080p BGR frames ->
    852x480.  Algorithmic bytes: source pixels with a non-zero tap weight + the small frames."""
    from oracle import resize_oracle
    dev = torch.device("cuda", 0)
    peak, _ = bench.measured_peak()
    g = torch.Generator(device=dev).manual_seed(1234)
    frames = torch.randint(0, 256, (n, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    for dsize in ((852, 480), (960, 540), (1280, 720)):
        out = torch.empty((n, dsize[1], dsize[0], 3), dtype=torch.uint8, device=dev)
        T = resize_oracle.touched_pixels((1920, 1080), dsize)
        algo = 3 * n * (T + dsize[0] * dsize[1])
        for _ in range(3):
            homo.resize(frames, dsize, dst=out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            homo.resize(frames, dsize, dst=out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        print("resize x%d 1080p -> %dx%d: %.3f ms %.0f Mpix/s (output) frac %.3f" % (
            n, dsize[0], dsize[1], ms, n * dsize[0] * dsize[1] / ms / 1e3, algo / (ms * 1e-3) / 1e9 / peak))


def iou_bench(n=8192, steps=10):
    """Rotated-box IoU matrix (tracker association, rbox_tracker.py:87-92): n x n float32 boxes.
    Compute-bound (float64 registers); the HBM figure is the n^2 * 4 B matrix it writes."""
    from bev_b200 import rbox_torch
    dev = torch.device("cuda", 0)
    peak, _ = bench.measured_peak()
    g = torch.Generator(device=dev).manual_seed(3)
    u = torch.rand((2, n, 5), device=dev, generator=g)
    lo = torch.tensor([0.0, 0.0, 1.0, 1.0, -3.2], device=dev)
    hi = torch.tensor([300.0, 300.0, 30.0, 30.0, 3.2], device=dev)
    a, b = (lo + u[0] * (hi - lo)).contiguous(), (lo + u[1] * (hi - lo)).contiguous()
    for _ in range(3):
        out = rbox_torch.iou_batch_rbox(a, b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = rbox_torch.iou_batch_rbox(a, b)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    print("iou %d x %d: %.3f ms %.1f Gpairs/s, matrix written at %.0f GB/s (%.2f of the HBM peak), %.1f %% pairs overlap"
          % (n, n, ms, n * n / ms / 1e6, n * n * 4 / ms / 1e6, n * n * 4 / ms / 1e6 / peak,
             100.0 * float((out > 0).float().mean())))


def host_single(steps=200):
    """The reference's own loop shape (vis_homo.py:85-89): ONE host frame per call, result back in
    host memory -- bevk_warp_perspective_host on pinned numpy-backed buffers, against cv2 on the
    same frame with all host threads."""
    import time
    import cv2
    H = bench.h_canon(1)
    dsize = (1024, 1024)
    rng = np.random.default_rng(0)
    frame = rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    h_src = torch.from_numpy(frame).pin_memory()
    h_dst = torch.empty((1024, 1024, 3), dtype=torch.uint8).pin_memory()
    for _ in range(5):
        _native.warp_perspective_host(h_src[None], H, dsize, dst=h_dst[None])
    t0 = time.perf_counter()
    for _ in range(steps):
        _native.warp_perspective_host(h_src[None], H, dsize, dst=h_dst[None])
    ours = (time.perf_counter() - t0) / steps
    assert np.array_equal(h_dst.numpy(), cv2.warpPerspective(frame, H, dsize))
    for _ in range(3):
        cv2.warpPerspective(frame, H, dsize)
    t0 = time.perf_counter()
    for _ in range(50):
        cv2.warpPerspective(frame, H, dsize)
    ref = (time.perf_counter() - t0) / 50
    print("one host frame per call: ours %.1f us (H2D + kernel + D2H, synchronous), cv2 %.1f us on %d threads"
          % (ours * 1e6, ref * 1e6, cv2.getNumThreads()))


def cams_uniform(n_frames=256, steps=5):
    """SURVEY 8d secondary variant of cfg 4: the eight BrnoCompSpeed-shaped cameras warped to a
    uniform 1024^2 BEV (their own BEV rectangle stretched to it), n_frames 1080p frames each."""
    import json
    cams = json.load(open(os.path.join(ROOT, "tests", "golden", "cfg4_cams.json")))
    peak, _ = bench.measured_peak()
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1234)
    frames = torch.randint(0, 256, (n_frames, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    out = torch.empty((n_frames, 1024, 1024, 3), dtype=torch.uint8, device=dev)
    for c in cams:
        u, v = int(c["bspec"]["u_size"]), int(c["bspec"]["v_size"])
        H = np.diag([1024.0 / u, 1024.0 / v, 1.0]) @ np.array(c["H_bev_img"])
        T, _, _ = _native.warp_touched_pixels((1920, 1080), (1024, 1024), H, 1)
        algo = (T + 1024 * 1024) * 3 * n_frames
        for _ in range(2):
            homo.warp_perspective(frames, H, (1024, 1024), dst=out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            homo.warp_perspective(frames, H, (1024, 1024), dst=out)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        print("cam %s -> 1024^2 x%d: T %.0fk px, %.3f ms %.0f Mpix/s frac %.3f" % (
            c["id"], n_frames, T / 1e3, ms, n_frames * 1024 * 1024 / ms / 1e3, algo / (ms * 1e-3) / 1e9 / peak))


def cfg1_cold_warm(steps=50):
    """BASELINE configs[0]: one 1080p frame -> 1024^2, per-call device time with the frame warm in
    L2 (back-to-back calls) and cold (a 512 MB buffer is rewritten between calls; SURVEY 8d)."""
    dev = torch.device("cuda", 0)
    H = bench.h_canon(1)
    g = torch.Generator(device=dev).manual_seed(1234)
    frame = torch.randint(0, 256, (1, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    out = torch.empty((1, 1024, 1024, 3), dtype=torch.uint8, device=dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    for _ in range(5):
        homo.warp_perspective(frame, H, (1024, 1024), dst=out)
    torch.cuda.synchronize()
    res = {}
    for mode in ("warm", "cold"):
        ev = []
        for _ in range(steps):  # everything is queued; only the warp calls are bracketed by events
            if mode == "cold":
                flush.fill_(1)
            torch.cuda._sleep(200000)  # ~100 us of device idle spin: the host runs ahead of the queue
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            homo.warp_perspective(frame, H, (1024, 1024), dst=out)
            e1.record()
            ev.append((e0, e1))
        torch.cuda.synchronize()
        res[mode] = sum(a.elapsed_time(b) for a, b in ev) / steps * 1e3
    print("cfg1 one 1080p frame -> 1024^2: warm %.1f us, cold (L2 flushed) %.1f us per call" % (res["warm"], res["cold"]))


def card():
    """Name and power limit of GPU 0 (read-only nvidia-smi query): part of every number printed."""
    import subprocess
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip() or r.stderr.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        return "unknown (%s)" % e


def _alternate(routes, rounds, steps):
    """ms per call of each route, timed with CUDA events in rounds that alternate the routes."""
    times = {name: [] for name in routes}
    for name, fn in routes.items():  # warm-up: module loads, allocations, the staged kernel's set-up
        for _ in range(2):
            fn()
    torch.cuda.synchronize()
    for _ in range(rounds):
        for name, fn in routes.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    return times


def _report(label, times, algo_bytes, peak):
    for name, t in times.items():
        t = np.array(t)
        med = float(np.median(t))
        print("%s | %s: median %.4f ms (min %.4f, max %.4f, spread %.1f %%), %.0f GB/s algorithmic = %.3f of %.1f GB/s"
              % (label, name, med, t.min(), t.max(), 100.0 * (t.max() - t.min()) / med,
                 algo_bytes / (med * 1e-3) / 1e9, algo_bytes / (med * 1e-3) / 1e9 / peak, peak), flush=True)
    names = list(times)
    if len(names) == 2:
        a, b = np.array(times[names[0]]), np.array(times[names[1]])
        print("%s | %s / %s per round: %s" % (label, names[0], names[1],
                                             " ".join("%.3f" % v for v in a / b)), flush=True)


def nv12_bench(rounds=5):
    """NV12 frames (GPU decoder output) to BGR BEVs: the fused warp against converting to BGR and
    then warping, alternating the two routes in one process; the conversion alone.  Algorithmic
    bytes: touched luma + 2 x touched chroma samples (oracle coordinate map, host) + 3 x dst pixels.
    Every frame set is larger than the 126 MB L2."""
    import json
    from oracle import nv12_oracle
    print("card: %s" % card(), flush=True)
    peak, src = bench.measured_peak()
    print("peak: %.1f GB/s (%s)" % (peak, src), flush=True)
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1234)

    # cfg 2: 256 x 1080p -> 1024^2, the canonical map
    n, dsize, H = 256, (1024, 1024), bench.h_canon(1)
    frames = torch.randint(0, 256, (n, 1620, 1920), dtype=torch.uint8, device=dev, generator=g)
    bgr = torch.empty((n, 1080, 1920, 3), dtype=torch.uint8, device=dev)
    out_a = torch.empty((n, 1024, 1024, 3), dtype=torch.uint8, device=dev)
    out_b = torch.empty_like(out_a)
    for flags, fname in ((1, "bilinear"), (0, "nearest")):
        luma, chroma = nv12_oracle.touched_samples((1920, 1080), dsize, H, flags)
        algo = n * (luma + 2 * chroma + 3 * dsize[0] * dsize[1])

        def fused():
            homo.warp_perspective_nv12(frames, H, dsize, dst=out_a, flags=flags)

        def two_pass():
            homo.nv12_to_bgr(frames, dst=bgr)
            homo.warp_perspective(bgr, H, dsize, dst=out_b, flags=flags, path="fast")
        times = _alternate({"fused": fused, "nv12_to_bgr + staged warp": two_pass}, rounds, 10)
        assert torch.equal(out_a, out_b), "routes differ"
        print("cfg2 %s: touched luma %d, chroma %d per frame, %.2f MB algorithmic per frame"
              % (fname, luma, chroma, algo / n / 1e6))
        _report("cfg2 x%d 1080p NV12 -> 1024^2 %s" % (n, fname), times, algo, peak)

    # the conversion alone: reads 1.5 B and writes 3 B per pixel
    conv_bytes = n * 1080 * 1920 * 9 // 2
    times = _alternate({"nv12_to_bgr": lambda: homo.nv12_to_bgr(frames, dst=bgr)}, rounds, 10)
    _report("conversion x%d 1080p" % n, times, conv_bytes, peak)
    del frames, bgr, out_a, out_b
    torch.cuda.empty_cache()

    # cfg 4: 8 cameras x 1000 frames, one homography and BEV size per camera
    cams = json.load(open(os.path.join(ROOT, "tests", "golden", "cfg4_cams.json")))
    n = 1000
    frames = torch.randint(0, 256, (n, 1620, 1920), dtype=torch.uint8, device=dev, generator=g)
    bgr = torch.empty((n, 1080, 1920, 3), dtype=torch.uint8, device=dev)
    jobs, algo = [], 0
    for c in cams:
        Hc = np.array(c["H_bev_img"])
        ds = (int(c["bspec"]["u_size"]), int(c["bspec"]["v_size"]))
        luma, chroma = nv12_oracle.touched_samples((1920, 1080), ds, Hc, 1)
        algo += n * (luma + 2 * chroma + 3 * ds[0] * ds[1])
        jobs.append((Hc, ds, torch.empty((n, ds[1], ds[0], 3), dtype=torch.uint8, device=dev)))

    def fused4():
        for Hc, ds, o in jobs:
            homo.warp_perspective_nv12(frames, Hc, ds, dst=o)

    def two_pass4():
        for Hc, ds, o in jobs:
            homo.nv12_to_bgr(frames, dst=bgr)
            homo.warp_perspective(bgr, Hc, ds, dst=o)
    times = _alternate({"fused": fused4, "nv12_to_bgr + warp per camera": two_pass4}, rounds, 2)
    _report("cfg4 8 cameras x%d 1080p NV12" % n, times, algo, peak)


def yuv420_bench(rounds=5):
    """YUV 4:2:0 BEVs for a video encoder (vis_homo.py:110-111): the fused warps to I420 against the
    BGR warp followed by bgr_to_yuv420, for BGR and NV12 frames, alternating the routes in one
    process; and the conversion alone.  Algorithmic bytes of a warp: the touched source bytes (3 per
    touched BGR pixel; touched luma + 2 x touched chroma samples for NV12) + 1.5 per dst pixel; of
    the conversion: 3 + 1.5 bytes per pixel.  Every frame set is larger than the 126 MB L2."""
    import json
    from oracle import nv12_oracle
    print("card: %s" % card(), flush=True)
    peak, src = bench.measured_peak()
    print("peak: %.1f GB/s (%s)" % (peak, src), flush=True)
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1234)

    def src_bytes(ds, Hm, flags, nv12):
        if nv12:
            luma, chroma = nv12_oracle.touched_samples((1920, 1080), ds, Hm, flags)
            return luma + 2 * chroma
        return 3 * _native.warp_touched_pixels((1920, 1080), ds, Hm, flags)[0]

    # cfg 2: 256 x 1080p -> 1024^2, the canonical map
    n, dsize, H = 256, (1024, 1024), bench.h_canon(1)
    bgr = torch.randint(0, 256, (n, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    nv12 = torch.randint(0, 256, (n, 1620, 1920), dtype=torch.uint8, device=dev, generator=g)
    bev = torch.empty((n, 1024, 1024, 3), dtype=torch.uint8, device=dev)
    out_a = torch.empty((n, 1536, 1024), dtype=torch.uint8, device=dev)
    out_b = torch.empty_like(out_a)
    for flags, fname in ((1, "bilinear"), (0, "nearest")):
        for nv, frames in ((False, bgr), (True, nv12)):
            algo = n * (src_bytes(dsize, H, flags, nv) + 3 * dsize[0] * dsize[1] // 2)
            if nv:
                routes = {"fused": lambda: homo.warp_perspective_nv12_yuv420(frames, H, dsize, dst=out_a, flags=flags),
                          "warp_perspective_nv12 + bgr_to_yuv420": lambda: (
                              homo.warp_perspective_nv12(frames, H, dsize, dst=bev, flags=flags),
                              homo.bgr_to_yuv420(bev, dst=out_b))}
            else:
                routes = {"fused": lambda: homo.warp_perspective_yuv420(frames, H, dsize, dst=out_a, flags=flags),
                          "staged warp + bgr_to_yuv420": lambda: (
                              homo.warp_perspective(frames, H, dsize, dst=bev, flags=flags, path="fast"),
                              homo.bgr_to_yuv420(bev, dst=out_b))}
            times = _alternate(routes, rounds, 10)
            assert torch.equal(out_a, out_b), "routes differ"
            _report("cfg2 x%d 1080p %s -> 1024^2 I420 %s" % (n, "NV12" if nv else "BGR", fname), times, algo, peak)
    del bgr, nv12, out_a, out_b
    torch.cuda.empty_cache()

    # the conversion alone, on 256 1024^2 BEVs
    yuv = torch.empty((n, 1536, 1024), dtype=torch.uint8, device=dev)
    bev.random_(0, 256, generator=g)
    for layout in ("i420", "nv12"):
        times = _alternate({"bgr_to_yuv420 " + layout: lambda: homo.bgr_to_yuv420(bev, layout, dst=yuv)}, rounds, 10)
        _report("conversion x%d 1024^2" % n, times, n * 1024 * 1024 * 9 // 2, peak)
    del bev, yuv
    torch.cuda.empty_cache()

    # cfg 4: 8 cameras x 1000 frames, one homography and BEV size per camera
    cams = json.load(open(os.path.join(ROOT, "tests", "golden", "cfg4_cams.json")))
    n = 1000
    for nv in (False, True):
        frames = torch.randint(0, 256, (n, 1620, 1920) if nv else (n, 1080, 1920, 3), dtype=torch.uint8, device=dev,
                               generator=g)
        jobs, algo = [], 0
        for c in cams:
            Hc = np.array(c["H_bev_img"])
            ds = (int(c["bspec"]["u_size"]), int(c["bspec"]["v_size"]))
            algo += n * (src_bytes(ds, Hc, 1, nv) + 3 * ds[0] * ds[1] // 2)
            jobs.append((Hc, ds, torch.empty((n, ds[1], ds[0], 3), dtype=torch.uint8, device=dev),
                         torch.empty((n, ds[1] * 3 // 2, ds[0]), dtype=torch.uint8, device=dev)))

        def fused4():
            for Hc, ds, _, o in jobs:
                (homo.warp_perspective_nv12_yuv420 if nv else homo.warp_perspective_yuv420)(frames, Hc, ds, dst=o)

        def two_pass4():
            for Hc, ds, b, o in jobs:
                (homo.warp_perspective_nv12 if nv else homo.warp_perspective)(frames, Hc, ds, dst=b)
                homo.bgr_to_yuv420(b, dst=o)
        times = _alternate({"fused": fused4, "warp + bgr_to_yuv420 per camera": two_pass4}, rounds, 2)
        _report("cfg4 8 cameras x%d 1080p %s -> I420" % (n, "NV12" if nv else "BGR"), times, algo, peak)
        del frames, jobs
        torch.cuda.empty_cache()


def resize_nv12_bench(rounds=5):
    """The small frame of the reference's frame loop (vis_homo.py:90) from NV12 frames: the fused
    resize against converting to BGR and then resizing, alternating the two routes in one process.
    Algorithmic bytes: touched luma + 2 x touched chroma samples (taps with a non-zero weight) +
    3 x dst pixels.  Every frame set is larger than the 126 MB L2."""
    from oracle import resize_nv12_oracle
    print("card: %s" % card(), flush=True)
    peak, src = bench.measured_peak()
    print("peak: %.1f GB/s (%s)" % (peak, src), flush=True)
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1234)
    for n, (h, w), dsize in ((256, (1080, 1920), (852, 480)), (256, (1080, 1920), (960, 540)),
                             (64, (2160, 3840), (1920, 1080))):
        frames = torch.randint(0, 256, (n, h * 3 // 2, w), dtype=torch.uint8, device=dev, generator=g)
        bgr = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
        out_a = torch.empty((n, dsize[1], dsize[0], 3), dtype=torch.uint8, device=dev)
        out_b = torch.empty_like(out_a)
        luma, chroma = resize_nv12_oracle.resize_touched_samples((w, h), dsize)
        algo = n * (luma + 2 * chroma + 3 * dsize[0] * dsize[1])

        def fused():
            homo.resize_nv12(frames, dsize, dst=out_a)

        def two_pass():
            homo.nv12_to_bgr(frames, dst=bgr)
            homo.resize(bgr, dsize, dst=out_b)
        times = _alternate({"fused": fused, "nv12_to_bgr + resize": two_pass}, rounds, 10)
        assert torch.equal(out_a, out_b), "routes differ"
        label = "x%d %dx%d NV12 -> %dx%d" % (n, w, h, dsize[0], dsize[1])
        print("%s: touched luma %d, chroma %d per frame, %.2f MB algorithmic per frame"
              % (label, luma, chroma, algo / n / 1e6))
        _report(label, times, algo, peak)
        del frames, bgr, out_a, out_b
        torch.cuda.empty_cache()


AREA_WORKLOADS = ((256, (1080, 1920), (852, 480)), (256, (1080, 1920), (960, 540)),
                  (64, (2160, 3840), (1920, 1080)), (256, (480, 852), (1920, 1080)))


def resize_area_bench(rounds=5):
    """INTER_AREA resize of BGR frames against the INTER_LINEAR kernel on the same shapes,
    alternating the two in one process; the last shape upscales.  Algorithmic bytes: 3 x (touched
    source pixels + dst pixels); a downscale touches the whole frame.  Every frame set is larger
    than the 126 MB L2.  Frame 0 of the area route is checked against the oracle."""
    from oracle import resize_area_oracle
    print("card: %s" % card(), flush=True)
    peak, src = bench.measured_peak()
    print("peak: %.1f GB/s (%s)" % (peak, src), flush=True)
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1234)
    for n, (h, w), dsize in AREA_WORKLOADS:
        frames = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device=dev, generator=g)
        out_a = torch.empty((n, dsize[1], dsize[0], 3), dtype=torch.uint8, device=dev)
        out_b = torch.empty_like(out_a)
        algo = n * 3 * (resize_area_oracle.touched_pixels((w, h), dsize) + dsize[0] * dsize[1])

        def area():
            homo.resize(frames, dsize, dst=out_a, interpolation=homo.INTER_AREA)

        def linear():
            homo.resize(frames, dsize, dst=out_b)
        times = _alternate({"area": area, "linear": linear}, rounds, 10)
        ref = resize_area_oracle.resize(frames[0].cpu().numpy(), dsize)
        assert np.array_equal(out_a[0].cpu().numpy(), ref), "area route differs from the oracle"
        label = "x%d %dx%d BGR -> %dx%d (%s)" % (n, w, h, dsize[0], dsize[1], resize_area_oracle.branch((w, h), dsize))
        print("%s: %.2f MB algorithmic per frame" % (label, algo / n / 1e6))
        _report(label, times, algo, peak)
        del frames, out_a, out_b
        torch.cuda.empty_cache()


def resize_nv12_area_bench(rounds=5):
    """INTER_AREA resize of NV12 frames: the fused kernel against the fused INTER_LINEAR kernel
    and against nv12_to_bgr + INTER_AREA resize, alternating the three in one process.
    Algorithmic bytes: touched luma + 2 x touched chroma samples + 3 x dst pixels.  Every frame set
    is larger than the 126 MB L2."""
    from oracle import resize_area_oracle
    print("card: %s" % card(), flush=True)
    peak, src = bench.measured_peak()
    print("peak: %.1f GB/s (%s)" % (peak, src), flush=True)
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1234)
    for n, (h, w), dsize in AREA_WORKLOADS:
        frames = torch.randint(0, 256, (n, h * 3 // 2, w), dtype=torch.uint8, device=dev, generator=g)
        bgr = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
        out_a = torch.empty((n, dsize[1], dsize[0], 3), dtype=torch.uint8, device=dev)
        out_b, out_c = torch.empty_like(out_a), torch.empty_like(out_a)
        luma, chroma = resize_area_oracle.touched_samples_nv12((w, h), dsize)
        algo = n * (luma + 2 * chroma + 3 * dsize[0] * dsize[1])

        def fused_area():
            homo.resize_nv12(frames, dsize, dst=out_a, interpolation=homo.INTER_AREA)

        def fused_linear():
            homo.resize_nv12(frames, dsize, dst=out_b)

        def two_pass_area():
            homo.nv12_to_bgr(frames, dst=bgr)
            homo.resize(bgr, dsize, dst=out_c, interpolation=homo.INTER_AREA)
        times = _alternate({"fused area": fused_area, "fused linear": fused_linear,
                            "nv12_to_bgr + area resize": two_pass_area}, rounds, 10)
        assert torch.equal(out_a, out_c), "area routes differ"
        label = "x%d %dx%d NV12 -> %dx%d (%s)" % (n, w, h, dsize[0], dsize[1], resize_area_oracle.branch((w, h), dsize))
        print("%s: touched luma %d, chroma %d per frame, %.2f MB algorithmic per frame"
              % (label, luma, chroma, algo / n / 1e6))
        _report(label, times, algo, peak)
        del frames, bgr, out_a, out_b, out_c
        torch.cuda.empty_cache()


def _duplex_ceiling(h_up, h_dn, dev):
    """ms(nu, nd): the best of three plain pinned copies of nu bytes up from h_up and nd bytes down
    to h_dn at the same time, on two streams -- the host link's ceiling for a route's bytes."""
    import time
    d_up = torch.empty(h_up.numel(), dtype=torch.uint8, device=dev)
    d_dn = torch.empty(h_dn.numel(), dtype=torch.uint8, device=dev)
    s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def ceiling(nu, nd):
        best = None
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            with torch.cuda.stream(s_up):
                d_up[:nu].copy_(h_up[:nu], non_blocking=True)
            with torch.cuda.stream(s_dn):
                h_dn[:nd].copy_(d_dn[:nd], non_blocking=True)
            s_up.synchronize()
            s_dn.synchronize()
            dt = (time.perf_counter() - t0) * 1e3
            best = dt if best is None else min(best, dt)
        return best
    return ceiling


def _kernel_ms(fn, names):
    """Sum of the device durations of the kernels one fn() runs whose names contain one of names
    (torch.profiler, in a run of its own)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    us = 0.0
    for e in prof.key_averages():
        if any(k in e.key for k in names):
            us += getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0.0)
    return us / 1e3


def video_host_bench(rounds=5, n=256):
    """Host video frames to host BEVs through bevk_warp_perspective_video_host (vis_homo.py:85-111
    with a CPU codec): cfg 2, n pinned 1080p frames -> 1024^2 bilinear with the canonical map, for
    every pair of frame formats that a CPU decoder / encoder / cv2 user takes.  Per route: the host
    clock around the synchronous call (warm-up first, routes alternated in rounds), the bytes the
    call moves up (the referenced row band, and the chroma rows under it) and down, the link ceiling
    for those bytes (plain pinned copies up and down at the same time, as bench.py does for e2e),
    and the route's share of it.  The kernel time per route is the sum of the device durations of
    the kernels one call runs (torch.profiler: the I420-source kernels have no device entry point
    to bracket with events).  Every route's output equals the device route on the same frames."""
    import time
    print("card: %s" % card(), flush=True)
    dev = torch.device("cuda", 0)
    H, ssize, dsize = bench.h_canon(1), (1920, 1080), (1024, 1024)
    w, h, dw, dh = ssize[0], ssize[1], dsize[0], dsize[1]
    r0, r1 = _native.warp_host_rows(ssize, dsize, H, 1)
    rows, crows = r1 - r0 + 1, r1 // 2 - r0 // 2 + 1
    up = {"bgr": 3 * w * rows, "i420": w * rows + w * crows, "nv12": w * rows + w * crows}
    down = {"bgr": 3 * dw * dh, "i420": dw * dh * 3 // 2, "nv12": dw * dh * 3 // 2}
    routes = [("bgr", "bgr"), ("bgr", "i420"), ("i420", "bgr"), ("i420", "i420"), ("nv12", "nv12")]
    print("cfg2 x%d 1080p -> 1024^2 bilinear, uploaded rows [%d, %d]" % (n, r0, r1), flush=True)

    g = torch.Generator().manual_seed(1234)
    bgr = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=g).pin_memory()
    i420 = torch.randint(0, 256, (n, h * 3 // 2, w), dtype=torch.uint8, generator=g).pin_memory()
    nv12 = torch.from_numpy(np.stack([yuv420_oracle.i420_to_nv12(f) for f in i420.numpy()])).pin_memory()
    src = {"bgr": bgr, "i420": i420, "nv12": nv12}
    out = {r: torch.empty((n, dh, dw, 3) if r[1] == "bgr" else (n, dh * 3 // 2, dw), dtype=torch.uint8).pin_memory()
           for r in routes}

    def call(r):
        homo.warp_perspective_video_host(src[r[0]], H, dsize, r[0], r[1], dst=out[r])

    for r in routes:  # warm-up: workspace allocations, module loads
        call(r)
    times = {r: [] for r in routes}
    for _ in range(rounds):
        for r in routes:
            t0 = time.perf_counter()
            call(r)
            times[r].append((time.perf_counter() - t0) * 1e3)

    # the device route on the same frames (I420 frames as their NV12 relayout)
    for r in routes:
        s = src["nv12" if r[0] == "i420" else r[0]].to(dev)
        if r[0] == "bgr":
            ref = (homo.warp_perspective(s, H, dsize) if r[1] == "bgr"
                   else homo.warp_perspective_yuv420(s, H, dsize, r[1]))
        else:
            ref = (homo.warp_perspective_nv12(s, H, dsize) if r[1] == "bgr"
                   else homo.warp_perspective_nv12_yuv420(s, H, dsize, r[1]))
        assert torch.equal(ref.cpu(), out[r]), "%s -> %s differs from the device route" % r
        del s, ref
    torch.cuda.empty_cache()

    # the link ceiling for each route's byte counts: plain pinned copies, both directions at once
    ceiling = _duplex_ceiling(bgr.view(-1), out[("bgr", "bgr")].view(-1), dev)

    def kernel_ms(r):
        return _kernel_ms(lambda: call(r), ("warp",))

    for r in routes:
        nu, nd = up[r[0]] * n, down[r[1]] * n
        ceil = ceiling(nu, nd)
        t = np.array(times[r])
        med = float(np.median(t))
        print("%s -> %s: median %.2f ms (min %.2f, max %.2f, spread %.1f %%), %.2f Gpix/s | H2D %.1f MB, D2H %.1f MB "
              "per step, ceiling %.2f ms (%.1f GB/s both ways) -> %.1f %% of it | kernels %.2f ms"
              % (r[0], r[1], med, t.min(), t.max(), 100.0 * (t.max() - t.min()) / med, n * dw * dh / med / 1e6,
                 nu / 1e6, nd / 1e6, ceil, (nu + nd) / ceil / 1e6, 100.0 * ceil / med, kernel_ms(r)), flush=True)


def frame_loop_bench(rounds=5, n=200):
    """The live-camera loop of vis_homo.py:85-111 for one frame at a time (cfg 1: launch-bound): the
    1024^2 BEV, the 852x480 small frame, its 1024^2 BEV and the YUV 4:2:0 (I420) frames of both BEVs
    for an encoder, from one 1080p BGR frame and from one NV12 frame of a GPU decoder.  Four routes
    per chain, alternated in rounds:
      ctypes    the bev_b200.homo functions (ctypes, one Python call per entry point)
      ops       the torch.ops.bev_cuda operators, eager
      compile   the operator chain under torch.compile(fullgraph=True)
      graph     one torch.cuda.graph replay of the operator chain
    Per route: the host time per frame (host clock around n frames that ends in a synchronise, median
    over the rounds) and the device time of the same work (the kernels' durations per frame,
    torch.profiler over n frames in a run of its own).  All routes must give the same bytes."""
    import time
    from torch.profiler import ProfilerActivity, profile
    from bev_b200 import torch_ops
    torch_ops.load()
    ops = torch.ops.bev_cuda
    print("card: %s" % card(), flush=True)
    dev = torch.device("cuda", 0)
    H, (w, h), (dw, dh), (sw, sh) = bench.h_canon(1), (1920, 1080), (1024, 1024), (852, 480)
    fx, fy = w / sw, h / sh  # Calib.scale(align_corners=False) of the calibration
    Hs = H @ np.array([[fx, 0.0, 0.5 * fx - 0.5], [0.0, fy, 0.5 * fy - 0.5], [0.0, 0.0, 1.0]])
    Ht, Hst = torch.from_numpy(H), torch.from_numpy(Hs)
    g = torch.Generator(device=dev).manual_seed(1234)
    bgr = torch.randint(0, 256, (h, w, 3), dtype=torch.uint8, device=dev, generator=g)
    nv12 = torch.randint(0, 256, (h * 3 // 2, w), dtype=torch.uint8, device=dev, generator=g)

    def bgr_ops(f):
        bev = ops.warp_perspective(f, Ht, dw, dh)
        small = ops.resize(f, sw, sh)
        bev_small = ops.warp_perspective(small, Hst, dw, dh)
        return bev, small, bev_small, ops.bgr_to_yuv420(bev), ops.bgr_to_yuv420(bev_small)

    def bgr_ctypes(f):
        bev = homo.warp_perspective(f, H, (dw, dh))
        small = homo.resize(f, (sw, sh))
        bev_small = homo.warp_perspective(small, Hs, (dw, dh))
        return bev, small, bev_small, homo.bgr_to_yuv420(bev), homo.bgr_to_yuv420(bev_small)

    def nv12_ops(f):
        bev = ops.warp_perspective_nv12(f, Ht, dw, dh)
        small = ops.resize_nv12(f, sw, sh)
        bev_small = ops.warp_perspective(small, Hst, dw, dh)
        return bev, small, bev_small, ops.warp_perspective_nv12_yuv420(f, Ht, dw, dh), ops.bgr_to_yuv420(bev_small)

    def nv12_ctypes(f):
        bev = homo.warp_perspective_nv12(f, H, (dw, dh))
        small = homo.resize_nv12(f, (sw, sh))
        bev_small = homo.warp_perspective(small, Hs, (dw, dh))
        return (bev, small, bev_small, homo.warp_perspective_nv12_yuv420(f, H, (dw, dh)),
                homo.bgr_to_yuv420(bev_small))

    for label, frame, eager, ctypes_chain in (("bgr 1080p", bgr, bgr_ops, bgr_ctypes),
                                              ("nv12 1080p", nv12, nv12_ops, nv12_ctypes)):
        compiled = torch.compile(eager, fullgraph=True)
        ref = eager(frame)
        for _ in range(3):  # warm-up on a side stream before capture, as torch.cuda.graph asks
            compiled(frame)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                eager(frame)
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            graph_out = eager(frame)
        routes = {"ctypes": lambda: ctypes_chain(frame), "ops": lambda: eager(frame),
                  "compile": lambda: compiled(frame), "graph": graph.replay}
        graph.replay()
        torch.cuda.synchronize()
        for name, out in (("ctypes", ctypes_chain(frame)), ("compile", compiled(frame)), ("graph", graph_out)):
            assert all(torch.equal(a, b) for a, b in zip(out, ref)), "%s route differs from the eager operators" % name
        host = {r: [] for r in routes}
        for _ in range(rounds):
            for r, fn in routes.items():
                fn()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(n):
                    fn()
                torch.cuda.synchronize()
                host[r].append((time.perf_counter() - t0) * 1e6 / n)
        for r, fn in routes.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(n):
                    fn()
                torch.cuda.synchronize()
            kern = sum(e.self_device_time_total for e in prof.key_averages()
                       if e.device_type == torch.autograd.DeviceType.CUDA) / n
            t = np.array(host[r])
            print("frame_loop %s -> 1024^2 + 852x480 + YUV | %-7s: host %.1f us/frame (min %.1f, max %.1f), "
                  "device %.1f us/frame" % (label, r, float(np.median(t)), t.min(), t.max(), kern), flush=True)
        del graph, graph_out, compiled


def video_host_small_bench(rounds=5, n=256):
    """The three images of vis_homo.py:85-111 -- the BEV, the 852x480 small frame and its BEV -- from
    n pinned host 1080p frames of a CPU codec, cfg 2 (1024^2 BEVs through the canonical map, the small
    frames' map scaled from it as Calib.scale(align_corners=False) scales a calibration), INTER_LINEAR
    resize, bilinear warps.  Routes, alternated in rounds (host clock around each synchronous call):
      bgr one pass    warp_perspective_video_host_small, BGR -> BGR
      bgr today       warp_perspective_host for the BEV, then the whole frames uploaded (pinned), resize,
                      warp_perspective of the small frames and the two downloads
      i420 one pass   warp_perspective_video_host_small, I420 -> I420
    Per route: the bytes it moves up and down, the link ceiling for them (plain pinned copies both
    ways at once, measured in the same run), its share of that ceiling, and its kernel time
    (torch.profiler).  The two BGR routes must give the same bytes."""
    import time
    print("card: %s" % card(), flush=True)
    dev = torch.device("cuda", 0)
    H, ssize, dsize, small_size = bench.h_canon(1), (1920, 1080), (1024, 1024), (852, 480)
    w, h, dw, dh, sw, sh = ssize[0], ssize[1], dsize[0], dsize[1], small_size[0], small_size[1]
    fx, fy = w / sw, h / sh  # small pixel centre x -> (x + 0.5) * fx - 0.5 in the frame
    Hs = H @ np.array([[fx, 0.0, 0.5 * fx - 0.5], [0.0, fy, 0.5 * fy - 0.5], [0.0, 0.0, 1.0]])
    r0, r1 = _native.warp_host_rows(ssize, dsize, H, 1)
    band = 3 * w * (r1 - r0 + 1)
    up = {"bgr one pass": 3 * w * h, "bgr today": band + 3 * w * h, "i420 one pass": w * h * 3 // 2}
    dn_bgr = 3 * dw * dh * 2 + 3 * sw * sh
    down = {"bgr one pass": dn_bgr, "bgr today": dn_bgr, "i420 one pass": dw * dh * 3 + 3 * sw * sh}
    print("cfg2 x%d 1080p -> 1024^2 and 852x480 -> 1024^2, bilinear, INTER_LINEAR resize; BEV band rows [%d, %d]"
          % (n, r0, r1), flush=True)

    g = torch.Generator().manual_seed(1234)
    bgr = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=g).pin_memory()
    i420 = torch.randint(0, 256, (n, h * 3 // 2, w), dtype=torch.uint8, generator=g).pin_memory()

    def outs(fmt):
        frame = (dh, dw, 3) if fmt == "bgr" else (dh * 3 // 2, dw)
        return [torch.empty((n,) + s, dtype=torch.uint8).pin_memory() for s in (frame, (sh, sw, 3), frame)]
    out = {r: outs(r.split()[0]) for r in up}
    d_frames = torch.empty((n, h, w, 3), dtype=torch.uint8, device=dev)
    d_small = torch.empty((n, sh, sw, 3), dtype=torch.uint8, device=dev)
    d_bev_small = torch.empty((n, dh, dw, 3), dtype=torch.uint8, device=dev)

    def today():
        o = out["bgr today"]
        _native.warp_perspective_host(bgr, H, dsize, dst=o[0])
        d_frames.copy_(bgr, non_blocking=True)
        homo.resize(d_frames, small_size, dst=d_small)
        homo.warp_perspective(d_small, Hs, dsize, dst=d_bev_small)
        o[1].copy_(d_small, non_blocking=True)
        o[2].copy_(d_bev_small, non_blocking=True)
        torch.cuda.synchronize()

    def one_pass(src, fmt, o):
        return lambda: homo.warp_perspective_video_host_small(src, H, Hs, dsize, small_size, fmt, fmt, dst=o[0],
                                                              small=o[1], dst_small=o[2])
    routes = {"bgr one pass": one_pass(bgr, "bgr", out["bgr one pass"]), "bgr today": today,
              "i420 one pass": one_pass(i420, "i420", out["i420 one pass"])}
    for fn in routes.values():  # warm-up: workspace allocations, module loads
        fn()
    times = {r: [] for r in routes}
    for _ in range(rounds):
        for r, fn in routes.items():
            t0 = time.perf_counter()
            fn()
            times[r].append((time.perf_counter() - t0) * 1e3)
    for a, b in zip(out["bgr one pass"], out["bgr today"]):
        assert torch.equal(a, b), "the one-pass BGR route differs from today's route"
    kernels = {r: _kernel_ms(fn, ("warp", "resize")) for r, fn in routes.items()}
    del routes, out, d_frames, d_small, d_bev_small
    torch.cuda.empty_cache()

    # plain pinned copies of each route's bytes, both directions at once
    ceiling = _duplex_ceiling(torch.empty(max(up.values()) * n, dtype=torch.uint8).pin_memory(),
                              torch.empty(max(down.values()) * n, dtype=torch.uint8).pin_memory(), dev)
    for r in up:
        nu, nd = up[r] * n, down[r] * n
        ceil = ceiling(nu, nd)
        t = np.array(times[r])
        med = float(np.median(t))
        print("%s: median %.2f ms (min %.2f, max %.2f, spread %.1f %%) | H2D %.1f MB, D2H %.1f MB per step, "
              "ceiling %.2f ms (%.1f GB/s both ways) -> %.1f %% of it | kernels %.2f ms"
              % (r, med, t.min(), t.max(), 100.0 * (t.max() - t.min()) / med, nu / 1e6, nd / 1e6, ceil,
                 (nu + nd) / ceil / 1e6, 100.0 * ceil / med, kernels[r]), flush=True)


def device_mats_bench(rounds=5):
    """Homographies in CUDA tensors (the *_dmat entry points, the operators given a CUDA M) against the
    same calls with host matrices, alternated in rounds in one process; every pair of routes must give
    the same bytes.  A device matrix is read and inverted by the kernels when they run, and always takes
    the direct-gather kernels.
      cfg 1  one torch.cuda.graph replay of the one-frame loop (1080p BGR frame -> 1024^2 BEV, 852x480
             small frame, its 1024^2 BEV), captured with CPU H / Hs and with CUDA H / Hs
      cfg 2  256 1080p frames -> 1024^2, bilinear and nearest: device matrices against the automatic
             host-matrix route (the staged kernel) and the host-matrix direct-gather kernels
      cfg 4  the 8 cameras of tests/golden/cfg4_cams.json x 1000 1080p frames, host against device"""
    import json
    from bev_b200 import torch_ops
    torch_ops.load()
    ops = torch.ops.bev_cuda
    print("card: %s" % card(), flush=True)
    peak, _ = bench.measured_peak()
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1234)

    # cfg 1: graph replays
    H, (w, h), (sw, sh) = bench.h_canon(1), (1920, 1080), (852, 480)
    fx, fy = w / sw, h / sh
    Hs = H @ np.array([[fx, 0.0, 0.5 * fx - 0.5], [0.0, fy, 0.5 * fy - 0.5], [0.0, 0.0, 1.0]])
    frame = torch.randint(0, 256, (1, h, w, 3), dtype=torch.uint8, device=dev, generator=g)
    graphs, outs = {}, {}
    for route, (Ht, Hst) in (("host H", (torch.from_numpy(H), torch.from_numpy(Hs))),
                             ("device H", (torch.from_numpy(H).to(dev), torch.from_numpy(Hs).to(dev)))):
        def loop(Ht=Ht, Hst=Hst):
            small = ops.resize(frame, sw, sh)
            return ops.warp_perspective(frame, Ht, 1024, 1024), small, ops.warp_perspective(small, Hst, 1024, 1024)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                loop()
        torch.cuda.current_stream().wait_stream(s)
        graphs[route] = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graphs[route]):
            outs[route] = loop()
        graphs[route].replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in zip(outs["host H"], outs["device H"])), "cfg 1: routes differ"
    times = _alternate({r: gr.replay for r, gr in graphs.items()}, rounds, 200)
    for r, t in times.items():
        t = np.array(t) * 1e3
        print("device_mats cfg1 graph replay | %-8s: median %.1f us (min %.1f, max %.1f)"
              % (r, float(np.median(t)), t.min(), t.max()), flush=True)
    del graphs, outs

    # cfg 2
    n, dsize = 256, (1024, 1024)
    frames = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device=dev, generator=g)
    Hd = torch.from_numpy(H).to(dev)
    for flags, label in ((1, "bilinear"), (0, "nearest")):
        outs = {r: torch.empty((n, 1024, 1024, 3), dtype=torch.uint8, device=dev) for r in ("auto", "generic", "dmat")}
        routes = {"host M auto (staged)": lambda: homo.warp_perspective(frames, H, dsize, dst=outs["auto"], flags=flags,
                                                                         path="auto"),
                  "host M direct gather": lambda: homo.warp_perspective(frames, H, dsize, dst=outs["generic"],
                                                                        flags=flags, path="generic"),
                  "device M": lambda: _native.warp_perspective_dmat(frames, Hd, dsize, dst=outs["dmat"], flags=flags)}
        for fn in routes.values():
            fn()
        torch.cuda.synchronize()
        assert torch.equal(outs["auto"], outs["dmat"]) and torch.equal(outs["generic"], outs["dmat"]), \
            "cfg 2 %s: routes differ" % label
        T, _, _ = _native.warp_touched_pixels((w, h), dsize, H, flags)
        _report("device_mats cfg2 %s 256 x 1080p -> 1024^2" % label, _alternate(routes, rounds, 10),
                (T + dsize[0] * dsize[1]) * 3 * n, peak)
        del outs
    del frames
    torch.cuda.empty_cache()

    # cfg 4
    cams = json.load(open(os.path.join(ROOT, "tests", "golden", "cfg4_cams.json")))
    n = 1000
    frames = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, device=dev, generator=g)
    tables = [(np.array(c["H_bev_img"]), (int(c["bspec"]["u_size"]), int(c["bspec"]["v_size"]))) for c in cams]
    outs = [(torch.empty((n, d[1], d[0], 3), dtype=torch.uint8, device=dev),
             torch.empty((n, d[1], d[0], 3), dtype=torch.uint8, device=dev)) for _, d in tables]
    dev_tables = [torch.from_numpy(Hc).to(dev) for Hc, _ in tables]

    def host_all():
        for (Hc, d), (o, _) in zip(tables, outs):
            homo.warp_perspective(frames, Hc, d, dst=o)

    def dev_all():
        for Hc, (_, d), (_, o) in zip(dev_tables, tables, outs):
            _native.warp_perspective_dmat(frames, Hc, d, dst=o)

    host_all()
    dev_all()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b) for a, b in outs), "cfg 4: routes differ"
    algo = sum((_native.warp_touched_pixels((w, h), d, Hc, 1)[0] + d[0] * d[1]) * 3 * n for Hc, d in tables)
    _report("device_mats cfg4 8 cameras x 1000 x 1080p", _alternate({"host M": host_all, "device M": dev_all},
                                                                    rounds, 2), algo, peak)


def compo_dmat_bench(rounds=5, n=64):
    """The fused BEV compositor with CUDA H_bg / H_fg (bevk_composite_bev_u8c3_dmat) against the same
    calls with host matrices, alternated in rounds in one process; each pair must give the same bytes.
      x64    n 1080p renders + masks over ONE 1080p background -> 1024^2 BEVs (compo_bench's row),
             with one shared homography pair and with one pair per frame
      graph  one torch.cuda.graph replay of a single 1080p composite, captured with CPU and with
             CUDA matrices"""
    from bev_b200 import torch_ops
    torch_ops.load()
    ops = torch.ops.bev_cuda
    print("card: %s" % card(), flush=True)
    peak, _ = bench.measured_peak()
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1234)
    ssize, dsize = (1920, 1080), (1024, 1024)
    B = torch.randint(0, 256, (1, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    F = torch.randint(0, 256, (n, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    M = torch.randint(0, 256, (n, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    H = bench.h_canon(1)
    T, _, _ = _native.warp_touched_pixels(ssize, dsize, H, 1)
    D = dsize[0] * dsize[1]
    algo = 3 * (T + n * (2 * T + D))  # as compo_bench: background once, render and mask per frame, output
    for label, Hh in (("shared pair", H), ("pair per frame", np.repeat(H[None], n, 0))):
        Hd = torch.from_numpy(np.ascontiguousarray(Hh)).to(dev)
        outs = [torch.empty((n, 1024, 1024, 3), dtype=torch.uint8, device=dev) for _ in range(2)]
        routes = {"host H": lambda: _native.composite_bev_u8c3(B, F, M, Hh, Hh, dsize, out=outs[0]),
                  "device H": lambda: _native.composite_bev_u8c3_dmat(B, F, M, Hd, Hd, dsize, out=outs[1])}
        for fn in routes.values():
            fn()
        torch.cuda.synchronize()
        assert torch.equal(outs[0], outs[1]), "x%d %s: routes differ" % (n, label)
        _report("compo_dmat x%d 1080p -> 1024^2 %s" % (n, label), _alternate(routes, rounds, 10), algo, peak)
        del outs
    del F, M
    torch.cuda.empty_cache()

    fg = torch.randint(0, 256, (1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    mask = torch.randint(0, 256, (1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    graphs, outs = {}, {}
    for route, Ht in (("host H", torch.from_numpy(H)), ("device H", torch.from_numpy(H).to(dev))):
        def one(Ht=Ht):
            return ops.composite_bev(B[0], fg, mask, Ht, Ht, 1024, 1024)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                one()
        torch.cuda.current_stream().wait_stream(s)
        graphs[route] = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graphs[route]):
            outs[route] = one()
        graphs[route].replay()
    torch.cuda.synchronize()
    assert torch.equal(outs["host H"], outs["device H"]), "graph: routes differ"
    times = _alternate({r: gr.replay for r, gr in graphs.items()}, rounds, 200)
    for r, t in times.items():
        t = np.array(t) * 1e3
        print("compo_dmat 1080p -> 1024^2 graph replay | %-8s: median %.1f us (min %.1f, max %.1f)"
              % (r, float(np.median(t)), t.min(), t.max()), flush=True)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "nv12":
        nv12_bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "yuv420":
        yuv420_bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "video_host":
        video_host_bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "video_host_small":
        video_host_small_bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "frame_loop":
        frame_loop_bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "device_mats":
        device_mats_bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "compo_dmat":
        compo_dmat_bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "resize_nv12":
        resize_nv12_bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "resize_area":
        resize_area_bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "resize_nv12_area":
        resize_nv12_area_bench()
    elif len(sys.argv) > 1 and sys.argv[1] == "cfg4":
        if len(sys.argv) > 3:
            _native.set_warp_path(sys.argv[3])
        cfg4(int(sys.argv[2]) if len(sys.argv) > 2 else 1000)
    elif len(sys.argv) > 1 and sys.argv[1] == "cams1024":
        if len(sys.argv) > 2:
            _native.set_warp_path(sys.argv[2])
        cams_uniform()
    elif len(sys.argv) > 1 and sys.argv[1] == "cfg1":
        cfg1_cold_warm()
    elif len(sys.argv) > 1 and sys.argv[1] == "host1":
        host_single()
    elif len(sys.argv) > 1 and sys.argv[1] == "iou":
        iou_bench(int(sys.argv[2]) if len(sys.argv) > 2 else 8192)
    elif len(sys.argv) > 1 and sys.argv[1] == "resize":
        resize_bench(int(sys.argv[2]) if len(sys.argv) > 2 else 256)
    elif len(sys.argv) > 1 and sys.argv[1] == "compo":
        compo_bench(int(sys.argv[2]) if len(sys.argv) > 2 else 64)
    else:
        main()
