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
                  (64, (2160, 3840), (1920, 1080)))


def resize_area_bench(rounds=5):
    """INTER_AREA resize of BGR frames against the INTER_LINEAR kernel on the same shapes,
    alternating the two in one process.  Algorithmic bytes: 3 x (touched source pixels + dst
    pixels); a downscale touches the whole frame.  Every frame set is larger than the 126 MB L2.
    Frame 0 of the area route is checked against the oracle."""
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


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "nv12":
        nv12_bench()
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
