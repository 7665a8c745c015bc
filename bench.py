#!/usr/bin/env python
"""bench.py -- headline benchmark of the bev_b200 hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]
                    [--dump-outputs DIR]

A "step" is one pass of the batched warp over one synthetic batch.  The default workload is
BASELINE.json configs[1]: 256 synthetic 1080p uint8 frames, one fixed homography (SURVEY.md 8d
H_canon), bilinear image->BEV warp to 1024x1024.  N > 1 runs one process per GPU (torchrun), each
with its own 256 frames (weak scaling, no data-path collective); rank 0 prints ONE JSON line.
The frames come from a seeded generator, so with --dump-outputs two builds run with the same
arguments can be compared output for output (see dump_output).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "BEV warp Mpix/s"
UNIT = "Mpix/s"

# name -> (n_frames, src (w,h), dst (w,h), channels, dtype, flags, homography scale, inverse)
WORKLOADS = {
    "cfg2_1080p_to_bev1024_u8c3_bilinear_x256": (256, (1920, 1080), (1024, 1024), 3, "uint8", 1, 1, False),
    "cfg2_nearest": (256, (1920, 1080), (1024, 1024), 3, "uint8", 0, 1, False),
    "cfg1_single_frame": (1, (1920, 1080), (1024, 1024), 3, "uint8", 1, 1, False),
    "cfg5_4k_to_bev2048_u8c3_x64": (64, (3840, 2160), (2048, 2048), 3, "uint8", 1, 2, False),
    "cfg5_4k_to_bev2048_f16c3_x64": (64, (3840, 2160), (2048, 2048), 3, "float16", 1, 2, False),
    "cfg5_inv_bev2048_to_4k_u8c3_x64": (64, (2048, 2048), (3840, 2160), 3, "uint8", 1, 2, True),
    "cfg5_inv_bev2048_to_4k_f16c3_x64": (64, (2048, 2048), (3840, 2160), 3, "float16", 1, 2, True),
    # the cfg-2 map on the other pixel formats of the staged kernel
    "cfg2_u8c1_x256": (256, (1920, 1080), (1024, 1024), 1, "uint8", 1, 1, False),
    "cfg2_u8c4_x256": (256, (1920, 1080), (1024, 1024), 4, "uint8", 1, 1, False),
    "cfg2_f32c3_x128": (128, (1920, 1080), (1024, 1024), 3, "float32", 1, 1, False),
}
DEFAULT_WORKLOAD = "cfg2_1080p_to_bev1024_u8c3_bilinear_x256"


def h_canon(scale):
    """SURVEY.md 8d canonical homography (1080p -> 1024^2; x2 for 4K -> 2048^2)."""
    from bev_b200 import homo
    src = np.array([[700, 420], [1220, 420], [1900, 1060], [20, 1060]], np.float64) * scale
    dst = np.array([[200, 0], [824, 0], [824, 1024], [200, 1024]], np.float64) * scale
    return homo.homo_from_pts(src, dst)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


DUMP_LIMIT = 64 * 10**6  # bytes written by --dump-outputs, all files together


def dump_output(out_dir, name, t, limit=DUMP_LIMIT):
    """Write tensor t (..., C) as out_dir/<name>.npy in float32, so that two builds run with the
    same arguments can be compared output for output.  If the whole tensor does not fit in `limit`
    bytes, a fixed sample of its pixels (whole rows of the last axis, positions drawn with seed 0
    and sorted) is written as (k, C), with their flat pixel indices as <name>_index.npy (float64).
    Returns the paths written."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    c = t.shape[-1]
    pixels = t.reshape(-1, c)
    path = os.path.join(out_dir, name + ".npy")
    data = limit - 4096  # the rest holds the .npy headers
    if t.numel() * 4 <= data:
        np.save(path, t.float().cpu().numpy())
        return [path]
    k = data // (4 * c + 8)
    idx = np.sort(np.random.default_rng(0).choice(pixels.shape[0], k, replace=False, shuffle=False))
    sample = pixels[torch.from_numpy(idx).to(t.device)].float().cpu().numpy()
    ipath = os.path.join(out_dir, name + "_index.npy")
    np.save(path, sample)
    np.save(ipath, idx.astype(np.float64))
    return [path, ipath]


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples taken while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"], stdout=f, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 7:
                    continue
                try:
                    sm.append(float(parts[0]))
                    mx.append(float(parts[1]))
                except ValueError:
                    continue
                for name, val in zip(names, parts[3:7]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


def reference_arm(args, wl):
    """--impl reference: the reference's CPU implementation (cv2 loop, all host threads) on a
    bounded sample of the same workload.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import ref_cpu
    from oracle.synth import seeded_frame
    n_frames, ssize, dsize, ch, dtype, flags, hscale, inverse = WORKLOADS[wl]
    H = h_canon(hscale)
    if inverse:
        H = np.linalg.inv(H)
    sample = n_frames  # the whole workload: every step is one pass of the reference loop over all frames
    np_dtype = "float32" if dtype == "float16" else dtype  # cv2 has no fp16 warp (SURVEY.md 0.4)
    frames = [seeded_frame(1234 + i, ssize[1], ssize[0], ch, np_dtype) for i in range(sample)]
    run, kind, cores = ref_cpu.make_warp_runner()
    for _ in range(max(args.warmup, 1)):  # full passes: thread pool, page cache and clocks warm
        run(frames, H, dsize, flags)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        run(frames, H, dsize, flags)
        times.append(time.perf_counter() - t0)
    ms = 1e3 * sum(times) / len(times)
    value = sample * dsize[0] * dsize[1] / (ms * 1e-3) / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8" if dtype == "uint8" else dtype,
        "data": "synthetic",
        "config": {"workload": wl, "frames_per_step": sample, "src": list(ssize), "dst": list(dsize),
                   "same_config": True,
                   "note": "each step = the reference loop (cv2.warpPerspective per frame, "
                           "vis_homo.py:85-89) over all %d frames of the workload" % sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": "%d steps x %d frames" % (args.steps, sample),
                         "cpu": ref_cpu.cpu_model()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def ours(args, wl):
    import torch
    import torch.distributed as dist
    from bev_b200 import _native, homo, sharding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # The only collective is the send/recv gather of BEV batches into rank 0: give NCCL's
        # point-to-point path all its channels (measured at N=2, tools/gather_probe.py: 543 GB/s
        # into rank 0 with the default channel count, 598 GB/s with 64, and no longer sensitive
        # to the slice size the pipelined gather uses).
        for k, v in (("NCCL_MIN_P2P_NCHANNELS", "64"), ("NCCL_MAX_P2P_NCHANNELS", "64"),
                     ("NCCL_MAX_NCHANNELS", "64")):
            os.environ.setdefault(k, v)
        dist.init_process_group("nccl", device_id=dev)

    n_frames, ssize, dsize, ch, dtype, flags, hscale, inverse = WORKLOADS[wl]
    H = h_canon(hscale)
    if inverse:
        H = np.linalg.inv(H)
    if args.path:
        _native.set_warp_path(args.path)
    tdtype = {"uint8": torch.uint8, "float16": torch.float16, "float32": torch.float32}[dtype]
    es = {"uint8": 1, "float16": 2, "float32": 4}[dtype]

    # synthetic frames: i.i.d. uniform noise, generated on the device, per-rank seed (SURVEY 8d)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    frames = torch.randint(0, 256, (n_frames, ssize[1], ssize[0], ch), dtype=torch.uint8, device=dev,
                           generator=g)
    if tdtype != torch.uint8:
        frames = (frames.to(torch.float32) / 255.0).to(tdtype)
    out = torch.empty((n_frames, dsize[1], dsize[0], ch), dtype=tdtype, device=dev)

    T, r0, r1 = _native.warp_touched_pixels(ssize, dsize, H, flags)
    algo_bytes_frame = (T + dsize[0] * dsize[1]) * ch * es
    algo_bytes_step = algo_bytes_frame * n_frames

    def step():
        homo.warp_perspective(frames, H, dsize, dst=out, flags=flags)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
        time.sleep(0.05)
    try:  # the nvidia-smi sampler must not outlive a failed step
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        barrier()
        ev[0].record()
        for i in range(args.steps):
            step()
            ev[i + 1].record()
        barrier()
    finally:
        clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_output(args.dump_outputs, "warp_output", out)
    total_ms = ev[0].elapsed_time(ev[-1])
    per_launch_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms_max = float(t.item())
    ms_per_step = total_ms_max / args.steps
    px_step = n_frames * dsize[0] * dsize[1]
    value = world * px_step / (ms_per_step * 1e-3) / 1e6

    # ---- e2e: same metric through the host-buffer C-ABI call, pinned host memory, H2D + D2H timed
    e2e_steps = max(1, min(args.e2e_steps, args.steps))
    if args.no_e2e:
        e2e_s = float("nan")
    else:
        h_src = torch.empty(frames.shape, dtype=tdtype).pin_memory()
        h_src.copy_(frames)
        h_dst = torch.empty(out.shape, dtype=tdtype).pin_memory()
        _native.warp_perspective_host(h_src, H, dsize, dst=h_dst, flags=flags)  # warm-up (allocs)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            _native.warp_perspective_host(h_src, H, dsize, dst=h_dst, flags=flags)
        torch.cuda.synchronize()
        e2e_s = (time.perf_counter() - t0) / e2e_steps
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * px_step / float(te.item()) / 1e6
    row_bytes = ssize[0] * ch * es
    up0, up1 = _native.warp_host_rows(ssize, dsize, H, flags)  # only referenced rows are uploaded
    h2d = n_frames * (up1 - up0 + 1) * row_bytes
    d2h = out.numel() * es
    # What the host link allows for these byte counts: plain pinned copies of h2d bytes up and
    # d2h bytes down at the same time, on every rank at once (the ranks share the host's memory
    # and PCIe root complexes) -- the ceiling of the e2e number at this N.
    pcie = None
    if not args.no_e2e:
        d_up = torch.empty(h2d, dtype=torch.uint8, device=dev)
        h_up = h_src.view(torch.uint8).reshape(-1)[:h2d]
        h_dn = h_dst.view(torch.uint8).reshape(-1)
        d_dn = out.view(torch.uint8).reshape(-1)
        s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
        best = None
        for _ in range(3):
            barrier()
            t0 = time.perf_counter()
            with torch.cuda.stream(s_up):
                d_up.copy_(h_up, non_blocking=True)
            with torch.cuda.stream(s_dn):
                h_dn.copy_(d_dn, non_blocking=True)
            s_up.synchronize()
            s_dn.synchronize()
            dt = time.perf_counter() - t0
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            best = float(tt.item()) if best is None else min(best, float(tt.item()))
        pcie = {"copy_ms": best * 1e3, "GBps_per_gpu_both_directions": (h2d + d2h) / best / 1e9,
                "GBps_box_total": world * (h2d + d2h) / best / 1e9,
                "ceiling_Mpix_s": world * px_step / best / 1e6,
                "e2e_frac_of_ceiling": e2e_value / (world * px_step / best / 1e6)}
        del d_up, h_src, h_dst

    # ---- gather of BEV outputs to rank 0 (reported separately from the warp scaling, SURVEY 8e):
    #      once after the warp, and once chunk-pipelined behind the warp on a side stream
    gather = None
    if world > 1:
        out_bytes = out.numel() * es
        sharding.gather_to_rank0(out[:2])  # connection set-up is not part of the measurement
        torch.cuda.synchronize()
        dist.barrier()

        def max_ms(ms):
            tg = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tg, op=dist.ReduceOp.MAX)
            return float(tg.item())

        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        gms = None
        for _ in range(3):  # the first pass also pays for the 1.6 GB receive buffer's allocation
            barrier()
            g0.record()
            gathered = sharding.gather_to_rank0(out, chunks=1)
            g1.record()
            torch.cuda.synchronize()
            ms_g = max_ms(g0.elapsed_time(g1))
            gms = ms_g if gms is None else min(gms, ms_g)
            del gathered

        def produce(b, e, dst):
            homo.warp_perspective(frames[b:e], H, dsize, dst=dst[b:e], flags=flags)

        best = None
        for _ in range(3):
            barrier()
            g0.record()
            _, gathered = sharding.pipelined_gather_to_rank0(
                produce, n_frames, tuple(out.shape[1:]), tdtype, dev, chunks=8, local_out=out)
            g1.record()
            torch.cuda.synchronize()
            pms = max_ms(g0.elapsed_time(g1))
            best = pms if best is None else min(best, pms)
            del gathered
        into0 = (world - 1) * out_bytes
        gather = {"ms": gms, "bytes_into_rank0": into0, "GBps_into_rank0": into0 / (gms * 1e-3) / 1e9,
                  "pipelined": {"ms_warp_and_gather": best, "chunks": 8,
                                "GBps_into_rank0": into0 / (best * 1e-3) / 1e9,
                                "Mpix_s_gathered_on_rank0": world * px_step / (best * 1e-3) / 1e6,
                                "note": "8 frame slices: warp of slice k+1 on the compute stream while "
                                        "slice k is gathered (NCCL send/recv) on a side stream"},
                  "ingress_peak_GBps": {"nominal": 900.0, "measured_peer_copy": 770.0},
                  "limiting": "rank 0's NVLink ingress: (N-1) x %.0f MB must enter one GPU, the warp "
                              "that produces them takes %.2f ms per rank" % (out_bytes / 1e6, ms_per_step)}

    # ---- the other sharded workloads of BASELINE.json at N > 1
    multi = None
    if world > 1 and not args.no_other_configs:
        del frames, out
        torch.cuda.empty_cache()
        multi = {"projection": projection_leg(dev, min(args.steps, 20), 0.0, False, world=world),
                 "cfg4_sharded": cfg4_sharded(dev, rank, world, min(args.steps, 5))}
        frames = out = None

    if rank == 0:
        peak, peak_src = measured_peak()
        launch_ms = statistics.mean(per_launch_ms)
        achieved = algo_bytes_step / (launch_ms * 1e-3) / 1e9
        traffic = None
        prof = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(prof):
            try:
                traffic = json.load(open(prof)).get(wl)
            except Exception:
                traffic = None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8" if dtype == "uint8" else dtype,
            "data": "synthetic",
            "config": {"workload": wl, "frames_per_gpu": n_frames, "src": list(ssize),
                       "dst": list(dsize), "channels": ch,
                       "interp": "bilinear" if flags & 1 else "nearest",
                       "homography": "H_canon (SURVEY 8d)", "parallelism": "frames sharded, %d per GPU" % n_frames,
                       "l2": "inputs %.0f MB per step >> 126 MB L2, no flush needed"
                             % (n_frames * ssize[0] * ssize[1] * ch * es / 1e6),
                       "kernel_path": args.path or "auto"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "api": "bevk_warp_perspective_host (pinned host src/dst)", "pcie": pcie},
            "gpu_launches": args.steps * 1,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "frac_of_nominal_8000": achieved / 8000.0,
                         "algo_bytes_per_launch": algo_bytes_step,
                         "algo_bytes_per_frame": algo_bytes_frame,
                         "launch_ms": launch_ms, "kernel": "bevk warp kernel (1 launch per step)"},
        }
        if gather:
            line["gather"] = gather
        if multi:
            line.update(multi)
        if world == 1 and not args.no_cpu_baseline:
            from oracle import ref_cpu
            sample = n_frames  # the same 256 frames the GPU arm warps (and --impl reference times)
            host = frames[:sample].cpu()
            if tdtype == torch.float16:
                host = host.to(torch.float32)
            cb = ref_cpu.time_warp(list(host.numpy()), H, tuple(dsize), flags,
                                   min_seconds=args.cpu_seconds)
            line["cpu_baseline"] = {"value": cb["value"], "unit": UNIT, "cores": cb["cores"],
                                    "kind": cb["kind"], "sample": cb["sample"], "cpu": cb["cpu"],
                                    "ms_per_frame": cb["ms_per_frame"]}
        if world == 1 and not args.no_projection:
            del frames, out
            torch.cuda.empty_cache()
            line["projection"] = projection_leg(dev, min(args.steps, 20), min(args.cpu_seconds, 5.0),
                                                not args.no_cpu_baseline)
        if world == 1 and not args.no_other_configs:
            torch.cuda.empty_cache()
            line["other_configs"] = other_configs(dev, min(args.steps, 10))
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def projection_leg(dev, steps, cpu_seconds, with_cpu, world=1):
    """BASELINE configs[2]: 10 M synthetic xywh-theta BEV boxes -> image corners and back (fp32),
    through bev_b200.rbox_torch (one fused CUDA kernel per direction).  Returns the `projection`
    object of the JSON line: projections/s (one box through one direction), the HBM roofline of
    the two kernels (52 B per box and direction, SURVEY.md 8d) and the reference's numpy float64
    chain timed on a bounded sample of the same boxes.  world > 1: every rank projects its own
    10 M boxes (weak scaling, no exchange), time = max over ranks, value = all ranks' boxes."""
    import torch
    import torch.distributed as dist
    from bev_b200 import rbox_torch
    n = 10_000_000
    seed = 0 + (dist.get_rank() if world > 1 else 0)
    g = torch.Generator(device=dev).manual_seed(seed)
    u = torch.rand((n, 5), dtype=torch.float32, device=dev, generator=g)
    lo = torch.tensor([0.0, 0.0, 4.0, 8.0, -np.pi], dtype=torch.float32, device=dev)
    hi = torch.tensor([1024.0, 1024.0, 40.0, 120.0, np.pi], dtype=torch.float32, device=dev)
    box = lo + u * (hi - lo)
    del u
    H_back = h_canon(1)             # image -> BEV
    H_fwd = np.linalg.inv(H_back)   # BEV -> image
    for _ in range(3):
        img = rbox_torch.xywhr_to_img_corners(box, H_fwd, "bev")
        back = rbox_torch.img_corners_to_xywhr(img, H_back, "bev")
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        img = rbox_torch.xywhr_to_img_corners(box, H_fwd, "bev")
        back = rbox_torch.img_corners_to_xywhr(img, H_back, "bev")
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    peak, peak_src = measured_peak()
    algo = 2 * 52 * n
    out = {"metric": "rbox projections/s", "value": world * 2 * n / (ms * 1e-3) / 1e6, "unit": "Mproj/s",
           "boxes_per_gpu": n, "n_gpus": world, "ms_fwd_plus_back": ms, "dtype": "f32 io, f64 registers",
           "gpu_launches_per_step": "2 bulk kernels (+ 2 one-block tail launches when n % 256 != 0)",
           "roofline": {"bound": "hbm", "achieved": algo / (ms * 1e-3) / 1e9, "peak": peak,
                        "unit": "GB/s", "frac": algo / (ms * 1e-3) / 1e9 / peak,
                        "algo_bytes_per_step": algo, "peak_source": peak_src, "per": "GPU"},
           "round_trip_max_abs_err": float((back[:, :4] - box[:, :4]).abs().max().item())}
    if with_cpu:
        from oracle import ref_cpu
        sample = box[:200_000].cpu().numpy()
        cb = ref_cpu.time_rbox_chain(sample, H_fwd, H_back, "bev", min_seconds=cpu_seconds)
        out["cpu_baseline"] = cb
    return out


def cfg4_sharded(dev, rank, world, steps, n_frames=1000):
    """BASELINE configs[3] on N GPUs: the eight BrnoCompSpeed-shaped camera streams of
    tests/golden/cfg4_cams.json, 1000 synthetic 1080p frames each, sharded two ways:
      by_frames  -- every rank takes the frame slice [r, r+1) * 1000 / N of EVERY stream (the
                    config's "frame-sharded": even work, eight launches of 1000 / N frames per rank);
      by_camera  -- whole streams dealt to the ranks by sharding.shard_cameras (N = 8: one stream per
                    GPU, SURVEY.md 8e): long launches, but the streams' BEVs differ in size.
    Nothing is exchanged; time = max over ranks of the rank's total over its launches."""
    import torch
    import torch.distributed as dist
    from bev_b200 import _native, homo, sharding
    cams = json.load(open(os.path.join(ROOT, "tests", "golden", "cfg4_cams.json")))
    peak, _ = measured_peak()

    def run(jobs):
        """jobs: (camera index, first frame, frames).  Returns this rank's (ms, pixels, algorithmic bytes)."""
        ms_tot, px, nbytes = 0.0, 0, 0
        for k, f0, nf in jobs:
            c = cams[k]
            H = np.array(c["H_bev_img"])
            dsize = (int(c["bspec"]["u_size"]), int(c["bspec"]["v_size"]))
            g = torch.Generator(device=dev).manual_seed(1234 + k)
            frames = torch.randint(0, 256, (nf, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
            dst = torch.empty((nf, dsize[1], dsize[0], 3), dtype=torch.uint8, device=dev)
            T, _, _ = _native.warp_touched_pixels((1920, 1080), dsize, H, 1)
            for _ in range(2):
                homo.warp_perspective(frames, H, dsize, dst=dst)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                homo.warp_perspective(frames, H, dsize, dst=dst)
            e1.record()
            torch.cuda.synchronize()
            ms_tot += e0.elapsed_time(e1) / steps
            px += nf * dsize[0] * dsize[1]
            nbytes += (T + dsize[0] * dsize[1]) * 3 * nf
            del frames, dst
            torch.cuda.empty_cache()
        return ms_tot, px, nbytes

    def reduce(ms, px, nbytes):
        t = torch.tensor([ms, float(px), float(nbytes)], dtype=torch.float64, device=dev)
        tmax, tsum = t.clone(), t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        return float(tmax[0].item()), float(tsum[0].item()), float(tsum[1].item()), float(tsum[2].item())

    out = {"cameras": len(cams), "frames_per_camera": n_frames}
    # whole streams per rank
    mine = sharding.shard_cameras(len(cams), rank, world)
    ms_max, ms_sum, px, nbytes = reduce(*run([(k, 0, n_frames) for k in mine]))
    n1_ms = ms_sum  # every camera's full-stream kernel time, summed over all ranks = one GPU doing all eight
    out["by_camera"] = {"ms": ms_max, "Mpix_s": px / ms_max / 1e3, "cameras_of_rank0": mine,
                        "roofline_frac_per_gpu": nbytes / world / (ms_max * 1e-3) / 1e9 / peak,
                        "efficiency": n1_ms / (world * ms_max)}
    # a frame slice of every stream per rank
    b, e = sharding.shard_range(n_frames, rank, world)
    ms_max, _, px, nbytes = reduce(*run([(k, b, e - b) for k in range(len(cams))]))
    out["by_frames"] = {"ms": ms_max, "Mpix_s": px / ms_max / 1e3, "frames_per_rank_and_camera": e - b,
                        "roofline_frac_per_gpu": nbytes / world / (ms_max * 1e-3) / 1e9 / peak,
                        "efficiency": n1_ms / (world * ms_max)}
    out["n1_equivalent_ms"] = n1_ms
    out["note"] = ("ms = slowest rank's total over its launches (one per camera); n1_equivalent_ms = sum over "
                   "the eight cameras of the single-GPU 1000-frame kernel time; efficiency = that / (N x ms). "
                   "by_camera loses to the uneven BEV sizes of the streams (192x320 ... 320x640), by_frames to "
                   "the shorter launches")
    return out


def other_configs(dev, steps):
    """Kernel-only numbers for the other BASELINE configs (inputs resident in HBM, CUDA events,
    3 warm-up launches each): cfg 2 nearest, cfg 5 both directions in uint8 and float16, cfg 4
    (8 cameras x 1000 frames, the homographies of tests/golden/cfg4_cams.json).  Reported inside
    the one JSON line as `other_configs`; the headline stays cfg 2."""
    import torch
    from bev_b200 import _native, homo
    peak, _ = measured_peak()
    out = {}

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    for wl in ("cfg2_nearest", "cfg5_4k_to_bev2048_u8c3_x64", "cfg5_inv_bev2048_to_4k_u8c3_x64",
               "cfg5_4k_to_bev2048_f16c3_x64", "cfg5_inv_bev2048_to_4k_f16c3_x64",
               "cfg2_u8c1_x256", "cfg2_u8c4_x256", "cfg2_f32c3_x128"):
        n, ssize, dsize, ch, dtype, flags, hscale, inverse = WORKLOADS[wl]
        H = np.linalg.inv(h_canon(hscale)) if inverse else h_canon(hscale)
        es = {"uint8": 1, "float16": 2, "float32": 4}[dtype]
        g = torch.Generator(device=dev).manual_seed(1234)
        frames = torch.randint(0, 256, (n, ssize[1], ssize[0], ch), dtype=torch.uint8, device=dev, generator=g)
        if dtype != "uint8":
            frames = (frames.to(torch.float32) / 255.0).to(torch.float16 if dtype == "float16" else torch.float32)
        dst = torch.empty((n, dsize[1], dsize[0], ch), dtype=frames.dtype, device=dev)
        T, _, _ = _native.warp_touched_pixels(ssize, dsize, H, flags)
        algo = (T + dsize[0] * dsize[1]) * ch * es * n
        ms = timed(lambda: homo.warp_perspective(frames, H, dsize, dst=dst, flags=flags))
        out[wl] = {"ms": ms, "Mpix_s": n * dsize[0] * dsize[1] / ms / 1e3, "roofline_frac": algo / (ms * 1e-3) / 1e9 / peak}
        del frames, dst
        torch.cuda.empty_cache()

    cams = json.load(open(os.path.join(ROOT, "tests", "golden", "cfg4_cams.json")))
    n = 1000
    g = torch.Generator(device=dev).manual_seed(1234)
    frames = torch.randint(0, 256, (n, 1080, 1920, 3), dtype=torch.uint8, device=dev, generator=g)
    tot_ms, tot_px, tot_bytes = 0.0, 0, 0
    for c in cams:
        H = np.array(c["H_bev_img"])
        dsize = (int(c["bspec"]["u_size"]), int(c["bspec"]["v_size"]))
        dst = torch.empty((n, dsize[1], dsize[0], 3), dtype=torch.uint8, device=dev)
        T, _, _ = _native.warp_touched_pixels((1920, 1080), dsize, H, 1)
        tot_ms += timed(lambda: homo.warp_perspective(frames, H, dsize, dst=dst))
        tot_px += n * dsize[0] * dsize[1]
        tot_bytes += (T + dsize[0] * dsize[1]) * 3 * n
        del dst
    out["cfg4_8cams_x1000_1080p_to_brno_bevs"] = {
        "ms": tot_ms, "Mpix_s": tot_px / tot_ms / 1e3, "roofline_frac": tot_bytes / (tot_ms * 1e-3) / 1e9 / peak,
        "note": "8 launches (one per camera); DRAM traffic is at the 64-byte-granular floor (DESIGN.md 3.2)"}
    del frames
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--path", default=None, choices=[None, "auto", "generic", "fast"])
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling aid: skip the host-buffer leg")
    ap.add_argument("--no-projection", action="store_true", help="skip the rbox projection leg")
    ap.add_argument("--no-other-configs", action="store_true",
                    help="skip the kernel-only numbers of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's warp output (rank 0) as "
                         "DIR/warp_output.npy in float32, a seeded sample if it exceeds 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the CUDA path (--impl ours)")

    if args.impl == "reference":
        reference_arm(args, args.workload)
        return
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # convenience: relaunch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1",
               "--nproc-per-node", str(args.gpus), "--master-addr", "127.0.0.1",
               "--master-port", str(29500 + os.getpid() % 500)] + sys.argv
        sys.exit(subprocess.call(cmd))
    ours(args, args.workload)


if __name__ == "__main__":
    main()
