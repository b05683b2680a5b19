#!/usr/bin/env python
"""bench.py — frames/sec of the ElasticFusion hot path (track + fuse + predict) on B200, with the ICP-reduction roofline.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload ...]

A *step* is one ElasticFusion::processFrame call on one frame of the synthetic ICL-NUIM-shaped room sequence; every rank (one
per GPU) tracks and fuses its own independent sequence, so `value` is the whole-job frames/sec (weak scaling, no data-path
collective; NCCL only for the two barriers and the max-over-ranks, through elasticfusion_b200/multi.py).

  value      frames/sec with the K frames already resident in HBM (ef_process_frame_device), one CUDA-event pair per frame on the
             context's stream; the stop event is recorded after the main stream has joined the look-ahead stream, so every
             kernel enqueued during the step -- including the staging of the next frame -- lies inside the timed span. L2 is
             flushed (256 MiB write) between frames, outside the spans.
  e2e        the same frames through the host-buffer calls: pinned copy + H2D of the step's frame and the D2H read of the pose
             inside the timed (wall-clock) region -- what a caller of libefusion.so sees.
  no_lookahead  both numbers with plain per-frame calls (the caller does not own frame i+1 while frame i runs).
  roofline   the ICP residual + Jacobian + 29-term reduction at level 0 (north_star's kernel): algorithmic 48 B/pixel + 116 B,
             average launch duration over a batch of launches whose inputs exceed L2, against MEASURED_PEAKS.json hbm_gbs;
             `full_iteration` is the complete Gauss-Newton iteration (k_iter1 + k_iter2) on the same bytes.
  value_1280x960, large_map   (rank 0, N=1 only) BASELINE configs[2] frames/sec, and frames/sec + per-pass GB/s with 5 M (640x480)
             and 20 M (1280x960) surfels RESIDENT: the map is pre-populated through ef_map_upload after the first frame.
  tracking_only  event-timed tracking stages of this library vs the reference's own CUDA tracking kernels (oracle/_ref) per frame.
  cpu_baseline   the reference arm on a bounded sample (reference CUDA tracking + CPU-oracle mapping; pure CPU port if oracle/_ref
             is absent).

--impl reference times the reference arm alone: the reference's CUDA tracking kernels compiled unmodified into oracle/_ref (driven
launch-for-launch like Core/Utils/RGBDOdometry.cpp) plus the CPU oracle for the GLSL mapping half, which cannot run without OpenGL
(BASELINE.md §3). Under torchrun rank 0 alone runs: it drives one sequence per GPU concurrently (one host thread each, the host
cores split between them), so its `value` is the whole-job aggregate for the same N-sequence job.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BIG = 2147483647 // 2
MAXD = 20.0
CLOCK_Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
           "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
METRIC = "frames/sec, full track+fuse+predict (processFrame)"

WORKLOADS = {
    # name: (scale, surfel capacity, resident surfels to pre-populate (0: map grows from the sequence), description)
    "640x480": (1, 5_000_000, 0, "640x480 synthetic planar-room sequence (ICL-NUIM-shaped), full track+fuse, 5M surfel cap"),
    "1280x960": (2, 20_000_000, 0, "1280x960 high-res synthetic sequence, full track+fuse, 20M surfel cap"),
    "640x480-5M": (1, 5_600_000, 5_000_000, "640x480 synthetic planar-room sequence, full track+fuse, 5M surfels resident (map pre-populated)"),
    "1280x960-20M": (2, 21_500_000, 20_000_000, "1280x960 high-res synthetic sequence, full track+fuse, 20M surfels resident (map pre-populated)"),
}


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, device_index: int):
        self.idx = device_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={CLOCK_Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_frames(K, n, seed):
    """First n frames of the synthetic sequence (frame i depends only on (seed, i), so a longer cached run serves any
    shorter request: the reference arm and repeated runs on one box do not render again)."""
    from elasticfusion_b200 import synth

    cache = os.path.join(os.environ.get("EF_BENCH_CACHE", "/tmp"), f"ef_bench_{K.width}x{K.height}_{seed}.npz")
    have_rgb = have_depth = None
    if os.path.exists(cache):
        try:
            z = np.load(cache)
            have_rgb, have_depth = z["rgb"], z["depth"]
        except Exception:
            have_rgb = have_depth = None
    m = 0 if have_rgb is None else len(have_rgb)
    if m >= n:
        return have_rgb[:n], have_depth[:n]
    rgb = np.empty((n, K.height, K.width, 3), np.uint8)
    depth = np.empty((n, K.height, K.width), np.uint16)
    if m:
        rgb[:m], depth[:m] = have_rgb, have_depth
    traj = synth.trajectory(n, seed=seed)
    for i in range(m, n):
        rgb[i], depth[i] = synth.render(traj[i], K, noise_seed=seed * 100003 + i)[:2]
    try:
        tmp = cache + f".{os.getpid()}.tmp.npz"
        np.savez(tmp, rgb=rgb, depth=depth)
        os.replace(tmp, cache)
    except Exception:
        pass
    return rgb, depth


def workload(name):
    from elasticfusion_b200 import synth

    if name not in WORKLOADS:
        raise SystemExit("unknown workload")
    scale, cap, resident, desc = WORKLOADS[name]
    K = synth.K_DEFAULT if scale == 1 else synth.K_DEFAULT.scaled(scale)
    return K, cap, resident, desc


def bench_config(wl_name, frames_per_gpu, world, la, flush, surfels_at_end=None, **extra):
    """The `config` object: ONE key set for both arms (the driver compares them), arm-specific values only."""
    cfg = {"workload": wl_name, "frames_per_gpu": frames_per_gpu, "parallelism": f"{world} independent sequences, one per GPU",
           "open_loop": True, "time_delta": "INT_MAX/2 (open loop: Ferns' time(0) seed cannot matter, SURVEY.md §8d)",
           "l2": "flushed between frames (256 MiB write, outside the timed spans)" if flush else "not flushed",
           "lookahead": ("next frame's upload + depth preprocess + pyramids + SO(3) loop staged on a side stream inside the timed span "
                         "of the frame in flight (ef_prefetch_frame); the span ends after both streams have joined") if la else "off",
           "skip_mid_predict": ("1: the predict() of Core/ElasticFusion.cpp:387, whose outputs only loop closure reads, is not executed "
                                "(the reference arm executes it)"),
           "surfels_at_end": surfels_at_end}
    cfg.update(extra)
    return cfg


def dump_outputs(ctx, out_dir, limit=64 << 20):
    """Writes what a caller of processFrame receives after the last timed frame to out_dir/<name>.npy: the camera pose, the
    model views predicted for the next frame (vertex, normal, colour), the surfel count and the surfel map. Above `limit` bytes in
    all, the map is a fixed seeded sample of its rows, kept in map order (the map's compaction preserves order). Every value is
    finite: the undefined normal of a surfel at a depth edge (NaN in the map) is written as the zero vector, which no unit normal
    can be."""
    os.makedirs(out_dir, exist_ok=True)
    out = {"pose": ctx.get_pose(), "surfel_count": np.array([ctx.map_count()], np.float64)}
    for name in ("VERTEX", "NORMAL", "IMAGE"):
        out[f"model_{name.lower()}"] = ctx.download(name).astype(np.float32)
    surfels = ctx.map_download()
    rows = max(0, limit - sum(a.nbytes for a in out.values())) // (12 * 4)
    if len(surfels) > rows:
        surfels = surfels[np.sort(np.random.default_rng(0).choice(len(surfels), rows, replace=False))]
    out["surfels"] = surfels
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.where(np.isfinite(a), a, 0).astype(a.dtype))


def populate_map(ctx, K, n_resident, seed, rgb0, depth0):
    """Frame 0 through the public call (tick 1 builds the map from the frame), then replaces the map by ~n_resident stable surfels
    tiling the room (the pose after frame 0 is the identity = the world frame of the sequence) and re-renders the model view."""
    from elasticfusion_b200 import synth

    ctx.process_frame(rgb0, depth0, 0)
    T_w_room = np.linalg.inv(synth.trajectory(1, seed=seed)[0])
    surf = synth.room_surfels(n_resident, T_w_room, view_depth=1.5, focal=K.fx)
    ctx.map_upload(surf)
    n = len(surf)
    del surf
    ctx.predict()
    ctx.sync()
    return n


# ------------------------------------------------------------------------------------------------------------------
def timed_sequence(ctx, torch, stream, dev, flush, rgb, depth, rgb_d, depth_d, first, warmup, steps, la, do_flush, host):
    """Runs frames first .. first+warmup+steps-1 (frame `first` must not have been processed yet; with look-ahead frame
    first+warmup+steps is staged as well). Device mode: CUDA-event time per frame (ms list). Host mode: wall seconds per frame."""
    def step(i):
        if host:
            if la:
                ctx.process_frame_device(None, None, i)
                ctx.prefetch_frame(rgb[i + 1], depth[i + 1])
                ctx.finish_frame()
            else:
                ctx.process_frame(rgb[i], depth[i], i)
        else:
            if la:
                ctx.process_frame_device(None, None, i)
                ctx.prefetch_frame_device(rgb_d[i + 1].data_ptr(), depth_d[i + 1].data_ptr())
                ctx.join_lookahead()
            else:
                ctx.process_frame_device(rgb_d[i].data_ptr(), depth_d[i].data_ptr(), i)

    with torch.cuda.stream(stream):
        if la:
            if host:
                ctx.prefetch_frame(rgb[first], depth[first])
            else:
                ctx.prefetch_frame_device(rgb_d[first].data_ptr(), depth_d[first].data_ptr())
        for i in range(first, first + warmup):
            step(i)
    ctx.sync()
    out = []
    l0 = ctx.launch_count()
    t0 = time.perf_counter()
    if host:
        for k in range(steps):
            i = first + warmup + k
            if do_flush:
                flush.fill_(k & 0xff)
                torch.cuda.synchronize(dev)
            t = time.perf_counter()
            step(i)
            out.append(time.perf_counter() - t)
    else:
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        with torch.cuda.stream(stream):
            for k in range(steps):
                i = first + warmup + k
                if do_flush:
                    flush.fill_(k & 0xff)
                ev[k][0].record(stream)
                step(i)
                ev[k][1].record(stream)
        ctx.sync()
        out = [s.elapsed_time(e) for s, e in ev]
    wall = time.perf_counter() - t0
    timed_sequence.last_launches = ctx.launch_count() - l0  # kernels launched inside the timed loop
    return out, wall


def run_ours(args, rank, world, dist):
    import torch

    from elasticfusion_b200 import capi, multi

    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    K, cap, resident, wl_name = workload(args.workload)
    n_total = args.warmup + args.steps
    seed = multi.sequence_seed(42, multi.shard_sequences(world, world, rank)[0])  # one sequence per rank
    rgb, depth = make_frames(K, n_total + 2, seed)  # +1 frame 0 of a pre-populated map, +1: the last timed frame stages its successor
    stream = torch.cuda.Stream(device=dev)
    la = not args.no_lookahead
    do_flush = not args.no_flush
    cfg = capi.default_config(K.width, K.height, K.fx, K.fy, K.cx, K.cy, capacity=cap, time_delta=BIG, device=local)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if dist is not None:
            multi.barrier(dist, dev)
        torch.cuda.synchronize(dev)

    rgb_d = torch.from_numpy(rgb).to(dev)
    depth_d = torch.from_numpy(depth.view(np.int16)).to(dev)
    torch.cuda.synchronize(dev)

    # ---------------- value: inputs resident in HBM ----------------
    ctx = capi.Context(cfg, stream=stream.cuda_stream)
    first = 0
    n_resident = 0
    if resident:
        n_resident = populate_map(ctx, K, resident, seed, rgb[0], depth[0])
        first = 1
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    # (the warm-up frames run inside timed_sequence, before its timed loop)
    frame_ms, t_wall = timed_sequence(ctx, torch, stream, dev, flush, rgb, depth, rgb_d, depth_d, first, args.warmup, args.steps, la, do_flush, False)
    barrier()
    launches = timed_sequence.last_launches
    dev_ms = float(sum(frame_ms))
    n_surfels = ctx.map_count()
    pose = ctx.get_pose()
    if args.dump_outputs and rank == 0:
        dump_outputs(ctx, args.dump_outputs)

    # ---------------- roofline: ICP reduction at level 0, cold L2 ----------------
    roof = icp_roofline(ctx, stream, flush, K, rgb, depth, local)
    stages = map_stage_rooflines(ctx, torch, stream, flush, K) if resident else None
    ctx.close()

    # ---------------- e2e: host buffers through the public call ----------------
    ctx2 = capi.Context(cfg, stream=stream.cuda_stream)
    if resident:
        populate_map(ctx2, K, resident, seed, rgb[0], depth[0])
    barrier()
    e2e_list, _ = timed_sequence(ctx2, torch, stream, dev, flush, rgb, depth, rgb_d, depth_d, first, args.warmup, args.steps, la, do_flush, True)
    e2e_s = float(sum(e2e_list))
    barrier()
    pose2 = ctx2.get_pose()
    ctx2.close()

    # ---------------- the same without look-ahead (plain per-frame calls), fewer frames ----------------
    nola = None
    if not args.quick:
        k_n = min(args.steps, 60)
        w_n = min(args.warmup, 10)
        c3 = capi.Context(cfg, stream=stream.cuda_stream)
        if resident:
            populate_map(c3, K, resident, seed, rgb[0], depth[0])
        ms3, _ = timed_sequence(c3, torch, stream, dev, flush, rgb, depth, rgb_d, depth_d, first, w_n, k_n, False, do_flush, False)
        c3.close()
        c4 = capi.Context(cfg, stream=stream.cuda_stream)
        if resident:
            populate_map(c4, K, resident, seed, rgb[0], depth[0])
        s4, _ = timed_sequence(c4, torch, stream, dev, flush, rgb, depth, rgb_d, depth_d, first, w_n, k_n, False, do_flush, True)
        c4.close()
        nola = {"value": k_n / (sum(ms3) / 1000.0), "e2e": k_n / sum(s4), "unit": "frames/s per GPU", "frames": k_n,
                "note": "plain ef_process_frame[_device] calls: frame i+1 is not available while frame i runs"}
    clocks = sampler.stop()  # sampled across the value, roofline and e2e loops
    del rgb_d, depth_d

    # max over ranks, whole-job aggregate (elasticfusion_b200/multi.py)
    if dist is not None:
        agg_v = multi.aggregate_throughput(dist, args.steps, dev_ms / 1000.0, dev)
        agg_e = multi.aggregate_throughput(dist, args.steps, e2e_s, dev)
    else:
        agg_v = {"frames": args.steps, "seconds": dev_ms / 1000.0, "fps": args.steps / (dev_ms / 1000.0)}
        agg_e = {"frames": args.steps, "seconds": e2e_s, "fps": args.steps / e2e_s}
    if rank != 0:
        return
    hbm, peak_src = load_peaks()
    out = {
        "metric": METRIC, "value": agg_v["fps"], "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": agg_v["seconds"] * 1000.0 / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(wl_name, args.steps, world, la, do_flush, int(n_surfels), surfels_resident_at_start=int(n_resident)),
        "e2e": {"value": agg_e["fps"], "unit": "frames/s", "h2d_bytes_per_step": int(K.width * K.height * 5),
                "d2h_bytes_per_step": 132, "ms_per_step": agg_e["seconds"] * 1000.0 / args.steps},
        "gpu_launches": int(round(launches)), "launches_per_frame": launches / args.steps,
        "clocks": clocks, "roofline": dict(roof, peak=hbm, frac=roof["achieved"] / hbm, peak_source=peak_src),
        "frame_ms": {"median": statistics.median(frame_ms), "p10": float(np.percentile(frame_ms, 10)), "p90": float(np.percentile(frame_ms, 90))},
        "wall_s_value_loop": t_wall, "wall_fps_value_loop": args.steps / t_wall, "pose_check": float(np.abs(pose - pose2).max()),
    }
    roof["full_iteration"]["frac"] = roof["full_iteration"]["achieved"] / hbm
    if nola:
        out["no_lookahead"] = nola
    if stages:
        for s in stages.values():
            s["frac"] = s["achieved"] / hbm
        out["map_stage_rooflines"] = stages
    if world == 1 and not args.quick and args.workload == "640x480":
        out.update(extras_single_gpu(args, torch, capi, stream, dev, flush, local, hbm, peak_src))
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_baseline(K, rgb, depth, cap)
        out["cpu_baseline"] = cb
        if cb.get("tracking_ms_per_frame"):
            ours = tracking_stage_ms(capi, stream, K, rgb, depth, local, cap)
            out["tracking_only"] = {"ours_ms": ours, "reference_ms": cb["tracking_ms_per_frame"], "ratio": cb["tracking_ms_per_frame"] / ours,
                                    "what": ("ours: CUDA-event time of the stages RGBDOdometry::init* + getIncrementalTransformation cover (live + model "
                                             "pyramids, SO(3) loop, Sobel + candidates, 19 Gauss-Newton iterations, finish), no look-ahead, median per frame; "
                                             "reference: the reference's own kernels and host loop (oracle/_ref), wall clock per frame")}
    print(json.dumps(out))


def extras_single_gpu(args, torch, capi, stream, dev, flush, local, hbm, peak_src):
    """Rank 0 at N=1 on the default workload: BASELINE configs[2] and the large-map workloads, bounded frame counts."""
    res = {}
    # --- 1280x960, map grown from the sequence (configs[2]) + the roofline kernel at that size
    Kh, cap_h, _, name_h = workload("1280x960")
    k_h, w_h = 40, 8
    rgb_h, depth_h = make_frames(Kh, k_h + w_h + 2, 42)
    rgb_hd = torch.from_numpy(rgb_h).to(dev)
    depth_hd = torch.from_numpy(depth_h.view(np.int16)).to(dev)
    cfg_h = capi.default_config(Kh.width, Kh.height, Kh.fx, Kh.fy, Kh.cx, Kh.cy, capacity=cap_h, time_delta=BIG, device=local)
    c = capi.Context(cfg_h, stream=stream.cuda_stream)
    ms, _ = timed_sequence(c, torch, stream, dev, flush, rgb_h, depth_h, rgb_hd, depth_hd, 0, w_h, k_h, True, True, False)
    roof_hi = icp_roofline(c, stream, flush, Kh, rgb_h, depth_h, local)
    n_h = c.map_count()
    c.close()
    c = capi.Context(cfg_h, stream=stream.cuda_stream)
    es, _ = timed_sequence(c, torch, stream, dev, flush, rgb_h, depth_h, rgb_hd, depth_hd, 0, w_h, k_h, True, True, True)
    c.close()
    res["value_1280x960"] = {"value": k_h / (sum(ms) / 1000.0), "e2e": k_h / sum(es), "unit": "frames/s", "frames": k_h, "warmup": w_h,
                             "workload": name_h, "surfels_at_end": int(n_h), "ms_per_step": sum(ms) / k_h}
    roof_hi["full_iteration"]["frac"] = roof_hi["full_iteration"]["achieved"] / hbm
    res["roofline_1280x960"] = dict(roof_hi, peak=hbm, frac=roof_hi["achieved"] / hbm, peak_source=peak_src)
    # --- maps at their stated size
    large = {}
    for name, (Kx, rgb_x, depth_x, rgb_xd, depth_xd) in (("640x480-5M", (None,) * 5), ("1280x960-20M", (Kh, rgb_h, depth_h, rgb_hd, depth_hd))):
        Kw, cap_w, resident, desc = workload(name)
        k_w, w_w = 40, 8
        if Kx is None:
            rgb_x, depth_x = make_frames(Kw, k_w + w_w + 2, 42)
            rgb_xd = torch.from_numpy(rgb_x).to(dev)
            depth_xd = torch.from_numpy(depth_x.view(np.int16)).to(dev)
        cfg_w = capi.default_config(Kw.width, Kw.height, Kw.fx, Kw.fy, Kw.cx, Kw.cy, capacity=cap_w, time_delta=BIG, device=local)
        c = capi.Context(cfg_w, stream=stream.cuda_stream)
        n0 = populate_map(c, Kw, resident, 42, rgb_x[0], depth_x[0])
        ms, _ = timed_sequence(c, torch, stream, dev, flush, rgb_x, depth_x, rgb_xd, depth_xd, 1, w_w, k_w, True, True, False)
        n1 = c.map_count()
        stages = map_stage_rooflines(c, torch, stream, flush, Kw)
        for s in stages.values():
            s["frac"] = s["achieved"] / hbm
        c.close()
        c = capi.Context(cfg_w, stream=stream.cuda_stream)
        populate_map(c, Kw, resident, 42, rgb_x[0], depth_x[0])
        es, _ = timed_sequence(c, torch, stream, dev, flush, rgb_x, depth_x, rgb_xd, depth_xd, 1, w_w, k_w, True, True, True)
        c.close()
        large[name] = {"value": k_w / (sum(ms) / 1000.0), "e2e": k_w / sum(es), "unit": "frames/s", "frames": k_w, "warmup": w_w, "workload": desc,
                       "surfels_resident_at_start": int(n0), "surfels_at_end": int(n1), "ms_per_step": sum(ms) / k_w, "peak": hbm,
                       "map_stage_rooflines": stages}
    res["large_map"] = large
    return res


def map_stage_rooflines(ctx, torch, stream, flush, K):
    """The full-map passes of one frame, each timed alone on the resident map with CUDA events on the launching stream, L2 flushed
    before every sample (the maps exceed L2 anyway at 5 M / 20 M). achieved = algorithmic bytes / time:
    index map 32 B/surfel + 52 B/pixel; clean 48 B/surfel read when nothing moves, 96 B/surfel when the whole map shifts down by
    one (a surfel near the start is culled); raycast 32 B/surfel + 16 B per surfel that survives the vertex stage (not counted)
    + 38 B/pixel."""
    n = ctx.map_count()
    npx = K.width * K.height
    tick = ctx.get_tick()

    def timed(fn, reps=7):
        ev = []
        with torch.cuda.stream(stream):
            for k in range(reps):
                flush.fill_(k)
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record(stream)
                fn()
                e.record(stream)
                ev.append((s, e))
        ctx.sync()
        return statistics.median([s.elapsed_time(e) * 1000.0 for s, e in ev])

    out = {}
    t = timed(lambda: ctx.map_predict_indices(None, tick, MAXD, BIG))
    b = 32 * n + 52 * npx
    out["index_map"] = {"kernels": "k_update_pose + k_index_scatter + k_index_resolve", "algorithmic_bytes": b, "duration_us": t, "achieved": b / t / 1e3, "unit": "GB/s"}
    t = timed(lambda: ctx.map_raycast(None, MAXD, 10.0, tick, tick, BIG, 0))
    b = 32 * n + 38 * npx
    out["raycast"] = {"kernels": "k_update_pose + k_splat_scatter + k_splat_resolve", "algorithmic_bytes": b, "duration_us": t, "achieved": b / t / 1e3, "unit": "GB/s"}
    ctx.map_predict_indices(None, tick, MAXD, BIG)
    ctx.map_clean(None, tick, 10.0, BIG, MAXD)  # settle: whatever this view culls is gone after one pass
    t = timed(lambda: ctx.map_clean(None, tick, 10.0, BIG, MAXD))
    b = 32 * ctx.map_count()  # (+16 B normal/radius for the surfels in view: not counted)
    out["clean_static"] = {"kernels": "k_update_pose + k_clean_flags + k_clean_move (nothing moves: position + colour/time read, one bit written)", "algorithmic_bytes": b, "duration_us": t, "achieved": b / t / 1e3,
                           "unit": "GB/s"}
    # whole-map shift: cull surfel 1 (lastTime = -1 -> `w == -1` rule, copy_unstable.vert:119), every later surfel moves down by one
    if n > 4096:
        import ctypes as C

        ts = []
        for k in range(5):
            cnt = ctx.map_count()
            one = np.zeros((1, 12), np.float32)
            one[0, 7] = -1.0
            ctx.map_upload_range(one, 1)
            ts.append(timed(lambda: ctx.map_clean(None, tick, 10.0, BIG, MAXD), reps=1))
            assert ctx.map_count() == cnt - 1
        t = statistics.median(ts)
        b = 128 * ctx.map_count()
        out["clean_shift"] = {"kernels": "k_update_pose + k_clean_flags + k_clean_move (every surfel moves down by one: 32 B test read + 48 B read + 48 B written)", "algorithmic_bytes": b, "duration_us": t,
                              "achieved": b / t / 1e3, "unit": "GB/s"}
    return out


def icp_roofline(ctx, stream, flush, K, rgb, depth, local):
    """Duration of the dominant kernel (k_iter1: ICP residual + Jacobian + per-CTA 29-term reduction, one Gauss-Newton
    iteration of level 0) and of the complete iteration (k_iter1 + k_iter2: + final sums, 6x6 solve, pose update).

    cold (the HBM-roofline number): the launch is repeated round-robin over R independent contexts whose level-0 maps
    together exceed the 126 MB L2 (R x 14.7 MB at 640x480, R x 59 MB at 1280x960), so every launch finds its inputs evicted;
    two CUDA events bracket the whole batch on the launching stream and the average per launch is reported -- inputs larger
    than L2, no flush inside the timed region, launch gaps included as in the frame loop. warm = the same batch on one
    context (L2 resident). single_launch_event_us = one launch between two events after a 256 MiB flush (adds the latency of
    an isolated launch + two event records, ~4 us)."""
    import torch

    from elasticfusion_b200 import capi

    T = ctx.get_pose()
    R = T[:3, :3].astype(np.float32)
    t = T[:3, 3].astype(np.float32)
    ctx.icp_step_async(0, R, t, np.linalg.inv(R).astype(np.float32), t)
    ctx.sync()
    nbytes = 48 * K.width * K.height + 116
    n_ctx = max(3, int(np.ceil(260e6 / nbytes)))  # level-0 maps in rotation: twice the 126 MB L2
    cfg = capi.default_config(K.width, K.height, K.fx, K.fy, K.cx, K.cy, capacity=400_000 * (K.width // 640) ** 2, time_delta=BIG, device=local)
    ring = []
    for j in range(n_ctx):
        c = capi.Context(cfg, stream=stream.cuda_stream)
        for i in range(2):
            c.process_frame(rgb[(i + j) % len(rgb)], depth[(i + j) % len(depth)], i)
        Tj = c.get_pose()
        Rj, tj = Tj[:3, :3].astype(np.float32), Tj[:3, 3].astype(np.float32)
        c.icp_step_async(0, Rj, tj, np.linalg.inv(Rj).astype(np.float32), tj)
        c.sync()
        ring.append(c)

    def batch(ctxs, rounds, full):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        call = (lambda c: c.icp_step_async(0)) if full else (lambda c: c.icp_dense_pass_async(0))
        with torch.cuda.stream(stream):
            for c in ctxs:  # untimed pass: instruction cache, TLBs
                call(c)
            s.record(stream)
            for _ in range(rounds):
                for c in ctxs:
                    call(c)
            e.record(stream)
        e.synchronize()
        return s.elapsed_time(e) * 1000.0 / (rounds * len(ctxs))

    cold = statistics.median([batch(ring, 4, False) for _ in range(5)])
    warm = statistics.median([batch([ctx], 4 * n_ctx, False) for _ in range(5)])
    full_cold = statistics.median([batch(ring, 4, True) for _ in range(5)])
    full_warm = statistics.median([batch([ctx], 4 * n_ctx, True) for _ in range(5)])
    for c in ring:
        c.close()

    def single(fn):
        ev = []
        with torch.cuda.stream(stream):
            for k in range(20):
                flush.fill_(k)
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record(stream)
                fn()
                e.record(stream)
                ev.append((s, e))
        ctx.sync()
        return statistics.median([s.elapsed_time(e) * 1000.0 for s, e in ev])

    single_cold = single(lambda: ctx.icp_dense_pass_async(0))
    full_single = single(lambda: ctx.icp_step_async(0))
    traffic = ncu_us = None
    for name in ("r02_traffic.json", "r01_traffic.json"):
        tp = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tp):
            try:
                tj = json.load(open(tp))
                traffic = tj.get(f"k_iter1_{K.width}x{K.height}")
                ncu_us = tj.get(f"k_iter1_{K.width}x{K.height}_ncu_duration_us")
                break
            except Exception:
                traffic = None
    return {"kernel": "k_iter1 (ICP residual + Jacobian + per-CTA 29-term reduction, level 0; ef_reduce.cu)", "bound": "hbm", "unit": "GB/s",
            "achieved": nbytes / (cold * 1e-6) / 1e9, "algorithmic_bytes": nbytes, "duration_us": cold,
            "achieved_warm_l2": nbytes / (warm * 1e-6) / 1e9, "duration_warm_us": warm,
            "single_launch_event_us": single_cold,
            "full_iteration": {"kernels": "k_iter1 + k_iter2 (dense rows -> per-CTA partials -> final double sums -> 6x6 LDL^T -> pose update), ICP term only",
                               "algorithmic_bytes": nbytes, "duration_us": full_cold, "achieved": nbytes / (full_cold * 1e-6) / 1e9,
                               "duration_warm_us": full_warm, "single_launch_event_us": full_single, "unit": "GB/s"},
            "traffic": traffic, "ncu_duration_us": ncu_us,
            "units_per_launch": f"{K.width * K.height} pixels (one Gauss-Newton iteration of pyramid level 0), 48 B each",
            "timing": (f"two CUDA events on the launching stream around a batch of 4 x {n_ctx} launches rotating over {n_ctx} contexts "
                       f"({n_ctx * nbytes / 1e6:.0f} MB of level-0 maps, twice the 126 MB L2, so every launch is L2-cold), average per launch, median of 5 batches")}


def tracking_stage_ms(capi, stream, K, rgb, depth, local, cap, frames=40):
    """Median per-frame CUDA-event time of the tracking stages (EF_STAGE_TIMING=1: stages 2..6), plain calls."""
    os.environ["EF_STAGE_TIMING"] = "1"
    try:
        c = capi.Context(capi.default_config(K.width, K.height, K.fx, K.fy, K.cx, K.cy, capacity=min(cap, 3_000_000), time_delta=BIG, device=local),
                         stream=stream.cuda_stream)
    finally:
        del os.environ["EF_STAGE_TIMING"]
    rows = []
    for i in range(min(frames, len(rgb))):
        c.process_frame(rgb[i], depth[i], i)
        ms = c.stage_ms()
        if i >= 5 and len(ms) >= 7:
            rows.append(sum(ms[2:7]))
    c.close()
    return float(statistics.median(rows)) if rows else None


def cpu_baseline(K, rgb, depth, cap, seconds=15.0):
    """The reference arm on a bounded sample of the same workload, rank 0 at N=1: the reference's CUDA tracking kernels
    (oracle/_ref, when present) + the CPU oracle (OpenMP over the host cores) for the GL mapping half; pure CPU port otherwise."""
    from oracle import ef_oracle as eo

    kind, f = "port", None
    try:
        from oracle import ef_ref

        if ef_ref.available():
            f = ef_ref.HybridFusion(K, capacity=min(cap, 3_000_000))
            kind = "reference"
    except Exception:
        f = None
    if f is None:
        f = eo.Fusion(K, capacity=min(cap, 3_000_000))
    n, t0 = 0, time.perf_counter()
    while n < len(rgb) and (time.perf_counter() - t0 < seconds or n < 5):
        f.process_frame(rgb[n], depth[n], n)
        n += 1
    dt = time.perf_counter() - t0
    st = f.timers()
    out = {"value": n / dt, "unit": "frames/s", "cores": eo.get_threads(), "kind": kind,
           "sample": (f"first {n} frames of the same sequence ({dt:.1f} s): " +
                      ("reference CUDA tracking kernels (oracle/_ref) + CPU-oracle mapping (the GL half cannot run here)" if kind == "reference"
                       else "CPU oracle pipeline (oracle/_ref absent)")),
           "stages_s": st}
    if kind == "reference" and n > 1:
        out["tracking_ms_per_frame"] = (st["ref_init_s"] + st["ref_track_s"]) / (n - 1) * 1000.0  # frame 0 is not tracked
    return out


# ------------------------------------------------------------------------------------------------------------------
def usable_cores():
    """Host threads this process may really use: affinity mask capped by the cgroup CPU quota (oversubscribing OpenMP
    beyond that makes the spin-waiting teams collapse)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(p))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // p))
        except Exception:
            pass
    return max(1, n)


def run_reference(args, rank, world):
    """Reference arm: reference CUDA tracking (oracle/_ref, unmodified kernels driven like RGBDOdometry.cpp) + CPU oracle
    for the GLSL mapping half. Falls back to the pure CPU oracle when oracle/_ref is absent. Rank 0 alone runs (the other
    ranks exit without work); at N > 1 it drives N sequences concurrently, one host thread and one GPU each, the host cores
    split between them: `value` is the aggregate frames/sec of the same N-sequence job the product arm ran."""
    if rank != 0:
        return
    from elasticfusion_b200 import multi

    K, cap, resident, wl_name = workload(args.workload)
    n_total = args.warmup + args.steps
    budget_frames = min(n_total, 150 if K.width <= 640 else 48)
    try:
        from oracle import ef_ref

        have_ref = ef_ref.available()
    except Exception:
        have_ref = False
    from oracle import ef_oracle as eo

    n_seq = max(1, world)
    n_dev = 1
    if have_ref:
        import torch

        n_dev = max(1, torch.cuda.device_count())
    cores = min(usable_cores(), 32 * n_seq)  # the oracle's row-parallel loops stop scaling (and can collapse) beyond ~32 threads
    per_thread = max(1, cores // n_seq)
    w = min(args.warmup, budget_frames // 4)
    k = min(args.steps, budget_frames - w)
    frames = [make_frames(K, w + k, multi.sequence_seed(42, s)) for s in range(n_seq)]
    kind = "reference" if have_ref else "port"
    sample = ("reference CUDA tracking kernels (oracle/_ref) + CPU-oracle mapping (GL half cannot run here)" if have_ref
              else "CPU oracle pipeline (oracle/_ref absent)")
    results = [None] * n_seq
    start = threading.Barrier(n_seq + 1)
    done_warm = threading.Barrier(n_seq + 1)

    def work(s):
        eo.set_threads(per_thread)
        if have_ref:
            import torch

            torch.cuda.set_device(s % n_dev)
            runner = ef_ref.HybridFusion(K, capacity=min(cap, 3_000_000))
        else:
            runner = eo.Fusion(K, capacity=min(cap, 3_000_000))
        rgb, depth = frames[s]
        for i in range(w):
            runner.process_frame(rgb[i], depth[i], i)
        t_w = runner.timers() if hasattr(runner, "timers") else {}
        done_warm.wait()
        start.wait()
        for i in range(w, w + k):
            runner.process_frame(rgb[i], depth[i], i)
        t_e = runner.timers() if hasattr(runner, "timers") else {}
        results[s] = {kk: t_e[kk] - t_w.get(kk, 0.0) for kk in t_e}

    threads = [threading.Thread(target=work, args=(s,)) for s in range(n_seq)]
    for th in threads:
        th.start()
    done_warm.wait()
    t0 = time.perf_counter()
    start.wait()
    for th in threads:
        th.join()
    dt = time.perf_counter() - t0
    v = n_seq * k / dt
    st = results[0] or {}
    track_ms = ((st.get("ref_init_s", 0.0) + st.get("ref_track_s", 0.0)) / k * 1000.0) if have_ref else None
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": world,
           "steps": k, "warmup": w, "ms_per_step": dt / k * 1000.0, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": bench_config(wl_name, k, world, False, False, None, surfels_resident_at_start=0),
           "cpu_baseline": {"value": v, "unit": "frames/s", "cores": per_thread * n_seq, "kind": kind,
                            "sample": sample + f"; {k} frames x {n_seq} sequence(s), {per_thread} host threads each"},
           "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "tracking_ms_per_frame": track_ms, "stages_s": st}
    # the reference arm executes the mid-frame predict and runs without look-ahead / flush: say so in the shared keys
    out["config"]["skip_mid_predict"] = "0: the reference's processFrame runs predict() twice per frame"
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="640x480", choices=sorted(WORKLOADS))
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--no-lookahead", action="store_true", help="process each frame without staging its successor on the side stream")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline numbers only: no 1280x960 / large-map / no-look-ahead extras")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed frames, write the last frame's outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.warmup < 3:
        args.warmup = 3
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
        import torch
        import torch.distributed as dist_mod

        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        dist_mod.init_process_group(backend="nccl")
        dist = dist_mod
    run_ours(args, rank, world, dist)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
