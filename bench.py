#!/usr/bin/env python
"""bench.py — frames/sec of the whole run_vo pipeline on B200 (BASELINE.json config 5; DESIGN.md §Measurement).

A STEP is one pass of the VisualOdometry state machine (mvo_vo_add_frame, reference src/vo/vo_addFrame.cpp:10-142) over
one synthetic 150-frame 640x480 sequence, from a BLANK state: ORB extract + grid-NMS (<= 2001 keypoints) on every frame,
two-view initialisation (essential + homography RANSAC, triangulation, E/H choice), then per frame the match of the map
points in view against the frame, RANSAC PnP, the 5-frame bundle adjustment (10 LM iterations, fixed map points as
shipped), and on every large move a keyframe: match with the previous keyframe, epipolar inliers, triangulation,
pushCurrPointsToMap_, optimizeMap_.  Initialisation and keyframes are inside the timed region.

  value   frames/s with the frame images already resident in HBM (150 slots = 138 MB > the 126 MB L2)
  e2e     the same metric through the C ABI with HOST images (page-locked): the H2D copy of every frame and the D2H read
          of its pose are inside the timed region; e2e_pageable: the same from ordinary (pageable) memory, as a cv::Mat is
  --impl reference   the reference's own CPU path on the host cores over the same sequence: oracle/vo_pipeline_oracle.py =
          the same state machine over cv2 (the OpenCV the reference calls) + oracle/ba_oracle.c (g2o restated); the
          reference binary itself cannot be built here (no OpenCV C++/g2o/...)

A step is ONE call of mvo_vo_run_sequence (include/mvo.h: run_vo.cpp's main loop over frames in memory).

One JSON line on stdout (rank 0).  --dump-outputs DIR: what the last timed step returned to its caller, as .npy files (rank 0).
Launch for N > 1:
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
      --master-port P bench.py --gpus N --steps K --warmup W
Multi-GPU = independent sequences per GPU (replicas only, SURVEY.md §8e): NCCL only carries the per-rank timings
(all_reduce MAX).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT / "monocular-visual-odometry_b200" / "python"))
sys.path.insert(0, str(ROOT))

W, H = 640, 480
# frames per sequence (BASELINE config 5: >= 150); MVO_BENCH_FRAMES is a test hook (tests/test_multirank_cpu.py runs the
# reference arm on a short sequence) and shows up in config.frames_per_step
N_FRAMES = int(os.environ.get("MVO_BENCH_FRAMES", "150"))
MAX_KPTS = 2000
BA_ITERS = 10
METRIC = "VO frames/sec @ 640x480, 2000 kpts, 5-frame BA"
WORKLOAD = ("full run_vo pipeline (VisualOdometry::addFrame state machine) over one synthetic 640x480 sequence per GPU: "
            "ORB extract+grid-NMS (<=2001 kpts), two-view initialisation (E+H RANSAC, triangulation), then per frame Hamming match "
            "vs map + RANSAC PnP (2 px) + 5-frame BA (10 LM it, Huber, fixed map points as shipped), keyframe insertion + "
            "triangulation + map culling on every large move")


def bench_config():
    """The configuration both arms run, verbatim in both JSON lines."""
    return {"workload": WORKLOAD, "frames_per_step": N_FRAMES, "image": "640x480 BGR u8",
            "sequence": f"mvo_synth.room_loop_sequence(seed=rank, {N_FRAMES} frames): ray-cast textured box room, closed-loop 6-dof trajectory",
            "l2": f"inputs larger than L2: {N_FRAMES} frames x 921,600 B = {N_FRAMES * H * W * 3 / 1e6:.0f} MB > 126 MB, each read once per step"}


# Algorithmic bytes per launch of each kernel class for ONE 640x480 frame (DESIGN.md §Kernels;
# SURVEY.md §8d gives the per-frame ORB figure 1,041,660 B = BGR in + keypoints + descriptors out).
PYR_PX = 640 * 480 + 533 * 400 + 444 * 333 + 370 * 278          # 771,112 gray pixels over 4 levels
ALGO_BYTES = {
    "k_gray": 640 * 480 * 3 + 640 * 480,
    "k_resize": None,                                            # 3 launches of different size: see DESIGN.md
    "k_fast": PYR_PX + 4 * 7300,                                  # read every level once + packed candidates out
    "k_select": 2 * 4 * 7300 + 8 * 2001,
    "k_blur": None,
    "k_describe": 2001 * (31 * 31 + 512) + 2001 * (28 + 32),
    "match_kernel": 32 * (2001 + 2001) + 4 * 2001,
    "k_pnp_hypotheses": 20 * 2000 + 96 * 4096,
    "k_pnp_score": 20 * 2000 + 100 * 4096,
    "k_pnp_finish": 20 * 2000 + 4 * 4096,
    "k_ba": 10000 * 16 + 2000 * 24 + 5 * 96,
    # match-list filter (the largest member of the class): keys + in-view flags + map points in, pairs + PnP arrays out
    "k_track_glue": 2001 * (4 + 1 + 12) + 1300 * (8 + 20),
    "k_epi": 2000 * 16 + 4096 * 72,
}


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake_slowdown": 0x80, "applications_clocks_setting": 0x2, "sync_boost": 0x10}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._halt.wait(0.05)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def nvml_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
    ids = [v for v in vis.split(",") if v.strip()]
    if local_rank < len(ids) and ids[local_rank].strip().isdigit():
        return int(ids[local_rank])
    return local_rank


def pin_to_gpu_numa_node(index):
    """Run this rank's threads (main thread, extraction worker) on the cores NVML reports as local to the GPU: a tracked
    frame is a chain of small dependent launches, so launch latency across the socket boundary shows."""
    if os.environ.get("MVO_BENCH_NO_PIN"):
        return
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception:
        pass


def build_sequence(seed):
    """The rank's sequence: N_FRAMES BGR frames of the ray-cast room + ground-truth camera->world poses."""
    import mvo_synth
    frames, truth = mvo_synth.cached_room_loop_sequence(seed, N_FRAMES)
    return [mvo_synth.gray_to_bgr(f) for f in frames], [np.asarray(T) for T in truth]


def trajectory_stats(poses, truth, states):
    """ATE of the estimated trajectory from the frame the VO initialised at (similarity-aligned: monocular scale)."""
    import mvo_synth
    init = states.index(2) if 2 in states else -1
    if init < 0 or len(poses) - init < 3:
        return {"initialised_at": init, "ate_rms": None}
    err, scale = mvo_synth.trajectory_error(poses[init:], truth[init:])
    return {"initialised_at": init, "ate_rms": err, "scale": scale}


# ------------------------------------------------------------------------- multi-rank plumbing
def sequence_seed(rank):
    """Replicas only (SURVEY.md §8e): rank r runs its own independent synthetic sequence, seed = r."""
    return int(rank)


def reduce_max_ms(ms, dist, device):
    """Per-rank elapsed milliseconds -> the slowest rank's (the time the whole job took)."""
    if dist is None:
        return float(ms)
    import torch
    t = torch.tensor([ms], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def whole_job_fps(world, steps, ms):
    """Aggregate throughput: every rank ran `steps` passes over its own N_FRAMES-frame sequence in `ms` (max over ranks)."""
    return world * steps * N_FRAMES / (ms / 1e3)


# ------------------------------------------------------------------------------- reference arm
def cpu_pass(imgs):
    """One pass of the reference's CPU path (the oracle pipeline) over the sequence; returns poses, states, keyframes."""
    import mvo_synth
    from oracle import vo_pipeline_oracle as vp
    cpu = vp.CpuVo(mvo_synth.K_DEFAULT, H, W, max_number_of_keypoints=MAX_KPTS, ba_iterations=BA_ITERS, init_calc_homography=True)
    poses, states, kf = [], [], 0
    for im in imgs:
        T, info = cpu.add_frame(im)
        poses.append(T); states.append(info["state_out"]); kf += int(info["keyframe"])
    return poses, states, kf


def cpu_sample_text(cv2, n_pass, dt):
    return (f"{n_pass} pass(es) over the {N_FRAMES}-frame sequence of seed 0 ({dt:.1f} s): the run_vo state machine restated in Python "
            f"(oracle/vo_pipeline_oracle.py, libstdc++ container order) over cv2 {cv2.__version__} — ORB detect/compute, BFMatcher, "
            f"findEssentialMat/recoverPose, findHomography/decomposeHomographyMat, triangulatePoints, solvePnPRansac(100 it, 2 px, 0.999): "
            f"the OpenCV routines the reference calls — + oracle/ba_oracle.c (g2o restated, {BA_ITERS} LM it); reference binary not buildable here")


def run_reference(args, rank, world):
    """The reference's CPU path on the host cores; rank 0 only."""
    if rank != 0:
        return
    import cv2
    cores = os.cpu_count() or 1
    cv2.setNumThreads(cores)
    imgs, truth = build_sequence(0)
    for _ in range(args.warmup):
        cpu_pass(imgs[:30])                 # warm-up: page in cv2 / the oracle library (a bounded prefix per warm-up step)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        poses, states, kf = cpu_pass(imgs)
    dt = time.perf_counter() - t0
    fps = args.steps * N_FRAMES / dt
    if args.dump_outputs:
        Path(args.dump_outputs).mkdir(parents=True, exist_ok=True)
        np.save(Path(args.dump_outputs) / "poses.npy", np.asarray(poses, dtype=np.float64))
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/f32/f64", "data": "synthetic", "config": bench_config(),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cv2.getNumThreads(), "host_cores": cores,
                         "kind": "port", "sample": cpu_sample_text(cv2, args.steps, dt)},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "trajectory": dict(trajectory_stats(poses, truth, states), keyframes=kf),
    }
    print(json.dumps(line), flush=True)


def cpu_baseline():
    """The same workload on the host cores (bounded sample: one pass = 150 frames), rank 0 / N=1 only."""
    import cv2
    cores = os.cpu_count() or 1
    cv2.setNumThreads(cores)
    imgs, truth = build_sequence(0)
    cpu_pass(imgs[:20])
    t0 = time.perf_counter()
    poses, states, kf = cpu_pass(imgs)
    dt = time.perf_counter() - t0
    return {"value": N_FRAMES / dt, "unit": "frames/s", "cores": cv2.getNumThreads(), "host_cores": cores, "kind": "port",
            "sample": cpu_sample_text(cv2, 1, dt), "trajectory": dict(trajectory_stats(poses, truth, states), keyframes=kf)}


# --------------------------------------------------------------------------------------- own arm
def run_gpu(args, rank, world, local_rank):
    import torch
    import mvo_b200
    import mvo_synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this framework has no CPU path (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    pin_to_gpu_numa_node(nvml_index(local_rank))
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # NCCL's version banner off stdout: one JSON line there
        import torch.distributed as dist_mod
        dist = dist_mod
        # NCCL prints its version banner on the C-level stdout when the communicator is created (NCCL_DEBUG=VERSION/INFO in the
        # environment): file descriptor 1 points at stderr until the first collective has run, so that stdout carries one JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    stream = torch.cuda.Stream()       # non-blocking: no implicit coupling with the legacy default stream
    ctx = mvo_b200.Context(local_rank, max_keypoints=MAX_KPTS, ba_iterations=BA_ITERS)
    ctx.set_stream(stream.cuda_stream)
    K = mvo_synth.K_DEFAULT
    imgs, truth = build_sequence(sequence_seed(rank))          # one independent sequence per rank / GPU
    vo = mvo_b200.VisualOdometry(ctx, K, H, W)
    if not vo.device_resident:
        raise SystemExit("bench.py: the state machine did not select the device-resident tracking path")

    # device-resident frames (> L2) and page-locked / pageable host frames
    frame_bytes = H * W * 3
    d_frames = torch.empty((N_FRAMES, H, W, 3), dtype=torch.uint8, device="cuda")
    h_frames = [torch.from_numpy(im).pin_memory() for im in imgs]
    for s in range(N_FRAMES):
        d_frames[s].copy_(h_frames[s], non_blocking=True)
    torch.cuda.synchronize()
    h_np = [t.numpy() for t in h_frames]          # views of the pinned buffers (stable pointers)
    p_np = [np.array(im, copy=True) for im in imgs]   # ordinary (pageable) memory, as a cv::Mat from cv::imread is

    def dev_args(i):
        return (d_frames[i].data_ptr(),), dict(channels=3, stride=W * 3, on_device=True)

    def host_args(i):
        return (h_np[i],), {}

    def pageable_args(i):
        return (p_np[i],), {}

    def run_pass(args_of):
        """One step: the whole sequence from a BLANK state through mvo_vo_run_sequence — run_vo.cpp's main loop (for every image:
        addFrame, record the pose) over frames in memory; frame i+1 is handed over (look-ahead) before frame i is added."""
        vo.reset()
        a = [args_of(i) for i in range(N_FRAMES)]
        poses, infos = vo.run_sequence([x[0][0] for x in a], **a[0][1])
        return list(poses), [inf.state_out for inf in infos], sum(inf.keyframe for inf in infos), infos

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(args_of, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        last = None
        for _ in range(n):
            last = run_pass(args_of)
        e1.record(stream)
        barrier()
        return reduce_max_ms(e0.elapsed_time(e1), dist, "cuda"), last

    # warm-up (>= 3 passes), then a calibration pass with every kernel class timed to find the dominant one
    warm = max(args.warmup, 3)
    for _ in range(warm):
        run_pass(dev_args)
    names = mvo_b200.kernel_names()
    vo.timing_enable((1 << len(names)) - 1)
    vo.timing_read()
    run_pass(dev_args)
    ms_k, cnt_k = vo.timing_read()
    stages = {names[k]: {"us_per_frame": 1e3 * ms_k[k] / N_FRAMES, "launches_per_frame": float(cnt_k[k]) / N_FRAMES}
              for k in range(len(names)) if cnt_k[k]}
    dominant = max(stages, key=lambda k: stages[k]["us_per_frame"])
    vo.timing_enable(0)

    # ---- timed region: K steps, images resident in HBM, no per-kernel events ----
    sampler = ClockSampler(nvml_index(local_rank))
    sampler.start()
    launches0 = vo.kernel_launches
    ms, (poses, states, kf, infos) = timed(dev_args, args.steps)
    launches = vo.kernel_launches - launches0
    clocks = sampler.stop()
    info_last = infos[-1]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, poses, infos, mvo_b200)
    # the dominant kernel's average launch duration: CUDA events around ITS launches only, same loop, separate pass
    kd = names.index(dominant)
    vo.timing_enable(1 << kd)
    vo.timing_read()
    run_pass(dev_args)
    ms_d, cnt_d = vo.timing_read()
    dom_us = 1e3 * ms_d[kd] / max(int(cnt_d[kd]), 1)
    vo.timing_enable(0)

    # ---- e2e: host images through the C ABI, H2D + D2H inside the timed region ----
    run_pass(host_args)
    ms_e2e, _ = timed(host_args, args.steps)
    n_pg = max(1, min(args.steps, 5))
    run_pass(pageable_args)
    ms_pg, _ = timed(pageable_args, n_pg)

    by_kind = None
    extra = None
    if rank == 0:
        # where the wall time of a pass goes, by kind of frame (host clock, one extra pass)
        vo.reset()
        kinds = {}
        vo.prefetch(*dev_args(0)[0], **dev_args(0)[1])
        for i in range(N_FRAMES):
            if i + 1 < N_FRAMES:
                vo.prefetch(*dev_args(i + 1)[0], **dev_args(i + 1)[1])
            t1 = time.perf_counter()
            _, inf = vo.add_frame(*dev_args(i)[0], **dev_args(i)[1])
            dt = time.perf_counter() - t1
            kind = "first" if inf.state_in == 0 else "initialisation" if inf.state_in == 1 else "keyframe" if inf.keyframe else "tracked"
            kinds.setdefault(kind, []).append(dt)
        by_kind = {k: {"n": len(v), "ms_mean": 1e3 * float(np.mean(v)), "ms_median": 1e3 * float(np.median(v))} for k, v in kinds.items()}
        extra = bench_extras(ctx, stream, d_frames, names, torch, mvo_b200, mvo_synth)

    ok = bool(info_last.state_out == 2) and kf >= 5 and info_last.n_inliers > 30

    if rank == 0:
        peak, peak_src = _peaks()
        fps = whole_job_fps(world, args.steps, ms)
        fps_e2e = whole_job_fps(world, args.steps, ms_e2e)
        fps_pg = whole_job_fps(world, n_pg, ms_pg)
        ab = ALGO_BYTES.get(dominant)
        traffic, issue = None, None
        tp = ROOT / "profiles" / "traffic.json"
        if tp.exists():
            traffic = json.loads(tp.read_text()).get(dominant)
        ip = ROOT / "profiles" / "issue.json"
        if ip.exists():
            issue = json.loads(ip.read_text()).get(dominant)
        roof = {"kernel": dominant, "bound": "hbm", "achieved": (ab / (dom_us * 1e-6) / 1e9) if ab else None,
                "peak": peak, "unit": "GB/s", "frac": (ab / (dom_us * 1e-6) / 1e9 / peak) if ab else None,
                "traffic": traffic, "us_per_launch": dom_us, "algorithmic_bytes_per_launch": ab, "peak_source": peak_src,
                "issue_frac": issue,
                "note": "single-frame launches are latency/issue-bound, not HBM-bound (DESIGN.md §Roofline); issue_frac = issue-active "
                        "share of the kernel's SM cycles x share of SMs it occupies, from the committed ncu capture (profiles/issue.json)"}
        d2h = 768 + 20 * 96
        line = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/f32/f64", "data": "synthetic", "config": bench_config(),
            "detail": {"sequences": "one independent synthetic sequence per GPU (seed = rank)",
                       "ms_per_frame": ms / args.steps / N_FRAMES,
                       "pipelining": "one mvo_vo_run_sequence call per step (run_vo.cpp's main loop in C): the next frame is handed over with "
                                     "mvo_vo_prefetch, its upload, ORB extraction and descriptor matching overlap the current frame (2 streams); results identical",
                       "device_resident": True, "tracking_ok": ok, "keyframes": int(kf),
                       "last_frame": {"keypoints": info_last.n_keypoints, "matches": info_last.n_matches,
                                      "inliers": info_last.n_inliers, "ba_frames": info_last.ba_frames, "map_points": info_last.map_points},
                       "ms_per_frame_by_kind": by_kind},
            "trajectory": dict(trajectory_stats(poses, truth, states), keyframes=int(kf)),
            "clocks": clocks,
            "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": frame_bytes * N_FRAMES, "d2h_bytes_per_step": d2h * N_FRAMES,
                    "ms_per_step": ms_e2e / args.steps, "host_memory": "page-locked (cudaHostAlloc) caller buffers"},
            "e2e_pageable": {"value": fps_pg, "unit": "frames/s", "steps": n_pg, "ms_per_step": ms_pg / n_pg,
                             "host_memory": "pageable caller buffers (as cv::imread's cv::Mat)"},
            "gpu_launches": int(launches),
            "roofline": roof,
            "stages": stages,
            "extra": extra,
        }
        if world == 1:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line), flush=True)
    vo.close()
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(out_dir, poses, infos, mvo_b200):
    """The last timed step's results as a caller of mvo_vo_run_sequence receives them: poses.npy (frames x 4 x 4 camera->world)
    and one info_<field>.npy per mvo_vo_frame_info field (frames, or frames x 16 for T_w_c_pnp), all float64 (< 100 KB)."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "poses.npy", np.asarray(poses, dtype=np.float64))
    for name, _ in mvo_b200.VoFrameInfo._fields_:
        if name != "pad":
            vals = [getattr(inf, name) for inf in infos]
            np.save(out / f"info_{name}.npy", np.array([list(v) if name == "T_w_c_pnp" else v for v in vals], dtype=np.float64))


def bench_extras(ctx, stream, d_frames, names, torch, mvo_b200, mvo_synth):
    """BASELINE configs 2-4 as stand-alone stage timings (rank 0): batched device-resident ORB extraction, RANSAC PnP on
    2000 correspondences x 4096 hypotheses, bundle adjustment of 5 frames x 2000 FREE points (Schur), 10 LM iterations."""
    out = {}
    peak_b, _ = _peaks()
    frame_bytes = H * W * 3

    def ev_time(fn, nrep):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for it in range(nrep):
            fn(it)
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / nrep        # us per call

    # ---- config 2: batched ORB (the only form of the path whose algorithmic bytes are comparable with the HBM roofline) ----
    B = 64
    cap = MAX_KPTS + 1
    d_k = torch.empty(B * cap * 28, dtype=torch.uint8, device="cuda")
    d_d = torch.empty(B * cap * 32, dtype=torch.uint8, device="cuda")
    d_c = torch.empty(B, dtype=torch.int32, device="cuda")

    def orb_batch_call(it):
        ctx.orb_extract_batch_dev(d_frames[(it % 2) * B].data_ptr(), B, H, W, 3, W * 3, frame_bytes, d_k.data_ptr(), d_d.data_ptr(),
                                  d_c.data_ptr(), cap)
    for w in range(3):
        orb_batch_call(w)
    us = ev_time(orb_batch_call, 10)                       # 2 x 64 different slots: 118 MB of input between revisits
    nk = int(d_c.sum().item())
    mvo_b200.timing_enable(ctx, (1 << len(names)) - 1)
    mvo_b200.timing_read(ctx)
    for it in range(2):
        orb_batch_call(it)
    ms_b, cnt_b = mvo_b200.timing_read(ctx)
    mvo_b200.timing_enable(ctx, 0)
    batch_stages = {names[k]: round(1e3 * ms_b[k] / (2 * B), 3) for k in range(len(names)) if cnt_b[k]}
    algo = B * (frame_bytes + 28 * (nk / B) + 32 * (nk / B))     # SURVEY §8d: BGR in + KeyPoint + descriptor out
    out["orb_batch"] = {"batch": B, "us_per_batch": us, "frames_per_s": B / (us * 1e-6), "keypoints_per_frame": nk / B,
                        "algorithmic_bytes_per_frame": algo / B, "achieved_GBps": algo / (us * 1e-6) / 1e9,
                        "hbm_frac": algo / (us * 1e-6) / 1e9 / peak_b, "kernel_us_per_frame": batch_stages,
                        "kernel_only_hbm_frac": (algo / B) / (sum(batch_stages.values()) * 1e-6) / 1e9 / peak_b if batch_stages else None,
                        "note": "mvo_orb_extract_batch_dev, 64 frames per call; integer-issue bound (FAST + BRIEF), not HBM bound — DESIGN.md §6"}

    # ---- config 3: RANSAC PnP, 2000 correspondences, 4096 hypotheses (host-array entry point, includes its copies) ----
    P, uv, _, _, _ = mvo_synth.pnp_problem(0, n=2000)
    hyp = int(ctx.params.pnp_hypotheses)
    for _ in range(3):
        ctx.solve_pnp_ransac(P, uv, mvo_synth.K_DEFAULT)
    t0 = time.perf_counter()
    nrep = 50
    for _ in range(nrep):
        rvec, tvec, inl = ctx.solve_pnp_ransac(P, uv, mvo_synth.K_DEFAULT)
    us_pnp = (time.perf_counter() - t0) / nrep * 1e6
    out["pnp_config3"] = {"correspondences": 2000, "hypotheses": int(hyp), "us_per_call": us_pnp, "reprojections_per_s": 2000 * hyp / (us_pnp * 1e-6),
                          "inliers": int(len(inl)), "timing": "host clock around mvo_solve_pnp_ransac (H2D of the points, 4 kernels, D2H of the result)"}

    # ---- config 4: BA, 5 frames x 2000 free points (Schur complement), 10 LM iterations ----
    pb = mvo_synth.ba_problem(0, n_frames=5, n_points=2000)
    ctx.set_params(ba_iterations=BA_ITERS)
    for _ in range(3):
        ctx.bundle_adjustment(pb["T_w_c"], pb["points"], pb["edge_frame"], pb["edge_point"], pb["obs"], pb["K"], fix_points=False, update_points=True)
    mvo_b200.timing_enable(ctx, 1 << names.index("k_ba"))
    mvo_b200.timing_read(ctx)
    t0 = time.perf_counter()
    nrep = 20
    for _ in range(nrep):
        _, _, st = ctx.bundle_adjustment(pb["T_w_c"], pb["points"], pb["edge_frame"], pb["edge_point"], pb["obs"], pb["K"], fix_points=False, update_points=True)
    us_ba = (time.perf_counter() - t0) / nrep * 1e6
    ms_ba, cnt_ba = mvo_b200.timing_read(ctx)
    mvo_b200.timing_enable(ctx, 0)
    kb = names.index("k_ba")
    E = len(pb["edge_frame"])
    k_us = 1e3 * ms_ba[kb] / max(int(cnt_ba[kb]), 1)
    out["ba_config4"] = {"frames": 5, "points": 2000, "edges": int(E), "lm_iterations": int(st[2]), "us_per_call": us_ba, "kernel_us": k_us,
                         "edge_iterations_per_s": E * float(st[2]) / (k_us * 1e-6), "algorithmic_GBps": ALGO_BYTES["k_ba"] * float(st[2]) / (k_us * 1e-6) / 1e9,
                         "timing": "kernel_us: CUDA events around k_ba (free points, Schur); us_per_call: host clock around mvo_bundle_adjustment"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (poses and per-frame results) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
