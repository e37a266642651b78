#!/usr/bin/env python
"""Felzenszwalb over-segmentation per call: the library's host code (pcm_felzenszwalb) against the GPU
(pcm_felzenszwalb_gpu).

    python tools/felzenszwalb_bench.py [--reps N] [--host-reps M] [--out DIR]

Input: SegTrack2 content at the sizes (w x h) the reference meets -- 139 x 224 (the soldier crop of the default config),
300 x 240 (a bmx crop), 480 x 264 (a whole frog frame) -- and 1920 x 1080 (a parachute frame resized), with the
reference's arguments (scale 100, sigma 0.5, min_size 50).

One JSON line per size: host and GPU milliseconds per call (median; wall clock around the synchronous call, the GPU one
including the crop upload and the label download), whether the two label maps are equal, the round counts of the merge
and min-size passes, and the GPU kernel time per call split by stage, from torch.profiler in a separate run (`--out DIR`
keeps its trace).  Then one line with the device name, its power limit and its maximum SM clock.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "non-rigid-object-tracking_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pcm  # noqa: E402,F401  (sets CUDA_DEVICE_MAX_CONNECTIONS before anything initialises CUDA)

import cv2 as cv  # noqa: E402
import numpy as np  # noqa: E402

ARGS = dict(scale=100, sigma=0.5, min_size=50)
# kernel name fragment -> stage
STAGES = [("slic_load", "smoothing"), ("slic_smooth", "smoothing"), ("fz_cost", "costs"), ("RadixSort", "sort (CUB)"),
          ("fz_init", "merge rounds"), ("fz_rounds_kernel<false>", "merge rounds"), ("fz_gather", "gather"),
          ("fz_rounds_kernel<true>", "min-size rounds"), ("qs_", "labels")]


def inputs():
    """(name, frame, rect) per size"""
    from helpers import read_video
    para = cv.resize(read_video("Video", "parachute")[5], (1920, 1080), interpolation=cv.INTER_LINEAR)
    return [("soldier crop", read_video("Video", "soldier")[0], (300, 0, 139, 224)),
            ("bmx crop", read_video("Video", "bmx")[10], (200, 60, 300, 240)),
            ("frog frame", read_video("Video", "frog")[0], (0, 0, 480, 264)),
            ("parachute 1080p", np.ascontiguousarray(para), (0, 0, 1920, 1080))]


def device_info(index=0):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit, clock = [s.strip() for s in out.split(",")]
        return dict(device=name, power_limit_w=float(limit), max_sm_clock_mhz=float(clock))
    except (OSError, ValueError, subprocess.TimeoutExpired):
        return dict(device=None, power_limit_w=None, max_sm_clock_mhz=None)


def stage_of(name):
    for frag, stage in STAGES:
        if frag in name:
            return stage
    return "other"


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--host-reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from pcm import capi
    if not torch.cuda.is_available():
        raise SystemExit("felzenszwalb_bench.py needs a CUDA device")
    h = capi.Handle(0)
    for name, frame, rect in inputs():
        w, hh = rect[2], rect[3]
        host_ms = []
        for _ in range(a.host_reps):
            t0 = time.perf_counter()
            want, n_want = capi.felzenszwalb(frame, rect, **ARGS)
            host_ms.append(1e3 * (time.perf_counter() - t0))
        for _ in range(3):                                        # warm-up: module load, buffer growth
            got, n = h.felzenszwalb(frame, rect, **ARGS)
        gpu_ms = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            got, n = h.felzenszwalb(frame, rect, **ARGS)
            gpu_ms.append(1e3 * (time.perf_counter() - t0))
        rounds = h.felzenszwalb_debug_last()["rounds"]
        from torch.profiler import ProfilerActivity, profile
        n_prof = 3
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n_prof):
                h.felzenszwalb(frame, rect, want_labels=False, **ARGS)
        split = {}
        for ev in prof.key_averages():
            if ev.device_type.name == "CUDA" or getattr(ev, "device_time_total", 0):
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                split[stage_of(ev.key)] = split.get(stage_of(ev.key), 0.0) + t / 1e3 / n_prof
        if a.out:
            os.makedirs(a.out, exist_ok=True)
            prof.export_chrome_trace(os.path.join(a.out, "felzenszwalb_trace_%dx%d.json" % (w, hh)))
        print(json.dumps(dict(input=name, size="%dx%d" % (w, hh), pixels=w * hh, host_ms=float(np.median(host_ms)),
                              gpu_ms=float(np.median(gpu_ms)), gpu_ms_min=float(np.min(gpu_ms)),
                              speedup=float(np.median(host_ms) / np.median(gpu_ms)),
                              equal=bool(n == n_want and np.array_equal(got, want)), n_labels=int(n),
                              merge_rounds=rounds[0], min_size_rounds=rounds[1],
                              gpu_kernel_ms_by_stage={k: round(v, 4) for k, v in sorted(split.items())})), flush=True)
    h.close()
    print(json.dumps(device_info(0)), flush=True)


if __name__ == "__main__":
    main()
