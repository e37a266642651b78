#!/usr/bin/env python
"""SLIC over-segmentation per call: the library's host code (pcm_slic) against the GPU (pcm_slic_gpu).

    python tools/slic_bench.py [--reps N] [--host-reps M] [--out DIR]

Input: one seeded, textured synthetic frame per size (colour ramps plus uniform noise), the crop = the whole frame, the
reference's arguments (n_segments 250, compactness 10, sigma 1, max_iter 10, start_label 0).  Sizes (w x h): 139 x 224
(the soldier crop of the default config), 480 x 264 (frog / worm) and 1920 x 1080.

One JSON line per size: host and GPU milliseconds per call (median; wall clock around the synchronous call, the GPU one
including the crop upload and the label download), whether the two label maps are equal, and the GPU kernel time per
call split by stage, from torch.profiler in a separate run (`--out DIR` keeps its trace).  Then one line with the device
name, its power limit and its maximum SM clock.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "non-rigid-object-tracking_b200"))
import pcm  # noqa: E402,F401  (sets CUDA_DEVICE_MAX_CONNECTIONS before anything initialises CUDA)

import numpy as np  # noqa: E402

SIZES = [(139, 224), (480, 264), (1920, 1080)]
ARGS = dict(n_segments=250, compactness=10.0, sigma=1.0, max_iter=10, start_label=0)
# kernel name fragment -> stage
STAGES = [("slic_load", "smooth+lab"), ("slic_smooth", "smooth+lab"), ("slic_lab", "smooth+lab"),
          ("slic_assign", "kmeans_assign"), ("slic_settle", "kmeans_assign"), ("slic_bounds", "kmeans_update"),
          ("slic_update", "kmeans_update"), ("RadixSort", "sort (CUB)"), ("Scan", "scan (CUB)"), ("slic_", "connectivity")]


def frame_of(w, h, seed=0):
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    base = np.stack([(xx * 255) // max(w - 1, 1), (yy * 255) // max(h - 1, 1), ((xx + yy) * 3) % 256], -1)
    return np.clip(base + rng.integers(-24, 25, base.shape), 0, 255).astype(np.uint8)


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
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from pcm import capi
    if not torch.cuda.is_available():
        raise SystemExit("slic_bench.py needs a CUDA device")
    h = capi.Handle(0)
    for w, hh in SIZES:
        frame = frame_of(w, hh)
        rect = (0, 0, w, hh)
        host_ms = []
        for _ in range(a.host_reps):
            t0 = time.perf_counter()
            want, n_want = capi.slic(frame, rect, **ARGS)
            host_ms.append(1e3 * (time.perf_counter() - t0))
        for _ in range(3):                                        # warm-up: module load, buffer growth
            got, n = h.slic(frame, rect, **ARGS)
        gpu_ms = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            got, n = h.slic(frame, rect, **ARGS)
            gpu_ms.append(1e3 * (time.perf_counter() - t0))
        from torch.profiler import ProfilerActivity, profile
        n_prof = 3
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n_prof):
                h.slic(frame, rect, want_labels=False, **ARGS)
        split = {}
        for ev in prof.key_averages():
            if ev.device_type.name == "CUDA" or getattr(ev, "device_time_total", 0):
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
                split[stage_of(ev.key)] = split.get(stage_of(ev.key), 0.0) + t / 1e3 / n_prof
        if a.out:
            os.makedirs(a.out, exist_ok=True)
            prof.export_chrome_trace(os.path.join(a.out, "slic_trace_%dx%d.json" % (w, hh)))
        print(json.dumps(dict(size="%dx%d" % (w, hh), pixels=w * hh, host_ms=float(np.median(host_ms)),
                              gpu_ms=float(np.median(gpu_ms)), gpu_ms_min=float(np.min(gpu_ms)),
                              speedup=float(np.median(host_ms) / np.median(gpu_ms)),
                              equal=bool(n == n_want and np.array_equal(got, want)), n_labels=int(n),
                              gpu_kernel_ms_by_stage={k: round(v, 4) for k, v in sorted(split.items())})), flush=True)
    h.close()
    print(json.dumps(device_info(0)), flush=True)


if __name__ == "__main__":
    main()
