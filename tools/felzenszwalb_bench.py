#!/usr/bin/env python
"""Felzenszwalb over-segmentation per call: the library's host code (pcm_felzenszwalb) against the GPU
(pcm_felzenszwalb_gpu), and per clip of the sweep: the host pool, single GPU calls and one GPU batch.

    python tools/felzenszwalb_bench.py [--reps N] [--host-reps M] [--out DIR] [--legs sizes,batch]

Input: SegTrack2 content at the sizes (w x h) the reference meets -- 139 x 224 (the soldier crop of the default config),
300 x 240 (a bmx crop), 480 x 264 (a whole frog frame) -- and 1920 x 1080 (a parachute frame resized), with the
reference's arguments (scale 100, sigma 0.5, min_size 50).

One JSON line per size: host and GPU milliseconds per call (median; wall clock around the synchronous call, the GPU one
including the crop upload and the label download), whether the two label maps are equal, the round counts of the merge
and min-size passes, and the GPU kernel time per call split by stage, from torch.profiler in a separate run (`--out DIR`
keeps its trace).

The batch leg, one JSON line per clip (soldier, bmx, frog, worm), on the crops the sweep builds (ClipContext.schedule with
config_benchmark.yaml): seconds for the whole clip with the host pool the sweep used before the batch (16 threads of
capi.felzenszwalb), with one pcm_felzenszwalb_device call per crop, and with one pcm_felzenszwalb_device_batch call
(median of --reps, wall clock around synchronous calls); whether all three give the same maps and counts, the round counts
of the batch (the largest over its crops) and the largest and summed round counts of the single calls, and the GPU kernel
time of the batch by stage, from torch.profiler in a separate run.

Then one line with the device name, its power limit and its maximum SM clock.
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
STAGES = [("fz_load", "smoothing"), ("fz_smooth", "smoothing"), ("fz_cost", "costs"), ("RadixSort", "sort (CUB)"),
          ("fz_init", "merge rounds"), ("fz_rounds_kernel<false>", "merge rounds"), ("fz_gather", "gather"),
          ("fz_rounds_kernel<true>", "min-size rounds"), ("qs_", "labels"), ("fz_label", "labels")]
CLIPS = ["soldier", "bmx", "frog", "worm"]


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


def kernel_split(prof, n_prof):
    split = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" or getattr(ev, "device_time_total", 0):
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            split[stage_of(ev.key)] = split.get(stage_of(ev.key), 0.0) + t / 1e3 / n_prof
    return {k: round(v, 4) for k, v in sorted(split.items())}


def sizes_leg(h, a):
    from pcm import capi
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
        if a.out:
            os.makedirs(a.out, exist_ok=True)
            prof.export_chrome_trace(os.path.join(a.out, "felzenszwalb_trace_%dx%d.json" % (w, hh)))
        print(json.dumps(dict(input=name, size="%dx%d" % (w, hh), pixels=w * hh, host_ms=float(np.median(host_ms)),
                              gpu_ms=float(np.median(gpu_ms)), gpu_ms_min=float(np.min(gpu_ms)),
                              speedup=float(np.median(host_ms) / np.median(gpu_ms)),
                              equal=bool(n == n_want and np.array_equal(got, want)), n_labels=int(n),
                              merge_rounds=rounds[0], min_size_rounds=rounds[1],
                              gpu_kernel_ms_by_stage=kernel_split(prof, n_prof))), flush=True)


def batch_leg(h, a):
    """Per clip: the sweep's crops through the host pool, single device calls and one batch."""
    import ctypes as C
    from concurrent.futures import ThreadPoolExecutor
    import torch
    import yaml
    from pcm import capi, fastseq, sweep
    pkg = os.path.join(ROOT, "non-rigid-object-tracking_b200")
    with open(os.path.join(pkg, "config_benchmark.yaml")) as f:
        base = yaml.full_load(f)
    with open(os.path.join(pkg, "polygons.yaml")) as f:
        polygons = yaml.full_load(f)
    lib = capi.load_library()
    for video in CLIPS:
        cfg = sweep.sequence_config(base, polygons, video, dict(over_segmentation="felzenszwalb"),
                                    os.path.join(pkg, "Input/SegTrack2/Video"), os.path.join(pkg, "Input/SegTrack2/Truth"))
        clip = fastseq.ClipContext(cfg["input_video"], cfg["input_truth"], cfg.get("resize_factor") or 1, 0)
        bboxes, switch = clip.selections(cfg)
        _, _, rects, _ = clip.schedule(cfg, bboxes, switch)
        T = len(rects[0])
        flat = [r for fr in rects for r in fr]
        fi = [k // T for k in range(len(flat))]
        sizes = [r[2] * r[3] for r in flat]
        offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
        H, W = clip.H, clip.W
        fb = H * W * 3
        d_frames = clip.d_frames.data_ptr()
        d = torch.empty(int(offsets[-1]), dtype=torch.int32, device="cuda")
        d_one = torch.empty(int(offsets[-1]), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()

        def pool():
            with ThreadPoolExecutor(max_workers=16) as ex:
                return list(ex.map(lambda k: capi.felzenszwalb(clip.frames[fi[k]], flat[k], **ARGS), range(len(flat))))

        def serial():
            counts, n = [], C.c_int(0)
            for k, r in enumerate(flat):
                rc = lib.pcm_felzenszwalb_device(h._h, C.c_void_p(d_frames + fi[k] * fb), H, W, W * 3, (C.c_int * 4)(*r), 100.0,
                                                 0.5, 50, None, 0, C.c_void_p(d_one.data_ptr() + 4 * int(offsets[k])), C.byref(n))
                assert rc == 0, lib.pcm_last_error()
                counts.append(n.value)
            return counts

        def batch():
            return h.felzenszwalb_device_batch(d_frames, fb, fi, H, W, W * 3, flat, d.data_ptr(), offsets[:-1], **ARGS)

        def timed(fn, reps):
            out, secs = None, []
            for _ in range(reps):
                t0 = time.perf_counter()
                out = fn()
                secs.append(time.perf_counter() - t0)
            return out, float(np.median(secs))
        host, host_s = timed(pool, max(1, a.host_reps // 2))
        batch()                                                   # warm-up: module load, buffer growth
        serial()
        one_counts, serial_s = timed(serial, max(1, a.reps // 10))
        counts, batch_s = timed(batch, max(1, a.reps // 4))
        rounds = h.felzenszwalb_debug_last()["rounds"]
        got, got_one = d.cpu().numpy(), d_one.cpu().numpy()
        equal = all(counts[k] == host[k][1] == one_counts[k] and
                    np.array_equal(got[offsets[k]:offsets[k + 1]], host[k][0].reshape(-1)) and
                    np.array_equal(got_one[offsets[k]:offsets[k + 1]], host[k][0].reshape(-1)) for k in range(len(flat)))
        single_rounds = []                                        # the round counts of each single call
        n = C.c_int(0)
        for k, r in enumerate(flat):
            lib.pcm_felzenszwalb_device(h._h, C.c_void_p(d_frames + fi[k] * fb), H, W, W * 3, (C.c_int * 4)(*r), 100.0, 0.5, 50,
                                        None, 0, None, C.byref(n))
            single_rounds.append(_last_rounds(lib, h))
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            batch()
        if a.out:
            os.makedirs(a.out, exist_ok=True)
            prof.export_chrome_trace(os.path.join(a.out, "felzenszwalb_batch_trace_%s.json" % video))
        print(json.dumps(dict(clip=video, crops=len(flat), pixels=int(offsets[-1]), host_pool_16_s=host_s, serial_device_s=serial_s,
                              batch_s=batch_s, batch_vs_host_pool=host_s / batch_s, batch_vs_serial=serial_s / batch_s,
                              equal=bool(equal), batch_rounds=list(rounds),
                              single_rounds_max=[max(r[0] for r in single_rounds), max(r[1] for r in single_rounds)],
                              single_rounds_sum=[sum(r[0] for r in single_rounds), sum(r[1] for r in single_rounds)],
                              batch_kernel_ms_by_stage=kernel_split(prof, 1))), flush=True)
        clip.close()


def _last_rounds(lib, h):
    """The round counts of the last call (the smoothed image is not fetched: its shape is not tracked for raw calls)."""
    import ctypes as C
    r = (C.c_int32 * 2)()
    assert lib.pcm_felzenszwalb_debug_last(h._h, None, r) == 0
    return r[0], r[1]


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--host-reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--legs", default="sizes,batch", help="comma-separated: sizes, batch")
    a = ap.parse_args()
    import torch
    from pcm import capi
    if not torch.cuda.is_available():
        raise SystemExit("felzenszwalb_bench.py needs a CUDA device")
    legs = set(a.legs.split(","))
    h = capi.Handle(0)
    if "sizes" in legs:
        sizes_leg(h, a)
    if "batch" in legs:
        batch_leg(h, a)
    h.close()
    print(json.dumps(device_info(0)), flush=True)


if __name__ == "__main__":
    main()
