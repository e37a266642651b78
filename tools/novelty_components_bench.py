#!/usr/bin/env python
"""Cost of PCA novelty detection by number of components at 1080p (device-resident frames).

    python tools/novelty_components_bench.py [--steps K] [--warmup W] [--frames NF] [--features "8 hsv_lab"]

Input as in bench.py's device leg: the seeded synthetic 1920x1080 sequence (pcm/synthetic.py, seed 0), NF frames and
their truth resident on the device, crop = full frame (2 073 600 px), 16x16 grid labels, 20 trees of depth 5.  The
models are synthetic (seeded random trees, random orthonormal PCA components) so that every case uses the same
forests.  Cases: novelty on, n_components k in {1, 2, 3, 5, 8}, one model alone and two models blended.

One JSON line per case: per-frame kernel times from CUDA events around every launch (pcm_profile_read), `score` (K1)
and `novelty` (the rank-k kernel, id 7; 0 for k = 1, whose error K1 computes in-line), the whole step (all kernels of a
frame, events on the stream with per-kernel timing off), the device name and its power limit.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "non-rigid-object-tracking_b200"))
import pcm  # noqa: E402,F401  (sets CUDA_DEVICE_MAX_CONNECTIONS before anything initialises CUDA)

import numpy as np  # noqa: E402

WIDTH, HEIGHT = 1920, 1080


def random_trees(rng, n_trees, depth, F):
    trees = []
    for _ in range(n_trees):
        feature, thr, left, right, val = [], [], [], [], []

        def rec(d):
            i = len(feature)
            feature.append(0); thr.append(0.0); left.append(-1); right.append(-1); val.append(rng.random())
            if d < depth:
                feature[i] = int(rng.integers(0, F))
                thr[i] = float((rng.integers(-1, 255) + 0.5) / 255)
                left[i] = rec(d + 1)
                right[i] = rec(d + 1)
            return i
        rec(0)
        trees.append((np.array(feature, np.int32), np.array(thr), np.array(left, np.int32), np.array(right, np.int32),
                      np.array(val)))
    return trees


def power_limit(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return float(out)
    except (OSError, ValueError, subprocess.TimeoutExpired):
        return None


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--frames", type=int, default=24)
    ap.add_argument("--features", default="8 hsv_lab")
    ap.add_argument("--ks", default="1,2,3,5,8")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("novelty_components_bench.py: no CUDA device")
    from pcm import capi
    from pcm.providers import grid_segments
    from pcm.synthetic import SyntheticSequence

    dev = torch.device("cuda", 0)
    name, limit = torch.cuda.get_device_name(0), power_limit(0)
    tok = args.features.split()
    n, spaces = int(tok[0]), tok[1].split("_")
    F = 3 * (1 + 8 * n) * len(spaces)
    seq = SyntheticSequence(WIDTH, HEIGHT, 300, seed=0)
    NF = args.frames
    d_frames = torch.from_numpy(np.stack([seq.frame(i) for i in range(NF)])).to(dev)
    d_truth = torch.from_numpy(np.stack([seq.truth(i) for i in range(NF)])).to(dev)
    labels = grid_segments(seq.frame(0), 16)
    S = int(labels.max()) + 1
    d_labels = torch.from_numpy(labels).to(dev)
    d_mask = torch.zeros((HEIGHT, WIDTH), dtype=torch.uint8, device=dev)
    d_counts = torch.zeros(2, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    rng = np.random.default_rng(0)
    forests = [random_trees(rng, 20, 5, F) for _ in range(2)]
    rect = (0, 0, WIDTH, HEIGHT)
    frame_bytes = WIDTH * HEIGHT * 3

    for k in [int(v) for v in args.ks.split(",")]:
        h = capi.Handle(0)
        h.set_features(n, spaces)
        for m in range(2):
            h.add_model_arrays(100 * m, forests[m])
            q, _ = np.linalg.qr(rng.normal(size=(F, k)))
            h.set_novelty(m, rng.random(F), np.ascontiguousarray(q.T))
        h.use_own_stream()
        stream = torch.cuda.ExternalStream(h.stream, device=dev)
        for blend in (False, True):
            prm = capi.Handle.make_params(0, 1 if blend else -1, 0.6 if blend else 1.0, 0.4 if blend else 0.0, novelty=True,
                                          dilation_kernel=7, outlier_threshold=5.0)

            def step(s):
                f = s % NF
                h.update_device(d_frames.data_ptr() + f * frame_bytes, HEIGHT, WIDTH, WIDTH * 3, rect, d_labels.data_ptr(),
                                S, 0, prm, d_mask.data_ptr(), WIDTH)
                h.iou_device(d_mask.data_ptr(), WIDTH, d_truth.data_ptr() + f * HEIGHT * WIDTH, WIDTH, 1, HEIGHT, WIDTH,
                             d_counts.data_ptr())

            for s in range(args.warmup):
                step(s)
            h.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for s in range(args.steps):
                step(s)
            e1.record(stream)
            h.synchronize()
            step_ms = e0.elapsed_time(e1) / args.steps
            h.profile_enable(True)
            h.profile_read(reset=True)
            for s in range(args.steps):
                step(s)
            prof = h.profile_read(reset=True, names=capi.ALL_KERNEL_NAMES)
            h.profile_enable(False)
            per = {kk: (v[0] / args.steps) for kk, v in prof.items()}
            print(json.dumps({"features": args.features, "n_components": k, "blend": blend, "steps": args.steps,
                              "score_ms": per["score"], "novelty_ms": per["novelty"], "step_ms": step_ms,
                              "novelty_launches_per_frame": prof["novelty"][1] / args.steps,
                              "device": name, "power_limit_w": limit}), flush=True)
        h.close()


if __name__ == "__main__":
    main()
