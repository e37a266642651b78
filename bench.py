#!/usr/bin/env python
"""bench.py -- PC masker frames/s at 1080p (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload: synthetic 1920x1080 BGR sequence (pcm/synthetic.py, seed 0, 300 frames),
default config.yaml params (20 trees, depth 5, "8 hsv_lab" -> 390 features/pixel,
novelty off, prior 0, dilation 7), three models at frames [0, 100, 200] with the
reference's temporal blending, tracker box (20, 20, 1880, 1040) so that the enlarged
crop is the full frame (2 073 600 px), 16x16 grid-block labels generated once.

A step = one frame through the per-frame hot path: update() (colour conversion,
star features, forest scoring, blend, superpixel decision, dilation) + the IoU of
the mask against the ground truth (computeBenchmark).

  value      device-resident: frames, labels, truth already in HBM; K steps timed with
             CUDA events on the launching stream; whole-job frames/s (all ranks)
  e2e        the same step through the public plugin API (Masker.update + IoU) with
             HOST numpy buffers, host<->device copies inside the timed region
  roofline   fused score kernel (K1): algorithmic bytes 11 B/pixel (3 B BGR read + 8 B
             float64 P(fg) written, SURVEY.md §8d) / its mean duration (CUDA events)
  cpu_baseline / --impl reference: oracle/ref_port.py (port of the reference's CPU
             path with the reference's cost structure), 1 core, bounded sample

--dump-outputs DIR writes what the last step of the `value` loop handed its caller: the
mask (DIR/mask.npy, float32 0/255) and its IoU counts (DIR/iou_counts.npy, float64
intersection and union).  Only that loop is dumped: it is the path whose speed the line
reports, and its seeded inputs are the same from run to run, so two builds compare output
for output.  The reference arm and the sweep workload refuse the option.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "non-rigid-object-tracking_b200")
sys.path.insert(0, PKG)
import pcm  # noqa: E402,F401  (sets CUDA_DEVICE_MAX_CONNECTIONS before anything initialises CUDA)

import numpy as np  # noqa: E402

WIDTH, HEIGHT, SEQ_FRAMES = 1920, 1080, 300
MODEL_FRAMES = [0, 100, 200]
TRACK_BOX = (20, 20, 1880, 1040)
ALGO_BYTES_PER_PX_K1 = 11
PARAMS = dict(n_estimators=20, max_depth=5, n_components=1, novelty_detection=False, over_segmentation="grid:16",
              features="8 hsv_lab", dilation_kernel=7, prior_weight=0.0)
CONFIG = dict(multi_selection=True, params=PARAMS)
METRIC = "PC masker frames/sec at 1080p"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML every few ms
    (nvidia-ml-py), or the `nvidia-smi --query-gpu` line of the profiling recipe if NVML is
    not importable."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, gpu_index):
        self.samples = []          # (sm_mhz, sm_max_mhz, [reason flags])
        self.stop = threading.Event()
        self.gpu = gpu_index
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(gpu_index))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.masks = [getattr(pynvml, n, 0) for n in ("nvmlClocksEventReasonHwSlowdown", "nvmlClocksEventReasonHwThermalSlowdown",
                                                          "nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksEventReasonSwPowerCap")]
            if not all(self.masks):
                self.masks = [0x8, 0x40, 0x20, 0x4]      # NVML bit values of the four reasons
        except Exception:
            self.nvml = None
        self.thread = threading.Thread(target=self.run, daemon=True)

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[i])
            except Exception:
                pass
        return i

    def sample_once(self):
        if self.nvml is not None:
            p = self.nvml
            mhz = float(p.nvmlDeviceGetClockInfo(self.handle, p.NVML_CLOCK_SM))
            try:
                bits = int(p.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                bits = int(p.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            self.samples.append((mhz, self.max_mhz, [bool(bits & m) for m in self.masks]))
        else:
            out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
            parts = [q.strip() for q in out.strip().split(",")]
            if len(parts) >= 6:
                self.samples.append((float(parts[0]), float(parts[1]), [q.lower().startswith("active") for q in parts[2:6]]))

    def run(self):
        while not self.stop.is_set():
            try:
                self.sample_once()
            except Exception:
                pass
            self.stop.wait(0.004 if self.nvml is not None else 0.1)

    def __enter__(self):
        self.thread.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.thread.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = [x[0] for x in self.samples]
        reasons = [n for i, n in enumerate(self.NAMES) if any(x[2][i] for x in self.samples)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(x[1] for x in self.samples), "reasons": reasons,
                "samples": len(self.samples), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def sequence_state(i, model_frames):
    """(current model, next model or -1, w_cur, w_next) at sequence index i
    (reference pixel_classification.py:81-87, :117-118)."""
    cur = 0
    while cur + 1 < len(model_frames) and i >= model_frames[cur + 1]:
        cur += 1
    if cur + 1 < len(model_frames):
        span = model_frames[cur + 1] - model_frames[cur]
        tmp = i - model_frames[cur]
        return cur, cur + 1, 1 - (tmp / span), tmp / span
    return cur, -1, 1.0, 0.0


def train_models(masker, seq):
    import cv2 as cv
    for f in MODEL_FRAMES:
        poly = seq.polygon(0, f)
        masker.addModel(frame=seq.frame(f), poly_roi=poly, bbox=cv.boundingRect(np.array(poly, np.int32)),
                        bbox_roni=seq.roni(), n_frame=f)


class CachedGrid:
    """16x16 grid-block labels, generated once per crop shape (SURVEY.md §8d config 2)."""

    def __init__(self, block=16):
        self.block, self.cache = block, {}

    def __call__(self, crop):
        key = crop.shape[:2]
        if key not in self.cache:
            from pcm.providers import grid_segments
            seg = grid_segments(crop, self.block)
            seg.setflags(write=False)           # the same read-only array every time: the plugin sends it to the device once
            self.cache[key] = seg
        return self.cache[key]


# ---------------------------------------------------------------------------------------
# CPU arm (oracle port): cpu_baseline of the default arm and `--impl reference`
# ---------------------------------------------------------------------------------------
def cpu_port_setup(seq, clfs):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from ref_port import RefPortMasker
    seg = CachedGrid(16)
    m = RefPortMasker(debug=False, frame=seq.frame(0), config=CONFIG, poly_roi=None, segment_fn=seg)
    for f, clf in zip(MODEL_FRAMES, clfs):
        m.models.append({"n_frame": f, "model": clf})
        m.novelty_det.append({"n_frame": f, "model": None, "threshold": 0.0})
    return m


def cpu_port_step(m, frame, truth, sample_w, sample_h, index):
    """One update() + IoU of the port on a sample_w x sample_h crop; returns seconds."""
    from ref_port import compute_benchmark
    m.index = index
    m.current_model = sequence_state(index, MODEL_FRAMES)[0]
    # tracker box whose 20 px enlargement gives exactly the sample crop at (200, 200)
    box = (220, 220, sample_w - 40, sample_h - 40)
    mask = np.zeros_like(frame)
    t0 = time.perf_counter()
    m.update(bbox=box, frame=frame, mask=mask)
    compute_benchmark(mask[:, :, 2], truth)
    return time.perf_counter() - t0


def sample_dims(px):
    """w x h (16:9-ish, multiples of 16) with about `px` pixels, capped at a quarter frame."""
    px = int(min(max(px, 16384), 960 * 540))
    h = max(64, int((px * 9 / 16) ** 0.5) // 16 * 16)
    w = max(64, (px // h) // 16 * 16)
    return min(w, 960), min(h, 540)


def sklearn_models(seq):
    """Train the three forests exactly as addModel does, on the CPU port's own features
    (used by `--impl reference`, which must not touch the CUDA library)."""
    import cv2 as cv
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from ref_port import RefPortMasker
    m = RefPortMasker(debug=False, frame=seq.frame(0), config=CONFIG, poly_roi=None, segment_fn=CachedGrid(16))
    for f in MODEL_FRAMES:
        poly = seq.polygon(0, f)
        m.addModel(frame=seq.frame(f), poly_roi=poly, bbox=cv.boundingRect(np.array(poly, np.int32)),
                   bbox_roni=seq.roni(), n_frame=f)
    return [d["model"] for d in m.models]


# ---- reference arm: every host core runs its own copy of the (single-threaded) CPU path ----
_W = {}


def _ref_worker_init(clf_blob, seed):
    """Pool initializer: each worker process owns a port masker, four frames and their truth."""
    import pickle
    from pcm.synthetic import SyntheticSequence
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    seq = SyntheticSequence(WIDTH, HEIGHT, SEQ_FRAMES, seed=seed)
    _W["m"] = cpu_port_setup(seq, pickle.loads(clf_blob))
    _W["frames"] = [seq.frame(i) for i in range(4)]
    _W["truths"] = [seq.truth(i) for i in range(4)]
    cpu_port_step(_W["m"], _W["frames"][0], _W["truths"][0], 64, 64, 0)          # numba JIT
    return True


def _ref_worker_step(job):
    s, sw, sh = job
    return cpu_port_step(_W["m"], _W["frames"][s % 4], _W["truths"][s % 4], sw, sh, s % SEQ_FRAMES)


def _ref_worker_ready(_):
    return "m" in _W


def run_reference(args, rank, world):
    """The reference's CPU implementation of the path (oracle/ref_port.py: same third-party
    calls and cost structure as maskers/pixel_classification.py:45-126) on ALL host cores: the
    path itself is single-threaded (plain numba @jit, sklearn n_jobs=None), so parallelism is
    across independent frames, one worker process per core, exactly how the reference's own
    benchmark.py:63-64 uses the machine (ThreadPool of `python main.py` processes)."""
    if rank != 0:
        return None
    import multiprocessing as mp
    import pickle
    from pcm.synthetic import SyntheticSequence
    cores = max(1, min(int(os.environ.get("PCM_REF_CORES", os.cpu_count() or 1)), 64))
    seq = SyntheticSequence(WIDTH, HEIGHT, SEQ_FRAMES, seed=0)
    log("[reference] training 3 forests with the CPU port ...")
    clfs = sklearn_models(seq)
    n_steps = args.steps + args.warmup
    # ~85 k px/s per core (BASELINE.md §2); every worker does one sample crop per step, so a
    # step lasts sample_px / 85k seconds; keep the whole run near two minutes
    # (and the float64 feature matrix of a worker, 3 120 B/px plus two transient copies, near 1 GB)
    sw, sh = sample_dims(min(85000 * 120 / max(n_steps, 1), 98304))
    ctx = mp.get_context("spawn")
    log("[reference] starting %d worker processes ..." % cores)
    with ctx.Pool(cores, initializer=_ref_worker_init, initargs=(pickle.dumps(clfs), 0)) as pool:
        assert all(pool.map(_ref_worker_ready, range(cores), chunksize=1))
        for s in range(args.warmup):
            pool.map(_ref_worker_step, [(s, sw, sh)] * cores, chunksize=1)
        t = 0.0
        for s in range(args.warmup, n_steps):
            t0 = time.perf_counter()
            pool.map(_ref_worker_step, [(s, sw, sh)] * cores, chunksize=1)
            t += time.perf_counter() - t0
    px_per_s = args.steps * cores * sw * sh / t
    value = px_per_s / (WIDTH * HEIGHT)
    sample = ("per step every one of %d worker processes runs update()+IoU on a %dx%d crop of a 1080p frame; "
              "frames/s = pixels/s of all workers / 2073600" % (cores, sw, sh))
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic",
        "config": workload_config(),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host_cores_available": os.cpu_count(),
    }
    if not args.no_sweep:
        log("[reference] sampling the CPU port of the sweep ...")
        try:
            out["sweep"] = cpu_sweep_sample(cores)
        except Exception as e:
            out["sweep"] = {"error": "%s: %s" % (type(e).__name__, e)}
    return out


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy, so that two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def workload_config():
    return {"workload": "synthetic 1920x1080 BGR sequence, 300 frames, crop = full frame (2073600 px), "
                        "3 models @ [0,100,200] blended, 16x16 grid labels",
            "params": PARAMS, "l2": "24 distinct resident frames (149 MB) cycled; inputs larger than the 126 MB L2",
            "parallelism": "one independent sequence per GPU (no data-path collective)"}


# ---------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)

    from maskers import getMaskerByName
    from pcm import capi
    from pcm.synthetic import SyntheticSequence

    seq = SyntheticSequence(WIDTH, HEIGHT, SEQ_FRAMES, seed=rank)
    seg = CachedGrid(16)
    t0 = time.time()
    masker = getMaskerByName("PC", debug=False, frame=seq.frame(0), config=CONFIG, poly_roi=seq.polygon(0, 0),
                             update_mask=False, segment_fn=seg, device=local_rank)
    train_models(masker, seq)
    log("[rank %d] trained %d models in %.1f s" % (rank, len(masker.models), time.time() - t0))
    h = masker.native
    NF = args.frames
    frames_h = [seq.frame(i) for i in range(NF)]
    truth_h = [seq.truth(i) for i in range(NF)]
    rect = capi.crop_rect(TRACK_BOX, HEIGHT, WIDTH)
    assert rect == (0, 0, WIDTH, HEIGHT)
    labels_h = seg(frames_h[0])
    S = int(labels_h.max()) + 1

    # ---- device-resident inputs ----------------------------------------------------------
    d_frames = torch.from_numpy(np.stack(frames_h)).to(dev)            # [NF, H, W, 3] u8
    d_truth = torch.from_numpy(np.stack(truth_h)).to(dev)              # [NF, H, W] u8
    d_labels = torch.from_numpy(labels_h).to(dev)                      # [H, W] i32
    d_mask = torch.zeros((HEIGHT, WIDTH), dtype=torch.uint8, device=dev)
    n_total = args.steps + args.warmup
    d_counts = torch.zeros((n_total, 2), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    # the handle's PRIVATE stream: only there may the next frame's colour conversion start under the previous frame's
    # last kernels (K0 "early" under programmatic dependent launch); events are recorded on it through an ExternalStream
    h.use_own_stream()
    stream = torch.cuda.ExternalStream(h.stream, device=dev)
    frame_bytes = HEIGHT * WIDTH * 3

    def device_step(s):
        cur, nxt, w0, w1 = sequence_state(s % SEQ_FRAMES, MODEL_FRAMES)
        p = capi.Handle.make_params(cur, nxt, w0, w1, novelty=False, dilation_kernel=PARAMS["dilation_kernel"],
                                    outlier_threshold=0.0, prior_weight=PARAMS["prior_weight"])
        f = s % NF
        h.update_device(d_frames.data_ptr() + f * frame_bytes, HEIGHT, WIDTH, WIDTH * 3, rect, d_labels.data_ptr(), S,
                        0, p, d_mask.data_ptr(), WIDTH)
        h.iou_device(d_mask.data_ptr(), WIDTH, d_truth.data_ptr() + f * HEIGHT * WIDTH, WIDTH, 1, HEIGHT, WIDTH,
                     d_counts.data_ptr() + 16 * s)

    def barrier():
        h.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for s in range(args.warmup):
        device_step(s)
    barrier()
    launches0 = h.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        e0.record(stream)
        for s in range(args.warmup, n_total):
            device_step(s)
        e1.record(stream)
        barrier()
    ms_total = e0.elapsed_time(e1)
    launches = h.launch_count - launches0
    if args.dump_outputs and rank == 0:
        # what the last timed step handed its caller: the mask (0 / 255) and its (intersection, union) with the truth
        dump_outputs(args.dump_outputs, {"mask": d_mask.cpu().numpy().astype(np.float32),
                                         "iou_counts": d_counts[n_total - 1].cpu().numpy().astype(np.float64)})
    if dist is not None:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    value = world * args.steps / (ms_total / 1e3)

    # ---- per-kernel timing over the same K steps (events around every launch) --------------
    h.profile_enable(True)
    h.profile_read(reset=True)
    for s in range(args.warmup, n_total):
        device_step(s)
    prof = h.profile_read(reset=True)
    h.profile_enable(False)
    k1_ms = prof["score"][0] / max(prof["score"][1], 1)
    step_kernel_ms = sum(v[0] for v in prof.values()) / max(prof["score"][1], 1)
    peak, peak_src = measured_peak_gbs()
    achieved = ALGO_BYTES_PER_PX_K1 * WIDTH * HEIGHT / (k1_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "score_kernel (fused convert+features+forest)", "achieved": achieved,
                "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "k1_ms": k1_ms, "kernel_share_of_step": k1_ms / step_kernel_ms if step_kernel_ms else None,
                "per_kernel_ms": {k: (v[0] / v[1] if v[1] else 0.0) for k, v in prof.items()},
                "limiter": "shared-memory instruction rate (1 LDS/clk/SM; 9.07 LDS per pixel-tree), see DESIGN.md section 4"}
    # the bound that actually binds K1: one shared-memory instruction per clock per SM.  Trees walked per pixel, averaged
    # over the timed steps (two blended 20-tree forests up to frame 199 of the sequence, one afterwards)
    trees = [PARAMS["n_estimators"] * (2 if sequence_state(s % SEQ_FRAMES, MODEL_FRAMES)[1] >= 0 else 1)
             for s in range(args.warmup, n_total)]
    sm_mhz = clocks.summary().get("sm_mhz") or 1965.0
    sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    lds_ms = 1e3 * WIDTH * HEIGHT * (sum(trees) / len(trees)) * 9.07 / 32 / (sm_count * sm_mhz * 1e6)
    roofline["lds_bound"] = {"lds_per_pixel_tree": 9.07, "trees_per_pixel_mean": sum(trees) / len(trees), "sm_mhz": sm_mhz,
                             "bound_ms": lds_ms, "frac": lds_ms / k1_ms if k1_ms else None,
                             "note": "K1 against its own binding resource (profiles/r01_b_k1_instruction_mix.txt): time the "
                                     "shared-memory pipe needs at one instruction per clock per SM / measured K1 time"}
    # DRAM / L2 bytes per launch of every kernel of the chain: from the committed ncu capture of this same command
    # (tools/ncu_traffic.py -> profiles/r02_traffic.json); `traffic` is K1's DRAM bytes per launch
    traffic_file = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.isfile(traffic_file):
        try:
            tr = json.load(open(traffic_file))
            # `traffic`: K1's DRAM bytes per launch from the `ncu --set full` capture (cold L2: every plane and label byte comes
            # from HBM once); `traffic_steady_state`: the same launch inside the running chain, where they are L2 hits
            roofline["traffic"] = tr["kernels"]["score"].get("dram_bytes_cold_cache", tr["kernels"]["score"]["dram_bytes"])
            roofline["traffic_steady_state"] = tr["kernels"]["score"]["dram_bytes"]
            roofline["traffic_by_kernel"] = tr["kernels"]
            roofline["traffic_frame"] = tr["frame"]
            roofline["traffic_source"] = "profiles/r02_traffic.json (ncu, per launch)"
        except Exception:
            pass

    # sanity: the timed steps produced real masks
    counts = d_counts.cpu().numpy()
    assert counts[args.warmup:, 1].min() > 0, "empty masks/truth in the timed region"
    mean_iou = float(np.mean(counts[args.warmup:, 0] / counts[args.warmup:, 1]))

    # ---- end to end through the plugin API with host buffers -------------------------------
    h.use_own_stream()
    e2e_steps = max(3, args.e2e_steps)
    mask_h = np.zeros_like(frames_h[0])
    # the contract's e2e leg copies its inputs "from pinned host memory": the long-lived host frames and truth images
    # are page-locked once (pcm_host_register), so the library's H2D copies read them in place
    if not args.no_register:
        for a in frames_h + truth_h:
            capi.host_register(a)

    t_split = [0.0, 0.0]

    def host_step(s):
        masker.index = s % SEQ_FRAMES
        masker.current_model = sequence_state(masker.index, MODEL_FRAMES)[0]
        f = s % NF
        ta = time.perf_counter()
        masker.update(bbox=TRACK_BOX, frame=frames_h[f], mask=mask_h, color=(0, 0, 255))
        tb = time.perf_counter()
        r = h.iou_counts(mask_h[:, :, 2], truth_h[f])
        t_split[0] += tb - ta
        t_split[1] += time.perf_counter() - tb
        return r

    for s in range(3):
        host_step(s)
    barrier()
    t_split[0] = t_split[1] = 0.0
    moved0 = h.transfer_bytes
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        host_step(s)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    moved1 = h.transfer_bytes
    ms_update, ms_iou = 1e3 * t_split[0] / e2e_steps, 1e3 * t_split[1] / e2e_steps
    # the same loop with the label-chunk cache off: all four inputs travel every step
    h.set_label_cache(False)
    masker.reuse_resident_labels = False
    n2 = max(3, e2e_steps // 3) if not args.no_resent else 1
    host_step(0)
    barrier()
    moved2 = h.transfer_bytes
    t0 = time.perf_counter()
    for s in range(n2):
        host_step(s)
    torch.cuda.synchronize()
    e2e_all_s = time.perf_counter() - t0
    moved3 = h.transfer_bytes
    h.set_label_cache(True)
    masker.reuse_resident_labels = True
    if not args.no_register:
        for a in frames_h + truth_h:
            capi.host_unregister(a)
    if dist is not None:
        t = torch.tensor([e2e_all_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_all_s = float(t.item())
    npx = WIDTH * HEIGHT
    # counted by the library from the copies it issued (pcm_transfer_bytes): frame crop 3 B/px, mask
    # 1 B/px and truth 1 B/px up, mask 1 B/px down; the int32 label map (4 B/px) travels only when a
    # chunk differs from the previous call's -- this workload's 16x16 grid labels are generated once
    e2e = {"value": world * e2e_steps / e2e_s, "unit": "frames/s", "steps": e2e_steps,
           "h2d_bytes_per_step": (moved1[0] - moved0[0]) // e2e_steps, "d2h_bytes_per_step": (moved1[1] - moved0[1]) // e2e_steps,
           "labels_resent_every_step": {"value": world * n2 / e2e_all_s, "unit": "frames/s", "steps": n2,
                                        "h2d_bytes_per_step": (moved3[0] - moved2[0]) // n2,
                                        "d2h_bytes_per_step": (moved3[1] - moved2[1]) // n2},
           "ms_update": ms_update, "ms_iou": ms_iou, "host_buffers_page_locked": not args.no_register,
           "api": "maskers.getMaskerByName('PC').update(bbox, frame, mask, color) + Handle.iou_counts(mask, truth)"}

    # ---- CPU baseline (rank 0, N = 1 only) ---------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        log("[cpu_baseline] timing the CPU port on a bounded sample ...")
        clfs = sklearn_models(seq)                     # the port scores with scikit-learn's predict_proba
        pm = cpu_port_setup(seq, clfs)
        cpu_port_step(pm, frames_h[0], truth_h[0], 64, 64, 0)          # numba JIT
        sw, sh = 640, 352
        reps, tt = 0, 0.0
        while reps < 2 or (tt < 8.0 and reps < 8):
            tt += cpu_port_step(pm, frames_h[reps % NF], truth_h[reps % NF], sw, sh, reps)
            reps += 1
        cpu = {"value": reps * sw * sh / tt / npx, "unit": "frames/s", "cores": 1, "kind": "port",
               "sample": "%d update()+IoU steps on a %dx%d crop of the 1080p frame (%.1f s), scaled to full-frame "
                         "frames/s by pixel count; the reference path is single-threaded" % (reps, sw, sh, tt),
               "host_cores_available": os.cpu_count()}

    # ---- the other BASELINE.json configs, timed on rank 0 (extra keys of the line) ----------------------------
    extras = {}
    if rank == 0 and not args.no_extras:
        h.synchronize()
        for name, fn in (("default_quickshift_1080p", lambda: extra_quickshift_1080p(h, d_frames, d_truth, d_mask, NF, args)),
                         ("config4_4k", lambda: extra_config_4k(local_rank, args)),
                         ("config0_soldier", lambda: extra_config0_soldier(local_rank))):
            t0 = time.time()
            try:
                extras[name] = fn()
            except Exception as e:            # an extra must never take the headline down with it
                extras[name] = {"error": "%s: %s" % (type(e).__name__, e)}
            log("[extra] %s: %.1f s" % (name, time.time() - t0))
    if cpu is not None and not args.no_sweep:
        log("[cpu_baseline] sampling the CPU port of the sweep ...")
        try:
            cpu["sweep"] = cpu_sweep_sample(max(1, os.cpu_count() or 1))
        except Exception as e:
            cpu["sweep"] = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---- second half of BASELINE.json's metric: the benchmark.py grid sweep, sharded over the ranks ----
    sweep_rec = None
    if not args.no_sweep:
        h.synchronize()
        sweep_rec = sweep_record(args, rank, world)

    out = None
    if rank == 0:
        out = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/f64", "data": "synthetic", "config": workload_config(),
            "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
            "cpu_baseline": cpu, "mean_iou_vs_truth": mean_iou, "impl": "b200", "sweep": sweep_rec,
        }
        out.update(extras)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return out



# ---------------------------------------------------------------------------------------
# the other BASELINE.json configs (extra keys; the headline stays configs[1])
# ---------------------------------------------------------------------------------------
def extra_quickshift_1080p(h, d_frames, d_truth, d_mask, NF, args):
    """configs[1] with the reference's DEFAULT over-segmentation (config.yaml:29 quickshift) instead of the cached
    16x16 grid labels: per frame pcm_quickshift_device (12-13 k segments at 1080p) + the K-chain + IoU, device resident."""
    import torch
    from pcm import capi
    dev = d_frames.device
    rect = (0, 0, WIDTH, HEIGHT)
    noise = torch.from_numpy(np.random.RandomState(42).normal(scale=0.00001, size=(HEIGHT, WIDTH))).to(dev)
    d_labels = torch.empty((HEIGHT, WIDTH), dtype=torch.int32, device=dev)
    n_steps = min(args.steps, 40)
    d_counts = torch.zeros((n_steps + 3, 2), dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    fb, S_seen = HEIGHT * WIDTH * 3, []

    def step(s):
        cur, nxt, w0, w1 = sequence_state(s % SEQ_FRAMES, MODEL_FRAMES)
        p = capi.Handle.make_params(cur, nxt, w0, w1, novelty=False, dilation_kernel=7, outlier_threshold=0.0, prior_weight=0.0)
        f = s % NF
        S = h.quickshift_device(d_frames.data_ptr() + f * fb, HEIGHT, WIDTH, WIDTH * 3, rect, 0.5, 3, 6, noise.data_ptr(),
                                d_labels.data_ptr())
        S_seen.append(S)
        h.update_device(d_frames.data_ptr() + f * fb, HEIGHT, WIDTH, WIDTH * 3, rect, d_labels.data_ptr(), S, 0, p,
                        d_mask.data_ptr(), WIDTH)
        h.iou_device(d_mask.data_ptr(), WIDTH, d_truth.data_ptr() + f * HEIGHT * WIDTH, WIDTH, 1, HEIGHT, WIDTH,
                     d_counts.data_ptr() + 16 * s)
    for s in range(3):
        step(s)
    h.synchronize()
    t0 = time.perf_counter()
    for s in range(3, 3 + n_steps):
        step(s)
    h.synchronize()
    dt = time.perf_counter() - t0
    c = d_counts.cpu().numpy()[3:]
    return {"value": n_steps / dt, "unit": "frames/s", "ms_per_step": 1e3 * dt / n_steps, "steps": n_steps,
            "segments_per_frame": int(np.mean(S_seen)), "mean_iou_vs_truth": float(np.mean(c[:, 0] / np.maximum(c[:, 1], 1))),
            "note": "device-resident; quickshift(kernel_size=3, max_dist=6, ratio=0.5) on the GPU every frame (one host sync per "
                    "frame for the segment count) + colour planes + forests + decision + dilation + IoU"}


def extra_config_4k(device, args):
    """BASELINE.json configs[4]: synthetic 3840x2160, FOUR targets (one masker each, 800x600 boxes -> 840x640 crops, shared
    mask, main.py:130-164,286-343), 100 frames, default params, three blended models per target."""
    import cv2 as cv
    import torch
    from maskers import getMaskerByName
    from pcm import capi
    from pcm.synthetic import SyntheticSequence
    W4, H4, NT, NG, STEPS = 3840, 2160, 4, 8, 100
    dev = torch.device("cuda", device)
    seq = SyntheticSequence(W4, H4, NG, seed=1, n_targets=NT)
    frames = [seq.frame(i) for i in range(NG)]
    truths = [seq.truth(i) for i in range(NG)]
    sel_frames, n_frames = [0, 3, 6], [0, 33, 66]
    seg = CachedGrid(16)
    maskers, boxes = [], []
    for t in range(NT):
        m = getMaskerByName("PC", debug=False, frame=frames[0], config=CONFIG, poly_roi=seq.polygon(t, 0), update_mask=False,
                            segment_fn=seg, device=device)
        for f, nf in zip(sel_frames, n_frames):
            poly = seq.polygon(t, f)
            m.addModel(frame=frames[f], poly_roi=poly, bbox=cv.boundingRect(np.array(poly, np.int32)), bbox_roni=seq.roni(), n_frame=nf)
        maskers.append(m)
        cx, cy = seq.centres[t][0]
        boxes.append((int(min(max(cx - 400, 0), W4 - 800)), int(min(max(cy - 300, 0), H4 - 600)), 800, 600))
    rects = [capi.crop_rect(b, H4, W4) for b in boxes]
    labels = [seg(frames[0][r[1]:r[1] + r[3], r[0]:r[0] + r[2]]) for r in rects]
    d_frames = torch.from_numpy(np.stack(frames)).to(dev)
    d_truth = torch.from_numpy(np.stack(truths)).to(dev)
    d_labels = [torch.from_numpy(l).to(dev) for l in labels]
    d_mask = torch.zeros((H4, W4), dtype=torch.uint8, device=dev)
    d_counts = torch.zeros((STEPS + 3, NT, 2), dtype=torch.int64, device=dev)
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    for m in maskers:
        m.native.set_stream(stream.cuda_stream)
    fb = H4 * W4 * 3

    def dev_step(s):
        f = s % NG
        with torch.cuda.stream(stream):
            d_mask.zero_()
        for t, m in enumerate(maskers):
            m.index = (s - 3) % STEPS if s >= 3 else 0
            m.current_model = sequence_state(m.index, n_frames)[0]
            m.update_resident(d_frames.data_ptr() + f * fb, H4, W4, W4 * 3, rects[t], d_labels[t].data_ptr(),
                              int(labels[t].max()) + 1, 0, d_mask.data_ptr(), W4)
            m.native.iou_device(d_mask.data_ptr(), W4, d_truth.data_ptr() + f * H4 * W4, W4, 1, H4, W4,
                                d_counts.data_ptr() + 16 * (s * NT + t))
    for s in range(3):
        dev_step(s)
    stream.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for s in range(3, 3 + STEPS):
        dev_step(s)
    e1.record(stream)
    stream.synchronize()
    ms = e0.elapsed_time(e1)
    c = d_counts.cpu().numpy()[3:]
    for m in maskers:
        m.native.use_own_stream()
    # end to end: Masker.update x 4 + IoU x 4 per frame with host buffers
    mask_h = np.zeros_like(frames[0])
    E2E = 12
    for a in frames + truths:
        capi.host_register(a)

    def host_step(s):
        f = s % NG
        mask_h[:, :, 2] = 0
        for t, m in enumerate(maskers):
            m.index = s % STEPS
            m.current_model = sequence_state(m.index, n_frames)[0]
            m.update(bbox=boxes[t], frame=frames[f], mask=mask_h, color=(0, 0, 255))
            m.native.iou_counts(mask_h[:, :, 2], truths[f])
    host_step(0)
    t0 = time.perf_counter()
    for s in range(E2E):
        host_step(s)
    e2e_s = time.perf_counter() - t0
    for a in frames + truths:
        capi.host_unregister(a)
    for m in maskers:
        m.close()
    px = sum(r[2] * r[3] for r in rects)
    return {"value": STEPS / (ms / 1e3), "unit": "frames/s", "ms_per_step": ms / STEPS, "steps": STEPS,
            "targets": NT, "crop_px_per_frame": px, "updates_per_s": NT * STEPS / (ms / 1e3),
            "e2e": {"value": E2E / e2e_s, "unit": "frames/s", "steps": E2E},
            "mean_iou_vs_truth": float(np.mean(c[..., 0] / np.maximum(c[..., 1], 1))),
            "note": "device-resident value: per frame 4 x (K0..K3 on an 840x640 crop) + 4 x IoU over the whole 4K frame, one "
                    "stream; %d distinct 4K frames (%.0f MB) cycled over 100 steps" % (NG, NG * fb / 1e6)}


def extra_config0_soldier(device):
    """BASELINE.json configs[0]: SegTrack2 soldier through the main.py flow with the default config.yaml (quickshift on the
    GPU, 4 blended models, host buffers through Masker.update)."""
    from pcm.sequence import load_config, run_sequence
    out = {}
    for provider in ("auto", "truth"):
        cfg = load_config(os.path.join(PKG, "config.yaml"))
        cfg["tracker_provider"] = provider
        run_sequence(cfg, device=device)                      # warm-up (library load, first-touch allocations)
        r = run_sequence(cfg, device=device)
        out[provider] = {"frames_per_s": r["n_frames"] / r["seconds"], "seconds": r["seconds"], "n_frames": r["n_frames"],
                         "mean_iou": r["mean_iou"], "tracker": r["tracker"], "train_seconds": r["train_seconds"]}
    return {"value": out["truth"]["frames_per_s"], "unit": "frames/s", "by_tracker_provider": out,
            "note": "main.py flow (pcm.sequence.run_sequence), 528x224 clip, 32 frames; `auto` = OpenCV tracker available in this "
                    "image (the reference's cv.legacy CSRT is not), `truth` = boxes from the ground-truth clip (no tracker cost)"}


def cpu_sweep_sample(cores):
    """CPU arm of the grid sweep on a bounded sample.  The reference runs every (hyper-parameters, clip) as a
    `python main.py cfg out` subprocess on a ThreadPool(cpu_count) (benchmark.py:16-24,63-84); here the CPU port
    oracle/ref_sequence.py is launched the same way for TWO opposite corners of the hyper-parameter grid per clip (all six
    binary factors low / all high: for a cost that is additive in the factors their mean is the grid mean), truncated to a few
    frames; a sequence's full cost is extrapolated as (imports + JIT + training) + frames * seconds per frame, and the
    sweep as the sum over the 256 sequences divided by the cores (perfect packing: optimistic for the CPU)."""
    import tempfile
    import yaml
    from multiprocessing.pool import ThreadPool
    from pcm import sweep
    with open(os.path.join(PKG, "config_benchmark.yaml")) as f:
        base = yaml.full_load(f)
    with open(os.path.join(PKG, "polygons.yaml")) as f:
        polygons = yaml.full_load(f)
    lo = dict(n_estimators=20, max_depth=7, n_components=1, novelty_detection=False, over_segmentation="felzenszwalb",
              features="6 lab", dilation_kernel=7, prior_weight=0.0)
    hi = dict(n_estimators=30, max_depth=10, n_components=1, novelty_detection=True, over_segmentation="quickshift",
              features="8 hsv_lab", dilation_kernel=7, prior_weight=0.1)
    K = 4
    tmp = tempfile.mkdtemp(prefix="pcm_cpu_sweep_")
    jobs = []
    for v in sweep.VIDEOS:
        for tag, prm in (("lo", lo), ("hi", hi)):
            cfg = sweep.sequence_config(base, polygons, v, prm, os.path.join(PKG, "Input/SegTrack2/Video"),
                                        os.path.join(PKG, "Input/SegTrack2/Truth"))
            cp, op = os.path.join(tmp, "config-%s-%s.yaml" % (tag, v)), os.path.join(tmp, "results-%s-%s.csv" % (tag, v))
            with open(cp, "w") as f:
                yaml.dump(cfg, f)
            jobs.append((v, tag, cp, op))

    def run(job):
        v, tag, cp, op = job
        subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_sequence.py"), cp, op, str(K)],
                       capture_output=True, text=True, timeout=900)
        l1, l2 = open(op).read().split("\n")[:2]
        secs = float(l1.split(";")[1])
        t_imp, t_train, n = l2.split(";")
        return v, tag, float(t_imp) + float(t_train), secs / int(n)
    t0 = time.time()
    with ThreadPool(min(cores, len(jobs))) as pool:
        res = pool.map(run, jobs)
    wall = time.time() - t0
    core_s, detail = 0.0, {}
    for v, tag, fixed, per_frame in res:
        full = fixed + sweep.CLIP_FRAMES[v] * per_frame
        core_s += 32 * full
        detail["%s_%s" % (v, tag)] = {"fixed_s": round(fixed, 2), "s_per_frame": round(per_frame, 3), "sequence_s": round(full, 1)}
    return {"value": 256 / (core_s / cores), "unit": "sequences/s", "cores": cores, "kind": "port",
            "core_seconds_256_sequences": core_s, "sample_wall_s": wall, "per_sequence": detail,
            "sample": "8 sequences (4 clips x the all-low / all-high corners of the hyper-parameter grid), %d frames each, as "
                      "concurrent `python oracle/ref_sequence.py cfg out` subprocesses (the reference's benchmark.py launches "
                      "`python main.py cfg out` the same way); extrapolated to full clips and 256 sequences" % K}


def sweep_run(args, rank, world):
    import yaml
    from pcm import sweep
    with open(os.path.join(PKG, "config_benchmark.yaml")) as f:
        base = yaml.full_load(f)
    with open(os.path.join(PKG, "polygons.yaml")) as f:
        polygons = yaml.full_load(f)
    return sweep.run(base, polygons, limit=args.sweep_limit or None, max_frames=args.sweep_max_frames or None, log=log,
                     seq_workers=args.sweep_workers or None)


def sweep_record(args, rank, world):
    """`sweep` sub-record of every bench line: the reference's benchmark.py grid (:26-89), 64 hyper-parameter
    combinations x 4 SegTrack2 clips = 256 sequences, sharded over the ranks, ONE final gather."""
    summary, table = sweep_run(args, rank, world)
    if rank != 0:
        return None
    return {"metric": "grid-sweep sequences/sec", "sequences_per_s": summary["sequences_per_s"], "unit": "sequences/s",
            "seconds": summary["seconds"], "n_sequences": summary["n_sequences"], "n_gpus": world, "scaling": "strong",
            "mean_iou": float(np.nanmean(table["avg_benchmark"])) if table is not None else None,
            "tracker_provider": summary.get("tracker_provider"), "host_cores": summary["host_cores"],
            "per_rank_sequences": summary["per_rank_sequences"], "seq_workers": summary["seq_workers"],
            "train_jobs": summary["train_jobs"], "per_stage_host_s": summary.get("per_stage_host_s_rank0"),
            "data": "SegTrack2 clips shipped with the reference (soldier, frog, worm, bmx)"}


def run_sweep(args, rank, world):
    """Second half of BASELINE.json's metric: the benchmark.py HYPERPARAMS x VIDEOS grid, whole
    sequences sharded over the ranks (one process per GPU), ONE final gather of the scores."""
    summary, table = sweep_run(args, rank, world)
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return None
    return {"metric": "grid-sweep sequences/sec", "value": summary["sequences_per_s"], "unit": "sequences/s",
            "n_gpus": world, "steps": summary["n_sequences"], "warmup": 0,
            "ms_per_step": 1e3 * summary["seconds"] / max(summary["n_sequences"], 1), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8/f64", "data": "SegTrack2 clips shipped with the reference",
            "config": {"workload": "benchmark.py grid: %d of 256 sequences (64 hyper-parameter combos x soldier/frog/"
                                   "worm/bmx), sharded by forest group, one final all_gather" % summary["n_sequences"],
                       "per_rank_sequences": summary["per_rank_sequences"], "train_jobs": summary["train_jobs"], "seq_workers": summary["seq_workers"],
                       "max_frames": args.sweep_max_frames or None},
            "per_stage_host_s": summary.get("per_stage_host_s_rank0"), "tracker_provider": summary.get("tracker_provider"),
            "mean_iou": float(np.nanmean(table["avg_benchmark"])) if table is not None else None, "impl": "b200"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=24, help="distinct device-resident frames cycled (24 x 6.2 MB > L2)")
    ap.add_argument("--e2e-steps", type=int, default=40)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--e2e-only", action="store_true", help="tuning aid: shorten the device-resident leg")
    ap.add_argument("--no-resent", action="store_true", help="tuning aid: shorten the labels-resent-every-step e2e leg")
    ap.add_argument("--no-register", action="store_true", help="e2e leg: do not page-lock the host frames (every input is staged)")
    ap.add_argument("--workload", default="1080p", choices=["1080p", "sweep"],
                    help="1080p: frames/s (default, the driver's metric); sweep: benchmark.py grid, sequences/s")
    ap.add_argument("--no-extras", action="store_true", help="skip the 4K / soldier / quickshift-1080p extra keys")
    ap.add_argument("--no-sweep", action="store_true", help="skip the grid-sweep sub-record of the default workload")
    ap.add_argument("--sweep-limit", type=int, default=0, help="only the first N sequences of the 256")
    ap.add_argument("--sweep-max-frames", type=int, default=0)
    ap.add_argument("--sweep-workers", type=int, default=0, help="sequence threads per rank (0: cores_per_rank / 3, at most 6)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the mask and IoU counts of the last timed step as DIR/<name>.npy (1080p workload of the b200 arm)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "1080p"):
        ap.error("--dump-outputs needs the 1080p workload of the b200 arm")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.e2e_only:
        args.steps = min(args.steps, 3)
    # the CPU port (oracle/) caches its numba compilations on disk: in a directory of this run, never in the tree,
    # which may be read-only
    numba_cache = None
    if "NUMBA_CACHE_DIR" not in os.environ:
        numba_cache = tempfile.TemporaryDirectory(prefix="pcm_bench_numba_")
        os.environ["NUMBA_CACHE_DIR"] = numba_cache.name
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line; everything else -> stderr.  Python-level prints
    # (sklearn, masker) are redirected through sys.stdout, C-level ones (NCCL prints its version
    # banner straight to file descriptor 1) through the descriptor itself.
    real_stdout = sys.stdout
    sys.stdout.flush()
    saved_fd = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = sys.stderr
    try:
        if args.impl == "reference":
            out = run_reference(args, rank, world)
        elif args.workload == "sweep":
            out = run_sweep(args, rank, world)
        else:
            out = run_b200(args, rank, world, local_rank)
    finally:
        sys.stdout = real_stdout
        os.dup2(saved_fd, 1)
        os.close(saved_fd)
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
