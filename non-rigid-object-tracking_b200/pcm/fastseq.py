"""Clip-resident sequence driver: the flow of `pcm.sequence.run_sequence` (reference main.py:72-368) for callers
that run MANY sequences over the same clip (the benchmark.py grid: 64 hyper-parameter sets per clip).

What is shared by all sequences of a clip is computed once per rank and kept on the device (`ClipContext`):
  * the decoded frames and the ground truth (gray, cv.cvtColor(BGR2GRAY) as main.py:285);
  * the tracker boxes of every frame -- they depend on the frames and on the (known) frames at which the masker
    switches models, never on the masks (main.py:287-339);
  * the over-segmentation of every frame's crop: quickshift or SLIC on the GPU (pcm_quickshift_device_batch,
    pcm_slic_device_batch) or felzenszwalb in the library's host code (pixel_classification.py:70-75) -- a function of
    frame and crop only;
  * the SIFT keypoints / descriptors of every crop (pixel_classification.py:129-163), when a prior is asked for.
A sequence is then ONE pass that enqueues, per frame, the masker kernels (`update_resident` -> pcm_update_device)
and the IoU kernel (pcm_iou_device) on a stream and synchronises once at the end -- unless the SIFT prior is on,
which needs the previous mask on the host every frame.

Results are the ones `run_sequence` gives for the same config (tests/test_gpu_sequence.py).  PyTorch is used for
device buffers and streams only.
"""
import threading
import time

import cv2 as cv
import numpy as np

from maskers import getMaskerByName
from . import capi, providers, stages
from . import sequence as seq_mod


class _Once:
    """dict whose values are computed once, by the first thread that asks (others wait)."""

    def __init__(self):
        self.values, self.locks, self.guard = {}, {}, threading.Lock()

    def get(self, key, make):
        with self.guard:
            if key in self.values:
                return self.values[key]
            lock = self.locks.setdefault(key, threading.Lock())
        with lock:
            with self.guard:
                if key in self.values:
                    return self.values[key]
            v = make()
            with self.guard:
                self.values[key] = v
            return v


class LabelArena:
    """Per-frame label maps of one (clip, box schedule, over-segmentation) on the device, back to back."""

    def __init__(self, d_labels, offsets, n_labels, host=None):
        self.d_labels, self.offsets, self.n_labels, self.host = d_labels, offsets, n_labels, host

    def ptr(self, k):
        return self.d_labels.data_ptr() + 4 * self.offsets[k]


class Share:
    """The ranks of a `torch.distributed` job that work on the same clip: per-frame host work of the clip (felzenszwalb
    label maps, SIFT detection) is split between them -- member i of m takes entries i, i + m, ... -- and the pieces are
    combined with an all-reduce (sum into zero-initialised buffers; NCCL over NVLink on GPUs, gloo in the CPU tests)."""

    def __init__(self, dist=None, group=None, index=0, size=1):
        self.dist, self.group, self.index, self.size = dist, group, index, max(1, size)

    def mine(self, n):
        return range(self.index, n, self.size)

    def combine(self, tensor):
        if self.size > 1:
            self.dist.all_reduce(tensor, op=self.dist.ReduceOp.SUM, group=self.group)
        return tensor


class ClipContext:
    def __init__(self, video_path, truth_path, resize_factor=1, device=0, max_frames=None, host_workers=4, share=None):
        import torch
        from concurrent.futures import ThreadPoolExecutor
        self.torch = torch
        self.device = device
        self.dev = torch.device("cuda", device)
        self.host_workers = max(1, int(host_workers))
        self.share = share or Share()
        with stages.stage("decode"):
            with ThreadPoolExecutor(max_workers=2) as pool:       # clip and ground truth decode side by side
                ft = pool.submit(seq_mod.read_clip, seq_mod.resolve_path(truth_path), resize_factor) if truth_path is not None else None
                frames = seq_mod.read_clip(seq_mod.resolve_path(video_path), resize_factor)
                truths = ft.result() if ft is not None else None
        if not frames:
            raise IOError("Fatal error! no frames in %s" % video_path)
        self.frames, self.truths = frames, truths
        self.n = len(frames) if max_frames is None else min(len(frames), max_frames)
        self.H, self.W = frames[0].shape[:2]
        with stages.stage("clip_upload"):
            self.d_frames = torch.from_numpy(np.stack(frames[:self.n])).to(self.dev)
            self.n_truth = 0
            self.d_truth = None
            if truths is not None:
                self.n_truth = min(len(truths), self.n)
                gray = np.stack([cv.cvtColor(t, cv.COLOR_BGR2GRAY) for t in truths[:self.n_truth]])
                self.d_truth = torch.from_numpy(gray).to(self.dev)
            torch.cuda.synchronize(self.dev)
        self.once = _Once()
        self.handle = capi.Handle(device)            # clip-level GPU work (quickshift and SLIC label maps)
        self.handle_lock = threading.Lock()

    def close(self):
        self.handle.close()

    @staticmethod
    def selections(config):
        """(bboxes[target][selection], switch_frames) of a sequence config, as main.py:146-163 derives them."""
        multi = config.get("multi_selection")
        bboxes = [[cv.boundingRect(np.array(sel)) for k, sel in enumerate(target) if multi or k == 0] for target in config["pts"]]
        switch = [config["pts_frame_numbers"][k] for k in range(len(bboxes[0]))] if multi else [0]
        return bboxes, switch

    def prepare(self, config, kinds, want_sift):
        """Everything the sequences of this clip share, computed NOW by the calling thread: tracker boxes, the label
        maps of the over-segmentations in `kinds`, SIFT features.  With a `share` of several ranks this is a collective:
        every member must call it with the same arguments, in the same order relative to its other clips.  (The
        quickshift and SLIC maps alone are no collective -- every rank computes them on its GPU -- and may be prepared
        from another thread at the same time.)"""
        bboxes, switch = self.selections(config)
        box_key, _, rects, _ = self.schedule(config, bboxes, switch)
        if not want_sift and set(kinds) <= {"quickshift", "SLIC"}:
            for kind in sorted(kinds):
                self.labels(kind, box_key, rects)
            return
        self._collective_ok = True
        try:
            for kind in sorted(kinds):
                self.labels(kind, box_key, rects)
            if want_sift:
                self.sift(box_key, rects, workers=self.host_workers)
        finally:
            self._collective_ok = False

    def _check_collective(self, what):
        if self.share.size > 1 and not getattr(self, "_collective_ok", False):
            raise RuntimeError("%s of a clip shared by %d ranks must be computed by ClipContext.prepare()" % (what, self.share.size))

    # ---- tracker boxes ------------------------------------------------------------------------------------
    def schedule(self, config, bboxes, switch_frames, tracker_provider=None):
        """Per-frame integer boxes of every target [(x, y, w, h)], for a masker that switches to model s + 1 after
        frame switch_frames[s] - 1 (pixel_classification.py:117-126); replays main.py:287-339 without the masks.
        Returns (key, boxes[n][targets], rects[n][targets], tracker name)."""
        provider = tracker_provider or config.get("tracker_provider") or "auto"
        first = tuple(tuple(int(v) for v in b[0]) for b in bboxes)
        key = (str(provider), config.get("tracker"), first, tuple(switch_frames),
               tuple(tuple(tuple(int(v) for v in b) for b in tb) for tb in bboxes))

        def make():
            with stages.stage("tracker_boxes"):
                factory, name = seq_mod.make_tracker(config, self.frames[0], [b[0] for b in bboxes], self.truths, provider)
                tracker = factory(self.frames[0], [b[0] for b in bboxes])
                out, rects = [], []
                cur = 0
                for index in range(self.n):
                    ok, boxes = tracker.update(self.frames[index])
                    ib = [seq_mod.int_box(b) for b in boxes]
                    out.append(ib)
                    rects.append([capi.crop_rect(b, self.H, self.W) for b in ib])
                    if cur + 1 < len(switch_frames) and index + 1 >= switch_frames[cur + 1]:
                        cur += 1
                        tracker = factory(self.frames[index], [bboxes[t][cur] for t in range(len(bboxes))], index + 1)
                return out, rects, name
        boxes, rects, name = self.once.get(("boxes", key), make)
        return key, boxes, rects, name

    # ---- over-segmentation ----------------------------------------------------------------------------------
    def labels(self, kind, box_key, rects, want_host=False):
        """LabelArena of `kind` in {"quickshift", "felzenszwalb", "SLIC"} for the crops `rects` (entry k = frame k // T,
        target k % T)."""
        torch = self.torch

        def make():
            flat = [r for fr in rects for r in fr]
            sizes = [r[2] * r[3] for r in flat]
            offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
            d = torch.empty(int(offsets[-1]), dtype=torch.int32, device=self.dev)
            n_labels = []
            T = len(rects[0])
            if kind == "quickshift":
                with stages.stage("quickshift_maps"), self.handle_lock:
                    # quickshift(crop, kernel_size=3, max_dist=6, ratio=0.5, random_seed=42) (:71): the tie-breaking
                    # noise RandomState(42).normal(scale=1e-5, size=(h, w)) is the first h*w values of ONE stream
                    noise = np.random.RandomState(42).normal(scale=0.00001, size=max(sizes))
                    d_noise = torch.from_numpy(noise).to(self.dev)
                    torch.cuda.current_stream(self.dev).synchronize()
                    fb = self.H * self.W * 3
                    # (one wait per crop, on purpose: enqueueing all crops of a clip at once was measured SLOWER -- thousands of
                    # queued launches on this stream block the launches of the fitting and sequence threads, round 2;
                    # and in ONE native call: a Python loop of short calls re-takes the interpreter lock once per crop,
                    # which under the fitting threads' load cost ten times the GPU work)
                    n_labels.extend(int(v) for v in self.handle.quickshift_device_batch(
                        self.d_frames.data_ptr(), fb, [k // T for k in range(len(flat))], self.H, self.W, self.W * 3, flat,
                        0.5, 3, 6, d_noise.data_ptr(), d.data_ptr(), offsets[:len(flat)]))
                host = None
            elif kind == "SLIC":
                with stages.stage("slic_maps"), self.handle_lock:
                    # slic(crop, n_segments=250, compactness=10, sigma=1, start_label=0) (:75), one native call for the clip
                    torch.cuda.current_stream(self.dev).synchronize()
                    n_labels.extend(int(v) for v in self.handle.slic_device_batch(
                        self.d_frames.data_ptr(), self.H * self.W * 3, [k // T for k in range(len(flat))], self.H, self.W,
                        self.W * 3, flat, d.data_ptr(), offsets[:len(flat)], n_segments=250, compactness=10.0, sigma=1.0,
                        start_label=0))
                host = None
            elif kind == "felzenszwalb":
                self._check_collective("felzenszwalb label maps")
                with stages.stage("felzenszwalb_maps"):
                    from concurrent.futures import ThreadPoolExecutor

                    def one(k):          # felzenszwalb(crop, scale=100, sigma=0.5, min_size=50) (:73), frames in parallel
                        t0 = time.perf_counter()
                        out = capi.felzenszwalb(self.frames[k // T], flat[k], scale=100, sigma=0.5, min_size=50)
                        stages.add("felzenszwalb_cpu", time.perf_counter() - t0)
                        return out
                    mine = list(self.share.mine(len(flat)))
                    with ThreadPoolExecutor(max_workers=self.host_workers) as pool:
                        res = dict(zip(mine, pool.map(one, mine)))
                    flat_host = np.zeros(int(offsets[-1]), np.int32)
                    counts = np.zeros(len(flat), np.int64)
                    for k, (seg, n_seg) in res.items():
                        flat_host[offsets[k]:offsets[k + 1]] = seg.reshape(-1)
                        counts[k] = n_seg
                    d.copy_(torch.from_numpy(flat_host))
                    d_counts = torch.from_numpy(counts).to(self.dev)
                    with stages.stage("share_allreduce"):
                        self.share.combine(d)               # the other members' frames arrive here
                        self.share.combine(d_counts)
                        n_labels.extend(int(v) for v in d_counts.cpu().numpy())
                    torch.cuda.current_stream(self.dev).synchronize()
                    host = None
            else:
                raise ValueError("no clip-resident over-segmentation for %r" % kind)
            return LabelArena(d, [int(o) for o in offsets], n_labels, host)
        arena = self.once.get(("labels", kind, box_key), make)
        if want_host and arena.host is None:
            def fetch():
                flat = [r for fr in rects for r in fr]
                h = arena.d_labels.cpu().numpy()
                return [h[arena.offsets[k]:arena.offsets[k + 1]].reshape(flat[k][3], flat[k][2]) for k in range(len(flat))]
            arena.host = self.once.get(("labels_host", kind, box_key), fetch)
        return arena


class SiftStore:
    """SIFT keypoints / descriptors of every crop of a box schedule: host arrays per entry and one device copy
    (pts float32 [M, 2], descriptors uint8 [M, 128]) for pcm_prior_device."""

    def __init__(self, pts, des, d_pts, d_des, offsets):
        self.pts, self.des, self.d_pts, self.d_des, self.offsets = pts, des, d_pts, d_des, offsets

    def count(self, k):
        return self.offsets[k + 1] - self.offsets[k]

    def pts_ptr(self, k):
        return self.d_pts.data_ptr() + 8 * self.offsets[k]

    def des_ptr(self, k):
        return self.d_des.data_ptr() + 128 * self.offsets[k]


_tls = threading.local()


def _sift_detect(crop):
    """cv.SIFT_create().detectAndCompute(crop, None) (:136) -> (pts float32 [m, 2], descriptors uint8 [m, 128])."""
    if getattr(_tls, "sift", None) is None:
        _tls.sift = cv.SIFT_create()
    kps, des = _tls.sift.detectAndCompute(np.ascontiguousarray(crop), None)
    pts = np.array([k.pt for k in kps], np.float32).reshape(-1, 2)
    if des is None or len(kps) == 0:
        return pts, np.zeros((0, 128), np.uint8)
    d8 = des.astype(np.uint8)
    if not np.array_equal(d8, des):
        raise ValueError("SIFT descriptors are expected to hold integers 0..255")
    return pts, d8


def _clip_sift(self, box_key, rects, workers=4):
    """SiftStore of the crops `rects` (computed once per clip and box schedule, frames in parallel)."""
    torch = self.torch

    def make():
        from concurrent.futures import ThreadPoolExecutor
        flat = [r for fr in rects for r in fr]
        T = len(rects[0])
        self._check_collective("SIFT features")
        with stages.stage("sift_detect"):
            def one(k):
                x, y, w, h = flat[k]
                t0 = time.perf_counter()
                out = _sift_detect(self.frames[k // T][y:y + h, x:x + w])
                stages.add("sift_detect_cpu", time.perf_counter() - t0)
                return out
            mine = list(self.share.mine(len(flat)))
            with ThreadPoolExecutor(max_workers=max(1, workers)) as pool:
                res = dict(zip(mine, pool.map(one, mine)))
        counts = np.zeros(len(flat), np.int64)
        for k, (p, _) in res.items():
            counts[k] = len(p)
        d_cnt = torch.from_numpy(counts).to(self.dev)
        with stages.stage("share_allreduce"):
            counts = self.share.combine(d_cnt).cpu().numpy()
        offsets = [0] + [int(v) for v in np.cumsum(counts)]
        M = max(offsets[-1], 1)
        pts = np.zeros((M, 2), np.float32)
        des = np.zeros((M, 128), np.uint8)
        for k, (p, d) in res.items():
            pts[offsets[k]:offsets[k + 1]] = p
            des[offsets[k]:offsets[k + 1]] = d
        d_pts = torch.from_numpy(pts).to(self.dev)
        d_des = torch.from_numpy(des).to(self.dev)
        with stages.stage("share_allreduce"):
            self.share.combine(d_pts)                   # zero everywhere but on the member that detected the entry
            self.share.combine(d_des)
        torch.cuda.current_stream(self.dev).synchronize()
        if self.share.size > 1:
            pts, des = d_pts.cpu().numpy(), d_des.cpu().numpy()
        host_pts = [pts[offsets[k]:offsets[k + 1]] for k in range(len(flat))]
        host_des = [des[offsets[k]:offsets[k + 1]] for k in range(len(flat))]
        return SiftStore(host_pts, host_des, d_pts, d_des, offsets)
    return self.once.get(("sift", box_key), make)


ClipContext.sift = _clip_sift


def _precomputable(config):
    if config.get("masker") != "PC" or config.get("manual_roi_selection"):
        return False
    if config.get("masker") in (config.get("custom_trackers") or []):
        return False
    return config["params"]["over_segmentation"] in ("quickshift", "felzenszwalb", "SLIC")


def _frame_loop(clip, maskers, rects, arena, sift, d_mask, d_counts, d_pri, gpu_prior, host_prior, model_cache, cache_tag):
    """Per-frame enqueue from Python: several targets share the mask plane (main.py:130-164,286-343), or the prior is
    computed on the host (FLANN) and needs the previous mask there."""
    torch = clip.torch
    frames = clip.frames
    T = len(maskers)
    n, H, W = clip.n, clip.H, clip.W
    fb = H * W * 3
    prev_rects = [None] * T
    prev_crops = [None] * T                         # the SAME array objects the prior saw one frame earlier (SiftPrior reuse)
    for index in range(n):
        prev_masks = None
        if gpu_prior and index > 0:
            # the priors of every target read the PREVIOUS frame's mask plane: queue them before it is cleared
            for i in range(T):
                k, kp = index * T + i, (index - 1) * T + i
                x, y, w, h = rects[index][i]
                px, py, pw, ph = prev_rects[i]
                maskers[i].native.prior_device(sift.pts_ptr(kp), sift.des_ptr(kp), sift.count(kp),
                                               d_mask.data_ptr() + py * W + px, W, pw, ph,
                                               sift.pts_ptr(k), sift.des_ptr(k), sift.count(k),
                                               arena.ptr(k), w, h, arena.n_labels[k], d_pri[i].data_ptr())
        if host_prior and index > 0:
            with stages.stage("prior_mask_d2h"):
                hm = d_mask.cpu().numpy()           # waits for the previous frame; its crops are the prevForegroundMasks
            prev_masks = [hm[r[1]:r[1] + r[3], r[0]:r[0] + r[2]] for r in prev_rects]
        if index > 0:
            d_mask.zero_()                          # main.py:286: a fresh mask per frame
        for i in range(T):
            rect = rects[index][i]
            k = index * T + i
            S = arena.n_labels[k]
            pri_ptr = d_pri[i].data_ptr() if (gpu_prior and index > 0) else 0
            m = maskers[i]
            if host_prior:
                x, y, w, h = rect
                crop = frames[index][y:y + h, x:x + w]
            if prev_masks is not None:
                with stages.stage("sift_prior"):
                    pri = m.prior_fn(prev_crops[i], prev_masks[i], crop, arena.host[k], S,
                                     cache=model_cache, key=(cache_tag, i, index, rect)) \
                        if cache_tag is not None else \
                        m.prior_fn(prev_crops[i], prev_masks[i], crop, arena.host[k], S)
                d_priors = torch.from_numpy(np.ascontiguousarray(pri, np.float32)).to(clip.dev)
                pri_ptr = d_priors.data_ptr()
            m.update_resident(clip.d_frames.data_ptr() + index * fb, H, W, W * 3, rect, arena.ptr(k), S, pri_ptr,
                              d_mask.data_ptr(), W)
            prev_rects[i] = rect
            if host_prior:
                prev_crops[i] = crop
            if index < clip.n_truth:
                m.native.iou_device(d_mask.data_ptr(), W, clip.d_truth.data_ptr() + index * H * W, W, 1, H, W,
                                    d_counts.data_ptr() + 16 * k)


JOB_DTYPE = np.dtype(capi.FrameJob)


def build_jobs(m, n, rects, frames_ptr, frame_bytes, arena, sift, priors_ptr, truth_ptr, n_truth, H, W, counts_ptr):
    """The `pcm_frame_job` records of the next `n` frames of the single-target masker `m` (whose state machine is
    advanced past them), as a numpy record array laid out like the C struct: frame k of the clip at `frames_ptr`,
    crop `rects[k]`, label map k of `arena`; with `sift` (a SiftStore) frames 1.. carry the prior step; the first
    `n_truth` frames carry the IoU step (truth planes H x W at `truth_ptr`, two int64 each at `counts_ptr`).  Filled
    column by column: a per-frame Python loop over ctypes fields held the interpreter lock for ~14 us per frame, which
    the sweep's 16 sequence threads share."""
    jobs = np.zeros(n, JOB_DTYPE)
    index = np.arange(n, dtype=np.uint64)
    rect = np.asarray(rects, np.int32).reshape(n, 4)
    jobs["d_frame"] = np.uint64(frames_ptr) + index * np.uint64(frame_bytes)
    jobs["rect"] = rect
    jobs["d_labels"] = np.uint64(arena.d_labels.data_ptr()) + np.uint64(4) * np.asarray(arena.offsets[:n], np.uint64)
    jobs["n_labels"] = np.asarray(arena.n_labels[:n], np.int32)
    jobs["clear_mask"][1:] = 2
    params = m.config["params"]
    p = jobs["params"]
    p["model_cur"], p["model_next"], p["w_cur"], p["w_next"], p["outlier_threshold"] = m._frame_schedule(n)
    p["novelty"] = int(bool(params["novelty_detection"]))
    p["dilation_kernel"] = int(params["dilation_kernel"])
    p["prior_weight"] = float(params["prior_weight"])
    if sift is not None and n > 1:
        off = np.asarray(sift.offsets[:n + 1], np.int64)
        pts, des = np.uint64(sift.d_pts.data_ptr()), np.uint64(sift.d_des.data_ptr())
        start = off[:-1].astype(np.uint64)
        count = (off[1:] - off[:-1]).astype(np.int32)
        jobs["d_pts_prev"][1:], jobs["d_des_prev"][1:] = pts + np.uint64(8) * start[:-1], des + np.uint64(128) * start[:-1]
        jobs["n_prev"][1:], jobs["prev_rect"][1:] = count[:-1], rect[:-1]
        jobs["d_pts"][1:], jobs["d_des"][1:] = pts + np.uint64(8) * start[1:], des + np.uint64(128) * start[1:]
        jobs["n_cur"][1:] = count[1:]
        jobs["d_priors_out"][1:] = priors_ptr
    t = min(n, n_truth)
    if t > 0:
        jobs["d_truth"][:t] = np.uint64(truth_ptr) + index[:t] * np.uint64(H * W)
        jobs["truth_stride"][:t] = W
        jobs["truth_channels"][:t] = 1
        jobs["d_counts"][:t] = np.uint64(counts_ptr) + np.uint64(16) * index[:t]
    return jobs


def run_sequence_fast(config, clip, device=0, model_cache=None, cache_tag=None, tracker_provider=None, stream=None,
                      out_path=None):
    """`run_sequence` over a ClipContext.  `stream`: a torch.cuda.Stream owned by the calling thread (created when
    omitted); the maskers enqueue on it."""
    torch = clip.torch
    t_wall = time.time()
    if not _precomputable(config):
        raise ValueError("run_sequence_fast: this config needs pcm.sequence.run_sequence")
    params = config["params"]
    pts, frame_numbers, ronis = config.get("pts"), config.get("pts_frame_numbers"), config.get("bboxes_roni")
    frames = clip.frames
    stream = stream or torch.cuda.Stream(device=clip.dev)

    t_train = time.time()
    maskers, bboxes = [], []
    for n_target, target_selection in enumerate(pts):
        bboxes.append([])
        m = getMaskerByName("PC", debug=False, frame=frames[0], config=config, poly_roi=pts[n_target][0],
                            update_mask=config.get("update_mask"), device=device, model_cache=model_cache,
                            cache_tag=(cache_tag, n_target) if cache_tag is not None else None,
                            train_jobs=config.get("train_jobs"), fit_estimators=config.get("fit_estimators"))
        maskers.append(m)
        for n_selection, selection in enumerate(target_selection):
            if not config.get("multi_selection") and n_selection > 0:
                continue
            bbox = cv.boundingRect(np.array(selection))
            bboxes[-1].append(bbox)
            n_frame = frame_numbers[n_selection]
            if n_frame >= len(frames):
                raise IOError("Fatal error! selection frame %d beyond the clip" % n_frame)
            m.addModel(frame=frames[n_frame], poly_roi=pts[n_target][n_selection], bbox=bbox,
                       bbox_roni=ronis[n_target][n_selection] if ronis is not None else None, n_frame=n_frame)
    t_train = time.time() - t_train

    switch_frames = [md["n_frame"] for md in maskers[0].models] if config.get("multi_selection") else [0]
    box_key, boxes, rects, tracker_name = clip.schedule(config, bboxes, switch_frames, tracker_provider)
    want_prior = params["prior_weight"] != 0.0
    # prior_provider "gpu" (default): exact 2-NN matching and everything after it on the device (pcm_prior_device), SIFT
    # detection once per clip frame on the host; "flann": the reference's own FLANN matcher on the host, per frame
    gpu_prior = want_prior and (config.get("prior_provider") or "gpu") == "gpu"
    host_prior = want_prior and not gpu_prior
    arena = clip.labels(params["over_segmentation"], box_key, rects, want_host=host_prior)
    sift = clip.sift(box_key, rects, workers=clip.host_workers) if gpu_prior else None
    T = len(maskers)
    n, H, W = clip.n, clip.H, clip.W
    fb = H * W * 3

    start = time.time()
    with torch.cuda.stream(stream):
        d_mask = torch.zeros((H, W), dtype=torch.uint8, device=clip.dev)
        d_counts = torch.zeros((n * T, 2), dtype=torch.int64, device=clip.dev)
        d_priors = None
        if gpu_prior:
            d_pri = [torch.empty(max(arena.n_labels), dtype=torch.float32, device=clip.dev) for _ in range(T)]
        for m in maskers:
            m.native.set_stream(stream.cuda_stream)
        if T == 1 and not host_prior:
            # single target, everything device-side: the whole sequence is ONE native call (pcm_run_frames)
            m = maskers[0]
            jobs = build_jobs(m, n, [r[0] for r in rects[:n]], clip.d_frames.data_ptr(), fb, arena, sift if gpu_prior else None,
                              d_pri[0].data_ptr() if gpu_prior else 0,
                              clip.d_truth.data_ptr() if clip.d_truth is not None else 0, clip.n_truth, H, W,
                              d_counts.data_ptr())
            mask_ptr = d_mask.data_ptr()
            with stages.stage("enqueue"):
                m.native.run_frames(H, W, W * 3, mask_ptr, W, jobs.ctypes.data, n)
        else:
            _frame_loop(clip, maskers, rects, arena, sift, d_mask, d_counts, d_pri if gpu_prior else None, gpu_prior,
                        host_prior, model_cache, cache_tag)
        with stages.stage("gpu_wait"):
            maskers[0].native.synchronize()
            counts = d_counts.cpu().numpy()
    seconds = time.time() - start
    stages.add("frame_loop", seconds)
    ious = []
    for k in range(min(n, clip.n_truth) * T):
        inter, union = int(counts[k, 0]), int(counts[k, 1])
        ious.append(inter / union if union else float("nan"))
    mean_iou = float(np.mean(ious)) if ious else float("nan")
    if out_path is not None:
        with open(out_path, "w") as f:
            f.write("%s;%s" % (mean_iou, seconds))
    for m in maskers:
        m.close()
    return dict(mean_iou=mean_iou, seconds=seconds, iou=ious, n_frames=n, n_updates=n * T, train_seconds=t_train,
                tracker=tracker_name, decode_seconds=0.0, wall_seconds=time.time() - t_wall)
