"""Hyper-parameter sweep of the reference's benchmark.py (:26-89), sharded over GPUs.

The reference runs VIDEOS x HYPERPARAMS sequences as `python main.py cfg out` subprocesses on
a thread pool and collects "{iou};{seconds}" files.  Here the same grid is split over the
ranks of a `torch.distributed` job -- one process per GPU, whole sequences per rank, no
per-pixel communication -- and the per-sequence scores are brought together with ONE
collective at the end (`all_gather` of a `[n, 3]` float64 tensor: sequence id, mean IoU,
seconds; NCCL on GPUs, gloo in the CPU tests).  Rank 0 writes `benchmark_results.csv` with the
reference's columns (`<video>_benchmark`, `<video>_time`, `avg_benchmark`).
"""
import itertools
import os
import threading
import time

import numpy as np

from . import sequence as seq_mod
from . import stages

# benchmark.py:41-51
VIDEOS = ["soldier", "frog", "worm", "bmx"]
HYPERPARAMS = {
    "n_estimators": [20, 30],
    "max_depth": [7, 10],
    "n_components": [1],
    "novelty_detection": [True, False],
    "over_segmentation": ["quickshift", "felzenszwalb"],
    "features": ["8 hsv_lab", "6 lab"],
    "dilation_kernel": [7],
    "prior_weight": [0.1, 0.0],
}
# frames per clip: only used to balance the shards
CLIP_FRAMES = {"soldier": 32, "frog": 279, "worm": 243, "bmx": 36, "parachute": 51, "bird_of_paradise": 98}


def params_list(hyper=None):
    """Cartesian product in the reference's order (benchmark.py:53-55)."""
    hyper = hyper or HYPERPARAMS
    keys, values = zip(*hyper.items())
    return [dict(zip(keys, v)) for v in itertools.product(*values)]


def build_items(videos=None, hyper=None):
    """[(sequence id, combo index i, video v, params)], id = i * len(videos) + position of v."""
    videos = videos or VIDEOS
    items = []
    for i, params in enumerate(params_list(hyper)):
        for k, v in enumerate(videos):
            items.append((i * len(videos) + k, i, v, params))
    return items


def item_cost(item):
    """Relative cost of a sequence on the resident GPU path, in "light frames" (31 us).  Calibrated on a B200 against a
    serial run of the whole grid (bench.py --workload sweep --sweep-workers 1, least squares over the 256 per-sequence
    times of benchmark_results.csv, 14 % rms error; profiles/README.md, round 2), per frame in us:
        31 + 64 novelty + 42 depth-10 + 31 30-trees + 18 prior + 86 novelty x hsv_lab
    plus a fixed 8 ms per sequence (masker and handle set-up, model export, job list, one synchronisation) = 260 light
    frames, which is what balances the 32-frame clips against the 280-frame ones."""
    _, _, v, p = item
    frames = CLIP_FRAMES.get(v, 100)
    nov = bool(p.get("novelty_detection"))
    per_frame = 1.0 + (2.1 if nov else 0.0) + (1.35 if int(p.get("max_depth") or 0) >= 10 else 0.0) + \
        (1.0 if int(p.get("n_estimators") or 0) >= 30 else 0.0) + (0.6 if p.get("prior_weight") else 0.0) + \
        (2.8 if nov and str(p.get("features")).endswith("hsv_lab") else 0.0)
    return frames * per_frame + 260.0


def forest_key(item):
    _, _, v, p = item
    return (v, p["features"], p["n_estimators"], p["max_depth"])


def fit_key(item):
    """Sequences with equal fit_key train on the same rows and share ONE fit: the forest is fitted with
    the grid's largest n_estimators and smaller forests are its first trees."""
    _, _, v, p = item
    return (v, p["features"], p["max_depth"])


class ModelCache:
    """Rank-wide cache of training rows, fitted forests and PCAs, safe for the sequence threads:
    a value is computed once, by the first thread that asks for it."""

    def __init__(self):
        self.values, self.locks, self.guard = {}, {}, threading.Lock()

    def get_or_compute(self, key, make):
        with self.guard:
            if key in self.values:
                return self.values[key]
            lock = self.locks.setdefault(key, threading.Lock())
        with lock:
            with self.guard:
                if key in self.values:
                    return self.values[key]
            value = make()
            with self.guard:
                self.values[key] = value
            return value


def clip_open_cost(video):
    """What a rank pays for every clip it touches, whatever its share of the clip's sequences: decoding and uploading the
    clip and waiting for the ranks it shares the clip with (measured: 0.23 s for the 279-frame clip = 16 light frames per
    clip frame)."""
    return 16.0 * CLIP_FRAMES.get(video, 100)


def clip_prepare_cost(video):
    """Host work that exists once per clip and is split between the ranks sharing it (over-segmentation maps, SIFT
    detection: ~11 ms of CPU per frame on the rank's four-odd cores); charged to the clip's sequences in equal parts."""
    return 55.0 * CLIP_FRAMES.get(video, 100)


def shard_cost(shard, all_items):
    """What `partition` balances: the shard's sequences, their part of the preparation of their clips, and the opening of
    every clip the shard touches."""
    clip_n = {}
    for it in all_items:
        clip_n[it[2]] = clip_n.get(it[2], 0) + 1
    return sum(item_cost(it) + clip_prepare_cost(it[2]) / clip_n[it[2]] for it in shard) + \
        sum(clip_open_cost(v) for v in {it[2] for it in shard})


def partition(items, world):
    """Contiguous split of the grid with CLIP LOCALITY: the sequences are ordered clip by clip (heaviest clip first; inside
    a clip by features, max_depth, ... so that neighbours share their fitted models) and the ordered list is cut into
    `world` runs that MINIMISE THE SLOWEST RANK, where a rank costs the sum of its sequences (`item_cost` plus the
    sequence's part of its clip's preparation) plus `clip_open_cost` for every clip it touches -- so a cut lands on a clip
    boundary whenever that is nearly balanced, instead of leaving one rank to open two long clips (dynamic programme over
    the cut positions).  Returns `world` lists of items; deterministic."""
    clip_cost, clip_n = {}, {}
    for it in items:
        clip_cost[it[2]] = clip_cost.get(it[2], 0.0) + item_cost(it)
        clip_n[it[2]] = clip_n.get(it[2], 0) + 1

    def key(it):
        p = it[3]
        return (-clip_cost[it[2]], it[2], str(p.get("features")), p.get("max_depth") or 0, p.get("n_estimators") or 0, it[0])
    ordered = sorted(items, key=key)
    n = len(ordered)
    shards = [[] for _ in range(world)]
    if not ordered:
        return shards
    if world >= n:                                   # one sequence per rank, the rest stay empty-handed
        for k, it in enumerate(ordered):
            shards[k].append(it)
        return shards
    cost = [item_cost(it) + clip_prepare_cost(it[2]) / clip_n[it[2]] for it in ordered]
    prefix = [0.0]
    for c in cost:
        prefix.append(prefix[-1] + c)
    clips = [it[2] for it in ordered]
    first_of_run = [k == 0 or clips[k] != clips[k - 1] for k in range(n)]     # the list is grouped by clip
    opens = [0.0] * (n + 1)                                                    # opens[k] = open cost of clip runs starting before k
    for k in range(n):
        opens[k + 1] = opens[k] + (clip_open_cost(clips[k]) if first_of_run[k] else 0.0)

    def run_cost(a, b):                              # items a .. b-1
        touched = opens[b] - opens[a] + (0.0 if first_of_run[a] else clip_open_cost(clips[a]))
        return prefix[b] - prefix[a] + touched
    INF = float("inf")
    best = [[INF] * (n + 1) for _ in range(world + 1)]      # best[r][k]: smallest possible maximum over r runs covering k items
    cut = [[0] * (n + 1) for _ in range(world + 1)]
    best[0][0] = 0.0
    for r in range(1, world + 1):
        for k in range(r, n - (world - r) + 1):
            for a in range(r - 1, k):
                if best[r - 1][a] == INF:
                    continue
                v = max(best[r - 1][a], run_cost(a, k))
                if v < best[r][k] - 1e-9:
                    best[r][k], cut[r][k] = v, a
    k = n
    for r in range(world, 0, -1):
        a = cut[r][k]
        shards[r - 1] = ordered[a:k]
        k = a
    return shards


def sequence_config(base, polygons, video, params, videos_path, truth_path):
    """The per-sequence config of benchmark.py:69-75."""
    return {**base, "input_video": "%s/%s.mp4" % (videos_path, video), "input_truth": "%s/%s.mp4" % (truth_path, video),
            "params": dict(params), **polygons[video]}


def clip_needs(all_items):
    """{clip: (over-segmentations, any SIFT prior)} over the WHOLE grid: what the ranks sharing a clip prepare together."""
    needs = {}
    for _, _, v, p in all_items:
        kinds, sift = needs.setdefault(v, (set(), [False]))
        kinds.add(p["over_segmentation"])
        sift[0] = sift[0] or bool(p.get("prior_weight"))
    return {v: (sorted(k), s[0]) for v, (k, s) in needs.items()}


def clip_order(all_items):
    """Clips, heaviest first: the order in which every rank opens and prepares the clips of its shard."""
    cost = {}
    for it in all_items:
        cost[it[2]] = cost.get(it[2], 0.0) + item_cost(it)
    return sorted(cost, key=lambda v: (-cost[v], v))


def run_shard(items, base, polygons, device=0, videos_path="Input/SegTrack2/Video", truth_path="Input/SegTrack2/Truth",
              max_frames=None, train_jobs=None, progress=None, seq_workers=1, resident=True, shares=None, all_items=None):
    """Run this rank's sequences; returns float64 [n, 3] = (sequence id, mean IoU, seconds).

    resident=True (default): every clip of the shard is decoded and uploaded ONCE (`fastseq.ClipContext`); its tracker
    boxes, over-segmentation maps and SIFT features are shared by all hyper-parameter sets, forests and PCAs are
    fitted on the GPU and shared through a rank-wide `ModelCache`, and a sequence is one asynchronous pass over the
    device-resident frames.  `seq_workers` threads run sequences concurrently, each on its own CUDA stream: the host
    stages of one sequence (SIFT priors, Python) overlap the kernels of the others; the fits run on threads of their
    own and the clips are prepared beside them (quickshift maps on a side thread, the host-side steps -- collectives
    when ranks share a clip -- on the calling thread), so a sequence starts as soon as what IT needs exists.  Every
    masker owns its own native context; results do not depend on the schedule.
    resident=False: the per-frame host-buffer path of `pcm.sequence.run_sequence` (what `main.py` runs)."""
    out = np.zeros((len(items), 3), np.float64)
    done = [0]
    lock = threading.Lock()
    cache = ModelCache()                            # rows / forests / PCAs / SIFT features, shared by the threads of this rank
    fit_estimators = max([int(it[3]["n_estimators"]) for it in items] or [0])
    videos = sorted({it[2] for it in items})
    from . import capi
    if items:
        capi.load_library()                                             # dlopen once, before the threads
    clips, order_v = {}, []
    if resident and items:
        from . import fastseq
        from concurrent.futures import ThreadPoolExecutor

        host_workers = max(2, min(16, (os.cpu_count() or 2) // max(int(os.environ.get("WORLD_SIZE", "1")), 1)))

        def open_clip(v):
            cfg = sequence_config(base, polygons, v, items[0][3], videos_path, truth_path)
            return fastseq.ClipContext(cfg["input_video"], cfg["input_truth"], cfg.get("resize_factor") or 1, device, max_frames,
                                       host_workers=host_workers, share=(shares or {}).get(v))
        # heaviest clips first; every clip opens (decodes, uploads) on its own thread
        order_v = [v for v in clip_order(all_items or items) if v in videos]
        with ThreadPoolExecutor(max_workers=max(1, len(videos))) as pool:
            clips = dict(zip(order_v, pool.map(open_clip, order_v)))

    gpu_prior = (base.get("prior_provider") or "gpu") == "gpu"
    PREPARE_STEPS = ("quickshift", "SLIC", "felzenszwalb", "sift")

    def prepare_clips(step):
        # (measured, round 2: preparing the clips of a single-GPU run side by side instead of one after the other made the
        # sweep SLOWER -- 55-64 instead of 79 sequences/s: every clip's frames are already spread over all host cores)
        """One kind of what all sequences of a clip share -- the label maps of an over-segmentation, or the SIFT features
        -- for every clip of the shard, in the same (step, clip) order on every rank: the ranks that share a clip split
        the per-frame host work and all-reduce the pieces (felzenszwalb, sift: calling thread of run_shard only; the
        quickshift and SLIC steps involve no collective and may run on another thread)."""
        needs = clip_needs(all_items or items)
        for v in order_v:
            cfg = sequence_config(base, polygons, v, items[0][3], videos_path, truth_path)
            with stages.stage("prepare_clips"):
                if step == "sift":
                    if needs[v][1] and gpu_prior:
                        clips[v].prepare(cfg, [], True)
                elif step in needs[v][0]:
                    clips[v].prepare(cfg, [step], False)

    def needs_of(k):
        """What sequence k waits for: the label maps of its over-segmentation, and the SIFT features if it uses the
        (device-side) prior."""
        p = items[k][3]
        need = {p["over_segmentation"]} & set(PREPARE_STEPS)
        if p.get("prior_weight") and gpu_prior:
            need.add("sift")
        return need

    local = threading.local()

    def run_one(k):
        sid, i, v, params = items[k]
        cfg = sequence_config(base, polygons, v, params, videos_path, truth_path)
        cfg["train_jobs"] = train_jobs
        cfg["fit_estimators"] = fit_estimators
        if resident:
            from . import fastseq
            if getattr(local, "stream", None) is None:
                import torch
                local.stream = torch.cuda.Stream(device=clips[v].dev)
            with stages.stage("sequence"):
                r = fastseq.run_sequence_fast(cfg, clips[v], device=device, model_cache=cache, cache_tag=v, stream=local.stream)
        else:
            r = seq_mod.run_sequence(cfg, device=device, model_cache=cache, cache_tag=v, max_frames=max_frames)
        out[k] = (sid, r["mean_iou"], r["seconds"])
        with lock:
            done[0] += 1
            if progress:
                progress(done[0], len(items), sid, r)

    def prefit_tasks():
        """One task per (clip, features, max_depth, polygon selection) of the shard: training rows, forest and (with the
        shallowest depth of a feature set, when any sequence asks for novelty detection) the PCA go into the rank-wide
        cache before the sequences ask for them, all in parallel instead of one sequence thread fitting while the
        others of its group wait."""
        seen, tasks = set(), []
        for it in items:
            _, _, v, p = it
            key = (v, p["features"], p["max_depth"])
            if key in seen:
                continue
            seen.add(key)
            novelty = any(q[2] == v and q[3]["features"] == p["features"] and q[3]["novelty_detection"] for q in items)
            first_depth = min(q[3]["max_depth"] for q in items if q[2] == v and q[3]["features"] == p["features"])
            cfg = sequence_config(base, polygons, v, dict(p, n_estimators=fit_estimators,
                                                           novelty_detection=bool(novelty and p["max_depth"] == first_depth)),
                                  videos_path, truth_path)
            n_sel = len(cfg["pts"][0]) if cfg.get("multi_selection") else 1
            for t in range(len(cfg["pts"])):
                for sel in range(n_sel):
                    tasks.append((v, cfg, t, sel))
        return tasks

    def prefit(task):
        import cv2 as cv
        from maskers import getMaskerByName
        v, cfg, t, sel = task
        frames = clips[v].frames
        with stages.stage("prefit"):
            m = getMaskerByName("PC", debug=False, frame=frames[0], config=cfg, poly_roi=cfg["pts"][t][0],
                                update_mask=cfg.get("update_mask"), device=device, model_cache=cache, cache_tag=(v, t),
                                fit_estimators=fit_estimators)
            pts = cfg["pts"][t][sel]
            n_frame = cfg["pts_frame_numbers"][sel]
            m.addModel(frame=frames[n_frame], poly_roi=pts, bbox=cv.boundingRect(np.array(pts)),
                       bbox_roni=cfg["bboxes_roni"][t][sel], n_frame=n_frame)
            m.close()

    # longest sequences first; sequences that share fits next to each other
    order = sorted(range(len(items)), key=lambda k: (-item_cost(items[k]), str(fit_key(items[k])), items[k][0]))
    if seq_workers <= 1 or len(order) <= 1:
        if resident:
            for step in PREPARE_STEPS:
                prepare_clips(step)
        for k in order:
            run_one(k)
    else:
        from concurrent.futures import ThreadPoolExecutor
        if not resident:
            for v in videos:                                            # decode every clip once, up front
                cfg = sequence_config(base, polygons, v, items[0][3], videos_path, truth_path)
                seq_mod.read_clip(seq_mod.resolve_path(cfg["input_video"]), cfg.get("resize_factor") or 1)
                seq_mod.read_clip(seq_mod.resolve_path(cfg["input_truth"]), cfg.get("resize_factor") or 1)
        tasks = prefit_tasks() if resident else []
        # The fits get threads of their own (half as many as there are sequence threads; PCM_SWEEP_FIT_WORKERS overrides),
        # so that the sequence threads are free for the sequences whose models and label maps are there.  Round 2
        # timelines (tools/sweep_ab.sh, profiles/README.md), 1 GPU + 16 cores: through the 16 sequence threads the 52
        # fits held all of them for the first 1.7 s of a 3.2 s sweep.  A fit is 6 ms of GPU time and otherwise host
        # work (training rows to the host and back, bootstrap draws, PCA): 8 fitting threads finish the 52 fits as soon
        # as 16 or 24 do (1.0 - 1.2 s) and leave the cores to the clip preparation; 48 thrash (1.8 - 3 s).
        fit_workers = int(os.environ.get("PCM_SWEEP_FIT_WORKERS", "0")) or max(4, seq_workers // 2)
        fit_workers = max(1, min(len(tasks), fit_workers)) if tasks else 1
        side_quickshift = resident and os.environ.get("PCM_SWEEP_SIDE_QUICKSHIFT", "1") != "0"
        with ThreadPoolExecutor(max_workers=seq_workers) as pool, ThreadPoolExecutor(max_workers=fit_workers) as fit_pool:
            futures = [fit_pool.submit(prefit, t) for t in tasks]               # GPU fits start at once ...
            pending, done_steps, guard = list(order), set(), threading.Lock()

            def release(step):
                """`step` is prepared: start the sequences that now have everything they need."""
                with guard:
                    done_steps.add(step)
                    ready = [k for k in pending if needs_of(k) <= done_steps]
                    gone = set(ready)
                    pending[:] = [k for k in pending if k not in gone]
                    futures.extend(pool.submit(run_one, k) for k in ready)

            if resident:
                # ... while the clips are prepared: the quickshift maps (GPU work, no collective) on a thread of their
                # own, the host-side steps (felzenszwalb maps, SIFT detection; collectives between the ranks that share
                # a clip) on this one.  Sequences start as soon as what THEY need is there.
                side, side_error = None, []
                if side_quickshift:
                    def quickshift_side():
                        try:
                            prepare_clips("quickshift")
                            release("quickshift")
                        except BaseException as e:          # re-raised on the main thread
                            side_error.append(e)
                    side = threading.Thread(target=quickshift_side, name="pcm-quickshift-maps")
                    side.start()
                for step in PREPARE_STEPS:
                    if side is not None and step == "quickshift":
                        continue
                    prepare_clips(step)
                    release(step)
                if side is not None:
                    side.join()
                    if side_error:
                        raise side_error[0]
            with guard:
                futures.extend(pool.submit(run_one, k) for k in pending)
                del pending[:]
            for f in futures:
                f.result()
    for c in clips.values():
        c.close()
    return out


def gather(local, world, dist=None, device=None):
    """ONE collective: every rank contributes its padded [n_max, 3] block; returns the [N, 3]
    array sorted by sequence id (on every rank)."""
    if world == 1 or dist is None:
        return local[np.argsort(local[:, 0])] if len(local) else local
    import torch
    n = torch.tensor([len(local)], dtype=torch.int64, device=device)
    sizes = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(sizes, n)
    n_max = max(int(s.item()) for s in sizes)
    block = torch.full((max(n_max, 1), 3), -1.0, dtype=torch.float64, device=device)
    if len(local):
        block[:len(local)] = torch.from_numpy(local).to(block.device)
    blocks = [torch.empty_like(block) for _ in range(world)]
    dist.all_gather(blocks, block)
    rows = [b[:int(s.item())].cpu().numpy() for b, s in zip(blocks, sizes)]
    allr = np.concatenate(rows, axis=0) if rows else np.zeros((0, 3))
    return allr[np.argsort(allr[:, 0])]


def results_table(all_rows, videos=None, hyper=None):
    """pandas frame with the reference's layout (benchmark.py:66-68,86-88)."""
    import pandas as pd
    videos = videos or VIDEOS
    plist = params_list(hyper)
    results = {i: dict(p) for i, p in enumerate(plist)}
    for sid, iou, secs in all_rows:
        i, k = divmod(int(sid), len(videos))
        results[i][videos[k] + "_benchmark"] = iou
        results[i][videos[k] + "_time"] = secs
    table = pd.DataFrame.from_dict(results, orient="index")
    cols = [v + "_benchmark" for v in videos if v + "_benchmark" in table]
    if cols:
        table["avg_benchmark"] = table[cols].mean(axis=1)
    return table


def run(base, polygons, videos=None, hyper=None, limit=None, max_frames=None, out_csv=None, backend=None,
        train_jobs=None, log=None, seq_workers=None, resident=True):
    """Entry point used by benchmark.py / bench.py --workload sweep.  Reads RANK / WORLD_SIZE /
    LOCAL_RANK; returns (summary dict, table or None) -- the table on rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    videos = videos or VIDEOS
    items = build_items(videos, hyper)
    if limit:
        items = items[:limit]
    shards = partition(items, world)
    dist = dev = None
    import torch
    if world > 1:
        import torch.distributed as dist
        backend = backend or ("nccl" if torch.cuda.is_available() else "gloo")
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
            dev = torch.device("cuda", local_rank)
            if not dist.is_initialized():
                dist.init_process_group("nccl", device_id=dev)
        elif not dist.is_initialized():
            dist.init_process_group(backend)
        dist.barrier()
    cores = max(1, (os.cpu_count() or 1) // max(world, 1))        # host cores of this rank
    if seq_workers is None:
        # resident sweep: a sequence thread spends its time inside native enqueue calls (GIL released) and every
        # thread owns a CUDA stream -- more threads than cores keeps more streams busy on the GPU
        seq_workers = max(4, min(16, 2 * cores)) if resident else max(1, min(6, cores // 3))
    if train_jobs is None:
        train_jobs = max(1, cores // seq_workers)
    try:
        import cv2
        cv2.setNumThreads(1 if resident else max(1, cores // seq_workers))   # resident: frames are detected in parallel instead
    except Exception:
        pass
    if torch.cuda.is_available():
        # the CUDA context and the library exist before the clock starts (process start-up is not sweep throughput)
        torch.cuda.set_device(local_rank)
        torch.zeros(1, device=torch.device("cuda", local_rank))
        torch.cuda.synchronize()
        from . import capi
        capi.Handle(local_rank).close()
    # ranks that work on the same clip form a group and split its per-frame host work (fastseq.Share)
    shares = {}
    if world > 1 and resident:
        from .fastseq import Share
        for v in clip_order(items):
            members = [r for r in range(world) if any(it[2] == v for it in shards[r])]
            if len(members) > 1:
                group = dist.new_group(ranks=members)          # collective: every rank creates every group, same order
                if rank in members:
                    shares[v] = Share(dist, group, members.index(rank), len(members))
        # a group's communicator is built by its first collective (NCCL: about a second with eight ranks): do that here,
        # with the process group itself, before the clock starts -- in the same clip order on every rank
        for v in clip_order(items):
            if v in shares:
                warm = torch.zeros(1, device=dev) if dev is not None else torch.zeros(1)
                dist.all_reduce(warm, group=shares[v].group)
        if dev is not None:
            torch.cuda.synchronize(dev)
        dist.barrier()
    blas_limit = None
    if resident:
        # the PCA fits call LAPACK from many threads at once: one BLAS thread each instead of a pool per call
        try:
            from threadpoolctl import threadpool_limits
            blas_limit = threadpool_limits(limits=1, user_api="blas")
        except Exception:
            pass
    stages.reset()
    t0 = time.time()
    local = run_shard(shards[rank], base, polygons, device=local_rank, max_frames=max_frames, train_jobs=train_jobs,
                      seq_workers=seq_workers, resident=resident, shares=shares, all_items=items,
                      progress=(lambda k, n, sid, r: log("[rank %d] %d/%d seq %d iou %.3f %.2fs (train %.2fs, decode %.2fs, wall %.2fs)" %
                                                         (rank, k, n, sid, r["mean_iou"], r["seconds"], r["train_seconds"],
                                                          r["decode_seconds"], r["wall_seconds"])))
                      if log else None)
    t_local = time.time() - t0
    if blas_limit is not None:
        blas_limit.restore_original_limits()
    stages.dump_timeline(".rank%d" % rank if world > 1 else "")
    all_rows = gather(local, world, dist, dev)
    t_all = t_local
    if world > 1:
        t = torch.tensor([t_local], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t_all = float(t.item())
    summary = dict(n_sequences=len(items), seconds=t_all, sequences_per_s=len(items) / t_all if t_all > 0 else 0.0,
                   n_gpus=world, per_rank_sequences=[len(s) for s in shards], train_jobs=train_jobs,
                   seq_workers=seq_workers, host_cores=os.cpu_count(), tracker_provider=base.get("tracker_provider"),
                   rank0_seconds=t_local, per_stage_host_s_rank0={k: round(v, 3) for k, v in sorted(stages.snapshot().items())})
    if log:
        log("[rank %d] sweep %.2f s; host stage seconds (summed over %d sequence threads): %s" %
            (rank, t_local, seq_workers, summary["per_stage_host_s_rank0"]))
    table = None
    if rank == 0:
        table = results_table(all_rows, videos, hyper)
        if out_csv:
            table.to_csv(out_csv, index=False)
    return summary, table
