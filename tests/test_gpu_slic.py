"""GPU SLIC (pcm_slic_gpu, pcm_slic.cuh) against the library's host SLIC (pcm_slic) and the restatement of scikit-image
0.17.2's algorithm in oracle/slic_oracle.py.

Bar: the label maps and counts are EQUAL.  Stage by stage: the smoothed image is bit-identical, the image the k-means sees
is within 1e-12 of the oracle's (CUDA's pow / cbrt are not glibc's; the fraction of values that differ at all is printed),
the centre map is the oracle's k-means run on the device's own image, and the labels are the oracle's connectivity pass
run on the device's own centre map."""
import ctypes as C
import os

import cv2 as cv
import numpy as np
import pytest
import yaml

import slic_oracle as so
from helpers import PKG, polygons, read_video

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def handle():
    from pcm import capi
    h = capi.Handle(0)
    yield h
    h.close()


def _params(h, w, n_segments):
    """(centers, step, step_y, step_x) of slic_oracle.slic for an h x w crop."""
    g = so.grid_steps(h, w, n_segments)
    if g is None:
        ys, xs, step_y, step_x = np.arange(h), np.arange(w), 1, 1
    else:
        sy, step_y, sx, step_x = g
        ys, xs = np.arange(sy, h, step_y), np.arange(sx, w, step_x)
    centers = np.zeros((len(ys) * len(xs), 6), np.float64)
    centers[:, 1] = np.repeat(ys, len(xs))
    centers[:, 2] = np.tile(xs, len(ys))
    return centers, float(max(1, step_y, step_x)), step_y, step_x


def _check(h, frame, rect, stages=True, **kw):
    """Device labels == host pcm_slic == oracle; with `stages`, every stage dump against the oracle."""
    from pcm import capi
    x, y, w, hh = rect
    crop = np.ascontiguousarray(frame[y:y + hh, x:x + w])
    args = dict(n_segments=250, compactness=10.0, sigma=1.0, max_iter=10, start_label=0)
    args.update(kw)
    got, n = h.slic(np.ascontiguousarray(frame), rect, **args)
    host, n_host = capi.slic(frame, rect, **args)
    assert n == n_host and np.array_equal(got, host), "device labels differ from pcm_slic"
    if not stages:
        return got, n
    want = so.slic(crop, **args)
    assert np.array_equal(got, want) and n == int(want.max()) + 1
    d = h.slic_debug_last()
    smooth = so.smooth(crop, float(args["sigma"]))
    assert np.array_equal(d["smoothed"], smooth), "smoothed image is not bit-identical"
    image = np.ascontiguousarray(so.rgb2lab_float(smooth) * (1.0 / args["compactness"]))
    err = np.abs(d["image"] - image)
    assert err.max() <= 1e-12
    print("rect %s: %.4f %% of the k-means image not bit-identical (max |diff| %.3g)"
          % (rect, 100.0 * np.mean(d["image"] != image), err.max()))
    centers, step, step_y, step_x = _params(hh, w, args["n_segments"])
    nearest = so._kmeans(np.ascontiguousarray(d["image"]), centers, step, step_y, step_x, int(args["max_iter"]))
    assert np.array_equal(d["nearest"], nearest), "centre map differs from the oracle's k-means on the device image"
    s = hh * w / args["n_segments"]
    lab = so._enforce_connectivity(nearest, int(0.5 * s), int(3 * s), int(args["start_label"]))
    assert np.array_equal(got, lab)
    return got, n


def test_slic_gpu_segtrack_crops(handle):
    _check(handle, read_video("Video", "soldier")[0], (300, 0, 139, 224))      # the default config's crop
    _check(handle, read_video("Video", "frog")[3], (150, 60, 133, 159))
    _check(handle, read_video("Video", "parachute")[5], (0, 0, 414, 352))


@pytest.mark.parametrize("case", ["noise", "flat", "gradient", "tiny", "other_params", "wide", "start_label", "no_sigma",
                                  "no_iter"])
def test_slic_gpu_synthetic(handle, case):
    """The synthetic cases of test_slic_cpu.py, plus start_label 1, sigma 0 and max_iter 0."""
    rng = np.random.default_rng(23)
    kw = {}
    if case == "noise":
        frame, rect = rng.integers(0, 256, (70, 90, 3), dtype=np.uint8), (3, 5, 81, 60)
    elif case == "flat":
        frame, rect = np.full((40, 50, 3), 99, np.uint8), (0, 0, 50, 40)
    elif case == "gradient":
        g = np.add.outer(np.arange(96), np.arange(120)).astype(np.uint8)
        frame, rect = np.stack([g, g[::-1], 255 - g], -1).copy(), (10, 7, 100, 80)
    elif case == "tiny":                       # fewer pixels than seeds: every pixel is its own cluster
        frame, rect = rng.integers(0, 256, (12, 14, 3), dtype=np.uint8), (1, 2, 11, 9)
    elif case == "wide":
        frame, rect = rng.integers(0, 256, (9, 900, 3), dtype=np.uint8), (0, 2, 900, 6)
    else:
        frame, rect = rng.integers(0, 64, (60, 60, 3), dtype=np.uint8), (0, 0, 60, 60)
        kw = dict(n_segments=75, compactness=10.0, sigma=1.0, start_label=0)   # optical_flow_masker.py:60's call
        if case == "start_label":
            kw["start_label"] = 1
        elif case == "no_sigma":
            kw["sigma"] = 0.0
        elif case == "no_iter":
            kw["max_iter"] = 0
    _check(handle, frame, rect, **kw)


def _truth_rects(video):
    """The crops of every frame of a clip for boxes taken from its ground truth (bounding box of the object)."""
    frames, truths = read_video("Video", video), read_video("Truth", video)
    from pcm import capi
    out = []
    for f, t in zip(frames, truths):
        pts = cv.findNonZero((cv.cvtColor(t, cv.COLOR_BGR2GRAY) > 0).astype(np.uint8))
        box = cv.boundingRect(pts) if pts is not None else (0, 0, f.shape[1], f.shape[0])
        out.append((f, capi.crop_rect(box, f.shape[0], f.shape[1])))
    return out


def test_slic_gpu_soldier_all_frames(handle):
    crops = _truth_rects("soldier")
    assert len(crops) >= 32
    for f, rect in crops:
        x, y, w, hh = rect
        got, n = _check(handle, f, rect, stages=False)
        want = so.slic(np.ascontiguousarray(f[y:y + hh, x:x + w]), n_segments=250, compactness=10.0, sigma=1.0, start_label=0)
        assert np.array_equal(got, want) and n == int(want.max()) + 1


def test_slic_gpu_1080p(handle):
    rng = np.random.default_rng(5)
    yy, xx = np.mgrid[0:1080, 0:1920]
    base = np.stack([(xx * 255) // 1919, (yy * 255) // 1079, ((xx + yy) * 3) % 256], -1)
    frame = np.clip(base + rng.integers(-24, 25, base.shape), 0, 255).astype(np.uint8)
    _check(handle, frame, (0, 0, 1920, 1080))


def _spiral(n):
    """A one-pixel path of label 1 winding inwards through label 0 (long BFS fronts in every direction)."""
    a = np.zeros((n, n), np.int32)
    dirs = [(0, 1), (1, 0), (0, -1), (-1, 0)]
    y = x = d = 0
    a[0, 0] = 1
    inside = lambda yy, xx: 0 <= yy < n and 0 <= xx < n
    while True:
        for _ in range(2):
            dy, dx = dirs[d]
            if inside(y + dy, x + dx) and not a[y + dy, x + dx] and not (inside(y + 2 * dy, x + 2 * dx) and a[y + 2 * dy, x + 2 * dx]):
                y, x = y + dy, x + dx
                a[y, x] = 1
                break
            d = (d + 1) % 4
        else:
            return a


@pytest.mark.parametrize("case", ["noise4", "noise2", "stripes_h", "stripes_v", "spiral", "single_capped", "tiny_max",
                                  "blocks_start1", "blocks_start0", "checker"])
def test_slic_connectivity_tap(handle, case):
    rng = np.random.default_rng(11)
    runs = []
    if case == "noise4":
        seg = rng.integers(0, 4, (61, 47))
        runs = [(5, 40, 0), (5, 40, 1), (0, 12, 0), (20, 7, 1)]
    elif case == "noise2":
        seg = rng.integers(0, 2, (90, 130))
        runs = [(30, 180, 0), (3, 9, 1)]
    elif case == "stripes_h":
        seg = (np.arange(40)[:, None] // 3 % 2) * np.ones((1, 57), np.int64)
        runs = [(100, 70, 0), (200, 40, 1)]
    elif case == "stripes_v":
        seg = (np.arange(57)[None, :] % 2) * np.ones((33, 1), np.int64)
        runs = [(40, 10, 0), (34, 34, 1)]
    elif case == "spiral":
        seg = _spiral(48)
        runs = [(30, 100, 0), (10, 50, 1), (500, 2000, 0)]
    elif case == "single_capped":
        seg = np.zeros((37, 41), np.int64)
        runs = [(0, 7, 0), (3, 10, 1), (9, 50, 0), (60, 13, 0)]
    elif case == "tiny_max":
        seg = rng.integers(0, 3, (20, 25))
        runs = [(0, 1, 0), (0, 0, 1), (0, -5, 0), (2, 1, 1)]
    else:
        seg = np.kron(rng.integers(0, 5, (9, 11)), np.ones((4, 3), np.int64))
        seg[rng.random(seg.shape) < 0.1] = 7
        start = 1 if case == "blocks_start1" else 0
        runs = [(6, 30, start), (13, 36, start), (0, 12, start)]
        if case == "checker":
            seg = (np.add.outer(np.arange(30), np.arange(31)) % 2)
            runs = [(2, 6, 0), (2, 6, 1), (0, 1, 0)]
    for min_size, max_size, start in runs:
        want = so._enforce_connectivity(np.ascontiguousarray(seg, np.int64), int(min_size), int(max_size), int(start))
        got, n = handle.slic_connectivity(seg, min_size, max_size, start)
        assert np.array_equal(got, want), (case, min_size, max_size, start)
        assert n == int(want.max()) + 1


def test_update_from_resident_slic_labels():
    """update(labels=None) after the GPU SLIC == update with the same labels passed from the host; after a SLIC of
    another rect the handoff is refused with PCM_E_STATE."""
    from pcm import capi
    from test_gpu_parity import _random_forest_arrays
    rng = np.random.default_rng(4)
    frame = read_video("Video", "worm")[10]
    rect = capi.crop_rect((120, 110, 140, 70), frame.shape[0], frame.shape[1])
    h = capi.Handle(0)
    h.set_features(6, ["lab"])
    h.add_model_arrays(0, _random_forest_arrays(rng, 10, 5, 3 * 49))
    prm = capi.Handle.make_params(0, dilation_kernel=7)
    labels, n = h.slic(frame, rect)
    m1 = np.zeros_like(frame)
    h.update(frame, rect, None, n, None, prm, m1)
    m2 = np.zeros_like(frame)
    h.update(frame, rect, labels, n, None, prm, m2)
    assert m1.any() and np.array_equal(m1, m2)
    other = (rect[0] + 2, rect[1], rect[2] - 2, rect[3])
    h.slic(frame, other, want_labels=False)
    with pytest.raises(capi.PcmError) as e:
        h.update(frame, rect, None, n, None, prm, m1)
    assert e.value.code == -3
    h.close()


def test_slic_limits(handle):
    from pcm import capi
    lib = capi.load_library()
    frame = np.zeros((16, 16, 3), np.uint8)
    n = C.c_int(0)

    def call(rect=(0, 0, 16, 16), H=16, W=16, n_segments=10, compactness=10.0, max_iter=10, start_label=0, kernel=None,
             radius=0):
        r = (C.c_int * 4)(*rect)
        return lib.pcm_slic_gpu(handle._h, frame.ctypes.data_as(C.c_void_p), H, W, W * 3, r, n_segments, compactness, 1.0,
                                kernel, radius, max_iter, start_label, None, C.byref(n))
    assert call() == 0 and n.value >= 1
    assert call(n_segments=0) == -1 and b"n_segments" in lib.pcm_last_error()
    assert call(compactness=0.0) == -1 and call(compactness=float("nan")) == -1
    assert call(max_iter=-1) == -1
    assert call(start_label=-1) == -1
    assert call(rect=(0, 0, 17, 16)) == -1 and call(rect=(0, 0, 0, 16)) == -1
    assert call(kernel=frame.ctypes.data_as(C.c_void_p), radius=-1) == -1
    big = 1 << 14
    assert call(rect=(0, 0, big + 1, big), H=big, W=big + 1) == -4           # more than 2^28 pixels
    d = lib.pcm_slic_device(handle._h, None, 16, 16, 48, (C.c_int * 4)(0, 0, 16, 16), 10, 10.0, 1.0, None, 0, 10, 0, None,
                            C.byref(n))
    assert d == -1 and b"pcm_slic_device" in lib.pcm_last_error()
    with pytest.raises(capi.PcmError):
        handle.slic_connectivity(np.zeros((4, 4), np.int32), 1, 3, -1)


def test_slic_device_batch_equals_host(handle):
    import torch
    from pcm import capi
    frames = read_video("Video", "frog")[:3]
    H, W = frames[0].shape[:2]
    d_frames = torch.from_numpy(np.stack(frames)).cuda()
    rects = [(150, 60, 133, 159), (100, 40, 200, 120), (0, 0, W, H)]
    sizes = [r[2] * r[3] for r in rects]
    offsets = np.concatenate([[0], np.cumsum(sizes)])[:3].astype(np.int64)
    d = torch.empty(int(sum(sizes)), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    counts = handle.slic_device_batch(d_frames.data_ptr(), H * W * 3, [0, 1, 2], H, W, W * 3, rects, d.data_ptr(), offsets)
    flat = d.cpu().numpy()
    for k, r in enumerate(rects):
        want, n = capi.slic(frames[k], r)
        assert counts[k] == n
        assert np.array_equal(flat[offsets[k]:offsets[k] + sizes[k]].reshape(r[3], r[2]), want)


@pytest.mark.parametrize("prior", [False, True])
def test_masker_gpu_slic_equals_host_slic(prior):
    """The plugin's SLIC on the GPU gives the masks of the same masker fed the host code's labels (capi.slic) through
    segment_fn, over a SegTrack2 sequence, with the prior off and on (a deterministic prior of the label map: what matters
    is that both paths hand it the same map)."""
    from pcm import capi
    from maskers import getMaskerByName
    from test_gpu_parity import _random_forest_arrays
    rng = np.random.default_rng(10)
    frames = read_video("Video", "soldier")

    def prior_fn(prev_frame, prev_mask, crop, segs, n):
        cnt = np.bincount(segs.ravel(), minlength=n)
        s = np.bincount(segs.ravel(), weights=crop[..., 0].ravel().astype(np.float64), minlength=n)
        return (s / np.maximum(cnt, 1) / 255.0).astype(np.float32)
    trees = _random_forest_arrays(rng, 12, 5, 3 * 49)

    def host_slic(crop):
        return capi.slic(crop, (0, 0, crop.shape[1], crop.shape[0]), n_segments=250, compactness=10.0, sigma=1.0, start_label=0)[0]

    def make(**kw):
        cfg = dict(multi_selection=False, params=dict(n_estimators=20, max_depth=5, n_components=1, novelty_detection=False,
                                                      over_segmentation="SLIC", features="6 lab", dilation_kernel=7,
                                                      prior_weight=0.1 if prior else 0.0))
        m = getMaskerByName("PC", debug=False, frame=frames[0], config=cfg, poly_roi=None, update_mask=False, prior_fn=prior_fn,
                            **kw)
        m.native.add_model_arrays(0, trees)
        m.models.append({"n_frame": 0, "model": None})
        m.novelty_det.append({"n_frame": 0, "model": None, "threshold": 0.0})
        return m
    a, b = make(), make(segment_fn=host_slic)
    assert a.native_seg == "SLIC" and b.native_seg is None
    any_mask = False
    for i in range(8):
        ma, mb = np.zeros_like(frames[i]), np.zeros_like(frames[i])
        box = (340 - 4 * i, 20, 90, 180)
        a.update(bbox=box, frame=frames[i], mask=ma, color=None)
        b.update(bbox=box, frame=frames[i], mask=mb, color=None)
        any_mask = any_mask or ma[..., 2].any()
        assert np.array_equal(ma, mb), i
    assert any_mask
    a.close(); b.close()


def test_clip_resident_slic_sequence_equals_the_per_frame_path():
    """run_sequence_fast with over_segmentation SLIC (label maps from pcm_slic_device_batch) gives run_sequence's
    per-frame IoUs."""
    from pcm import fastseq, sweep
    from pcm.sequence import run_sequence
    with open(os.path.join(PKG, "config_benchmark.yaml")) as f:
        base = yaml.full_load(f)
    base["tracker_provider"] = "truth"
    params = dict(n_estimators=20, max_depth=7, n_components=1, novelty_detection=False, over_segmentation="SLIC",
                  features="6 lab", dilation_kernel=7, prior_weight=0.0)
    cfg = sweep.sequence_config(base, polygons(), "soldier", params, "Input/SegTrack2/Video", "Input/SegTrack2/Truth")
    assert fastseq._precomputable(cfg)
    n = 20
    want = run_sequence(cfg, max_frames=n)
    clip = fastseq.ClipContext(cfg["input_video"], cfg["input_truth"], 1, 0, max_frames=n)
    got = fastseq.run_sequence_fast(cfg, clip)
    clip.close()
    assert got["n_frames"] == want["n_frames"]
    assert np.array_equal(np.asarray(got["iou"]), np.asarray(want["iou"]), equal_nan=True)
