"""GPU Felzenszwalb (pcm_felzenszwalb_gpu, pcm_felzenszwalb.cuh) against the library's host code (pcm_felzenszwalb) and the
round rule restated in oracle/felzenszwalb_rounds.py.

Bar: the label maps and counts are EQUAL, the smoothed image is bit-identical, and the device takes exactly the rounds the
restated rule takes (the rule is deterministic: this pins the rule itself, not only its result)."""
import ctypes as C

import cv2 as cv
import numpy as np
import pytest

import felzenszwalb_oracle as fo
import felzenszwalb_rounds as fr
from helpers import read_video
from test_felzenszwalb_rounds_cpu import graph_cases, image_cases, image_edges

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def handle():
    from pcm import capi
    h = capi.Handle(0)
    yield h
    h.close()


def _check(h, frame, rect, rounds=True, **kw):
    """Device labels == host pcm_felzenszwalb; with `rounds`, the round counts == merge_rounds's and the smoothed image
    == the oracle's, bit for bit."""
    from pcm import capi
    args = dict(scale=100, sigma=0.5, min_size=50)
    args.update(kw)
    got, n = h.felzenszwalb(np.ascontiguousarray(frame), rect, **args)
    want, n_want = capi.felzenszwalb(frame, rect, **args)
    assert n == n_want and np.array_equal(got, want), "device labels differ from pcm_felzenszwalb"
    if rounds:
        x, y, w, hh = rect
        crop = np.ascontiguousarray(frame[y:y + hh, x:x + w])
        d = h.felzenszwalb_debug_last()
        assert np.array_equal(d["smoothed"], fo.smooth(crop, float(args["sigma"]))), "smoothed image is not bit-identical"
        e0, e1, costs, nv = image_edges(crop, float(args["sigma"]))
        _, r_merge, r_small = fr.merge_rounds(e0, e1, costs, nv, args["scale"] / 255.0, args["min_size"])
        assert d["rounds"] == (r_merge, r_small)
    return got, n


@pytest.mark.parametrize("case", image_cases(), ids=lambda c: c[0])
def test_felzenszwalb_gpu_cases(handle, case):
    """Every case of test_felzenszwalb_cpu.py: SegTrack2 crops, synthetic images, other parameters, degenerate crops."""
    name, frame, rect, kw = case
    _, n = _check(handle, frame, rect, **kw)
    if name == "flat":
        assert n == 1


@pytest.mark.parametrize("sigma", [0.0, 0.5, 0.8, 2.0])
def test_felzenszwalb_gpu_smoothing(handle, sigma):
    frame = read_video("Video", "frog")[3]
    _check(handle, frame, (150, 60, 133, 159), sigma=sigma)


def _truth_rects(video, step=1):
    """The crops of every `step`-th frame of a clip for boxes taken from its ground truth (the sweep's crops)."""
    from pcm import capi
    frames, truths = read_video("Video", video), read_video("Truth", video)
    out = []
    for f, t in list(zip(frames, truths))[::step]:
        pts = cv.findNonZero((cv.cvtColor(t, cv.COLOR_BGR2GRAY) > 0).astype(np.uint8))
        box = cv.boundingRect(pts) if pts is not None else (0, 0, f.shape[1], f.shape[0])
        out.append((f, capi.crop_rect(box, f.shape[0], f.shape[1])))
    return out


@pytest.mark.parametrize("video,step", [("soldier", 1), ("bmx", 1), ("frog", 10), ("worm", 10)])
def test_felzenszwalb_gpu_sweep_crops(handle, video, step):
    crops = _truth_rects(video, step)
    assert len(crops) >= 5
    for f, rect in crops:
        _check(handle, f, rect)


def test_felzenszwalb_gpu_1080p(handle):
    rng = np.random.default_rng(5)
    yy, xx = np.mgrid[0:1080, 0:1920]
    base = np.stack([(xx * 255) // 1919, (yy * 255) // 1079, ((xx + yy) * 3) % 256], -1)
    frame = np.clip(base + rng.integers(-24, 25, base.shape), 0, 255).astype(np.uint8)
    _check(handle, frame, (0, 0, 1920, 1080), rounds=False)


@pytest.mark.parametrize("case", graph_cases(), ids=lambda c: c[0])
def test_felzenszwalb_graph_tap(handle, case):
    """The device passes on explicit edge lists == pcm_felzenszwalb_graph, in merge_rounds's rounds; a path whose rising
    costs all stay below the limits takes one merge round per edge."""
    from pcm import capi
    name, n, e0, e1, costs, scale, min_size = case
    got, count = handle.felzenszwalb_graph(n, e0, e1, costs, scale, min_size)
    want, n_want = capi.felzenszwalb_graph(n, e0, e1, costs, scale, min_size)
    assert count == n_want and np.array_equal(got, want)
    _, r_merge, r_small = fr.merge_rounds(e0, e1, costs, n, scale, min_size)
    d = handle.felzenszwalb_debug_last()
    assert d["smoothed"] is None and d["rounds"] == (r_merge, r_small)
    if name == "path_merging":
        assert r_merge == e0.size and count == 1


def test_update_from_resident_felzenszwalb_labels():
    """update(labels=None) after the GPU Felzenszwalb == update with the same labels passed from the host; after a
    Felzenszwalb of another rect the handoff is refused with PCM_E_STATE."""
    from pcm import capi
    from test_gpu_parity import _random_forest_arrays
    rng = np.random.default_rng(4)
    frame = read_video("Video", "worm")[10]
    rect = capi.crop_rect((120, 110, 140, 70), frame.shape[0], frame.shape[1])
    h = capi.Handle(0)
    h.set_features(6, ["lab"])
    h.add_model_arrays(0, _random_forest_arrays(rng, 10, 5, 3 * 49))
    prm = capi.Handle.make_params(0, dilation_kernel=7)
    labels, n = h.felzenszwalb(frame, rect)
    host, n_host = capi.felzenszwalb(frame, rect)
    assert n == n_host and np.array_equal(labels, host)
    m1 = np.zeros_like(frame)
    h.update(frame, rect, None, n, None, prm, m1)
    m2 = np.zeros_like(frame)
    h.update(frame, rect, host, n, None, prm, m2)
    assert m1.any() and np.array_equal(m1, m2)
    other = (rect[0] + 2, rect[1], rect[2] - 2, rect[3])
    h.felzenszwalb(frame, other, want_labels=False)
    with pytest.raises(capi.PcmError) as e:
        h.update(frame, rect, None, n, None, prm, m1)
    assert e.value.code == -3 and "pcm_felzenszwalb_gpu" in str(e.value)
    h.close()


def test_felzenszwalb_device_batch_equals_single_calls(handle):
    import torch
    from pcm import capi
    lib = capi.load_library()
    frames = read_video("Video", "frog")[:3]
    H, W = frames[0].shape[:2]
    d_frames = torch.from_numpy(np.stack(frames)).cuda()
    rects = [(150, 60, 133, 159), (100, 40, 200, 120), (0, 0, W, H)]
    sizes = [r[2] * r[3] for r in rects]
    offsets = np.concatenate([[0], np.cumsum(sizes)])[:3].astype(np.int64)
    d = torch.empty(int(sum(sizes)), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    counts = handle.felzenszwalb_device_batch(d_frames.data_ptr(), H * W * 3, [0, 1, 2], H, W, W * 3, rects, d.data_ptr(), offsets)
    flat = d.cpu().numpy()
    n = C.c_int(0)
    for k, r in enumerate(rects):
        one = torch.empty(sizes[k], dtype=torch.int32, device="cuda")
        rc = lib.pcm_felzenszwalb_device(handle._h, C.c_void_p(d_frames[k].data_ptr()), H, W, W * 3, (C.c_int * 4)(*r), 100.0, 0.5,
                                         50, None, 0, C.c_void_p(one.data_ptr()), C.byref(n))
        assert rc == 0 and n.value == counts[k]
        assert np.array_equal(flat[offsets[k]:offsets[k] + sizes[k]], one.cpu().numpy())
        rc = lib.pcm_felzenszwalb_device(handle._h, C.c_void_p(d_frames[k].data_ptr()), H, W, W * 3, (C.c_int * 4)(*r), 100.0, 0.5,
                                         50, None, 0, None, C.byref(n))
        assert rc == 0 and n.value == counts[k]
        want, n_want = capi.felzenszwalb(frames[k], r)
        assert n_want == counts[k] and np.array_equal(flat[offsets[k]:offsets[k] + sizes[k]].reshape(r[3], r[2]), want)


def test_felzenszwalb_gpu_errors(handle):
    from pcm import capi
    lib = capi.load_library()
    frame = np.zeros((16, 16, 3), np.uint8)
    fp = frame.ctypes.data_as(C.c_void_p)
    n = C.c_int(0)

    def gpu(rect=(0, 0, 16, 16), H=16, W=16, stride=48, kernel=None, radius=0, f=fp):
        return lib.pcm_felzenszwalb_gpu(handle._h, f, H, W, stride, (C.c_int * 4)(*rect), 100.0, 0.5, 50, kernel, radius, None,
                                        C.byref(n))

    def dev(rect=(0, 0, 16, 16), H=16, W=16, stride=48, kernel=None, radius=0, f=fp):
        return lib.pcm_felzenszwalb_device(handle._h, f, H, W, stride, (C.c_int * 4)(*rect), 100.0, 0.5, 50, kernel, radius, None,
                                           C.byref(n))
    assert gpu() == 0 and n.value >= 1
    for call, who in ((gpu, b"pcm_felzenszwalb_gpu"), (dev, b"pcm_felzenszwalb_device")):
        assert call(f=None) == -1 and who in lib.pcm_last_error()
        assert call(rect=(0, 0, 17, 16)) == -1 and who in lib.pcm_last_error()
        assert call(rect=(0, 0, 0, 16)) == -1 and who in lib.pcm_last_error()
        assert call(stride=45) == -1 and who in lib.pcm_last_error()
        assert call(kernel=fp, radius=-1) == -1 and who in lib.pcm_last_error()
        big = 1 << 14
        assert call(rect=(0, 0, big + 1, big), H=big, W=big + 1, stride=3 * (big + 1)) == -4 and who in lib.pcm_last_error()
    a = np.array([0, 1], np.int32)
    c = np.array([0.5, 0.25])
    assert lib.pcm_felzenszwalb_graph_gpu(handle._h, 2, 2, a.ctypes.data_as(C.c_void_p), None, c.ctypes.data_as(C.c_void_p), 1.0,
                                          1, a.ctypes.data_as(C.c_void_p), C.byref(n)) == -1
    with pytest.raises(capi.PcmError, match="pcm_felzenszwalb_graph_gpu"):
        handle.felzenszwalb_graph(2, [0], [2], [0.5], 1.0, 1)            # vertex out of range
    with pytest.raises(capi.PcmError, match="pcm_felzenszwalb_graph_gpu"):
        handle.felzenszwalb_graph(2, [0], [1], [-0.5], 1.0, 1)           # negative cost
    with pytest.raises(capi.PcmError, match="pcm_felzenszwalb_graph_gpu"):
        handle.felzenszwalb_graph(0, [], [], [], 1.0, 1)                 # no vertices
    fresh = capi.Handle(0)
    with pytest.raises(capi.PcmError) as e:
        fresh.felzenszwalb_debug_last()
    assert e.value.code == -3
    fresh.close()


@pytest.mark.parametrize("prior", [False, True])
def test_masker_gpu_felzenszwalb_equals_host_felzenszwalb(prior):
    """The plugin's Felzenszwalb on the GPU gives the masks of the same masker fed the host code's labels
    (capi.felzenszwalb) through segment_fn, over a SegTrack2 sequence, with the prior off and on."""
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

    def host_felzenszwalb(crop):
        return capi.felzenszwalb(crop, (0, 0, crop.shape[1], crop.shape[0]), scale=100, sigma=0.5, min_size=50)[0]

    def make(**kw):
        cfg = dict(multi_selection=False, params=dict(n_estimators=20, max_depth=5, n_components=1, novelty_detection=False,
                                                      over_segmentation="felzenszwalb", features="6 lab", dilation_kernel=7,
                                                      prior_weight=0.1 if prior else 0.0))
        m = getMaskerByName("PC", debug=False, frame=frames[0], config=cfg, poly_roi=None, update_mask=False, prior_fn=prior_fn,
                            **kw)
        m.native.add_model_arrays(0, trees)
        m.models.append({"n_frame": 0, "model": None})
        m.novelty_det.append({"n_frame": 0, "model": None, "threshold": 0.0})
        return m
    a, b = make(), make(segment_fn=host_felzenszwalb)
    assert a.native_seg == "felzenszwalb" and b.native_seg is None
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

