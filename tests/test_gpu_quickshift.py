"""GPU quickshift (pcm_quickshift, SURVEY §8 row f-1) against the restatement of
scikit-image 0.17.2's algorithm in oracle/quickshift_oracle.py (PARITY UNPINNED against
scikit-image itself: not installed, not vendored, no reference golden vectors).

Bar: the label maps are equal (same partition, same np.unique numbering).  The float64 window
sums run in the same order with the same un-fused operations on both sides; only exp() / cbrt()
come from different math libraries (last-ulp), which could flip a comparison only on an exact
near-tie, so a disagreement on more than 0.1 % of the pixels fails the test outright and any
smaller one is reported by the strict assertion."""
import numpy as np
import pytest

import quickshift_oracle as qso
from helpers import read_video

pytestmark = pytest.mark.gpu


def _check(h, frame, rect, **kw):
    x, y, w, hh = rect
    crop = frame[y:y + hh, x:x + w]
    want = qso.quickshift(crop, ratio=kw.get("ratio", 0.5), kernel_size=kw.get("kernel_size", 3),
                          max_dist=kw.get("max_dist", 6), random_seed=42)
    got, n = h.quickshift(frame, rect, noise=qso.tie_noise((hh, w), 42), **kw)
    assert got.shape == want.shape and n == int(want.max()) + 1 == int(got.max()) + 1
    agree = qso.partition_agreement(want, got)
    assert agree > 0.999, "partitions differ on %.3f %% of the pixels" % (100 * (1 - agree))
    assert np.array_equal(got, want)
    return got, n


def test_quickshift_segtrack_crops():
    from pcm import capi
    h = capi.Handle(0)
    h.set_features(8, ["hsv", "lab"])
    f = read_video("Video", "soldier")[0]
    _check(h, f, (300, 0, 139, 224))                       # the default config's crop size
    _check(h, read_video("Video", "frog")[3], (150, 60, 133, 159))
    _check(h, read_video("Video", "parachute")[5], (0, 0, 414, 352))   # whole frame, touches every border
    h.close()


@pytest.mark.parametrize("case", ["noise", "flat", "gradient", "tiny", "odd_params"])
def test_quickshift_synthetic(case):
    from pcm import capi
    rng = np.random.default_rng(7)
    h = capi.Handle(0)
    h.set_features(1, ["rgb"])
    kw = {}
    if case == "noise":
        frame, rect = rng.integers(0, 256, (70, 90, 3), dtype=np.uint8), (3, 5, 81, 60)
    elif case == "flat":                                   # every tie is broken by the seeded noise only
        frame, rect = np.full((50, 64, 3), 77, np.uint8), (0, 0, 64, 50)
    elif case == "gradient":
        g = np.add.outer(np.arange(96), np.arange(120)).astype(np.uint8)
        frame, rect = np.stack([g, g[::-1], 255 - g], -1).copy(), (10, 7, 100, 80)
    elif case == "tiny":
        frame, rect = rng.integers(0, 256, (9, 7, 3), dtype=np.uint8), (1, 2, 5, 4)
    else:
        frame, rect = rng.integers(0, 64, (60, 60, 3), dtype=np.uint8), (0, 0, 60, 60)
        kw = dict(ratio=1.0, kernel_size=5, max_dist=10)   # scikit-image's own defaults, window +-15
    _check(h, frame, rect, **kw)
    h.close()


def test_update_from_resident_quickshift_labels():
    """update(labels=None) after quickshift == update with the same labels passed from the host;
    a stale handoff (other frame / rect) is refused."""
    from pcm import capi
    from test_gpu_parity import _random_forest_arrays
    rng = np.random.default_rng(4)           # a forest that switches 40 of the 57 segments on
    frame = read_video("Video", "worm")[10]
    rect = capi.crop_rect((120, 110, 140, 70), frame.shape[0], frame.shape[1])
    h = capi.Handle(0)
    h.set_features(6, ["lab"])
    h.add_model_arrays(0, _random_forest_arrays(rng, 10, 5, 3 * 49))
    prm = capi.Handle.make_params(0, dilation_kernel=7)
    labels, n = h.quickshift(frame, rect, noise=qso.tie_noise((rect[3], rect[2]), 42))
    m1 = np.zeros_like(frame)
    h.update(frame, rect, None, n, None, prm, m1)
    m2 = np.zeros_like(frame)
    h.update(frame, rect, labels, n, None, prm, m2)
    assert m1.any() and np.array_equal(m1, m2)
    # labels == NULL with no quickshift pending: the label map the host-label update above left on the device is reused
    m3 = np.zeros_like(frame)
    h.update(frame, rect, None, n, None, prm, m3)
    assert np.array_equal(m3, m2)
    h.quickshift(frame, rect, noise=None, want_labels=False)   # noise reused for the same crop size
    other = frame.copy()
    with pytest.raises(capi.PcmError):
        h.update(other, rect, None, n, None, prm, m1)
    h.close()


def test_masker_native_seg_quickshift():
    """config over_segmentation: quickshift -> the plugin API segments on the GPU and produces
    the same mask as the same masker fed the oracle's label map through segment_fn."""
    from maskers import getMaskerByName
    from test_gpu_parity import _random_forest_arrays
    rng = np.random.default_rng(10)          # a forest with a non-trivial mask on all three frames
    frames = read_video("Video", "soldier")
    cfg = dict(multi_selection=False, params=dict(n_estimators=20, max_depth=5, n_components=1, novelty_detection=False,
                                                  over_segmentation="quickshift", features="6 lab", dilation_kernel=7,
                                                  prior_weight=0.0))
    trees = _random_forest_arrays(rng, 12, 5, 3 * 49)

    def make(**kw):
        m = getMaskerByName("PC", debug=False, frame=frames[0], config=cfg, poly_roi=None, update_mask=False, **kw)
        m.native.add_model_arrays(0, trees)
        m.models.append({"n_frame": 0, "model": None})
        m.novelty_det.append({"n_frame": 0, "model": None, "threshold": 0.0})
        return m
    a = make()
    b = make(segment_fn=lambda crop: qso.quickshift(crop, ratio=0.5, kernel_size=3, max_dist=6, random_seed=42))
    assert a.native_seg == "quickshift" and b.native_seg is None
    for i in range(3):
        ma, mb = np.zeros_like(frames[i]), np.zeros_like(frames[i])
        box = (340 - 4 * i, 20, 90, 180)
        assert a.update(bbox=box, frame=frames[i], mask=ma, color=None) is None
        assert b.update(bbox=box, frame=frames[i], mask=mb, color=None) is None
        assert ma[..., 2].any() and np.array_equal(ma, mb)
    a.close(); b.close()


def test_masker_native_seg_slic():
    """config over_segmentation: SLIC -> the plugin segments on the GPU (pcm_slic_gpu) and produces the same mask as the
    same masker fed the oracle's label map through segment_fn (oracle/slic_oracle.py; parity unpinned against
    scikit-image itself)."""
    import slic_oracle as so
    from maskers import getMaskerByName
    from test_gpu_parity import _random_forest_arrays
    rng = np.random.default_rng(10)
    frames = read_video("Video", "soldier")
    cfg = dict(multi_selection=False, params=dict(n_estimators=20, max_depth=5, n_components=1, novelty_detection=False,
                                                  over_segmentation="SLIC", features="6 lab", dilation_kernel=7,
                                                  prior_weight=0.0))
    trees = _random_forest_arrays(rng, 12, 5, 3 * 49)

    def make(**kw):
        m = getMaskerByName("PC", debug=False, frame=frames[0], config=cfg, poly_roi=None, update_mask=False, **kw)
        m.native.add_model_arrays(0, trees)
        m.models.append({"n_frame": 0, "model": None})
        m.novelty_det.append({"n_frame": 0, "model": None, "threshold": 0.0})
        return m
    a = make()
    b = make(segment_fn=lambda crop: so.slic(crop, n_segments=250, compactness=10, sigma=1, start_label=0))
    assert a.native_seg == "SLIC" and b.native_seg is None
    for i in range(3):
        ma, mb = np.zeros_like(frames[i]), np.zeros_like(frames[i])
        box = (340 - 4 * i, 20, 90, 180)
        assert a.update(bbox=box, frame=frames[i], mask=ma, color=None) is None
        assert b.update(bbox=box, frame=frames[i], mask=mb, color=None) is None
        assert ma[..., 2].any() and np.array_equal(ma, mb)
    a.close(); b.close()


def test_quickshift_device_refuses_short_stride():
    """pcm_quickshift_device refuses a row stride below 3 * W, as pcm_quickshift and the GPU SLIC entry points do."""
    import ctypes as C
    import torch
    from pcm import capi
    H, W = 24, 32
    d_frame = torch.zeros(H * W * 3, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    h = capi.Handle(0)
    n = C.c_int(0)
    rc = h.lib.pcm_quickshift_device(h._h, C.c_void_p(d_frame.data_ptr()), H, W, 3 * W - 3, (C.c_int * 4)(0, 0, W, H), 0.5, 3.0,
                                     6.0, None, None, C.byref(n))
    assert rc == -1 and b"pcm_quickshift_device" in h.lib.pcm_last_error()
    h.close()


def test_quickshift_device_batch_equals_single_crops():
    """pcm_quickshift_device_batch (the label maps of many crops of a device-resident clip in one native call, what the
    sweep uses per clip) against pcm_quickshift per crop on the host frames: same maps, same counts, crops of
    different sizes and frames in any order; the sequence tie noise is the first h*w values of one stream."""
    import torch
    from pcm import capi
    frames = read_video("Video", "frog")[:4]
    H, W = frames[0].shape[:2]
    rects = [(150, 60, 133, 159), (10, 5, 64, 48), (200, 100, 90, 120), (0, 0, 40, 33), (301, 77, 55, 61)]
    index = [0, 3, 1, 2, 3]
    sizes = [r[2] * r[3] for r in rects]
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    noise = np.random.RandomState(42).normal(scale=0.00001, size=max(sizes))
    d_frames = torch.from_numpy(np.stack(frames)).cuda()
    d_noise = torch.from_numpy(noise).cuda()
    d_labels = torch.full((int(offsets[-1]),), -7, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    h = capi.Handle(0)
    h.set_features(8, ["hsv", "lab"])
    counts = h.quickshift_device_batch(d_frames.data_ptr(), H * W * 3, index, H, W, W * 3, rects, 0.5, 3, 6,
                                       d_noise.data_ptr(), d_labels.data_ptr(), offsets[:-1])
    got = d_labels.cpu().numpy()
    for k, r in enumerate(rects):
        want, n = h.quickshift(frames[index[k]], r, noise=noise[:sizes[k]].reshape(r[3], r[2]))
        assert counts[k] == n
        assert np.array_equal(got[offsets[k]:offsets[k + 1]].reshape(r[3], r[2]), want)
    assert len(h.quickshift_device_batch(d_frames.data_ptr(), H * W * 3, [], H, W, W * 3, [], 0.5, 3, 6, d_noise.data_ptr(),
                                         d_labels.data_ptr(), [])) == 0
    with pytest.raises(capi.PcmError):
        h.quickshift_device_batch(d_frames.data_ptr(), H * W * 3, [0], H, W, W * 3, [(470, 0, 40, 40)], 0.5, 3, 6, d_noise.data_ptr(),
                                  d_labels.data_ptr(), [0])
    h.close()
