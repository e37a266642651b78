"""The batched GPU Felzenszwalb (pcm_felzenszwalb_device_batch: many crops in one pass, their merge rounds shared) gives,
crop for crop, the labels and count of the host pcm_felzenszwalb, and the round counts of oracle/felzenszwalb_rounds.py."""
import ctypes as C

import numpy as np
import pytest

import felzenszwalb_oracle as fo
import felzenszwalb_rounds as fr
from helpers import read_video
from test_felzenszwalb_rounds_cpu import image_edges
from test_gpu_felzenszwalb import _truth_rects

pytestmark = pytest.mark.gpu

CHUNK_PIXELS = 1 << 23                  # the chunk bound of pcm_felzenszwalb_device_batch (include/pcm_b200.h)
SENTINEL = -7


@pytest.fixture(scope="module")
def handle():
    from pcm import capi
    h = capi.Handle(0)
    yield h
    h.close()


def _run_batch(h, frames, items, scale=100, sigma=0.5, min_size=50, offsets=None, total=None):
    """items: (frame index, rect).  Uploads the frames, runs one batch into a sentinel-filled buffer and returns
    (flat labels on the host, counts, offsets)."""
    import torch
    H, W = frames[0].shape[:2]
    d_frames = torch.from_numpy(np.stack(frames)).cuda()
    sizes = [r[2] * r[3] for _, r in items]
    if offsets is None:
        offsets = np.concatenate([[0], np.cumsum(sizes)])[:len(items)].astype(np.int64)
        total = int(sum(sizes))
    d = torch.full((max(total, 1),), SENTINEL, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    counts = h.felzenszwalb_device_batch(d_frames.data_ptr(), H * W * 3, [i for i, _ in items], H, W, W * 3, [r for _, r in items],
                                         d.data_ptr(), offsets, scale=scale, sigma=sigma, min_size=min_size)
    return d.cpu().numpy(), counts, offsets


def _assert_host_equal(frames, items, flat, counts, offsets, **kw):
    from pcm import capi
    for k, (i, r) in enumerate(items):
        want, n_want = capi.felzenszwalb(frames[i], r, **kw)
        got = flat[offsets[k]:offsets[k] + r[2] * r[3]].reshape(r[3], r[2])
        assert counts[k] == n_want and np.array_equal(got, want), "crop %d %s differs from pcm_felzenszwalb" % (k, r)


@pytest.mark.parametrize("video", ["soldier", "bmx", "frog", "worm"])
def test_batch_equals_host_on_every_sweep_crop(handle, video):
    """Every frame of the clip, cropped by the box of its ground truth, in one batch."""
    crops = _truth_rects(video)
    frames = [f for f, _ in crops]
    items = [(k, r) for k, (_, r) in enumerate(crops)]
    flat, counts, offsets = _run_batch(handle, frames, items)
    _assert_host_equal(frames, items, flat, counts, offsets)


@pytest.mark.parametrize("args", [dict(sigma=0.0), dict(sigma=0.5), dict(sigma=2.0), dict(scale=300, sigma=0.8, min_size=20)],
                         ids=["sigma0", "sigma0.5", "sigma2", "other_params"])
def test_batch_of_mixed_crops(handle, args):
    """1x1, 1xN, Nx1 and flat crops among SegTrack2 crops; a frame used several times; label offsets out of order, with
    gaps that the batch must leave untouched."""
    frames = read_video("Video", "bmx")[:3]
    flat_frame = np.full_like(frames[0], 77)
    frames = frames + [flat_frame]
    H, W = frames[0].shape[:2]
    items = [(0, (10, 20, 1, 1)), (1, (200, 60, 300, 240)), (1, (0, 5, 1, 90)), (2, (40, 100, 120, 1)),
             (3, (0, 0, 64, 48)), (1, (150, 30, 200, 200)), (0, (W - 1, H - 1, 1, 1)), (2, (0, 0, W, H))]
    sizes = [r[2] * r[3] for _, r in items]
    gap = 13
    order = [5, 2, 7, 0, 3, 6, 1, 4]                        # where crop k's map goes, back to front with gaps
    offsets = np.zeros(len(items), np.int64)
    at = 0
    for k in order:
        offsets[k] = at
        at += sizes[k] + gap
    flat, counts, offsets = _run_batch(handle, frames, items, offsets=offsets, total=at, **args)
    kw = dict(scale=100, sigma=0.5, min_size=50)
    kw.update(args)
    _assert_host_equal(frames, items, flat, counts, offsets, **kw)
    written = np.zeros(at, bool)
    for k, s in enumerate(sizes):
        written[offsets[k]:offsets[k] + s] = True
    assert (flat[~written] == SENTINEL).all(), "the batch wrote into the gaps between label maps"
    assert counts[4] == 1                                   # the flat crop is one segment


def _hd_frames(n):
    rng = np.random.default_rng(11)
    yy, xx = np.mgrid[0:1080, 0:1920]
    out = []
    for i in range(n):
        base = np.stack([(xx * 255) // 1919, (yy * 255) // 1079, ((xx + yy) * (3 + i)) % 256], -1)
        out.append(np.clip(base + rng.integers(-24, 25, base.shape), 0, 255).astype(np.uint8))
    return out


def test_batch_above_the_chunk_bound(handle):
    """Five 1080p frames and small crops: more pixels than one chunk holds, so the batch runs in several chunks."""
    frames = _hd_frames(5)
    items = [(0, (5, 7, 60, 40)), (0, (0, 0, 1920, 1080)), (1, (0, 0, 1920, 1080)), (2, (300, 200, 1, 1)),
             (2, (0, 0, 1920, 1080)), (3, (0, 0, 1920, 1080)), (4, (100, 50, 90, 120)), (4, (0, 0, 1920, 1080)),
             (1, (1000, 500, 33, 1))]
    assert sum(r[2] * r[3] for _, r in items) > CHUNK_PIXELS
    flat, counts, offsets = _run_batch(handle, frames, items)
    _assert_host_equal(frames, items, flat, counts, offsets, scale=100, sigma=0.5, min_size=50)


def test_debug_last_after_a_batch(handle):
    """Round counts = the largest of merge_rounds's over the batch's crops; smoothed = the last crop's, bit for bit."""
    crops = _truth_rects("soldier")[::5]
    frames = [f for f, _ in crops]
    items = [(k, r) for k, (_, r) in enumerate(crops)]
    _run_batch(handle, frames, items)
    d = handle.felzenszwalb_debug_last()
    rounds = []
    for f, (x, y, w, h) in crops:
        crop = np.ascontiguousarray(f[y:y + h, x:x + w])
        _, r_merge, r_small = fr.merge_rounds(*image_edges(crop, 0.5), 100 / 255.0, 50)
        rounds.append((r_merge, r_small))
    assert d["rounds"] == (max(r[0] for r in rounds), max(r[1] for r in rounds))
    x, y, w, h = crops[-1][1]
    assert np.array_equal(d["smoothed"], fo.smooth(np.ascontiguousarray(frames[-1][y:y + h, x:x + w]), 0.5))


def test_batch_launches_grow_with_chunks_not_crops(handle):
    frame = read_video("Video", "frog")[0]
    one = [(0, (40, 30, 100, 80))]
    many = [(0, (40 + k % 50, 30 + k % 40, 100, 80)) for k in range(279)]
    deltas = []
    for items, frames in ((one, [frame]), (many, [frame]), (one, [frame])):
        before = handle.launch_count
        _run_batch(handle, frames, items)
        deltas.append(handle.launch_count - before)
    assert deltas[0] == deltas[1] == deltas[2] > 0          # 279 crops, one chunk: the launches of one crop
    before = handle.launch_count
    hd = [(k, (0, 0, 1920, 1080)) for k in range(5)]
    _run_batch(handle, _hd_frames(5), hd)
    assert handle.launch_count - before == 2 * deltas[0]  # two chunks


def test_batch_errors(handle):
    import torch
    from pcm import capi
    lib = capi.load_library()
    H, W = 16, 20
    d_frames = torch.zeros((2, H, W, 3), dtype=torch.uint8, device="cuda")
    d = torch.zeros(4 * H * W, dtype=torch.int32, device="cuda")
    counts = np.zeros(2, np.int32)

    def batch(n=2, frames=True, fi=(0, 1), rects=((0, 0, W, H), (2, 3, 5, 4)), offsets=(0, H * W), out=True):
        fi = np.asarray(fi, np.int32)
        rc = np.asarray(rects, np.int32).reshape(-1)
        off = np.asarray(offsets, np.int64)
        return lib.pcm_felzenszwalb_device_batch(handle._h, n, C.c_void_p(d_frames.data_ptr()) if frames else None, H * W * 3,
                                                 fi.ctypes.data_as(C.c_void_p), H, W, 3 * W, rc.ctypes.data_as(C.c_void_p),
                                                 100.0, 0.5, 50, None, 0, C.c_void_p(d.data_ptr()),
                                                 off.ctypes.data_as(C.c_void_p), counts.ctypes.data_as(C.c_void_p) if out else None)
    assert batch() == 0 and counts[0] >= 1 and counts[1] >= 1
    assert batch(frames=False) == -1 and b"pcm_felzenszwalb_device_batch" in lib.pcm_last_error()
    assert batch(out=False) == -1 and b"pcm_felzenszwalb_device_batch" in lib.pcm_last_error()
    assert batch(fi=(0, -1)) == -1 and b"negative index" in lib.pcm_last_error()
    assert batch(offsets=(-4, 0)) == -1 and b"negative index" in lib.pcm_last_error()
    assert batch(rects=((0, 0, W, H), (2, 3, W, 4))) == -1
    msg = lib.pcm_last_error()
    assert b"pcm_felzenszwalb_device_batch" in msg and b"crop 1" in msg
    assert batch(rects=((0, 0, 0, H), (2, 3, 5, 4))) == -1 and b"crop 0" in lib.pcm_last_error()
    assert batch(n=-1) == -1
    assert batch(n=0) == 0


def test_batch_ends_a_pending_handoff():
    """A handle with no pcm_update yet whose last call (Handle.felzenszwalb) left a handoff pending: after a batch,
    update(labels=None) is refused with PCM_E_STATE."""
    import torch
    from pcm import capi
    from test_gpu_parity import _random_forest_arrays
    rng = np.random.default_rng(4)
    frame = read_video("Video", "worm")[10]
    rect = capi.crop_rect((120, 110, 140, 70), frame.shape[0], frame.shape[1])
    h = capi.Handle(0)
    h.set_features(6, ["lab"])
    h.add_model_arrays(0, _random_forest_arrays(rng, 10, 5, 3 * 49))
    prm = capi.Handle.make_params(0, dilation_kernel=7)
    _, n = h.felzenszwalb(frame, rect)
    H, W = frame.shape[:2]
    d_frames = torch.from_numpy(frame[None].copy()).cuda()
    d = torch.empty(rect[2] * rect[3], dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    counts = h.felzenszwalb_device_batch(d_frames.data_ptr(), H * W * 3, [0], H, W, W * 3, [rect], d.data_ptr(), [0])
    assert counts[0] == n
    with pytest.raises(capi.PcmError) as e:
        h.update(frame, rect, None, n, None, prm, np.zeros_like(frame))
    assert e.value.code == -3
    h.close()
