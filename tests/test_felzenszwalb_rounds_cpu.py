"""The round rule of the GPU Felzenszwalb (oracle/felzenszwalb_rounds.py, the rule csrc/pcm_felzenszwalb.cuh runs) gives
the partition of the sequential passes of oracle/felzenszwalb_oracle.py, and the GPU entry points refuse NULL arguments
before touching a device.  Runs without a GPU."""
import ctypes as C

import numpy as np
import pytest

import felzenszwalb_oracle as fo
import felzenszwalb_rounds as fr
from helpers import read_video


def image_edges(img, sigma):
    """The edges of an HxWx3 u8 image as felzenszwalb_oracle.felzenszwalb builds them, in the stable cost order:
    (e0, e1, costs, n_vertices)."""
    image = fo.smooth(img, sigma)
    h, w = image.shape[:2]

    def cost(a, b):
        d = a - b
        return np.sqrt((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2])
    seg = np.arange(h * w).reshape(h, w)
    costs = np.concatenate([cost(image[:, 1:], image[:, :w - 1]).ravel(), cost(image[1:], image[:h - 1]).ravel(),
                            cost(image[1:, 1:], image[:h - 1, :w - 1]).ravel(),
                            cost(image[1:, :w - 1], image[:h - 1, 1:]).ravel()])
    e0 = np.concatenate([seg[:, 1:].ravel(), seg[1:].ravel(), seg[1:, 1:].ravel(), seg[:h - 1, 1:].ravel()])
    e1 = np.concatenate([seg[:, :w - 1].ravel(), seg[:h - 1].ravel(), seg[:h - 1, :w - 1].ravel(), seg[1:, :w - 1].ravel()])
    order = np.argsort(costs, kind="stable")
    return e0[order], e1[order], costs[order], h * w


def image_cases():
    """(name, frame, rect, kwargs) of every case of test_felzenszwalb_cpu.py."""
    rng = np.random.default_rng(17)
    g = np.add.outer(np.arange(96), np.arange(120)).astype(np.uint8)
    out = [("soldier", read_video("Video", "soldier")[0], (300, 0, 139, 224), {}),
           ("frog", read_video("Video", "frog")[3], (150, 60, 133, 159), {}),
           ("parachute", read_video("Video", "parachute")[5], (0, 0, 414, 352), {}),
           ("noise", rng.integers(0, 256, (70, 90, 3), dtype=np.uint8), (3, 5, 81, 60), {}),
           ("flat", np.full((40, 50, 3), 99, np.uint8), (0, 0, 50, 40), {}),
           ("gradient", np.stack([g, g[::-1], 255 - g], -1).copy(), (10, 7, 100, 80), {}),
           ("tiny", rng.integers(0, 256, (6, 7, 3), dtype=np.uint8), (1, 2, 3, 2), {}),
           ("other_params", rng.integers(0, 64, (60, 60, 3), dtype=np.uint8), (0, 0, 60, 60),
            dict(scale=1, sigma=0.8, min_size=20))]
    frame = np.random.default_rng(23).integers(0, 256, (32, 40, 3), dtype=np.uint8)
    for rect in [(4, 3, 1, 20), (2, 5, 30, 1), (7, 7, 1, 1), (0, 0, 2, 2)]:
        out.append(("degenerate_%dx%d" % (rect[2], rect[3]), frame, rect, dict(scale=100, sigma=0.5, min_size=3)))
    return out


def graph_cases():
    """(name, n_vertices, e0, e1, costs in the stable cost order, scale, min_size) of the explicit edge lists: the four
    edge-order cases of test_felzenszwalb_cpu.py, a path with strictly increasing costs (all merged / all rejected),
    scale 0 and min_size above the vertex count."""
    rng = np.random.default_rng(5)
    h, w = 30, 41
    seg = np.arange(h * w).reshape(h, w)
    e0 = np.concatenate([seg[:, 1:].ravel(), seg[1:].ravel(), seg[1:, 1:].ravel(), seg[:h - 1, 1:].ravel()])
    e1 = np.concatenate([seg[:, :w - 1].ravel(), seg[:h - 1].ravel(), seg[:h - 1, :w - 1].ravel(), seg[1:, :w - 1].ravel()])
    n = e0.size
    lists = {"lower_half_ties": (np.float64(0.25).view(np.uint64) + rng.integers(0, 2 ** 32, n, dtype=np.uint64)).view(np.float64),
             "few_distinct": rng.choice(np.array([0.0, 0.125, 0.1250000001, 0.3, 1.7]), n),
             "zeros_and_tiny": np.where(rng.random(n) < 0.5, 0.0, rng.random(n) * 1e-300),
             "wide_range": np.exp(rng.uniform(-40, 1, n))}
    out = []
    for name, costs in lists.items():
        order = np.argsort(costs, kind="stable")
        for scale, min_size in ((0.4, 1), (0.05, 12)):
            out.append(("%s_%g_%d" % (name, scale, min_size), h * w, e0[order], e1[order], costs[order], scale, min_size))
    m = 300
    path = np.arange(m - 1)
    rising = (path + 1) * 1e-4
    out.append(("path_merging", m, path, path + 1, rising, 1000.0, 1))
    out.append(("path_rejecting", m, path, path + 1, rising, 1e-6, 1))
    costs = lists["wide_range"]
    order = np.argsort(costs, kind="stable")
    out.append(("scale_0", h * w, e0[order], e1[order], costs[order], 0.0, 5))
    out.append(("min_size_above_n", h * w, e0[order], e1[order], costs[order], 0.05, h * w + 7))
    return out


def _same_partition_as_merge(e0, e1, costs, n, scale, min_size):
    root, merge, small = fr.merge_rounds(e0, e1, costs, n, scale, min_size)
    want = fo._merge(np.asarray(e0, np.int64), np.asarray(e1, np.int64), np.asarray(costs, np.float64), n, scale, min_size)
    assert np.array_equal(root, want)
    return merge, small


@pytest.mark.parametrize("case", image_cases(), ids=lambda c: c[0])
def test_rounds_give_the_sequential_partition_on_images(case):
    name, frame, rect, kw = case
    x, y, w, h = rect
    e0, e1, costs, n = image_edges(frame[y:y + h, x:x + w], kw.get("sigma", 0.5))
    merge, small = _same_partition_as_merge(e0, e1, costs, n, kw.get("scale", 100) / 255.0, kw.get("min_size", 50))
    if name == "flat":                         # every cost is zero: all merges, no min-size work
        assert small == 0


@pytest.mark.parametrize("case", graph_cases(), ids=lambda c: c[0])
def test_rounds_give_the_sequential_partition_on_edge_lists(case):
    name, n, e0, e1, costs, scale, min_size = case
    merge, small = _same_partition_as_merge(e0, e1, costs, n, scale, min_size)
    if name == "path_merging":                 # each edge waits for the previous one: one merge round per edge
        assert merge == e0.size
    elif name == "path_rejecting":             # every edge is a certain rejection in the first round
        assert merge == 1


def test_gpu_entry_points_refuse_null_without_a_device():
    from pcm import capi
    lib = capi.load_library()
    r = (C.c_int * 4)(0, 0, 4, 4)
    n = C.c_int(0)
    assert lib.pcm_felzenszwalb_gpu(None, None, 4, 4, 12, r, 100.0, 0.5, 50, None, 0, None, C.byref(n)) == -1
    assert b"pcm_felzenszwalb_gpu" in lib.pcm_last_error()
    assert lib.pcm_felzenszwalb_device(None, None, 4, 4, 12, r, 100.0, 0.5, 50, None, 0, None, C.byref(n)) == -1
    assert b"pcm_felzenszwalb_device" in lib.pcm_last_error()
    assert lib.pcm_felzenszwalb_device_batch(None, 1, None, 48, None, 4, 4, 12, None, 100.0, 0.5, 50, None, 0, None, None,
                                             None) == -1
    assert b"pcm_felzenszwalb_device_batch" in lib.pcm_last_error()
    assert lib.pcm_felzenszwalb_graph_gpu(None, 4, 0, None, None, None, 1.0, 1, None, C.byref(n)) == -1
    assert b"pcm_felzenszwalb_graph_gpu" in lib.pcm_last_error()
    assert lib.pcm_felzenszwalb_debug_last(None, None, None) == -1
    assert b"pcm_felzenszwalb_debug_last" in lib.pcm_last_error()
