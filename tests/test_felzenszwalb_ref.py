"""pcm_felzenszwalb against the Felzenszwalb-Huttenlocher code the reference vendors
(prim/src/FelzenSegment: segment-graph.h:48-81, segment_image_index.h:14-121), compiled from a
checkout of the reference named by PCM_REFERENCE_ROOT into oracle/_ref/libfelzen_ref.so; without
one, against oracle/felzen_fh_restated.cpp, the published algorithm restated with the same
arithmetic and entry points (oracle/build_ref.py).  SURVEY §8 row f-1.

What coincides between that code and the scikit-image variant the product implements is checked
EXACTLY on identical edge lists: the cost-ordered greedy merge with the k/|C| threshold, the
union-find bookkeeping and the min-size pass (`pcm_felzenszwalb_graph`, a parity tap of the
library that runs the same code as `pcm_felzenszwalb` after its edge construction).  What does
not coincide (float32 vs float64 pixels, Gaussian normalisation and border, tie order of equal
costs, `<=` vs `<`) is checked structurally on SegTrack2 crops; against scikit-image itself the
stage stays "parity unpinned".  Runs without a GPU."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from helpers import read_video

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "oracle"))
import build_ref  # noqa: E402


@pytest.fixture(scope="module")
def ref():
    path, _ = build_ref.build()
    lib = C.CDLL(path)
    P, I, F = C.c_void_p, C.c_int, C.c_float
    lib.felzen_ref_graph.restype = I
    lib.felzen_ref_graph.argtypes = [I, I, P, P, P, F, I, P]
    lib.felzen_ref_image.restype = I
    lib.felzen_ref_image.argtypes = [P, I, I, F, F, I, P]
    return lib


def first_appearance(labels):
    """Relabel so that components are numbered in order of first appearance."""
    _, first, inv = np.unique(labels, return_index=True, return_inverse=True)
    order = np.argsort(np.argsort(first))
    return order[inv].astype(np.int32)


def grid_edges(h, w, rng):
    """8-connected grid graph with DISTINCT float32 costs (no ties: the sort order is unique)."""
    idx = np.arange(h * w).reshape(h, w)
    a = np.concatenate([idx[:, 1:].ravel(), idx[1:, :].ravel(), idx[1:, 1:].ravel(), idx[:-1, 1:].ravel()])
    b = np.concatenate([idx[:, :-1].ravel(), idx[:-1, :].ravel(), idx[:-1, :-1].ravel(), idx[1:, :-1].ravel()])
    # smooth field + noise so that real multi-pixel components form
    field = rng.random((h, w)).astype(np.float64)
    for _ in range(3):
        field = (field + np.roll(field, 1, 0) + np.roll(field, 1, 1)) / 3
    cost = (np.abs(field.ravel()[a] - field.ravel()[b]) * 40 + rng.random(a.size) * 1e-3).astype(np.float32)
    # force distinct values: sort, and nudge duplicates up by one ulp until all differ
    order = np.argsort(cost, kind="stable")
    s = cost[order]
    for i in range(1, s.size):
        if s[i] <= s[i - 1]:
            s[i] = np.nextafter(s[i - 1], np.float32(np.inf))
    cost[order] = s
    assert np.unique(cost).size == cost.size
    return a.astype(np.int32), b.astype(np.int32), cost


@pytest.mark.parametrize("seed,h,w,c,min_size", [(0, 40, 60, 1.0, 20), (1, 64, 48, 0.5, 50), (2, 33, 77, 3.0, 1),
                                                  (3, 90, 90, 0.2, 50), (4, 25, 31, 100.0, 10)])
def test_merge_unionfind_minsize_equal_the_reference_on_identical_edges(ref, seed, h, w, c, min_size):
    from pcm import capi
    rng = np.random.default_rng(seed)
    a, b, cost = grid_edges(h, w, rng)
    perm = rng.permutation(a.size)                      # neither side may depend on the input order
    a, b, cost = a[perm].copy(), b[perm].copy(), cost[perm].copy()
    want = np.empty(h * w, np.int32)
    n_ref = ref.felzen_ref_graph(h * w, a.size, a.ctypes.data, b.ctypes.data, cost.ctypes.data, c, min_size, want.ctypes.data)
    assert n_ref > 0
    got, n = capi.felzenszwalb_graph(h * w, a, b, cost.astype(np.float64), c, min_size)
    assert n == n_ref
    assert 1 < n < h * w or c >= 100.0
    assert np.array_equal(first_appearance(got), want)


@pytest.mark.parametrize("clip", ["soldier", "frog", "parachute", "worm", "bmx"])
def test_whole_image_agrees_with_the_reference(ref, clip):
    """Same parameters as the masker's call (scale 100 == k 100 on 0..255 pixels, sigma 0.5, min_size 50).
    The two variants are not the same arithmetic (float32 vs float64 pixels, Gaussian normalisation and
    border, `<=` vs `<`, tie order), yet on SegTrack2 crops they carve the image into the SAME partition
    almost always: measured here over 12 crops per clip, 56 of 60 partitions are identical and the others
    differ in < 1.3 % of the pixels with equal segment counts.  Asserted: equal counts within 1 %, at most
    2 % of the pixels in differently numbered segments, and most crops of a clip identical."""
    from pcm import capi
    video = read_video("Video", clip)
    H, W = video[0].shape[:2]
    identical = total = 0
    for frame in (0, 5, 11, 17):
        for rect in ((0, 0, W, H), (W // 4, H // 4, W // 2, H // 2), (10, 7, min(150, W - 10), min(131, H - 7))):
            img = video[frame]
            x, y, w, h = rect
            got, n = capi.felzenszwalb(img, rect, scale=100, sigma=0.5, min_size=50)
            crop_rgb = np.ascontiguousarray(img[y:y + h, x:x + w, ::-1])
            want = np.empty((h, w), np.int32)
            n_ref = ref.felzen_ref_image(crop_rgb.ctypes.data, h, w, 0.5, 100.0, 50, want.ctypes.data)
            assert n_ref > 0 and abs(n - n_ref) <= max(1, n_ref // 100), (clip, frame, rect, n, n_ref)
            differing = float(np.mean(first_appearance(got.ravel()) != want.ravel()))
            assert differing <= 0.02, (clip, frame, rect, differing)
            identical += differing == 0.0
            total += 1
    assert identical >= total - 3, (clip, identical, total)
