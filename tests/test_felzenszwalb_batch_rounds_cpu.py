"""The batched GPU Felzenszwalb (pcm_felzenszwalb_device_batch) runs many crops as one graph of disjoint pieces: their edge
lists concatenated with index offsets and sorted once, stably.  Restated here with oracle/felzenszwalb_rounds.py: the
partition of that union, restricted to each crop, is the crop's own, and the union takes as many merge and min-size
rounds as its slowest crop.  Runs without a GPU."""
import cv2 as cv
import numpy as np
import pytest

import felzenszwalb_oracle as fo
import felzenszwalb_rounds as fr
from helpers import read_video
from test_felzenszwalb_rounds_cpu import image_cases, image_edges


def edge_order_edges(img, sigma):
    """The edges of an HxWx3 u8 image in the host's edge order (right, down, down-right, up-right; raster order within
    a class), before the sort: (e0, e1, costs, n_vertices)."""
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
    return e0, e1, costs, h * w


def segtrack_crops(video, frames):
    """(name, frame, rect) of the sweep's crops of `video` at the given frames: boxes from the ground truth."""
    from pcm import capi
    out = []
    for i in frames:
        f, t = read_video("Video", video)[i], read_video("Truth", video)[i]
        pts = cv.findNonZero((cv.cvtColor(t, cv.COLOR_BGR2GRAY) > 0).astype(np.uint8))
        box = cv.boundingRect(pts) if pts is not None else (0, 0, f.shape[1], f.shape[0])
        out.append(("%s_%d" % (video, i), f, capi.crop_rect(box, f.shape[0], f.shape[1])))
    return out


def batches():
    """(name, [(frame, rect)], scale, sigma, min_size): the image cases of test_felzenszwalb_rounds_cpu.py grouped by
    their arguments (a batch shares them), with SegTrack2 crops and 1x1 / 1xN / Nx1 crops."""
    groups = {}
    for name, frame, rect, kw in image_cases():
        key = (kw.get("scale", 100), kw.get("sigma", 0.5), kw.get("min_size", 50))
        groups.setdefault(key, []).append((frame, rect))
    out = []
    for (scale, sigma, min_size), crops in sorted(groups.items()):
        out.append(("cases_%g_%g_%d" % (scale, sigma, min_size), crops, scale, sigma, min_size))
    rng = np.random.default_rng(31)
    frame = rng.integers(0, 256, (24, 30, 3), dtype=np.uint8)
    thin = [(frame, (0, 0, 1, 1)), (frame, (5, 2, 1, 17)), (frame, (3, 9, 25, 1)), (frame, (29, 23, 1, 1))]
    seg = [(f, r) for _, f, r in segtrack_crops("bmx", [0, 9, 18]) + segtrack_crops("worm", [4, 40])]
    out.append(("segtrack2_and_thin", thin[:2] + seg[:3] + thin[2:] + seg[3:], 100, 0.5, 50))
    out.append(("thin_only", thin, 100, 0.5, 50))
    out.append(("segtrack2_sigma0", seg[:3], 300, 0.0, 20))
    return out


@pytest.mark.parametrize("batch", batches(), ids=lambda b: b[0])
def test_batch_is_the_disjoint_union_of_its_crops(batch):
    _, crops, scale, sigma, min_size = batch
    parts, solo, base = [], [], 0
    for frame, (x, y, w, h) in crops:
        crop = np.ascontiguousarray(frame[y:y + h, x:x + w])
        e0, e1, costs, n = edge_order_edges(crop, sigma)
        parts.append((e0 + base, e1 + base, costs))
        solo.append((base, n, fr.merge_rounds(*image_edges(crop, sigma), scale / 255.0, min_size)))
        base += n
    e0 = np.concatenate([p[0] for p in parts])
    e1 = np.concatenate([p[1] for p in parts])
    costs = np.concatenate([p[2] for p in parts])
    order = np.argsort(costs, kind="stable")          # crop after crop before the sort: each crop keeps its own order
    root, merge, small = fr.merge_rounds(e0[order], e1[order], costs[order], base, scale / 255.0, min_size)
    for b, n, (root_k, _, _) in solo:
        assert np.array_equal(root[b:b + n] - b, root_k)
    assert merge == max(s[2][1] for s in solo)
    assert small == max(s[2][2] for s in solo)
