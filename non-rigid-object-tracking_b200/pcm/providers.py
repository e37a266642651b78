"""Pluggable providers for the two third-party stages the reference takes from
packages that are not in this image (SURVEY.md §8c "parity unpinned"):

  * over-segmentation (skimage quickshift/felzenszwalb/slic,
    reference maskers/pixel_classification.py:70-75)  -> label providers here;
  * the rigid tracker (cv.legacy CSRT, reference main.py:258-261,287)
    -> bbox providers here.

Both sides of every parity test consume the SAME provider output.
"""
import cv2 as cv
import numpy as np


def grid_segments(crop, block=16):
    """Deterministic block-grid label map, labels 0..S-1 in raster order of blocks."""
    h, w = crop.shape[:2]
    nbx = (w + block - 1) // block
    r = np.arange(h, dtype=np.int32)[:, None] // block
    c = np.arange(w, dtype=np.int32)[None, :] // block
    return (r * nbx + c).astype(np.int32)


def voronoi_segments(crop, n_sites=200, seed=0):
    """Seeded random-Voronoi label map (irregular superpixel shapes), labels 0..S-1."""
    h, w = crop.shape[:2]
    rng = np.random.default_rng(seed + 7919 * h + w)
    n = max(1, min(n_sites, h * w))
    sy = rng.integers(0, h, n)
    sx = rng.integers(0, w, n)
    yy, xx = np.mgrid[0:h, 0:w]
    best = np.full((h, w), np.iinfo(np.int64).max, np.int64)
    lab = np.zeros((h, w), np.int32)
    for i in range(n):
        d = (yy - sy[i]) ** 2 + (xx - sx[i]) ** 2
        m = d < best
        best[m] = d[m]
        lab[m] = i
    _, inv = np.unique(lab, return_inverse=True)
    return inv.reshape(h, w).astype(np.int32)


def make_segment_provider(name, **kw):
    """Resolve `params.over_segmentation` (config.yaml:29) to a label provider.

    'grid[:block]' and 'voronoi[:sites]' are deterministic test providers.  The reference's names ('quickshift',
    'felzenszwalb', 'SLIC') normally never get here -- the masker runs all three natively on the GPU (pcm_quickshift /
    pcm_felzenszwalb_gpu / pcm_slic_gpu, SURVEY.md §8 f-1); asked for explicitly they map to the grid
    provider with a block size giving a comparable superpixel count.
    """
    name = str(name)
    if name.startswith("grid"):
        block = int(name.split(":")[1]) if ":" in name else kw.get("block", 16)
        return lambda crop: grid_segments(crop, block)
    if name.startswith("voronoi"):
        sites = int(name.split(":")[1]) if ":" in name else kw.get("n_sites", 200)
        return lambda crop: voronoi_segments(crop, sites, kw.get("seed", 0))
    if name in ("quickshift", "felzenszwalb", "SLIC"):
        block = {"quickshift": 6, "felzenszwalb": 10, "SLIC": 12}[name]
        return lambda crop: grid_segments(crop, block)
    raise ValueError("unknown over_segmentation %r" % name)


def truth_boxes(truth_frames, fallback):
    """Per-frame (x, y, w, h) = bounding rectangle of the ground-truth mask
    (gray > 127); frames with an empty truth reuse the previous box."""
    boxes = []
    prev = tuple(int(v) for v in fallback)
    for t in truth_frames:
        # OpenCV end to end (no index arrays, no interpreter lock held for the frame): the sweep computes the boxes of
        # a clip on the thread every sequence of the clip waits for
        g = t if t.ndim == 2 else cv.extractChannel(t, 0)
        x, y, w, h = cv.boundingRect(cv.threshold(np.ascontiguousarray(g), 127, 255, cv.THRESH_BINARY)[1])
        if w > 0 and h > 0:
            prev = (int(x), int(y), int(w), int(h))
        boxes.append(prev)
    return boxes


class ScriptedBoxTracker:
    """Stand-in for cv.legacy.MultiTracker (main.py:258-261,287): replays a list
    of per-frame boxes for each target."""

    def __init__(self, boxes_per_target):
        self.boxes = boxes_per_target
        self.i = 0

    def update(self, frame):
        i = min(self.i, len(self.boxes[0]) - 1)
        self.i += 1
        return True, [b[i] for b in self.boxes]
