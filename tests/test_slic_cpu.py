"""pcm_slic (host code of the library, SURVEY §8 row f-1) against the restatement of scikit-image 0.17.2's SLIC in
oracle/slic_oracle.py -- PARITY UNPINNED against scikit-image itself (not installed, not vendored, no reference vectors);
the Gaussian step of the oracle is the scipy-exact one of the felzenszwalb oracle.  Runs without a GPU."""
import numpy as np
import pytest
import scipy.ndimage as ndi

import slic_oracle as so
from helpers import read_video


def test_oracle_gaussian_step_equals_scipy():
    rng = np.random.default_rng(3)
    for shape in [(37, 53, 3), (5, 4, 3), (64, 9, 3)]:
        img = rng.integers(0, 256, shape, dtype=np.uint8)
        want = ndi.gaussian_filter((img.astype(np.float64) / 255.0)[np.newaxis], sigma=[1, 1, 1, 0])[0]
        assert np.array_equal(so.smooth(img, 1.0), want), shape


def test_oracle_grid_is_regular_grid():
    # 224 x 139 crop, 250 seeds: step = round(sqrt(224 * 139 / 250)) = 11, start = 11.16 // 2 = 5
    assert so.grid_steps(224, 139, 250) == (5, 11, 5, 11)
    assert so.grid_steps(10, 10, 250) is None
    sy, ty, sx, tx = so.grid_steps(3, 4000, 250)            # the short axis is shorter than the square-root step
    assert (sy, ty) == (1, 3) and tx == round(4000 / 250)


def _check(frame, rect, **kw):
    from pcm import capi
    x, y, w, h = rect
    want = so.slic(frame[y:y + h, x:x + w], n_segments=kw.get("n_segments", 250), compactness=kw.get("compactness", 10.0),
                   sigma=kw.get("sigma", 1.0), max_iter=kw.get("max_iter", 10), start_label=kw.get("start_label", 0))
    got, n = capi.slic(frame, rect, **kw)
    assert n == int(want.max()) + 1
    assert np.array_equal(got, want)
    return got, n


def test_slic_segtrack_crops():
    got, n = _check(read_video("Video", "soldier")[0], (300, 0, 139, 224))      # the default config's crop
    assert 150 < n < 300                                                        # about the 250 segments asked for
    # every segment is 4-connected (that is what the connectivity pass is for)
    lab, cnt = ndi.label(np.ones_like(got))
    for s in range(n):
        assert ndi.label(got == s)[1] == 1, s
    _check(read_video("Video", "frog")[3], (150, 60, 133, 159))
    _check(read_video("Video", "parachute")[5], (0, 0, 414, 352))


@pytest.mark.parametrize("case", ["noise", "flat", "gradient", "tiny", "other_params", "wide"])
def test_slic_synthetic(case):
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
    _check(frame, rect, **kw)


def test_slic_refuses_bad_arguments():
    """pcm_slic checks its arguments before it runs: PCM_E_INVALID (-1), or PCM_E_LIMIT (-4) above 2^28 pixels, with a
    message that names it."""
    import ctypes as C
    from pcm import capi
    lib = capi.load_library()
    frame = np.zeros((16, 16, 3), np.uint8)
    out = np.empty(16 * 16, np.int32)
    weights = np.full(3, 1.0 / 3)
    n = C.c_int(0)

    def call(rect=(0, 0, 16, 16), H=16, W=16, n_segments=10, compactness=10.0, max_iter=10, start_label=0, kernel=None,
             radius=0):
        rc = lib.pcm_slic(frame.ctypes.data_as(C.c_void_p), H, W, W * 3, (C.c_int * 4)(*rect), n_segments, compactness, 1.0,
                          kernel, radius, max_iter, start_label, out.ctypes.data_as(C.c_void_p), C.byref(n))
        assert rc == 0 or b"pcm_slic" in lib.pcm_last_error(), lib.pcm_last_error()
        return rc
    assert call() == 0 and n.value >= 1
    assert call(n_segments=0) == -1
    assert call(compactness=0.0) == -1 and call(compactness=float("nan")) == -1
    assert call(max_iter=-1) == -1
    assert call(start_label=-1) == -1
    assert call(rect=(0, 0, 0, 16)) == -1 and call(rect=(0, 0, 17, 16)) == -1
    assert call(kernel=weights.ctypes.data_as(C.c_void_p), radius=-1) == -1
    big = 1 << 14
    assert call(rect=(0, 0, big + 1, big), H=big, W=big + 1) == -4           # more than 2^28 pixels
