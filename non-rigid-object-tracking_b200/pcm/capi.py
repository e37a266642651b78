"""ctypes binding of libpcm_b200.so (include/pcm_b200.h) -- the same pattern the
reference uses for its own native component (prim/__init__.py:7-38).

There is no CPU fallback: if the library or a CUDA device is missing, creating a
`Handle` raises.
"""
import ctypes as C
import os

import numpy as np

from . import build as _build

SPACE_IDS = {"rgb": 0, "hsv": 1, "lab": 2}

_lib = None


class PcmError(RuntimeError):
    def __init__(self, code, msg):
        RuntimeError.__init__(self, "pcm_b200 error %d: %s" % (code, msg))
        self.code = code


class UpdateParams(C.Structure):
    _fields_ = [("model_cur", C.c_int32), ("model_next", C.c_int32),
                ("w_cur", C.c_double), ("w_next", C.c_double),
                ("novelty", C.c_int32), ("dilation_kernel", C.c_int32),
                ("outlier_threshold", C.c_double), ("prior_weight", C.c_double)]


class FrameJob(C.Structure):
    """pcm_frame_job (include/pcm_b200.h)."""
    _fields_ = [("d_frame", C.c_void_p), ("rect", C.c_int32 * 4), ("d_labels", C.c_void_p), ("n_labels", C.c_int32),
                ("clear_mask", C.c_int32), ("params", UpdateParams),
                ("d_pts_prev", C.c_void_p), ("d_des_prev", C.c_void_p), ("n_prev", C.c_int32), ("prev_rect", C.c_int32 * 4),
                ("d_pts", C.c_void_p), ("d_des", C.c_void_p), ("n_cur", C.c_int32), ("reserved", C.c_int32),
                ("d_priors_out", C.c_void_p), ("d_priors", C.c_void_p),
                ("d_truth", C.c_void_p), ("truth_stride", C.c_int64), ("truth_channels", C.c_int32), ("reserved2", C.c_int32),
                ("d_counts", C.c_void_p)]


P, I, L, D = C.c_void_p, C.c_int, C.c_int64, C.c_double
# (restype, argtypes) of every entry point of include/pcm_b200.h
_SIGNATURES = {
    "pcm_abi_version": (I, []),
    "pcm_last_error": (C.c_char_p, []),
    "pcm_create": (I, [I, C.POINTER(P)]),
    "pcm_destroy": (None, [P]),
    "pcm_set_stream": (I, [P, P]),
    "pcm_use_own_stream": (I, [P]),
    "pcm_get_stream": (I, [P, C.POINTER(P)]),
    "pcm_synchronize": (I, [P]),
    "pcm_set_features": (I, [P, I, I, P]),
    "pcm_num_features": (I, [P]),
    "pcm_add_model": (I, [P, I, I, P, P, P, P, P, P, C.POINTER(I)]),
    "pcm_set_novelty": (I, [P, I, P, P, I]),
    "pcm_set_novelty_k": (I, [P, I, P, P, I, I]),
    "pcm_num_models": (I, [P]),
    "pcm_crop_rect": (I, [P, I, I, P]),
    "pcm_update": (I, [P, P, I, I, L, P, P, I, P, C.POINTER(UpdateParams), P, L, L]),
    "pcm_update_device": (I, [P, P, I, I, L, P, P, I, P, C.POINTER(UpdateParams), P, L]),
    "pcm_iou": (I, [P, P, L, L, P, L, I, I, I, P]),
    "pcm_iou_device": (I, [P, P, L, P, L, I, I, I, P]),
    "pcm_quickshift": (I, [P, P, I, I, L, P, D, D, D, P, P, C.POINTER(I)]),
    "pcm_quickshift_device": (I, [P, P, I, I, L, P, D, D, D, P, P, C.POINTER(I)]),
    "pcm_quickshift_device_batch": (I, [P, I, P, L, P, I, I, L, P, D, D, D, P, P, P, P]),
    "pcm_felzenszwalb": (I, [P, I, I, L, P, D, D, I, P, I, P, C.POINTER(I)]),
    "pcm_felzenszwalb_graph": (I, [I, I, P, P, P, D, I, P, C.POINTER(I)]),
    "pcm_slic": (I, [P, I, I, L, P, I, D, D, P, I, I, I, P, C.POINTER(I)]),
    "pcm_slic_gpu": (I, [P, P, I, I, L, P, I, D, D, P, I, I, I, P, C.POINTER(I)]),
    "pcm_slic_device": (I, [P, P, I, I, L, P, I, D, D, P, I, I, I, P, C.POINTER(I)]),
    "pcm_slic_device_batch": (I, [P, I, P, L, P, I, I, L, P, I, D, D, P, I, I, I, P, P, P]),
    "pcm_slic_connectivity": (I, [P, P, I, I, C.c_longlong, C.c_longlong, I, P, C.POINTER(I)]),
    "pcm_slic_debug_last": (I, [P, P, P, P]),
    "pcm_host_register": (I, [P, C.c_size_t]),
    "pcm_host_unregister": (I, [P]),
    "pcm_run_frames": (I, [P, I, I, L, P, L, P, I]),
    "pcm_prior_device": (I, [P, P, P, I, P, L, I, I, P, P, I, P, I, I, I, P]),
    "pcm_fit_rows": (I, [P, P, P, I, I, C.c_longlong]),
    "pcm_pca_moments": (I, [P, C.c_longlong, P, P, P]),
    "pcm_pca_residuals": (I, [P, C.c_longlong, P, P, P]),
    "pcm_pca_residuals_k": (I, [P, C.c_longlong, P, P, I, P]),
    "pcm_fit_forest": (I, [P, P, P, I, I, C.c_longlong, I, I, I, P, P, I, P, P, P, P, P, P, P]),
    "pcm_convert": (I, [P, P, I, I, L, I, P, L]),
    "pcm_gather_features": (I, [P, P, I, I, L, P, P]),
    "pcm_set_debug": (I, [P, I]),
    "pcm_debug_last": (I, [P, P, P, P, P, P, P]),
    "pcm_debug_tables": (I, [P, P, P, P, P]),
    "pcm_launch_count": (L, [P]),
    "pcm_transfer_bytes": (I, [P, P]),
    "pcm_set_label_cache": (I, [P, I]),
    "pcm_profile_enable": (I, [P, I]),
    "pcm_profile_read": (I, [P, P, P, I, I]),
}
del P, I, L, D
EXPORTED_SYMBOLS = list(_SIGNATURES)


def library_path():
    return _build.LIB


def load_library():
    """dlopen the in-tree library (building it first if nvcc is available and the
    sources are newer).  Raises if it cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    if _build.needs_build():
        _build.build()
    lib = C.CDLL(_build.LIB)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.pcm_abi_version() != 1:
        raise RuntimeError("libpcm_b200.so ABI version mismatch")
    _lib = lib
    return lib


KERNEL_NAMES = ["score", "segment_reduce", "segment_decide", "segment_resolve", "mask_dilate", "iou", "planes"]
# every profile id of pcm_profile_read: KERNEL_NAMES plus the novelty kernel of PCAs with two or more components (id 7)
ALL_KERNEL_NAMES = KERNEL_NAMES + ["novelty"]
MAX_PCA_COMPONENTS = 8                 # PCM_MAX_PCA_COMPONENTS


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def class1_fraction(tree):
    """Per-node P(class 1) as `DecisionTreeClassifier.predict_proba` reports it.  scikit-learn >= 1.4 stores
    class FRACTIONS in `tree_.value` and returns them unchanged; older versions (the reference pins 0.24.1,
    environment.yaml:14) store weighted class COUNTS and predict_proba divides by their sum
    (`normalizer[normalizer == 0.0] = 1.0; proba /= normalizer`).  Both are reproduced bit for bit: values
    whose rows all sum to 1 are fractions (or single-sample counts, for which the division is the identity)
    and are taken as they are; anything else is normalised exactly like the old predict_proba."""
    v = np.asarray(tree.value[:, 0, :], np.float64)
    s = v.sum(axis=1)
    if np.all(np.abs(s - 1.0) < 1e-9):
        return v[:, 1].copy()
    s[s == 0.0] = 1.0
    return v[:, 1] / s


def crop_rect(bbox, frame_h, frame_w):
    """(x, y, w, h) of the crop the reference slices (pixel_classification.py:49-51)."""
    lib = load_library()
    b = (C.c_int * 4)(*[int(v) for v in bbox])
    out = (C.c_int * 4)()
    rc = lib.pcm_crop_rect(b, int(frame_h), int(frame_w), out)
    if rc:
        raise PcmError(rc, lib.pcm_last_error().decode())
    return tuple(out)


def _packed(frame):                    # an HxWx3 uint8 array with packed pixels: the library reads it in place
    return frame.dtype == np.uint8 and frame.ndim == 3 and frame.shape[2] == 3 and frame.strides[2] == 1 and frame.strides[1] == 3


def _batch_args(frame_index, rects, label_offsets):
    fi, off = np.ascontiguousarray(frame_index, np.int32), np.ascontiguousarray(label_offsets, np.int64)
    rc = np.ascontiguousarray(rects, np.int32).reshape(-1, 4)
    if not (len(fi) == len(rc) == len(off)):
        raise ValueError("frame_index, rects and label_offsets must have one entry per crop")
    return fi, rc, off, np.zeros(len(fi), np.int32)


def _gaussian_weights(sigma):
    """(weights, radius) of the 1-D Gaussian filter scipy.ndimage applies for `sigma` (truncated at 4 sigma);
    (None, 0) when sigma is not positive."""
    if not sigma > 0:
        return None, 0
    radius = int(4.0 * float(sigma) + 0.5)
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    return np.ascontiguousarray(phi / phi.sum(), np.float64), radius


def felzenszwalb(frame, rect, scale=100, sigma=0.5, min_size=50):
    """Felzenszwalb-Huttenlocher segmentation of the crop `rect` (defaults = the reference's call,
    pixel_classification.py:73).  Host code in the library; returns (labels int32 HxW, n_labels).
    The Gaussian weights are computed here the way scipy.ndimage does."""
    lib = load_library()
    if not _packed(frame):
        frame = np.ascontiguousarray(frame, np.uint8)
    r = (C.c_int * 4)(*[int(v) for v in rect])
    kernel, radius = _gaussian_weights(sigma)
    out = np.empty((rect[3], rect[2]), np.int32)
    n = C.c_int(0)
    rc = lib.pcm_felzenszwalb(_ptr(frame), frame.shape[0], frame.shape[1], frame.strides[0], r, float(scale), float(sigma),
                              int(min_size), _ptr(kernel), radius, _ptr(out), C.byref(n))
    if rc:
        raise PcmError(rc, lib.pcm_last_error().decode())
    return out, n.value


def slic(frame, rect, n_segments=250, compactness=10.0, sigma=1.0, max_iter=10, start_label=0):
    """SLIC superpixels of the crop `rect` (defaults = the reference's call, pixel_classification.py:75).  Host code in the
    library; returns (labels int32 HxW, n_labels).  The Gaussian weights are computed here the way scipy.ndimage does."""
    lib = load_library()
    if not _packed(frame):
        frame = np.ascontiguousarray(frame, np.uint8)
    r = (C.c_int * 4)(*[int(v) for v in rect])
    kernel, radius = _gaussian_weights(sigma)
    out = np.empty((rect[3], rect[2]), np.int32)
    n = C.c_int(0)
    rc = lib.pcm_slic(_ptr(frame), frame.shape[0], frame.shape[1], frame.strides[0], r, int(n_segments), float(compactness),
                      float(sigma), _ptr(kernel), radius, int(max_iter), int(start_label), _ptr(out), C.byref(n))
    if rc:
        raise PcmError(rc, lib.pcm_last_error().decode())
    return out, n.value


def host_register(arr):
    """Page-lock a long-lived C-contiguous array (cudaHostRegister): `Handle.update` / `Handle.iou_counts` then copy a
    frame or truth image inside it straight from this memory instead of staging it.  Keep the array alive until
    `host_unregister(arr)`."""
    lib = load_library()
    if not arr.flags.c_contiguous:
        raise ValueError("host_register needs a C-contiguous array")
    rc = lib.pcm_host_register(C.c_void_p(arr.ctypes.data), arr.nbytes)
    if rc:
        raise PcmError(rc, lib.pcm_last_error().decode())
    return arr


def host_unregister(arr):
    lib = load_library()
    rc = lib.pcm_host_unregister(C.c_void_p(arr.ctypes.data))
    if rc:
        raise PcmError(rc, lib.pcm_last_error().decode())


def felzenszwalb_graph(n_vertices, a, b, cost, scale, min_size):
    """Parity tap: the merge / union-find / min-size passes of `felzenszwalb` on an explicit edge list.
    Returns (labels int32[n_vertices], n_labels)."""
    lib = load_library()
    a = np.ascontiguousarray(a, np.int32)
    b = np.ascontiguousarray(b, np.int32)
    cost = np.ascontiguousarray(cost, np.float64)
    assert a.shape == b.shape == cost.shape and a.ndim == 1
    out = np.empty(int(n_vertices), np.int32)
    n = C.c_int(0)
    rc = lib.pcm_felzenszwalb_graph(int(n_vertices), a.size, _ptr(a), _ptr(b), _ptr(cost), float(scale), int(min_size), _ptr(out),
                                    C.byref(n))
    if rc:
        raise PcmError(rc, lib.pcm_last_error().decode())
    return out, n.value


class Handle:
    """One native masker context (one per tracked target)."""

    def __init__(self, device=0, debug=False):
        self.lib = load_library()
        self._h = C.c_void_p()
        self._check(self.lib.pcm_create(int(device), C.byref(self._h)))
        self.device = device
        if debug:
            self.set_debug(True)

    def set_debug(self, on=True, force_exact=False):
        """on: keep the stage buffers `debug_last` reports (P(fg) / novelty maps, pre-dilation map); force_exact: every
        label takes the exact sequential-float32 path of the decision kernel (test hook)."""
        self._check(self.lib.pcm_set_debug(self._h, int(bool(on)) | (2 if force_exact else 0)))

    def debug_scores(self, n_labels):
        """Per-label results of the last update that exist without `set_debug`: scores, areas, number of labels that took
        the exact path."""
        scores = np.empty(n_labels, np.float32)
        areas = np.empty(n_labels, np.int64)
        nx = C.c_int32(0)
        self._check(self.lib.pcm_debug_last(self._h, None, None, _ptr(scores), _ptr(areas), None, C.byref(nx)))
        return dict(scores=scores, areas=areas, n_exact=nx.value)

    def _check(self, rc):
        if rc:
            raise PcmError(rc, self.lib.pcm_last_error().decode())

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.pcm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- configuration ------------------------------------------------------
    def set_features(self, n_neighbors, spaces):
        ids = (C.c_int * len(spaces))(*[SPACE_IDS[s] for s in spaces])
        self._check(self.lib.pcm_set_features(self._h, int(n_neighbors), len(spaces), ids))

    @property
    def num_features(self):
        return self.lib.pcm_num_features(self._h)

    @property
    def num_models(self):
        return self.lib.pcm_num_models(self._h)

    @property
    def launch_count(self):
        return int(self.lib.pcm_launch_count(self._h))

    @property
    def transfer_bytes(self):
        """(host->device, device->host) bytes copied by the host-buffer entry points so far."""
        out = np.zeros(2, np.int64)
        self._check(self.lib.pcm_transfer_bytes(self._h, _ptr(out)))
        return int(out[0]), int(out[1])

    def set_label_cache(self, on=True):
        """Re-send only changed 1 MiB chunks of the label map between update() calls (default on)."""
        self._check(self.lib.pcm_set_label_cache(self._h, int(bool(on))))

    def set_stream(self, cuda_stream):
        """Enqueue on this cudaStream_t (integer handle; 0 = legacy default stream)."""
        self._check(self.lib.pcm_set_stream(self._h, C.c_void_p(int(cuda_stream))))

    def use_own_stream(self):
        self._check(self.lib.pcm_use_own_stream(self._h))

    @property
    def stream(self):
        """cudaStream_t (integer) the handle currently enqueues on."""
        out = C.c_void_p()
        self._check(self.lib.pcm_get_stream(self._h, C.byref(out)))
        return int(out.value or 0)

    def synchronize(self):
        self._check(self.lib.pcm_synchronize(self._h))

    def add_model_arrays(self, n_frame, tree_arrays):
        """tree_arrays: list of (feature, threshold_f64, left, right, value1) per tree."""
        offs = np.cumsum([0] + [len(t[0]) for t in tree_arrays]).astype(np.int64)
        feature = np.ascontiguousarray(np.concatenate([t[0] for t in tree_arrays]), np.int32)
        thr = np.ascontiguousarray(np.concatenate([t[1] for t in tree_arrays]), np.float64)
        left = np.ascontiguousarray(np.concatenate([t[2] for t in tree_arrays]), np.int32)
        right = np.ascontiguousarray(np.concatenate([t[3] for t in tree_arrays]), np.int32)
        val = np.ascontiguousarray(np.concatenate([t[4] for t in tree_arrays]), np.float64)
        idx = C.c_int(-1)
        self._check(self.lib.pcm_add_model(self._h, int(n_frame), len(tree_arrays), _ptr(offs), _ptr(feature),
                                           _ptr(thr), _ptr(left), _ptr(right), _ptr(val), C.byref(idx)))
        return idx.value

    def add_forest(self, n_frame, clf, n_trees=None):
        """Export a fitted sklearn RandomForestClassifier (binary, classes {0,1}); `n_trees`: only
        its first n_trees estimators (with a fixed random_state they ARE the smaller forest)."""
        if list(clf.classes_) != [0, 1]:
            raise ValueError("forest must be a binary {0,1} classifier (the reference indexes probs[:,1])")
        if hasattr(clf, "tree_arrays"):            # pcm.train.GpuForest: already raw arrays in scikit-learn's layout
            return self.add_model_arrays(n_frame, clf.tree_arrays(n_trees))
        arrays = []
        for est in clf.estimators_[:n_trees]:
            t = est.tree_
            arrays.append((t.feature, t.threshold, t.children_left, t.children_right, class1_fraction(t)))
        return self.add_model_arrays(n_frame, arrays)

    def set_novelty(self, model_index, mean, component):
        """PCA novelty detector of a model: `component` is components_[0] (1-D, pcm_set_novelty) or the whole
        components_ array, shape (n_components, F) (pcm_set_novelty_k)."""
        mean = np.ascontiguousarray(mean, np.float64).reshape(-1)
        comp = np.asarray(component, np.float64)
        if comp.ndim == 2:
            comp = np.ascontiguousarray(comp)
            if comp.shape[1] != len(mean):
                raise ValueError("components has %d features, mean %d" % (comp.shape[1], len(mean)))
            self._check(self.lib.pcm_set_novelty_k(self._h, int(model_index), _ptr(mean), _ptr(comp), comp.shape[0],
                                                   len(mean)))
            return
        comp = np.ascontiguousarray(comp).reshape(-1)
        self._check(self.lib.pcm_set_novelty(self._h, int(model_index), _ptr(mean), _ptr(comp), len(mean)))

    # -- hot path -------------------------------------------------------------
    @staticmethod
    def make_params(model_cur, model_next=-1, w_cur=1.0, w_next=0.0, novelty=False, dilation_kernel=7,
                    outlier_threshold=0.0, prior_weight=0.0):
        return UpdateParams(int(model_cur), int(model_next), float(w_cur), float(w_next), int(bool(novelty)),
                            int(dilation_kernel), float(outlier_threshold), float(prior_weight))

    def update(self, frame, rect, labels, n_labels, priors, params, mask, channel=2):
        """Host-buffer update: writes channel `channel` of `mask` (HxWxC u8) inside `rect`."""
        if not _packed(frame):
            frame = np.ascontiguousarray(frame, np.uint8)
        if mask.dtype != np.uint8 or mask.strides[-1] != 1 and mask.ndim == 3:
            raise ValueError("mask must be a uint8 array with unit channel stride")
        if labels is not None:
            labels = np.ascontiguousarray(labels, np.int32)
            if labels.size != rect[2] * rect[3]:
                raise ValueError("labels has %d elements, crop has %d" % (labels.size, rect[2] * rect[3]))
        n_labels = int(n_labels or 0)          # 0 / None: the library takes max(label) + 1
        pr = None if priors is None else np.ascontiguousarray(priors, np.float32)
        if pr is not None and pr.size != n_labels:
            raise ValueError("priors must have n_labels entries")
        r = (C.c_int * 4)(*[int(v) for v in rect])
        if mask.ndim == 3:
            mptr = C.c_void_p(mask.ctypes.data + channel * mask.strides[2])
            row, pix = mask.strides[0], mask.strides[1]
        else:
            mptr, row, pix = C.c_void_p(mask.ctypes.data), mask.strides[0], mask.strides[1]
        self._check(self.lib.pcm_update(self._h, _ptr(frame), frame.shape[0], frame.shape[1], frame.strides[0], r,
                                        _ptr(labels), int(n_labels), _ptr(pr), C.byref(params), mptr, row, pix))

    def quickshift(self, frame, rect, ratio=0.5, kernel_size=3, max_dist=6, noise=None, want_labels=True):
        """quickshift over-segmentation of the crop `rect` (defaults = the reference's call,
        pixel_classification.py:71).  Returns (labels int32 HxW or None, n_labels); the map also
        stays on the device for `update(..., labels=None)`.  `noise`: h*w float64 tie-breaking
        noise, or None to reuse the previous call's (same crop size)."""
        if not _packed(frame):
            raise ValueError("frame must be an HxWx3 uint8 array with packed pixels")
        r = (C.c_int * 4)(*[int(v) for v in rect])
        nz = None if noise is None else np.ascontiguousarray(noise, np.float64)
        if nz is not None and nz.size != rect[2] * rect[3]:
            raise ValueError("noise must have one value per crop pixel")
        out = np.empty((rect[3], rect[2]), np.int32) if want_labels else None
        n = C.c_int(0)
        self._check(self.lib.pcm_quickshift(self._h, _ptr(frame), frame.shape[0], frame.shape[1], frame.strides[0], r,
                                            float(ratio), float(kernel_size), float(max_dist), _ptr(nz), _ptr(out),
                                            C.byref(n)))
        return out, n.value

    def quickshift_device(self, d_frame, frame_h, frame_w, stride, rect, ratio, kernel_size, max_dist, d_noise, d_labels_out):
        """quickshift of the crop `rect` of a DEVICE frame into a device label map (integers = device addresses;
        d_noise: float64 tie-breaking noise, h*w values, or 0).  Waits for the segment count, which it returns."""
        r = (C.c_int * 4)(*[int(v) for v in rect])
        n = C.c_int(0)
        self._check(self.lib.pcm_quickshift_device(self._h, C.c_void_p(d_frame), int(frame_h), int(frame_w), int(stride), r,
                                                   float(ratio), float(kernel_size), float(max_dist),
                                                   C.c_void_p(d_noise) if d_noise else None,
                                                   C.c_void_p(d_labels_out) if d_labels_out else None, C.byref(n)))
        return n.value

    def quickshift_device_batch(self, d_frames, frame_bytes, frame_index, frame_h, frame_w, stride, rects, ratio, kernel_size,
                                max_dist, d_noise, d_labels_out, label_offsets):
        """quickshift_device for many crops of a device-resident clip in ONE native call (pcm_quickshift_device_batch):
        crop k = rects[k] of frame frame_index[k], label map at d_labels_out + 4 * label_offsets[k].  Returns the
        segment counts (int32 array)."""
        fi, rc, off, counts = _batch_args(frame_index, rects, label_offsets)
        self._check(self.lib.pcm_quickshift_device_batch(self._h, len(fi), C.c_void_p(d_frames), int(frame_bytes), _ptr(fi), int(frame_h),
                                                         int(frame_w), int(stride), _ptr(rc), float(ratio), float(kernel_size),
                                                         float(max_dist), C.c_void_p(d_noise) if d_noise else None,
                                                         C.c_void_p(d_labels_out), _ptr(off), _ptr(counts)))
        return counts

    def slic(self, frame, rect, n_segments=250, compactness=10.0, sigma=1.0, max_iter=10, start_label=0, want_labels=True,
             kernel=None):
        """SLIC over-segmentation of the crop `rect` on the GPU (pcm_slic_gpu; defaults = the reference's call,
        pixel_classification.py:75): the labels and count of the host `capi.slic`.  Returns (labels int32 HxW or None,
        n_labels); the map also stays on the device for `update(..., labels=None)`.  `kernel`: Gaussian weights, or None
        to compute them from sigma as scipy.ndimage does."""
        if not _packed(frame):
            raise ValueError("frame must be an HxWx3 uint8 array with packed pixels")
        r = (C.c_int * 4)(*[int(v) for v in rect])
        weights, radius = self._slic_weights(sigma, kernel)
        out = np.empty((rect[3], rect[2]), np.int32) if want_labels else None
        n = C.c_int(0)
        self._check(self.lib.pcm_slic_gpu(self._h, _ptr(frame), frame.shape[0], frame.shape[1], frame.strides[0], r,
                                          int(n_segments), float(compactness), float(sigma), _ptr(weights), radius,
                                          int(max_iter), int(start_label), _ptr(out), C.byref(n)))
        self._slic_shape = (int(rect[3]), int(rect[2]))
        return out, n.value

    @staticmethod
    def _slic_weights(sigma, kernel):
        if kernel is None:
            return _gaussian_weights(sigma)
        k = np.ascontiguousarray(kernel, np.float64).reshape(-1)
        if k.size % 2 != 1:
            raise ValueError("kernel must have 2 * radius + 1 weights")
        return k, k.size // 2

    def slic_device_batch(self, d_frames, frame_bytes, frame_index, frame_h, frame_w, stride, rects, d_labels_out, label_offsets,
                          n_segments=250, compactness=10.0, sigma=1.0, max_iter=10, start_label=0):
        """SLIC of many crops of a device-resident clip in ONE native call (pcm_slic_device_batch), laid out like
        quickshift_device_batch.  Returns the segment counts (int32 array)."""
        fi, rc, off, counts = _batch_args(frame_index, rects, label_offsets)
        weights, radius = _gaussian_weights(sigma)
        self._check(self.lib.pcm_slic_device_batch(self._h, len(fi), C.c_void_p(d_frames), int(frame_bytes), _ptr(fi), int(frame_h),
                                                   int(frame_w), int(stride), _ptr(rc), int(n_segments), float(compactness),
                                                   float(sigma), _ptr(weights), radius, int(max_iter), int(start_label),
                                                   C.c_void_p(d_labels_out), _ptr(off), _ptr(counts)))
        if len(fi):
            self._slic_shape = (int(rc[-1, 3]), int(rc[-1, 2]))
        return counts

    def slic_connectivity(self, nearest, min_size, max_size, start_label=0):
        """Parity tap: the device connectivity enforcement of SLIC on a centre map (HxW ints).  Returns (labels int32 HxW,
        n_labels)."""
        seg = np.ascontiguousarray(nearest, np.int32)
        if seg.ndim != 2:
            raise ValueError("nearest must be HxW")
        out = np.empty_like(seg)
        n = C.c_int(0)
        self._check(self.lib.pcm_slic_connectivity(self._h, _ptr(seg), seg.shape[1], seg.shape[0], int(min_size), int(max_size),
                                                   int(start_label), _ptr(out), C.byref(n)))
        return out, n.value

    def slic_debug_last(self):
        """Stage results of the last SLIC on this handle: smoothed (HxWx3 float64), image (HxWx3 float64, what the
        k-means sees) and nearest (HxW int32, the centre map after the last iteration)."""
        h, w = getattr(self, "_slic_shape", (0, 0))
        smoothed, image = np.empty((h, w, 3), np.float64), np.empty((h, w, 3), np.float64)
        nearest = np.empty((h, w), np.int32)
        self._check(self.lib.pcm_slic_debug_last(self._h, _ptr(smoothed), _ptr(image), _ptr(nearest)))
        return dict(smoothed=smoothed, image=image, nearest=nearest)

    def prior_device(self, d_pts_prev, d_des_prev, n_prev, d_prev_mask, prev_stride, prev_w, prev_h, d_pts, d_des, n_cur,
                     d_labels, crop_w, crop_h, n_labels, d_priors):
        """SIFT-match priors of one frame on the device (pcm_prior_device; integers = device addresses); asynchronous."""
        v = lambda x: C.c_void_p(x) if x else None
        self._check(self.lib.pcm_prior_device(self._h, v(d_pts_prev), v(d_des_prev), int(n_prev), v(d_prev_mask), int(prev_stride),
                                              int(prev_w), int(prev_h), v(d_pts), v(d_des), int(n_cur), v(d_labels),
                                              int(crop_w), int(crop_h), int(n_labels), v(d_priors)))

    def run_frames(self, frame_h, frame_w, frame_stride, d_mask, mask_stride, jobs, n_jobs):
        """Enqueue `n_jobs` FrameJob records (a ctypes array, or the address of records laid out like one) back to back;
        asynchronous (pcm_run_frames)."""
        self._check(self.lib.pcm_run_frames(self._h, int(frame_h), int(frame_w), int(frame_stride), C.c_void_p(d_mask),
                                            int(mask_stride), jobs, int(n_jobs)))

    def update_device(self, d_frame, frame_h, frame_w, stride, rect, d_labels, n_labels, d_priors, params, d_mask,
                      mask_stride):
        """Device-pointer update (integers are raw device addresses); asynchronous."""
        r = (C.c_int * 4)(*[int(v) for v in rect])
        self._check(self.lib.pcm_update_device(self._h, C.c_void_p(d_frame), int(frame_h), int(frame_w), int(stride), r,
                                               C.c_void_p(d_labels), int(n_labels),
                                               C.c_void_p(d_priors) if d_priors else None, C.byref(params),
                                               C.c_void_p(d_mask), int(mask_stride)))

    def iou_counts(self, mask, truth):
        """(intersection, union) of mask != 0 and truth != 0; truth HxW gray or HxWx3 BGR."""
        if mask.ndim != 2 or mask.dtype != np.uint8:
            raise ValueError("mask must be HxW uint8")
        tch = 1 if truth.ndim == 2 else truth.shape[2]
        if truth.dtype != np.uint8 or truth.strides[1] != tch or (truth.ndim == 3 and truth.strides[2] != 1):
            truth = np.ascontiguousarray(truth, np.uint8)
        if truth.shape[:2] != mask.shape:
            raise ValueError("mask / truth shapes differ")
        out = np.zeros(2, np.int64)
        self._check(self.lib.pcm_iou(self._h, C.c_void_p(mask.ctypes.data), mask.strides[0], mask.strides[1],
                                     _ptr(truth), truth.strides[0], tch, mask.shape[0], mask.shape[1], _ptr(out)))
        return int(out[0]), int(out[1])

    def iou_device(self, d_mask, mask_stride, d_truth, truth_stride, truth_channels, h, w, d_counts):
        self._check(self.lib.pcm_iou_device(self._h, C.c_void_p(d_mask), int(mask_stride), C.c_void_p(d_truth),
                                            int(truth_stride), int(truth_channels), int(h), int(w),
                                            C.c_void_p(d_counts)))

    # -- parity taps ------------------------------------------------------------
    def convert(self, bgr, space):
        bgr = np.ascontiguousarray(bgr, np.uint8)
        out = np.empty_like(bgr)
        self._check(self.lib.pcm_convert(self._h, _ptr(bgr), bgr.shape[0], bgr.shape[1], bgr.strides[0],
                                         SPACE_IDS[space], _ptr(out), out.strides[0]))
        return out

    def gather_features(self, frame, rect):
        frame = np.ascontiguousarray(frame, np.uint8)
        X = np.empty((rect[2] * rect[3], self.num_features), np.int16)
        r = (C.c_int * 4)(*[int(v) for v in rect])
        self._check(self.lib.pcm_gather_features(self._h, _ptr(frame), frame.shape[0], frame.shape[1],
                                                 frame.strides[0], r, _ptr(X)))
        return X

    def debug_last(self, crop_h, crop_w, n_labels):
        n = crop_h * crop_w
        p1 = np.empty(n, np.float64)
        sa = np.empty(n, np.float64)
        scores = np.empty(n_labels, np.float32)
        areas = np.empty(n_labels, np.int64)
        pre = np.empty((crop_h, crop_w), np.uint8)
        nx = C.c_int32(0)
        self._check(self.lib.pcm_debug_last(self._h, _ptr(p1), _ptr(sa), _ptr(scores), _ptr(areas), _ptr(pre),
                                            C.byref(nx)))
        return dict(p1=p1, sa=sa, scores=scores, areas=areas, pre=pre, n_exact=nx.value)

    def profile_enable(self, on=True):
        self._check(self.lib.pcm_profile_enable(self._h, int(bool(on))))

    def profile_read(self, reset=False, names=None):
        """{kernel name: (total ms, launches)} measured with CUDA events on the handle's stream; `names`: the first
        len(names) profile ids (default KERNEL_NAMES; ALL_KERNEL_NAMES includes the novelty kernel)."""
        names = KERNEL_NAMES if names is None else names
        ms = np.zeros(len(names), np.float64)
        cnt = np.zeros(len(names), np.int64)
        self._check(self.lib.pcm_profile_read(self._h, _ptr(ms), _ptr(cnt), len(names), int(bool(reset))))
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(names)}

    def tables(self):
        gamma = np.empty(256, np.uint16)
        cb = np.empty(2041, np.uint16)
        sdiv = np.empty(256, np.int32)
        hdiv = np.empty(256, np.int32)
        self._check(self.lib.pcm_debug_tables(self._h, _ptr(gamma), _ptr(cb), _ptr(sdiv), _ptr(hdiv)))
        return gamma, cb, sdiv, hdiv
