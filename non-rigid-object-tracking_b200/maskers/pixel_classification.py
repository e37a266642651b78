"""B200-native PixelClassification masker behind the reference's plugin API.

Interface and state machine follow the reference class
PixelClassificationNonRigidMasker (maskers/pixel_classification.py:24-228):
same constructor keywords, `addModel(...) -> bbox_roni`, `update(bbox, frame,
mask, color) -> None | model index`, same public attributes (`index`, `models`,
`novelty_det`, `current_model`, `prevFrame`, `prevForegroundMask`).

What differs is where the per-frame work runs: colour conversion, star-tap
features, forest scoring, PCA novelty error, temporal blend, per-superpixel
decision and dilation are CUDA kernels in libpcm_b200.so, reached through the C
ABI of include/pcm_b200.h (pcm/capi.py).  There is no CPU fallback for that path.
Training (`addModel`) stays with scikit-learn on the host, as in the reference;
its feature rows come from the same device code (pcm_gather_features).
"""
import copy

import cv2 as cv
import numpy as np
from sklearn.decomposition import PCA
from sklearn.ensemble import RandomForestClassifier
from sklearn.metrics import f1_score

from pcm import capi, stages, train
from pcm.providers import make_segment_provider
from pcm.priors import SiftPrior
from .masker import Masker


class PixelClassificationNonRigidMasker(Masker):
    _rows_ids = iter(range(1, 1 << 62))          # process-wide ids of training-row sets (device residency)

    def __init__(self, poly_roi=None, update_mask=None, segment_fn=None, prior_fn=None, device=0,
                 model_cache=None, cache_tag=None, train_jobs=None, fit_estimators=None, train_provider=None, **args):
        """Reference keywords: debug, frame, config, poly_roi, update_mask (main.py:138-144).
        Extra, all optional: `segment_fn(crop) -> int32 labels` and `prior_fn` (providers for the
        stages outside the hot path), `device` (CUDA ordinal), `model_cache` + `cache_tag` (a dict
        shared between maskers of a hyper-parameter sweep: training rows, fitted forests and PCAs
        are reused when (tag, frame, features, n_estimators, max_depth) repeat -- fits are
        deterministic, random_state=42), `train_jobs` (sklearn n_jobs for the fit; the fitted
        forest does not depend on it), `fit_estimators` (a sweep's largest n_estimators: the forest
        is fitted once with that many trees and every smaller n_estimators uses its first trees --
        with random_state=42 tree i is the same tree in both, tests/test_sweep_host.py),
        `train_provider`: "gpu" grows the forest and fits the PCA on the device (pcm/train.py: the same trees
        scikit-learn grows, tests/test_gpu_forest_fit.py), "sklearn" calls scikit-learn on the host as the
        reference does; default: "gpu" when the installed scikit-learn is the series the GPU trainer restates."""
        Masker.__init__(self, **args)
        import os
        provider = train_provider or self.config.get("train_provider") or os.environ.get("PCM_TRAIN") or "auto"
        if provider == "auto":
            provider = "gpu" if train.gpu_fit_supported() else "sklearn"
        if provider not in ("gpu", "sklearn"):
            raise ValueError("train_provider must be auto, gpu or sklearn")
        self.train_provider = provider
        self._resident_rows = 0
        self.model_cache = model_cache
        self.cache_tag = cache_tag
        self.train_jobs = train_jobs
        self.fit_estimators = fit_estimators
        self.poly_roi = copy.deepcopy(poly_roi)
        self.index = 0
        self.models = []
        self.novelty_det = []
        self.current_model = 0
        self.multi_selection = self.config.get("multi_selection")

        params = self.config["params"]
        tokens = params["features"].split()
        self.n_neighbors = int(tokens[0])
        self.spaces = tokens[1].split("_")
        self.native = capi.Handle(device)
        self.native.set_features(self.n_neighbors, self.spaces)
        # over-segmentation (:70-75), SURVEY §8 f-1, by the library unless segment_fn is given: native_seg is the
        # algorithm it runs, or None.  All three run on the GPU (pcm_quickshift, pcm_slic_gpu, pcm_felzenszwalb_gpu)
        method = params["over_segmentation"]
        self.native_seg = method if segment_fn is None and method in ("quickshift", "SLIC", "felzenszwalb") else None
        self.segment_fn = segment_fn or (None if self.native_seg else make_segment_provider(method))
        self._qs_noise_shape = None
        self._seg_prev = None                  # (provider's array object, crop shape) of the label map resident on the device
        self.reuse_resident_labels = True      # False: every update sends its label map, whatever the provider returns
        self._prior_fn = prior_fn              # SiftPrior() on first use (SIFT + FLANN objects are not free to build)
        self.prevForegroundMask = None

    @property
    def prior_fn(self):
        if self._prior_fn is None:
            self._prior_fn = SiftPrior()
        return self._prior_fn

    @prior_fn.setter
    def prior_fn(self, fn):
        self._prior_fn = fn

    # -- training (reference :166-228) -------------------------------------------
    @staticmethod
    def _n_components(params):
        """params.n_components as the native novelty path takes it: an integer in 1..PCM_MAX_PCA_COMPONENTS.  A fraction
        of explained variance (0 < n < 1) or "mle", which scikit-learn would also accept, is refused."""
        k = params.get("n_components")
        if isinstance(k, (bool, np.bool_)) or not isinstance(k, (int, np.integer)) or not 1 <= k <= capi.MAX_PCA_COMPONENTS:
            raise ValueError("n_components must be an integer between 1 and %d (PCM_MAX_PCA_COMPONENTS), got %r"
                             % (capi.MAX_PCA_COMPONENTS, k))
        return int(k)

    def _rows(self, frame, rect):
        """Raw feature rows of a rectangle, int16 in -1..255; the reference trains on these / 255 (:54-55, :192-196)."""
        return self.native.gather_features(frame, rect)

    def addModel(self, frame, poly_roi, bbox, n_frame, bbox_roni=None, show_prob_map=False):
        if bbox_roni is None:
            raise ValueError("bbox_roni is required (the reference opens a GUI selector here, :287)")
        params = self.config["params"]
        n_components = self._n_components(params) if params["novelty_detection"] else None
        cache = self.model_cache if self.model_cache is not None and self.cache_tag is not None else None

        def cached(key, make):
            """cache[key], computing it at most once (also across threads when the cache offers get_or_compute)."""
            if cache is None:
                return make()
            if hasattr(cache, "get_or_compute"):
                return cache.get_or_compute(key, make)
            if key not in cache:
                cache[key] = make()
            return cache[key]

        def make_rows():
            x, y, w, h = [int(v) for v in bbox]
            roi = np.zeros((h, w), np.uint8)
            cv.fillPoly(roi, np.array([[(p[0] - x, p[1] - y) for p in poly_roi]], dtype=np.int32), 255)
            X = self._rows(frame, (x, y, w, h))
            labels = (roi.reshape(-1) > 0).astype(np.int64)
            Xn = self._rows(frame, tuple(int(v) for v in bbox_roni))
            return (np.concatenate([X, Xn], axis=0), np.concatenate([labels, np.zeros(len(Xn), np.int64)]),
                    next(PixelClassificationNonRigidMasker._rows_ids))

        with stages.stage("train_rows"):
            Xi, labels, rows_id = cached((self.cache_tag, n_frame, params["features"], "rows"), make_rows)
        gpu = self.train_provider == "gpu"

        def resident():
            """True when this handle already holds the row set; it does after the call."""
            had = self._resident_rows == rows_id
            self._resident_rows = rows_id
            return had

        n_trees = int(params["n_estimators"])
        n_fit = max(n_trees, int(self.fit_estimators or 0))

        def make_forest():
            if gpu:
                return train.fit_forest(self.native, Xi, labels, n_fit, params["max_depth"], rows_id=rows_id,
                                        rows_resident=resident())
            X = Xi.astype(np.float64) / 255
            clf = RandomForestClassifier(random_state=42, n_estimators=n_fit, max_depth=params["max_depth"],
                                         n_jobs=self.train_jobs).fit(X, labels)
            if n_fit == n_trees:
                print("F1 score classifier for frame {}= {}".format(n_frame, round(f1_score(labels, clf.predict(X)), 2)))
            return clf

        with stages.stage("fit_forest"):
            clf = cached((self.cache_tag, n_frame, params["features"], n_fit, params["max_depth"], "forest"), make_forest)

        if params["novelty_detection"]:
            def make_pca():
                if gpu:
                    if not resident():
                        train.upload_rows(self.native, Xi, labels, rows_id)
                    return train.fit_pca(self.native, rows_id, len(labels), Xi.shape[1], n_components)
                X = Xi.astype(np.float64) / 255
                pca = PCA(n_components=n_components).fit(X[labels == 1])
                residual = np.sum(np.sqrt(np.power(X - pca.inverse_transform(pca.transform(X)), 2)), axis=1)
                return pca, np.percentile(residual, 90)
            with stages.stage("fit_pca"):
                pca, threshold = cached((self.cache_tag, n_frame, params["features"], params["n_components"], "pca"), make_pca)
        else:
            pca, threshold = None, 0.0

        with stages.stage("export_model"):
            m = self.native.add_forest(n_frame, clf, n_trees)
            if pca is not None:
                self.native.set_novelty(m, pca.mean_, pca.components_)
        self.models.append({"n_frame": n_frame, "model": clf, "n_trees": n_trees})
        self.novelty_det.append({"n_frame": n_frame, "model": pca, "threshold": threshold})
        return bbox_roni

    def close(self):
        """Release the native context (device buffers, stream)."""
        self.native.close()

    # -- per-frame hot path (reference :45-126) --------------------------------------
    def update(self, bbox, frame, mask, color=None):
        x, y, w, h = capi.crop_rect(bbox, frame.shape[0], frame.shape[1])
        if w <= 0 or h <= 0:
            raise ValueError("empty crop for bbox %r" % (bbox,))
        ys, xs = slice(y, y + h), slice(x, x + w)
        crop = frame[ys, xs]
        params = self.config["params"]

        want_prior = self.index != 0 and params["prior_weight"] != 0.0

        def prior(segs, n):
            if isinstance(self.prior_fn, SiftPrior) and self.cache_tag is not None:
                return self.prior_fn(self.prevFrame, self.prevForegroundMask, crop, segs, n, cache=self.model_cache,
                                     key=(self.cache_tag, self.index, (x, y, w, h)))
            return self.prior_fn(self.prevFrame, self.prevForegroundMask, crop, segs, n)
        n_labels, priors = 0, None             # 0: the library takes max(label) + 1 while staging
        same_labels, self._seg_next = False, None
        if self.native_seg is not None:
            # quickshift(crop, kernel_size=3, max_dist=6, ratio=0.5, random_seed=42) (:71),
            # felzenszwalb(crop, scale=100, sigma=0.5, min_size=50) (:73) or
            # slic(crop, n_segments=250, compactness=10, sigma=1, start_label=0) (:75) on the GPU; the label
            # map stays on the device and only travels to the host when the SIFT prior needs it
            if frame.strides[2] != 1 or frame.strides[1] != 3:
                frame = np.ascontiguousarray(frame)
            if self.native_seg == "quickshift":
                noise = None
                if self._qs_noise_shape != (h, w):
                    noise = np.random.RandomState(42).normal(scale=0.00001, size=(h, w))
                    self._qs_noise_shape = (h, w)
                with stages.stage("gpu_quickshift_call"):
                    segments, n_labels = self.native.quickshift(frame, (x, y, w, h), ratio=0.5, kernel_size=3, max_dist=6,
                                                                noise=noise, want_labels=want_prior)
            elif self.native_seg == "felzenszwalb":
                with stages.stage("gpu_felzenszwalb_call"):
                    segments, n_labels = self.native.felzenszwalb(frame, (x, y, w, h), scale=100, sigma=0.5, min_size=50,
                                                                  want_labels=want_prior)
            else:
                with stages.stage("gpu_slic_call"):
                    segments, n_labels = self.native.slic(frame, (x, y, w, h), n_segments=250, compactness=10.0, sigma=1.0,
                                                          start_label=0, want_labels=want_prior)
            if want_prior:
                with stages.stage("sift_prior"):
                    priors = prior(segments, n_labels)
            segments = None                    # update() continues from the device-resident map
        else:
            raw = self.segment_fn(crop)
            # a provider that hands back the very same READ-ONLY array vouches that the map has not changed: it is
            # still on the device from the previous update and does not travel again (pcm_update, labels == NULL)
            same_labels = (self.reuse_resident_labels and self._seg_prev is not None and raw is self._seg_prev[0] and self._seg_prev[1] == (h, w)
                           and isinstance(raw, np.ndarray) and not raw.flags.writeable)
            self._seg_next = (raw, (h, w))
            segments = np.ascontiguousarray(raw, np.int32)
            if want_prior:
                n_labels = int(segments.max()) + 1
                with stages.stage("sift_prior"):
                    priors = prior(segments, n_labels)

        p, blend = self._frame_params()
        self._seg_prev = None
        with stages.stage("gpu_update_call"):
            self.native.update(frame, (x, y, w, h), None if same_labels else segments, n_labels, priors, p, mask, channel=2)
        self._seg_prev, self._seg_next = self._seg_next, None
        return self._advance(blend, crop, mask[ys, xs, 2])

    # -- state machine shared by update() and update_resident() (reference :81-87, :114-126) ----------
    def _frame_params(self):
        """(pcm_update_params of the frame about to be processed, blend flag)."""
        params = self.config["params"]
        cur = self.current_model
        blend = bool(self.multi_selection) and len(self.models) > cur + 1
        w_cur, w_next = 1.0, 0.0
        if blend:
            span = self.models[cur + 1]["n_frame"] - self.models[cur]["n_frame"]
            tmp = self.index - self.models[cur]["n_frame"]
            w_cur, w_next = 1 - (tmp / span), tmp / span
        p = capi.Handle.make_params(cur, cur + 1 if blend else -1, w_cur, w_next,
                                    novelty=params["novelty_detection"],
                                    dilation_kernel=params["dilation_kernel"],
                                    outlier_threshold=self.novelty_det[cur]["threshold"],
                                    prior_weight=params["prior_weight"])
        return p, blend

    def _frame_schedule(self, n):
        """The pcm_update_params columns of the next `n` frames -- (model_cur, model_next, w_cur, w_next,
        outlier_threshold), one numpy array each -- and the state after them: what n rounds of
        _frame_params() / _advance(quiet=True) produce, computed per model span instead of per frame
        (reference :81-87, :114-118)."""
        cur_a, next_a = np.empty(n, np.int32), np.empty(n, np.int32)
        w_cur, w_next, thr = np.empty(n, np.float64), np.empty(n, np.float64), np.empty(n, np.float64)
        done = 0
        while done < n:
            cur = self.current_model
            blend = bool(self.multi_selection) and len(self.models) > cur + 1
            if blend:
                first, last = self.models[cur]["n_frame"], self.models[cur + 1]["n_frame"]
                k = min(n - done, max(1, last - self.index))    # the frame that reaches `last` switches models
                tmp = np.arange(self.index, self.index + k, dtype=np.int64) - first
                frac = tmp / np.float64(last - first)
                w_cur[done:done + k], w_next[done:done + k] = 1 - frac, frac
            else:
                k = n - done
                w_cur[done:done + k], w_next[done:done + k] = 1.0, 0.0
            cur_a[done:done + k], next_a[done:done + k] = cur, cur + 1 if blend else -1
            thr[done:done + k] = self.novelty_det[cur]["threshold"]
            self.index += k
            done += k
            if blend and self.index >= last:
                self.current_model += 1
        self.prevFrame = self.prevForegroundMask = None
        return cur_a, next_a, w_cur, w_next, thr

    def _advance(self, blend, crop, mask_crop, quiet=False):
        cur = self.current_model
        self.index += 1
        self.prevFrame = crop
        self.prevForegroundMask = mask_crop
        if blend and self.index >= self.models[cur + 1]["n_frame"]:
            self.current_model += 1
            if not quiet:
                print("\n \n CHANGE OF MODEL \n \n")
            return self.current_model   # tells the caller to re-initialise the tracker
        return None

    def update_resident(self, d_frame, frame_h, frame_w, frame_stride, rect, d_labels, n_labels, d_priors, d_mask,
                        mask_stride):
        """update() for a caller that keeps the frame, the label map of the crop `rect` (from pcm_crop_rect), the
        optional priors and the mask plane ON THE DEVICE (integers = device addresses): the same state machine and
        the same kernels as update(), enqueued on the handle's stream without waiting (pcm_update_device).  The
        caller provides what update() derives on the host (over-segmentation labels, SIFT priors) and owns
        prevFrame / prevForegroundMask bookkeeping.  Returns None or the new model index, like update()."""
        p, blend = self._frame_params()
        self.native.update_device(d_frame, frame_h, frame_w, frame_stride, rect, d_labels, n_labels, d_priors, p,
                                  d_mask, mask_stride)
        return self._advance(blend, None, None, quiet=True)
