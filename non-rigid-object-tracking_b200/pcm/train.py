"""Training side of addModel (reference maskers/pixel_classification.py:166-228) on the GPU.

The reference fits `RandomForestClassifier(random_state=42, n_estimators, max_depth).fit(X, labels)` (:199-200).
`fit_forest` grows the SAME trees with `pcm_fit_forest` (csrc/pcm_forest_fit.cuh): the per-tree seeds, bootstrap
counts and splitter seeds are drawn here with numpy exactly as scikit-learn draws them
(sklearn/ensemble/_base.py:77-84 `_set_random_states`, _forest.py:95-103,148-153 `_generate_sample_indices` +
`np.bincount`, tree/_splitter.pyx:155 `rand_r_state`), the trees themselves are grown on the device.  The growing
procedure restates scikit-learn 1.9's; it is used when the installed scikit-learn is of that series (the tests compare
the result with scikit-learn's `tree_` arrays) and `RandomForestClassifier` itself is used otherwise.
"""
import ctypes as C
import threading

import numpy as np

VALIDATED_SKLEARN = ("1.9.",)          # series whose tree builder csrc/pcm_forest_fit.cuh restates
MAX_INT32 = np.iinfo(np.int32).max
RAND_R_MAX = 2147483647


def gpu_fit_supported():
    import sklearn
    return sklearn.__version__.startswith(VALIDATED_SKLEARN)


_draws, _draw_locks, _draws_guard = {}, {}, threading.Lock()


def tree_draws(n_samples, n_estimators, random_state=42):
    """(counts uint8 [T, n], splitter seeds uint32 [T]) of the forest's trees.  They depend on the number of rows, trees
    and the seed only, and are computed ONCE per such triple, also when several threads ask at the same time (the fits
    of one row set -- two feature sets x two depths in the sweep -- start together; a plain memo let every one of them
    spend its 30 ms under the interpreter lock, which serialised the fitting threads of a whole sweep)."""
    key = (int(n_samples), int(n_estimators), int(random_state))
    with _draws_guard:
        if key in _draws:
            return _draws[key]
        lock = _draw_locks.setdefault(key, threading.Lock())
    with lock:
        with _draws_guard:
            if key in _draws:
                return _draws[key]
        rs = np.random.RandomState(random_state)
        tree_rs = np.random.RandomState(0)          # re-seeded per tree: RandomState(seed) without the construction
        counts = np.empty((n_estimators, n_samples), np.uint8)
        seeds = np.empty(n_estimators, np.uint32)
        for t in range(n_estimators):
            seed = rs.randint(MAX_INT32)
            tree_rs.seed(seed)
            c = np.bincount(tree_rs.randint(0, n_samples, n_samples), minlength=n_samples)
            if c.max() > 127:
                raise ValueError("bootstrap count above 127")
            counts[t] = c
            tree_rs.seed(seed)
            seeds[t] = tree_rs.randint(0, RAND_R_MAX)
        with _draws_guard:
            if len(_draws) >= 64:                   # bounded like the memo it replaces
                _draws.pop(next(iter(_draws)))
            _draws[key] = (counts, seeds)
            _draw_locks.pop(key, None)
        return counts, seeds


class GpuForest:
    """Fitted forest as raw per-tree arrays [(feature, threshold, left, right, value1)] in scikit-learn's node
    order; `classes_` / `n_estimators` / `n_features_in_` mirror the estimator attributes the masker reads."""

    def __init__(self, trees, n_features, max_depth):
        self.trees = trees
        self.n_estimators = len(trees)
        self.n_features_in_ = n_features
        self.max_depth = max_depth
        self.classes_ = np.array([0, 1])

    def tree_arrays(self, n_trees=None):
        return self.trees[:n_trees]


def fit_forest(handle, X, y, n_estimators, max_depth, random_state=42, rows_id=0, rows_resident=False, draws=None):
    """X: int16 [n, F] raw feature values (-1..255) as `Handle.gather_features` returns them; y: 0/1 labels.
    rows_id / rows_resident: a non-zero id names the row set; with rows_resident=True the rows the handle still holds
    from its previous fit with that id are reused instead of uploaded again.  Returns a GpuForest."""
    X = np.ascontiguousarray(X, np.int16)
    n, F = X.shape
    y8 = np.ascontiguousarray(y, np.uint8)
    if y8.min() != 0 or y8.max() != 1:
        raise ValueError("binary {0,1} labels with both classes present are required (the reference indexes probs[:,1])")
    counts, seeds = draws if draws is not None else tree_draws(n, n_estimators, random_state)
    max_features = max(1, int(np.sqrt(F)))
    cap = int(min(2 ** (max_depth + 1) - 1, 2 * n - 1)) if max_depth <= 24 else 2 * n - 1
    T = n_estimators
    node_count = np.empty(T, np.int32)
    feature = np.empty((T, cap), np.int32)
    left = np.empty((T, cap), np.int32)
    right = np.empty((T, cap), np.int32)
    thr = np.empty((T, cap), np.float64)
    val = np.empty((T, cap), np.float64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    handle._check(handle.lib.pcm_fit_forest(handle._h, None if rows_resident else p(X), p(y8), n, F, int(rows_id), T,
                                            int(max_depth), max_features, p(counts), p(seeds), cap, p(node_count),
                                            p(feature), p(thr), p(left), p(right), p(val), None))
    trees = []
    for t in range(T):
        k = int(node_count[t])
        trees.append((feature[t, :k].copy(), thr[t, :k].copy(), left[t, :k].copy(), right[t, :k].copy(), val[t, :k].copy()))
    return GpuForest(trees, F, max_depth)


class GpuPCA:
    """The attributes of sklearn.decomposition.PCA(n_components=k) the masker reads: mean_ [F], components_ [k, F]."""

    def __init__(self, mean, components):
        self.mean_ = mean
        self.components_ = components.reshape(-1, len(mean))
        self.n_components = self.components_.shape[0]


def upload_rows(handle, X, y, rows_id):
    X = np.ascontiguousarray(X, np.int16)
    y8 = np.ascontiguousarray(y, np.uint8)
    handle._check(handle.lib.pcm_fit_rows(handle._h, X.ctypes.data_as(C.c_void_p), y8.ctypes.data_as(C.c_void_p),
                                          X.shape[0], X.shape[1], int(rows_id)))


def pca_from_moments(gram, sums, n_class1, k=1):
    """(mean [F], components [k, F]) of PCA(n_components=k).fit(X / 255) from the moments pcm_pca_moments returns for the
    class-1 rows X (gram = X^T X and sums over the raw integer values, n_class1 rows), computed the way scikit-learn
    1.9's covariance_eigh solver computes them (decomposition/_pca.py `_fit_full`): C = X^T X - n mean mean^T,
    C /= n - 1, eigenvectors of C by decreasing eigenvalue, each with the sign that makes its largest-magnitude entry
    positive (svd_flip, u_based_decision=False).  The Gram matrix is scaled by 1/255^2 here."""
    m = int(n_class1)
    mean = sums / 255.0 / m
    Cov = gram / (255.0 * 255.0)
    Cov -= m * mean.reshape(-1, 1) * mean.reshape(1, -1)
    Cov /= m - 1
    _, vecs = np.linalg.eigh(Cov)
    comps = np.ascontiguousarray(vecs[:, ::-1][:, :k].T)
    rows = np.arange(k)
    signs = np.where(comps[rows, np.argmax(np.abs(comps), axis=1)] < 0, -1.0, 1.0)
    comps *= signs[:, None]
    return mean, comps


def fit_pca(handle, rows_id, n_rows, n_features, n_components=1):
    """PCA(n_components).fit(X[labels == 1]) and the 90th percentile of the L1 reconstruction error of every
    training row (reference :203-213) from the rows resident on `handle` under rows_id: the Gram matrix is accumulated
    on the device over the raw integer feature values (exact), the eigen-decomposition is `pca_from_moments`, the
    residuals are pcm_pca_residuals_k.  Like scikit-learn, n_components may not exceed min(class-1 rows, features).
    Returns (GpuPCA, threshold)."""
    F = n_features
    k = int(n_components)
    G = np.empty((F, F), np.float64)
    S = np.empty(F, np.float64)
    n1 = np.zeros(1, np.int64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    handle._check(handle.lib.pcm_pca_moments(handle._h, int(rows_id), p(G), p(S), p(n1)))
    m = int(n1[0])
    if m < 2:
        raise ValueError("PCA needs at least two foreground rows")
    if not 1 <= k <= min(m, F):
        raise ValueError("n_components=%r must be between 1 and min(n_samples, n_features)=%d with svd_solver='covariance_eigh'"
                         % (n_components, min(m, F)))
    mean, comps = pca_from_moments(G, S, m, k)
    err = np.empty(n_rows, np.float64)
    handle._check(handle.lib.pcm_pca_residuals_k(handle._h, int(rows_id), p(mean), p(comps), k, p(err)))
    return GpuPCA(mean, comps), float(np.percentile(err, 90))
