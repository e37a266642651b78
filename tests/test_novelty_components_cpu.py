"""PCA novelty detection with more than one component (params.n_components > 1), the parts that need no GPU: the host
eigen-decomposition of the GPU trainer against scikit-learn, the oracle's rank-k error against scikit-learn's
inverse_transform, argument checks of the new C entry points and of addModel."""
import ctypes as C

import numpy as np
import pytest
from sklearn.decomposition import PCA

import pcm_oracle as orc
from helpers import read_video

# (video, frame, features, crop x, y, w, h) of SegTrack2 crops; the first box of each is foreground-rich
CROPS = [("parachute", 0, "8 hsv_lab", 100, 40, 90, 60), ("frog", 3, "6 lab", 60, 50, 80, 70)]


def _rows(video, frame, features, x, y, w, h):
    crop = read_video("Video", video)[frame][y:y + h, x:x + w]
    n, spaces = orc.parse_features(features)
    return orc.get_features_int(orc.build_planes(crop, spaces), n)


def _moments(Xint):
    Xl = Xint.astype(np.int64)
    return (Xl.T @ Xl).astype(np.float64), Xl.sum(axis=0).astype(np.float64), len(Xint)


@pytest.mark.parametrize("crop", CROPS, ids=[c[0] for c in CROPS])
@pytest.mark.parametrize("k", [1, 2, 3, 8])
def test_pca_from_moments_is_sklearns_covariance_eigh(crop, k):
    from pcm import train
    Xint = _rows(*crop)
    G, S, m = _moments(Xint)
    mean, comps = train.pca_from_moments(G, S, m, k)
    ref = PCA(n_components=k, svd_solver="covariance_eigh").fit(Xint.astype(np.float64) / 255)
    assert comps.shape == (k, Xint.shape[1])
    np.testing.assert_allclose(mean, ref.mean_, rtol=1e-12, atol=0)
    np.testing.assert_allclose(comps, ref.components_, rtol=1e-7, atol=1e-9)


@pytest.mark.parametrize("crop", CROPS, ids=[c[0] for c in CROPS])
def test_pca_from_moments_rank_1_keeps_the_rank_1_arithmetic(crop):
    """k = 1 gives the bits of the rank-1 trainer: leading eigenvector of the same covariance, sign flipped by negation."""
    from pcm import train
    G, S, m = _moments(_rows(*crop))
    mean = S / 255.0 / m
    Cov = G / (255.0 * 255.0)
    Cov -= m * mean.reshape(-1, 1) * mean.reshape(1, -1)
    Cov /= m - 1
    _, vecs = np.linalg.eigh(Cov)
    comp = np.ascontiguousarray(vecs[:, -1])
    if comp[np.argmax(np.abs(comp))] < 0:
        comp = -comp
    got_mean, got = train.pca_from_moments(G, S, m, 1)
    assert got_mean.tobytes() == mean.tobytes()
    assert got.shape == (1, len(comp)) and got[0].tobytes() == comp.tobytes()
    assert train.GpuPCA(got_mean, got).n_components == 1


@pytest.mark.parametrize("k", [1, 2, 3, 5, 8])
def test_oracle_novelty_error_is_sklearns_inverse_transform(k):
    Xint = _rows(*CROPS[0])
    X = Xint.astype(np.float64) / 255
    pca = PCA(n_components=k, svd_solver="covariance_eigh").fit(X[: len(X) // 2])
    want = np.sum(np.abs(X - pca.inverse_transform(pca.transform(X))), axis=1)
    got = orc.novelty_error(Xint, pca.mean_, pca.components_)
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)


def test_rank_k_entry_points_reject_null_arguments_without_a_device():
    from pcm import capi
    lib = capi.load_library()
    mean = np.zeros(27)
    comps = np.zeros((3, 27))
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    for args in [(None, 0, p(mean), p(comps), 3, 27), (None, 0, None, None, 3, 27)]:
        assert lib.pcm_set_novelty_k(*args) == -1               # PCM_E_INVALID
        assert b"pcm_set_novelty_k" in lib.pcm_last_error()
    err = np.zeros(10)
    for args in [(None, 1, p(mean), p(comps), 3, p(err)), (None, 1, None, None, 3, None)]:
        assert lib.pcm_pca_residuals_k(*args) == -1
        assert b"pcm_pca_residuals_k" in lib.pcm_last_error()
    assert lib.pcm_set_novelty(None, 0, None, None, 27) == -1
    assert lib.pcm_pca_residuals(None, 1, None, None, None) == -1


@pytest.mark.parametrize("value", [0, 9, 0.95, 3.0, "mle", None, True])
def test_addmodel_refuses_n_components_outside_1_to_8(value):
    from maskers.pixel_classification import PixelClassificationNonRigidMasker as M
    with pytest.raises(ValueError, match="between 1 and 8"):
        M._n_components(dict(n_components=value))


@pytest.mark.parametrize("value", [1, 3, 8, np.int64(5)])
def test_addmodel_accepts_integer_n_components(value):
    from maskers.pixel_classification import PixelClassificationNonRigidMasker as M
    assert M._n_components(dict(n_components=value)) == int(value)
