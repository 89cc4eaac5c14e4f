"""The estimators fitting.py builds from fitted arrays are real scikit-learn objects that carry every attribute a
host fit sets (same names, dtypes, shapes) and compute what the host fit computes.  No GPU: the arrays come from
scikit-learn's own fits."""
import pickle
import warnings

import numpy as np
import pytest
from sklearn.decomposition import PCA
from sklearn.exceptions import ConvergenceWarning
from sklearn.preprocessing import RobustScaler
from sklearn.svm import OneClassSVM

from cell_image_analysis_b200 import artifacts, fitting


def _same_layout(a, b):
    va, vb = vars(a), vars(b)
    assert set(va) == set(vb), set(va) ^ set(vb)
    for k in va:
        x, y = va[k], vb[k]
        assert type(x) is type(y), (k, type(x), type(y))
        if isinstance(x, (np.ndarray, np.generic)):
            assert x.dtype == y.dtype and x.shape == y.shape, (k, x.dtype, y.dtype, x.shape, y.shape)


def _features(n=400, F=64, seed=0):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n, F)) @ rng.standard_normal((F, F)) * 0.3).astype(np.float32)


def _points(l=600, d=10, seed=1):
    rng = np.random.default_rng(seed)
    centers = rng.standard_normal((4, d)) * 3
    return centers[rng.integers(0, 4, l)] + rng.standard_t(3, (l, d))


def test_robust_scaler_from_arrays_is_the_fitted_scaler():
    X = _features()
    ref = RobustScaler().fit(X)
    est = fitting.robust_scaler_from_arrays(ref.center_, ref.scale_)
    _same_layout(est, ref)
    assert np.array_equal(est.transform(X), ref.transform(X))
    est2 = pickle.loads(pickle.dumps(est))
    assert np.array_equal(est2.transform(X), ref.transform(X))


def test_pca_from_spectrum_matches_the_full_svd():
    X = _features()
    n_components = 20
    X64 = X.astype(np.float64)
    mean = X64.mean(axis=0)
    Xc = X64 - mean
    w, v = np.linalg.eigh(Xc.T @ Xc / (len(X) - 1))
    est = fitting.pca_from_spectrum(mean, w[::-1], v[:, ::-1].T, len(X), n_components)
    _same_layout(est, PCA(n_components).fit(X))          # the attribute set and dtypes of a float32 fit
    ref = PCA(n_components, svd_solver="full").fit(X64)
    assert np.allclose(est.explained_variance_, ref.explained_variance_, rtol=1e-6)
    assert np.allclose(est.noise_variance_, ref.noise_variance_, rtol=1e-6)
    assert np.allclose(est.singular_values_, ref.singular_values_, rtol=1e-6)
    assert np.allclose(est.explained_variance_ratio_, ref.explained_variance_ratio_, rtol=1e-6)
    cos = np.sum(est.components_.astype(np.float64) * ref.components_, axis=1)
    assert np.all(cos > 1 - 1e-6), cos                  # the same sign as svd_flip gives the full solver
    z, zr = est.transform(X), ref.transform(X64)
    assert np.abs(z - zr).max() <= 1e-5 * np.abs(zr).max()
    sp = artifacts.scaler_pca_arrays(RobustScaler().fit(X), est)
    assert sp["f32_flow"] and sp["C"] == n_components


@pytest.mark.parametrize("nu", [0.05, 0.5])
def test_one_class_svm_from_solution_is_the_fitted_detector(nu):
    X = _points()
    ref = OneClassSVM(kernel="rbf", gamma="scale", nu=nu).fit(X)
    alpha = np.zeros(len(X))
    alpha[ref.support_] = ref.dual_coef_[0]
    est = fitting.one_class_svm_from_solution(X, alpha, -ref.intercept_[0], ref.n_iter_, ref.fit_status_, nu)
    _same_layout(est, ref)
    assert est._gamma == ref._gamma
    for k in ("support_", "support_vectors_", "_n_support", "dual_coef_", "intercept_", "offset_", "_num_iter"):
        assert np.array_equal(getattr(est, k), getattr(ref, k)), k
    assert est.n_iter_ == ref.n_iter_ and est.shape_fit_ == ref.shape_fit_
    Y = _points(200, seed=7)
    for f in ("decision_function", "score_samples", "predict"):
        assert np.array_equal(getattr(est, f)(Y), getattr(ref, f)(Y)), f
    est2 = pickle.loads(pickle.dumps(est))
    assert np.array_equal(est2.decision_function(Y), ref.decision_function(Y))
    a, b = artifacts.svm_arrays(est), artifacts.svm_arrays(ref)
    assert all(np.array_equal(a[k], b[k]) for k in a)


def test_max_iter_sets_fit_status_and_warns():
    X = _points()
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        ref = OneClassSVM(nu=0.1, max_iter=3).fit(X)
        alpha = np.zeros(len(X))
        alpha[ref.support_] = ref.dual_coef_[0]
        est = fitting.one_class_svm_from_solution(X, alpha, -ref.intercept_[0], ref.n_iter_, ref.fit_status_, 0.1,
                                                  max_iter=3)
    assert ref.fit_status_ == est.fit_status_ == 1
    assert sum(issubclass(x.category, ConvergenceWarning) for x in w) == 2
