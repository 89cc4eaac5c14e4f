"""The device fits of fitting.py against scikit-learn's host fits: RobustScaler exactly, PCA to the exact subspace,
OneClassSVM iteration for iteration (libsvm's SMO), and create_anomaly_detector_on_device against
create_anomaly_detector."""
import os
import pickle

import numpy as np
import pytest
from sklearn.decomposition import PCA
from sklearn.preprocessing import RobustScaler
from sklearn.svm import OneClassSVM

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from cell_image_analysis_b200.screening import Engine
    return Engine(device=0)


def scores_like(l, d=100, seed=0):
    """Clustered, heavy-tailed points with decaying scales, rounded to float32 and widened (PCA scores)."""
    rng = np.random.default_rng(seed)
    scales = 3.0 / np.sqrt(1 + np.arange(d))
    centers = rng.standard_normal((8, d)) * scales * 2
    X = centers[rng.integers(0, 8, l)] + rng.standard_t(4, (l, d)) * scales
    return X.astype(np.float32).astype(np.float64)


# ---- RobustScaler ----------------------------------------------------------------------------------------------

SCALER_CASES = {
    "n1": (1, 16, "normal"), "n2": (2, 16, "normal"), "n3": (3, 16, "normal"), "odd": (1001, 33, "normal"),
    "even": (1000, 33, "normal"), "ties": (777, 40, "ties"), "relu": (600, 40, "relu"),
    "2048x60000": (60000, 2048, "normal"),
}


@pytest.mark.parametrize("case", sorted(SCALER_CASES))
def test_robust_scaler_equals_sklearn(engine, case):
    from cell_image_analysis_b200 import fitting
    n, F, kind = SCALER_CASES[case]
    rng = np.random.default_rng(n + F)
    if kind == "ties":
        X = rng.integers(0, 5, (n, F)).astype(np.float32) * np.float32(0.25)
    elif kind == "relu":
        X = np.maximum(rng.standard_normal((n, F)), 0).astype(np.float32)
    else:
        X = (rng.standard_normal((n, F)) * rng.uniform(0.01, 10, F)).astype(np.float32)
    est, scaled = fitting.fit_robust_scaler_device(X, engine)
    ref = RobustScaler().fit(X)
    assert est.center_.dtype == ref.center_.dtype and est.scale_.dtype == ref.scale_.dtype
    assert np.array_equal(est.center_, ref.center_) and np.array_equal(est.scale_, ref.scale_)
    assert np.array_equal(scaled.cpu().numpy(), ref.transform(X))


def test_robust_scaler_refuses_nan(engine):
    from cell_image_analysis_b200 import _lib, fitting
    X = np.ones((10, 4), np.float32)
    X[3, 2] = np.nan
    with pytest.raises(_lib.CiaError) as e:
        fitting.fit_robust_scaler(X, engine)
    assert e.value.code == _lib.CIA_E_ARG


# ---- PCA -------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("n,F", [(5000, 2048), (60, 300), (101, 128)])
def test_pca_matches_the_full_svd(engine, n, F):
    from cell_image_analysis_b200 import fitting
    rng = np.random.default_rng(F)
    X = (rng.standard_normal((n, 64)) @ rng.standard_normal((64, F)) + 0.1 * rng.standard_normal((n, F)))
    X = (X * np.exp(-np.arange(F) / F)).astype(np.float32)
    n_components = min(100, F, n - 1)                    # train:412
    est = fitting.fit_pca(X, n_components, engine)
    ref = PCA(n_components, svd_solver="full").fit(X.astype(np.float64))
    assert est.components_.dtype == np.float32 and est.mean_.dtype == np.float32
    assert est.n_components_ == n_components and est.components_.shape == (n_components, F)
    ev, evr = est.explained_variance_.astype(np.float64), ref.explained_variance_
    assert np.abs(ev / evr - 1).max() <= 1e-6
    # relative to the leading eigenvalue as well: with n <= F the discarded spectrum is zero up to rounding
    assert abs(float(est.noise_variance_) - ref.noise_variance_) <= 1e-6 * ref.noise_variance_ + 1e-12 * evr[0]
    full = PCA(svd_solver="full").fit(X.astype(np.float64)).explained_variance_
    gap = np.minimum(np.abs(np.diff(full, prepend=np.inf)), np.abs(np.diff(full, append=-np.inf)))[:n_components] / full[:n_components]
    cos = np.sum(est.components_.astype(np.float64) * ref.components_, axis=1)
    assert np.all(1 - cos[gap >= 1e-3] <= 1e-8 + 2e-7), (1 - cos)[gap >= 1e-3].max()   # + float32 storage
    z, zr = est.transform(X), ref.transform(X.astype(np.float64))
    good = gap >= 1e-3
    assert np.abs(z[:, good] - zr[:, good]).max() <= 1e-5 * np.abs(zr).max()


# ---- OneClassSVM -----------------------------------------------------------------------------------------------

def _check_parity(est, ref, X, Y):
    assert est.n_iter_ == ref.n_iter_, (est.n_iter_, ref.n_iter_)
    assert np.array_equal(est.support_, ref.support_)
    assert est._gamma == ref._gamma
    assert np.abs(est.dual_coef_ - ref.dual_coef_).max() <= 1e-9
    off = abs(float(ref.offset_[0]))
    assert abs(float(est.offset_[0] - ref.offset_[0])) <= 1e-9 * off
    for Z in (X, Y):
        assert np.abs(est.decision_function(Z) - ref.decision_function(Z)).max() <= 1e-8 * off
        assert np.array_equal(est.predict(Z), ref.predict(Z))


@pytest.mark.parametrize("l", [4000, 12000, 60000])
@pytest.mark.parametrize("nu", [0.05, 0.10])
def test_one_class_svm_follows_libsvm(engine, l, nu):
    from cell_image_analysis_b200 import fitting
    X, Y = scores_like(l, seed=l), scores_like(2000, seed=l + 1)
    est = fitting.fit_one_class_svm(X, nu, engine=engine)
    ref = OneClassSVM(kernel="rbf", gamma="scale", nu=nu).fit(X)
    _check_parity(est, ref, X, Y)


def test_one_class_svm_tight_tolerance(engine):
    from cell_image_analysis_b200 import fitting
    X, Y = scores_like(4000, seed=5), scores_like(1000, seed=6)
    est = fitting.fit_one_class_svm(X, 0.05, tol=1e-8, engine=engine)
    ref = OneClassSVM(kernel="rbf", gamma="scale", nu=0.05, tol=1e-8).fit(X)
    _check_parity(est, ref, X, Y)


CORNERS = {
    "integer_nu_l": (2000, 0.05, None), "fractional_nu_l": (1999, 0.05, None), "nu_l_below_1": (10, 0.05, None),
    "nu_1": (300, 1.0, None), "duplicates": (900, 0.1, "dup"), "l1": (1, 0.5, None), "l2": (2, 0.5, None),
    "max_iter": (3000, 0.1, "max_iter"),
}


@pytest.mark.parametrize("case", sorted(CORNERS))
def test_one_class_svm_corner_cases(engine, case):
    import warnings
    from cell_image_analysis_b200 import fitting
    l, nu, kind = CORNERS[case]
    X = scores_like(l, d=20, seed=l)
    if kind == "dup":
        X = np.concatenate([X[:300]] * 3)                  # quad_coef = 0 between copies: TAU
    max_iter = 25 if kind == "max_iter" else -1
    if nu == 1.0:                                          # every alpha at 1: rho = inf, which sklearn refuses
        with pytest.raises(ValueError, match="not finite"):
            OneClassSVM(kernel="rbf", gamma="scale", nu=nu).fit(X)
        with pytest.raises(ValueError, match="not finite"):
            fitting.fit_one_class_svm(X, nu, engine=engine)
        return
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        est = fitting.fit_one_class_svm(X, nu, max_iter=max_iter, engine=engine)
        ref = OneClassSVM(kernel="rbf", gamma="scale", nu=nu, max_iter=max_iter).fit(X)
    assert est.fit_status_ == ref.fit_status_
    _check_parity(est, ref, X, X[: min(l, 50)])


def test_one_class_svm_is_deterministic(engine):
    from cell_image_analysis_b200 import fitting
    X = scores_like(8000, seed=3)
    a = fitting.fit_one_class_svm(X, 0.1, engine=engine)
    b = fitting.fit_one_class_svm(X, 0.1, engine=engine)
    assert np.array_equal(a.dual_coef_, b.dual_coef_) and np.array_equal(a.offset_, b.offset_)
    assert a.n_iter_ == b.n_iter_


# ---- end to end ------------------------------------------------------------------------------------------------

def test_create_anomaly_detector_on_device(tmp_path, model_dir, artifacts):
    from cell_image_analysis_b200 import synth
    from cell_image_analysis_b200.screening import ProductionMutantScreening
    from cell_image_analysis_b200.training import ImprovedAnomalyDetectionTraining
    s = ProductionMutantScreening(model_dir, segmenter=lambda ch: None, device=0, precision=0)
    cells = []
    for seed in range(4):
        green, labels = synth.make_field(seed)
        cells += s.extract_quality_cells_from_labels(green, labels)[0]
    cells = np.array(cells)
    assert len(cells) > 150
    enc = os.path.join(model_dir, "encoder.keras")
    host_dir, dev_dir = tmp_path / "host", tmp_path / "dev"
    t_host = ImprovedAnomalyDetectionTraining(str(host_dir))
    _, sc_ref, _ = t_host.create_anomaly_detector(enc, cells)
    t_dev = ImprovedAnomalyDetectionTraining(str(dev_dir))
    dets, sc, pca = t_dev.create_anomaly_detector_on_device(enc, cells)
    assert sorted(os.listdir(dev_dir)) == sorted(os.listdir(host_dir))
    with open(dev_dir / "scaler.pkl", "rb") as f:
        sc_dev = pickle.load(f)
    assert np.array_equal(sc_dev.center_, sc_ref.center_) and np.array_equal(sc_dev.scale_, sc_ref.scale_)
    # the detectors equal sklearn's fit on the device's PCA scores (the scoring path, fitted arrays loaded)
    import torch
    eng = t_dev.engine
    x = torch.from_numpy(np.ascontiguousarray(cells, np.float32)).to(eng.tdev)
    feat = eng.cae_forward(x, len(cells))[2]
    z = eng.svm_decision(feat, len(cells), want_pca=True, precision=0)[4][:len(cells)].cpu().numpy()
    for name, nu in (("Conservative", 0.05), ("Moderate", 0.10)):
        ref = OneClassSVM(kernel="rbf", gamma="scale", nu=nu).fit(z)
        _check_parity(dets[name], ref, z, z[:50])
    # a screener loaded from the device-written folder scores like sklearn on the same pickles
    for fname in ("best_autoencoder.keras", "encoder.keras"):
        os.symlink(os.path.join(model_dir, fname), dev_dir / fname)
    s2 = ProductionMutantScreening(str(dev_dir), segmenter=lambda ch: None, device=0, precision=0)
    r = s2.compute_anomaly_scores(cells)
    zz = s2.pca.transform(s2.scaler.transform(s2.encode_features(cells)))
    dec = s2.detector_conservative.decision_function(zz)
    assert np.abs(-r["conservative_scores"] - dec).max() <= 1e-4
