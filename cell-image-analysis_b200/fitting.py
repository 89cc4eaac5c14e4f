"""The fits of ``create_anomaly_detector`` (CAE_improved_modeltrain.py:404-423) on the GPU, returning real
scikit-learn estimators whose fitted attributes carry the names, dtypes and shapes a host ``fit`` gives them, so
that ``pickle``, ``artifacts.load_model_dir`` and scikit-learn's own ``transform`` / ``decision_function`` use them
unchanged.

* ``fit_robust_scaler(features)``      RobustScaler().fit           train:408      exact (csrc/fit.cu)
* ``fit_pca(features_scaled, n)``      PCA(n_components=n).fit      train:412-414  the exact subspace (fp64 covariance,
                                                                                   torch.linalg.eigh) that the
                                                                                   reference's randomized solver
                                                                                   approximates
* ``fit_one_class_svm(X, nu)``         OneClassSVM(kernel="rbf").fit train:420-423 libsvm's SMO iteration for iteration

Inputs are NumPy arrays or CUDA tensors; ``engine`` is a ``screening.Engine`` (one on cuda:0 when omitted).
"""
from __future__ import annotations

import ctypes as C

import numpy as np


def _engine(engine):
    if engine is None:
        from .screening import Engine
        engine = Engine(device=0)
    return engine


def _on_device(engine, x, dtype):
    import torch
    t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
    return t.to(device=engine.tdev, dtype=dtype).contiguous()


def _ptr(t):
    return C.c_void_p(t.data_ptr())


# ---- estimators from fitted arrays (no GPU) ----------------------------------------------------------------

def robust_scaler_from_arrays(center, scale):
    """A fitted ``RobustScaler()``: center_ float32, scale_ float64 as a fit on float32 features sets them."""
    from sklearn.preprocessing import RobustScaler
    est = RobustScaler()
    est.n_features_in_ = int(np.asarray(center).shape[0])
    est.center_ = np.asarray(center, np.float32).copy()
    est.scale_ = np.asarray(scale, np.float64).copy()
    return est


def pca_from_spectrum(mean, eigenvalues, eigenvectors, n_samples, n_components):
    """A fitted ``PCA(n_components)`` from the eigendecomposition of the covariance (sklearn's covariance_eigh,
    _pca.py): ``eigenvalues`` descending [k >= n_components], ``eigenvectors`` the matching rows [k, F].  Negative
    eigenvalues are clipped to 0, signs follow svd_flip(u_based_decision=False), and the spectrum is cut to
    min(n_samples, F) values as the full SVD has them.  Arrays are stored as float32, as a fit on float32 features
    stores them."""
    from sklearn.decomposition import PCA
    from sklearn.utils.extmath import svd_flip
    F = int(np.asarray(mean).shape[0])
    k = min(int(n_samples), F)
    ev = np.array(eigenvalues, np.float64)[:k]
    ev[ev < 0.0] = 0.0
    _, vt = svd_flip(None, np.array(eigenvectors, np.float64)[:n_components], u_based_decision=False)
    total_var = ev.sum()
    est = PCA(n_components=n_components)
    est.n_features_in_ = F
    est._fit_svd_solver = "covariance_eigh"
    est.mean_ = np.asarray(mean, np.float64).astype(np.float32)
    est.n_samples_ = int(n_samples)
    est.n_components_ = int(n_components)
    est.components_ = vt.astype(np.float32)
    est.explained_variance_ = ev[:n_components].astype(np.float32)
    est.explained_variance_ratio_ = (ev[:n_components] / total_var).astype(np.float32)
    est.singular_values_ = np.sqrt(ev[:n_components] * (n_samples - 1)).astype(np.float32)
    est.noise_variance_ = np.float32(ev[n_components:].mean() if n_components < k else 0.0)
    return est


def scale_gamma(X):
    """sklearn's gamma="scale" for dense X: 1 / (n_features * X.var())."""
    X_var = X.var()
    return 1.0 / (X.shape[1] * X_var) if X_var != 0 else 1.0


def one_class_svm_from_solution(X, alpha, rho, n_iter, fit_status, nu, gamma="scale", tol=1e-3, max_iter=-1,
                                gamma_value=None):
    """A fitted ``OneClassSVM(kernel="rbf")`` from libsvm's solution on X (float64 [l, d]): alpha [l] (support
    vectors are the nonzero entries, svm.cpp svm_train), rho and the iteration count.  A ``fit_status`` of 1
    (max_iter reached) issues sklearn's own ConvergenceWarning."""
    from sklearn.svm import OneClassSVM
    X = np.ascontiguousarray(X, np.float64)
    alpha = np.asarray(alpha, np.float64)
    est = OneClassSVM(kernel="rbf", gamma=gamma, nu=nu, tol=tol, max_iter=max_iter)
    sv = np.flatnonzero(alpha != 0).astype(np.int32)
    est._sparse = False
    est.n_features_in_ = X.shape[1]
    est._effective_probability = False
    est._gamma = scale_gamma(X) if gamma_value is None else gamma_value
    est.support_ = sv
    est.support_vectors_ = X[sv]
    est._n_support = np.array([len(sv), len(sv)], np.int32)
    est.dual_coef_ = alpha[sv].reshape(1, -1)
    est.intercept_ = np.array([-float(rho)])
    est._probA = np.empty(0, np.float64)
    est._probB = np.empty(0, np.float64)
    est.fit_status_ = int(fit_status)
    est._num_iter = np.array([int(n_iter)], np.int32)
    est.shape_fit_ = X.shape
    est._intercept_ = est.intercept_.copy()
    est._dual_coef_ = est.dual_coef_
    if not (np.isfinite(est._intercept_).all() and np.isfinite(est._dual_coef_).all()):   # as BaseLibSVM.fit
        raise ValueError("The dual coefficients or intercepts are not finite. The input data may contain large "
                         "values and need to be preprocessed.")
    est.n_iter_ = est._num_iter.item()
    est.offset_ = -est._intercept_
    est._warn_from_fit_status()
    return est


# ---- device fits ---------------------------------------------------------------------------------------------

def fit_robust_scaler_device(features, engine=None):
    """RobustScaler().fit on the device; returns (estimator, scaled) with scaled = transform(features), float32
    [n, F] on the device.  NaN is not supported (CIA_E_ARG)."""
    import torch
    eng = _engine(engine)
    x = _on_device(eng, features, torch.float32)
    n, F = x.shape
    center = torch.empty(F, dtype=torch.float32, device=eng.tdev)
    scale = torch.empty(F, dtype=torch.float64, device=eng.tdev)
    scaled = torch.empty_like(x)
    eng._check(eng.lib.cia_fit_robust_scaler(eng.h, _ptr(x), n, F, _ptr(center), _ptr(scale), _ptr(scaled),
                                             eng._stream()))
    eng.check_status()
    return robust_scaler_from_arrays(center.cpu().numpy(), scale.cpu().numpy()), scaled


def fit_robust_scaler(features, engine=None):
    """``RobustScaler().fit(features)`` (train:408) on the GPU: center_ and scale_ equal the host fit's."""
    return fit_robust_scaler_device(features, engine)[0]


def fit_pca(features_scaled, n_components, engine=None):
    """``PCA(n_components).fit(features_scaled)`` (train:412-414) on the GPU: fp64 covariance (csrc/fit.cu) and
    torch.linalg.eigh in float64 on the device, then sklearn's covariance_eigh post-processing."""
    import torch
    eng = _engine(engine)
    x = _on_device(eng, features_scaled, torch.float32)
    n, F = x.shape
    if not 1 <= n_components <= min(n, F):
        raise ValueError(f"n_components={n_components} must be between 1 and min(n_samples, n_features)={min(n, F)}")
    mean = torch.empty(F, dtype=torch.float64, device=eng.tdev)
    cov = torch.empty((F, F), dtype=torch.float64, device=eng.tdev)
    eng._check(eng.lib.cia_fit_pca_gram(eng.h, _ptr(x), n, F, _ptr(mean), _ptr(cov), eng._stream()))
    evals, evecs = torch.linalg.eigh(cov)
    k = min(n, F)
    evals = torch.flip(evals, (0,))[:k]
    vt = torch.flip(evecs, (1,))[:, :n_components].T
    return pca_from_spectrum(mean.cpu().numpy(), evals.cpu().numpy(), vt.cpu().numpy(), n, n_components)


def fit_one_class_svm(X, nu, gamma="scale", tol=1e-3, max_iter=-1, engine=None):
    """``OneClassSVM(kernel="rbf", gamma=gamma, nu=nu, tol=tol, max_iter=max_iter).fit(X)`` with libsvm's SMO run
    on the GPU (csrc/fit.cu): the same working sets, updates and stopping rule, hence the same iterations, support
    vectors and, to rounding of the kernel values, the same dual coefficients and offset.  X: float64 [l, d]
    (float32 is widened like sklearn's validate_data), d <= 512."""
    import torch
    eng = _engine(engine)
    x = _on_device(eng, X, torch.float64)
    X_host = x.cpu().numpy()
    l, d = x.shape
    g = scale_gamma(X_host) if gamma == "scale" else float(gamma)
    alpha = torch.empty(l, dtype=torch.float64, device=eng.tdev)
    result = torch.empty(4, dtype=torch.float64, device=eng.tdev)
    eng._check(eng.lib.cia_ocsvm_fit(eng.h, _ptr(x), l, d, C.c_double(nu), C.c_double(g), C.c_double(tol),
                                     int(max_iter), _ptr(alpha), _ptr(result), eng._stream()))
    rho, _obj, n_iter, status = result.cpu().numpy().tolist()
    return one_class_svm_from_solution(X_host, alpha.cpu().numpy(), rho, int(n_iter), int(status), nu, gamma=gamma,
                                       tol=tol, max_iter=max_iter, gamma_value=g)
