"""Times the device fits of fitting.py (RobustScaler, PCA, both one-class SVMs) at 20k / 60k / 200k cells
(2048 features -> 100 components), and scikit-learn's host fits at 20k / 60k in the same run.

    python tools/fit_probe.py [--sizes 20000,60000,200000] [--host-sizes 20000,60000] [--out DIR]

Prints the card name and power limit, each fit's wall time (host clock around work that ends in a device
synchronise), libsvm's iteration count and microseconds per iteration.  Features are synthetic, clustered and
heavy-tailed (seeded), so the SVM sees the shape of real PCA scores."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def features(n, F=2048, seed=0):
    rng = np.random.default_rng(seed)
    basis = rng.standard_normal((64, F)).astype(np.float32)
    centers = rng.standard_normal((8, 64)).astype(np.float32) * 2
    lat = centers[rng.integers(0, 8, n)] + rng.standard_t(4, (n, 64)).astype(np.float32)
    return np.maximum(lat @ basis * 0.1 + 0.05 * rng.standard_normal((n, F)).astype(np.float32), 0).astype(np.float32)


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="20000,60000,200000")
    ap.add_argument("--host-sizes", default="20000,60000")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from cell_image_analysis_b200 import fitting
    from cell_image_analysis_b200.screening import Engine
    eng = Engine(device=0)
    print(f"card: {card()}")
    sync = torch.cuda.synchronize
    rows = []
    warm = features(2000, seed=99)
    sc, xs = fitting.fit_robust_scaler_device(warm, eng)
    fitting.fit_pca(xs, 100, eng)
    for n in [int(s) for s in a.sizes.split(",") if s]:
        f = torch.from_numpy(features(n, seed=n)).to(eng.tdev)
        sync()
        t0 = time.perf_counter(); sc, xs = fitting.fit_robust_scaler_device(f, eng); sync(); t_sc = time.perf_counter() - t0
        t0 = time.perf_counter(); pca = fitting.fit_pca(xs, 100, eng); sync(); t_pca = time.perf_counter() - t0
        z = torch.from_numpy(pca.transform(sc.transform(f.cpu().numpy())).astype(np.float64)).to(eng.tdev)
        row = dict(cells=n, scaler_s=t_sc, pca_s=t_pca)
        for nu in (0.05, 0.10):
            sync()
            t0 = time.perf_counter(); det = fitting.fit_one_class_svm(z, nu, engine=eng); sync()
            t = time.perf_counter() - t0
            row[f"svm_{nu}_s"], row[f"svm_{nu}_iter"] = t, det.n_iter_
            row[f"svm_{nu}_us_per_iter"] = 1e6 * t / max(det.n_iter_, 1)
        print(json.dumps(row), flush=True)
        rows.append(row)
    from sklearn.decomposition import PCA
    from sklearn.preprocessing import RobustScaler
    from sklearn.svm import OneClassSVM
    for n in [int(s) for s in a.host_sizes.split(",") if s]:
        f = features(n, seed=n)
        t0 = time.perf_counter(); sc = RobustScaler().fit(f); xs = sc.transform(f); t_sc = time.perf_counter() - t0
        t0 = time.perf_counter(); pca = PCA(100).fit(xs); t_pca = time.perf_counter() - t0
        z = pca.transform(xs).astype(np.float64)
        row = dict(host=True, cells=n, scaler_s=t_sc, pca_s=t_pca)
        for nu in (0.05, 0.10):
            t0 = time.perf_counter(); det = OneClassSVM(kernel="rbf", gamma="scale", nu=nu).fit(z)
            row[f"svm_{nu}_s"], row[f"svm_{nu}_iter"] = time.perf_counter() - t0, det.n_iter_
        print(json.dumps(row), flush=True)
        rows.append(row)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "fit_probe.json"), "w") as fh:
            json.dump(dict(card=card(), rows=rows), fh, indent=1)


if __name__ == "__main__":
    main()
