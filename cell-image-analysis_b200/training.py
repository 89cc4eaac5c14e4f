"""Training-side users of the hot path (SURVEY.md §8b B5 / §8f row N4): the methods of
``ImprovedAnomalyDetectionTraining`` (CAE_improved_modeltrain.py:25) that run the SAME per-cell
extraction and CAE arithmetic as the screener, on the GPU:

* ``extract_quality_cells(image_path, stardist_model)``      train:39-111  (adds 'solidity' and 'file')
* ``create_training_dataset(folder_path)``                  train:113-157 (cell_statistics.csv, file_summary.csv)
* ``generate_data_quality_report``                          train:159-182
* ``evaluate_reconstruction_quality(autoencoder, cells)``   train:328-339 (the arithmetic; plots stay with the caller)
* ``create_anomaly_detector(encoder, cells)``               train:394-446 (features on the GPU; the scikit-learn
                                                            fits are the reference's own library calls)
* ``create_anomaly_detector_on_device(encoder, cells)``     train:394-446 with the four fits on the GPU too
                                                            (fitting.py, csrc/fit.cu)

Out of scope (SURVEY.md §2 C12-C14): the Keras model definition and ``fit`` loop
(``create_improved_autoencoder`` / ``train_autoencoder``) -- they define the weight-file contract the
loader reads, nothing on the screening path.  ``autoencoder`` / ``encoder`` arguments are therefore
paths to ``.keras`` files (or weight dicts as ``artifacts.load_keras_cae`` returns them), not Keras models.
"""
from __future__ import annotations

import os
import pickle
from datetime import datetime
from glob import glob

import numpy as np

from .artifacts import load_keras_cae
from .screening import Engine, ProductionMutantScreening, UnsupportedImageError, _default_imread


def normalize_percentile(x, pmin=3, pmax=99.8, eps=1e-20):
    """csbdeep.utils.normalize with its defaults (train:54, det:62): percentile-based scaling to
    float32, ``(x - p_lo) / (p_hi - p_lo + eps)`` without clipping.  Used when csbdeep is absent."""
    lo, hi = np.percentile(x, pmin), np.percentile(x, pmax)
    x = x.astype(np.float32, copy=False)
    return (x - np.float32(lo)) / (np.float32(hi) - np.float32(lo) + np.float32(eps))


def _normalize(x):
    try:
        from csbdeep.utils import normalize          # train:21
        return normalize(x)
    except ImportError:
        return normalize_percentile(x)


class _Extractor(ProductionMutantScreening):
    """The extraction half of the drop-in without the scoring artifacts."""

    def __init__(self, device=0, imread=None):
        self.model_dir, self.segmenter = None, None
        self.imread = imread or _default_imread
        self.engine = Engine(device=device)


class ImprovedAnomalyDetectionTraining:
    """Mirror of the reference class of the same name (train:25) for the methods listed above."""

    def __init__(self, output_dir, device: int = 0, imread=None):
        self.output_dir = output_dir                     # train:26-29
        os.makedirs(output_dir, exist_ok=True)
        self._x = _Extractor(device=device, imread=imread)
        self.engine = self._x.engine

    # train:39-111
    def extract_quality_cells(self, image_path, stardist_model):
        try:
            image = self._x.imread(image_path)
            if image.ndim == 3 and image.shape[-1] >= 3:          # train:45-51
                seg_channel, green_channel = image[..., 2], image[..., 1]
            else:
                seg_channel = green_channel = image
            if hasattr(stardist_model, "segment_device") and np.asarray(seg_channel).dtype in (np.uint8, np.uint16):
                labels, _n = stardist_model.segment_device(seg_channel)      # train:54-55 on the GPU, labels stay there
            else:
                labels, _details = stardist_model.predict_instances(_normalize(seg_channel))   # train:54-55
            cells, stats = self._x.extract_quality_cells_from_labels(green_channel, labels)
            for s in stats:
                s["file"] = os.path.basename(image_path)          # train:104
            return cells, stats
        except UnsupportedImageError:
            raise
        except Exception as e:                                     # train:109-111
            print(f"Error processing {image_path}: {e}")
            return [], []

    # train:113-157
    def create_training_dataset(self, folder_path, stardist_model=None):
        import pandas as pd
        print("=== Creating High-Quality Training Dataset ===")
        if stardist_model is None:
            from stardist.models import StarDist2D
            stardist_model = StarDist2D.from_pretrained("2D_versatile_fluo")       # train:118
        file_paths = sorted(glob(os.path.join(folder_path, "*.tif")))
        print(f"Found {len(file_paths)} image files")
        all_cells, all_stats, file_summary = [], [], []
        for i, file_path in enumerate(file_paths):
            filename = os.path.basename(file_path)
            print(f"Processing {i + 1}/{len(file_paths)}: {filename}")
            cells, stats = self.extract_quality_cells(file_path, stardist_model)
            all_cells.extend(cells)
            all_stats.extend(stats)
            file_summary.append({"filename": filename, "cells_extracted": len(cells),
                                 "mean_cell_intensity": np.mean([s["mean_intensity"] for s in stats]) if stats else 0})
            print(f"  Extracted {len(cells)} quality cells")
        print(f"\nTotal quality cells extracted: {len(all_cells)}")
        stats_df = pd.DataFrame(all_stats)
        file_summary_df = pd.DataFrame(file_summary)
        stats_df.to_csv(os.path.join(self.output_dir, "cell_statistics.csv"), index=False)
        file_summary_df.to_csv(os.path.join(self.output_dir, "file_summary.csv"), index=False)
        self.generate_data_quality_report(stats_df, file_summary_df)
        return np.array(all_cells), stats_df

    # train:159-182 (the on-disk layout of data_quality_report.txt is the contract; built as a line list)
    _REPORT_COLUMNS = (("CELL MORPHOLOGY STATISTICS:", (("Area", "area", 1), ("Eccentricity", "eccentricity", 3),
                                                        ("Solidity", "solidity", 3))),
                       ("INTENSITY STATISTICS:", (("Mean intensity", "mean_intensity", 3),
                                                  ("Std intensity", "std_intensity", 3))))

    def generate_data_quality_report(self, stats_df, file_summary_df):
        n_files, n_cells = len(file_summary_df), len(stats_df)
        lines = ["=== TRAINING DATA QUALITY REPORT ===", "",
                 "Generated: " + datetime.now().strftime("%Y-%m-%d %H:%M:%S"), "",
                 "OVERALL STATISTICS:",
                 f"Total files processed: {n_files}",
                 f"Total cells extracted: {n_cells}",
                 f"Average cells per file: {n_cells / n_files:.1f}", ""]
        for title, columns in self._REPORT_COLUMNS:
            lines.append(title)
            for label, column, digits in columns:           # pandas' sample std (ddof = 1), like the reference
                col = stats_df[column]
                lines.append(f"{label}: {col.mean():.{digits}f} ± {col.std():.{digits}f}")
            lines.append("")
        lines.append("FILE-WISE SUMMARY:")
        lines += [f"{name}: {count} cells, avg intensity: {mean:.3f}"
                  for name, count, mean in zip(file_summary_df["filename"], file_summary_df["cells_extracted"],
                                               file_summary_df["mean_cell_intensity"])]
        with open(os.path.join(self.output_dir, "data_quality_report.txt"), "w") as f:
            f.write("\n".join(lines) + "\n")

    def _weights(self, model, n_conv):
        w = load_keras_cae(model) if isinstance(model, (str, os.PathLike)) else model
        if w["n_conv"] not in (n_conv, 7):
            raise ValueError(f"expected a {n_conv}-conv CAE, got {w['n_conv']}")
        return w

    def _load(self, autoencoder=None, encoder=None):
        """Upload CAE weights; scaler / PCA / detectors are placeholders (never evaluated here)."""
        from sklearn.decomposition import PCA
        from sklearn.preprocessing import RobustScaler
        from sklearn.svm import OneClassSVM
        from . import artifacts as A
        rng = np.random.default_rng(0)
        f = rng.standard_normal((8, 2048)).astype(np.float32)
        sc, pca = RobustScaler().fit(f), PCA(n_components=2).fit(f)
        det = OneClassSVM(kernel="rbf", gamma="scale", nu=0.5).fit(pca.transform(sc.transform(f)))
        ae = autoencoder if autoencoder is not None else encoder
        if ae["n_conv"] != 7:
            # encoder only: the decoder half is never read for features; pad with zeros to satisfy the loader
            from .artifacts import FILTERS
            cin = [1] + FILTERS[:-1]
            ae = dict(ae, n_conv=7,
                      kernels=list(ae["kernels"]) + [np.zeros((3, 3, cin[i], FILTERS[i]), np.float32) for i in range(3, 7)],
                      biases=list(ae["biases"]) + [np.zeros(FILTERS[i], np.float32) for i in range(3, 7)],
                      bns=list(ae["bns"]) + [tuple(np.ones(FILTERS[i], np.float32) for _ in range(4)) for i in range(3, 6)])
        arts = dict(autoencoder=ae, encoder_same=True, scaler_pca=A.scaler_pca_arrays(sc, pca),
                    svm_conservative=A.svm_arrays(det), svm_moderate=A.svm_arrays(det))
        self._arts = arts
        self.engine.load_artifacts(arts)

    # train:328-339
    def evaluate_reconstruction_quality(self, autoencoder, cell_images):
        import torch
        print("=== Evaluating Reconstruction Quality ===")
        self._load(autoencoder=self._weights(autoencoder, 7))
        X = np.expand_dims(np.asarray(cell_images), axis=-1).astype("float32")         # train:332
        x = torch.from_numpy(np.ascontiguousarray(X[..., 0])).to(self.engine.tdev)
        mse, mae, _ = self.engine.cae_forward(x, len(X))
        self.engine.check_status()
        mse_errors, mae_errors = mse[:len(X)].cpu().numpy(), mae[:len(X)].cpu().numpy()
        print(f"MSE - Mean: {np.mean(mse_errors):.6f}, Std: {np.std(mse_errors):.6f}")
        print(f"MAE - Mean: {np.mean(mae_errors):.6f}, Std: {np.std(mae_errors):.6f}")
        return mse_errors, mae_errors

    def encode_features(self, encoder, cell_images):
        """train:398-402: ``encoder.predict(X)`` flattened HWC, float32 [N, 2048]."""
        import torch
        self._load(encoder=self._weights(encoder, 3))
        X = np.expand_dims(np.asarray(cell_images), axis=-1).astype("float32")
        x = torch.from_numpy(np.ascontiguousarray(X[..., 0])).to(self.engine.tdev)
        _mse, _mae, feat = self.engine.cae_forward(x, len(X))
        self.engine.check_status()
        return feat[:len(X)].cpu().numpy()

    # train:394-446
    def create_anomaly_detector(self, encoder, cell_images):
        from sklearn.decomposition import PCA
        from sklearn.preprocessing import RobustScaler
        from sklearn.svm import OneClassSVM
        print("=== Creating Anomaly Detector ===")
        features_flat = self.encode_features(encoder, cell_images)
        print(f"Encoded features shape: {(len(features_flat), 8, 8, 32)}")
        print(f"Flattened features shape: {features_flat.shape}")
        scaler = RobustScaler()                                                       # train:408
        features_scaled = scaler.fit_transform(features_flat)
        n_components = min(100, features_scaled.shape[1], features_scaled.shape[0] - 1)   # train:412
        pca = PCA(n_components=n_components)
        features_reduced = pca.fit_transform(features_scaled)
        print(f"PCA reduced to {n_components} components")
        print(f"Explained variance ratio (first 5): {pca.explained_variance_ratio_[:5]}")
        detectors = {"Conservative": OneClassSVM(kernel="rbf", gamma="scale", nu=0.05),
                     "Moderate": OneClassSVM(kernel="rbf", gamma="scale", nu=0.10)}   # train:420-423
        for detector in detectors.values():
            detector.fit(features_reduced)
        print("\nBaseline anomaly rates:")
        for name, detector in detectors.items():
            predictions = detector.predict(features_reduced)
            print(f"{name}: {np.sum(predictions == -1) / len(predictions) * 100:.2f}%")
        for fname, obj in (("scaler.pkl", scaler), ("pca.pkl", pca)):               # train:437-444
            with open(os.path.join(self.output_dir, fname), "wb") as f:
                pickle.dump(obj, f)
        for name, detector in detectors.items():
            with open(os.path.join(self.output_dir, f"detector_{name.lower()}.pkl"), "wb") as f:
                pickle.dump(detector, f)
        return detectors, scaler, pca

    # train:394-446, every fit on the GPU: the features stay on the device from the encoder to the SVM fits
    def create_anomaly_detector_on_device(self, encoder, cell_images):
        import torch
        from . import artifacts as A
        from . import fitting
        print("=== Creating Anomaly Detector ===")
        self._load(encoder=self._weights(encoder, 3))
        X = np.expand_dims(np.asarray(cell_images), axis=-1).astype("float32")
        x = torch.from_numpy(np.ascontiguousarray(X[..., 0])).to(self.engine.tdev)
        _mse, _mae, feat = self.engine.cae_forward(x, len(X))
        self.engine.check_status()
        n = len(X)
        feat = feat[:n]
        print(f"Encoded features shape: {(n, 8, 8, 32)}")
        print(f"Flattened features shape: {tuple(feat.shape)}")
        scaler, features_scaled = fitting.fit_robust_scaler_device(feat, self.engine)        # train:408
        n_components = min(100, feat.shape[1], n - 1)                                      # train:412
        pca = fitting.fit_pca(features_scaled, n_components, self.engine)
        print(f"PCA reduced to {n_components} components")
        print(f"Explained variance ratio (first 5): {pca.explained_variance_ratio_[:5]}")
        # the PCA scores of the scoring path (scaler.transform -> pca.transform, the exact fp64 kernels) with the
        # fitted arrays loaded; the detectors are placeholders here and their outputs unused
        placeholder = dict(sv=np.zeros((1, n_components)), coef=np.ones(1), gamma=1.0, rho=0.0)
        arts = dict(self._arts, scaler_pca=A.scaler_pca_arrays(scaler, pca), svm_conservative=placeholder,
                    svm_moderate=placeholder)
        self.engine.load_artifacts(arts)
        features_reduced = self.engine.svm_decision(feat, n, want_pca=True, precision=0)[4][:n]
        detectors = {"Conservative": fitting.fit_one_class_svm(features_reduced, 0.05, engine=self.engine),
                     "Moderate": fitting.fit_one_class_svm(features_reduced, 0.10, engine=self.engine)}   # train:420-423
        arts.update(svm_conservative=A.svm_arrays(detectors["Conservative"]),
                    svm_moderate=A.svm_arrays(detectors["Moderate"]))
        self.engine.load_artifacts(arts)
        _dc, _dm, pred_c, pred_m, _ = self.engine.svm_decision(feat, n, precision=0)
        print("\nBaseline anomaly rates:")
        for name, pred in (("Conservative", pred_c), ("Moderate", pred_m)):
            predictions = pred[:n].cpu().numpy()
            print(f"{name}: {np.sum(predictions == -1) / len(predictions) * 100:.2f}%")
        for fname, obj in (("scaler.pkl", scaler), ("pca.pkl", pca)):               # train:437-444
            with open(os.path.join(self.output_dir, fname), "wb") as f:
                pickle.dump(obj, f)
        for name, detector in detectors.items():
            with open(os.path.join(self.output_dir, f"detector_{name.lower()}.pkl"), "wb") as f:
                pickle.dump(detector, f)
        return detectors, scaler, pca

    def create_improved_autoencoder(self, *a, **k):
        raise NotImplementedError("CAE definition / fit (train:184-302) is out of scope: train with the reference "
                                  "script and point the screener at the saved .keras files")

    train_autoencoder = create_improved_autoencoder
