"""Diagnostic (GPU box): decision / feature error of every CAE precision mode against the oracle
on held-out synthetic autoencoders.  Usage: python tests/diagnostics/heldout_probe.py [modes...]"""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from helpers import artifacts_from, fit_detectors, synth_cae_weights
from oracle import scoring as oscoring
from cell_image_analysis_b200 import synth
from cell_image_analysis_b200.screening import Engine, ProductionMutantScreening

SETS = [(7, 1.0, 3), (11, 1.0, 3), (23, 0.3, 3), (37, 3.0, 8), (51, 1.0, 0)]
modes = [int(m) for m in sys.argv[1:]] or [0, 1, 3]
s0 = ProductionMutantScreening(os.path.join(ROOT, "tests", "golden", "model_dir"), segmenter=lambda c: None, precision=0)
train = []
for seed in (200, 201, 202):
    g, l = synth.make_field(seed)
    train.extend(s0.extract_quality_cells_from_labels(g, l)[0])
g, l = synth.make_field(0)
test = s0.extract_quality_cells_from_labels(g, l)[0]
rng = np.random.default_rng(0)
dummy = fit_detectors(rng.standard_normal((64, 2048)).astype(np.float32))
for seed, scale, nneg in SETS:
    w = synth_cae_weights(seed, scale, nneg)
    eng = Engine(device=0, precision=1)
    eng.load_artifacts(artifacts_from(w, *dummy))
    xt = torch.from_numpy(np.array(train).astype(np.float32)).to(eng.tdev)
    _, _, feat = eng.cae_forward(xt, len(train), precision=0)
    scaler, pca, cons, mod = fit_detectors(feat[:len(train)].cpu().numpy())
    eng.load_artifacts(artifacts_from(w, scaler, pca, cons, mod))
    ref = oscoring.compute_anomaly_scores(test, w, w, scaler, pca, cons, mod)
    n = len(test)
    x = torch.from_numpy(np.array(test).astype(np.float32)).to(eng.tdev)
    iqr = scaler.scale_
    for mode in modes:
        for deb in ((0.5, 2.4, 1.2), (0, 0, 0)) if mode in (1, 3) else ((0, 0, 0),):
            for name, v in zip(("cae_l1_debias", "cae_l2_debias", "cae_l3_debias"), deb):
                eng.set_option(name, v)
            mse, mae, feat = eng.cae_forward(x, n, precision=mode)
            dc, dm, pc, pm, _ = eng.svm_decision(feat, n)
            f = feat[:n].cpu().numpy()
            df = f - ref["_features"]
            fe = np.abs(df).mean() / np.abs(ref["_features"]).mean()
            se = np.abs(df / iqr).max()
            print(f"set {seed}/{scale}/{nneg} mode {mode} debias {deb}: max|d dec| cons {np.abs(dc[:n].cpu().numpy() + ref['conservative_scores']).max():.2e} "
                  f"mod {np.abs(dm[:n].cpu().numpy() + ref['moderate_scores']).max():.2e}  mean rel feat err {fe:.2e}  signed bias {df.mean() / np.abs(ref['_features']).mean():+.2e}  max |df/iqr| {se:.2e}", flush=True)
    eng.close()
