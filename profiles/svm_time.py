"""Times cia_svm_decision (scaler/PCA + both detectors) at the default artifact sizes and at
config 4 (20k SVs x 256-d)."""
import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cell_image_analysis_b200.artifacts import load_model_dir
from cell_image_analysis_b200.screening import Engine

def run(tag, arts, n, reps=5):
    eng = Engine(device=0, precision=1)
    eng.load_artifacts(arts)
    rng = np.random.default_rng(0)
    feat = torch.from_numpy((rng.standard_normal((n, 2048)) * 3.0).astype(np.float32)).to(eng.tdev)
    z = torch.from_numpy(rng.standard_normal((n, arts["scaler_pca"]["C"]))).to(eng.tdev)
    for _ in range(2): out = eng.svm_decision(feat, n)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): out = eng.svm_decision(feat, n)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    sv = sum(arts[k]["sv"].shape[0] for k in ("svm_conservative", "svm_moderate"))
    D = arts["scaler_pca"]["C"]
    print(f"{tag}: n={n} D={D} nSV(total)={sv} "
          f"{ms:.3f} ms per call (PCA + 2 SVM), SVM GEMM-form {2*D*sv*n/ms/1e9:.2f} TFLOP/s if SVM-only, "
          f"checksum {float(out[0][:n].sum()):.12e}")
    eng.close()

root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
arts = load_model_dir(os.path.join(root, "tests", "golden", "model_dir"))
run("default", arts, 15130)
rng = np.random.default_rng(1)
DIM, NSV = 256, 20000
q, _ = np.linalg.qr(rng.standard_normal((2048, DIM)))
sp = dict(arts["scaler_pca"], C=DIM, center=None, scale=None, components=np.ascontiguousarray(q.T),
          offset=np.zeros(DIM), f32_flow=True)
a4 = dict(arts); a4["scaler_pca"] = sp
for k in ("svm_conservative", "svm_moderate"):
    sv = rng.standard_normal((NSV, DIM)) * 3.0
    a4[k] = dict(sv=sv, coef=rng.uniform(0, 1, NSV), gamma=1.0 / (DIM * 9.0), rho=1.0)
run("config4", a4, 4736)
