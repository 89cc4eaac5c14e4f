"""GPU debugging aid (not a pytest module): layer-by-layer comparison of the tensor-core
CAE path against the oracle, through the cia_debug_copy_workspace tap.

    python tests/diagnostics/debug_tc.py [precision]      # on the B200 box
"""
import ctypes as C
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from cell_image_analysis_b200.screening import ProductionMutantScreening  # noqa: E402
from oracle import cae as ocae  # noqa: E402
from test_gpu_cae_layers import PASS_CELLS, ws_layout  # noqa: E402


def oracle_layers(X, w):
    outs = []
    x = torch.from_numpy(np.ascontiguousarray(X))[:, None]
    for i in range(7):
        x = ocae._conv(x, w["kernels"][i], w["biases"][i], True)
        if i < 6:
            x = ocae._bn(torch.relu(x), w["bns"][i])
            if i < 3:
                x = F.max_pool2d(x, 2)
            outs.append(x.permute(0, 2, 3, 1).numpy().copy())
            if i >= 3:
                x = F.interpolate(x, scale_factor=2, mode="nearest")
        else:
            outs.append(torch.sigmoid(x)[:, 0].numpy().copy())
    return outs


def planar_to_nhwc(buf, n, nch, r):
    return buf.reshape(n, nch, r, r, 8).transpose(0, 2, 3, 1, 4).reshape(n, r, r, nch * 8)


def main():
    prec = int(sys.argv[1]) if len(sys.argv) > 1 else 1
    s = ProductionMutantScreening(os.path.join(ROOT, "tests", "golden", "model_dir"), segmenter=lambda c: None)
    g = np.load(os.path.join(ROOT, "tests", "golden", "tiny_field.npz"))
    X = g["crops"].astype(np.float32)
    n = len(X)
    eng = s.engine
    ae = s.artifacts["autoencoder"]
    w = {"kernels": ae["kernels"], "biases": ae["biases"], "bns": ae["bns"]}
    ref = oracle_layers(X, w)
    x = torch.from_numpy(X).to(eng.tdev)
    mse, mae, feat = eng.cae_forward(x, n, precision=prec)
    torch.cuda.synchronize()
    # buffer offsets of k_cae_forward_tc at the handle's default pass size (one pass for this field)
    _, layout, c0, chunk = ws_layout(n, PASS_CELLS)
    assert (c0, chunk) == (0, n)
    bufs = {}
    for name, (off, per, _, _) in layout.items():
        dst = np.empty(n * per, np.float16)
        rc = eng.lib.cia_debug_copy_workspace(eng.h, 5, C.c_size_t(off * 2), C.c_void_p(dst.ctypes.data),
                                              C.c_size_t(dst.nbytes))
        assert rc == 0, rc
        bufs[name] = dst.astype(np.float32)

    def rep(name, got, want):
        d = np.abs(got - want)
        print(f"{name:6s} max|d| {d.max():.3e}  rel-to-max {d.max() / max(np.abs(want).max(), 1e-30):.3e}  "
              f"mean|d| {d.mean():.3e}  mean d {np.mean(got - want):+.3e} (rel {np.mean(got - want) / max(np.abs(want).mean(), 1e-30):+.2e})  |ref|max {np.abs(want).max():.3f}")

    a1 = planar_to_nhwc(bufs["A1h"], n, 4, 32)
    rep("A1 hi", a1, ref[0])
    if prec == 1:
        rep("A1 h+l", a1 + planar_to_nhwc(bufs["A1l"], n, 4, 32), ref[0])
    a2 = planar_to_nhwc(bufs["A2h"], n, 8, 16)
    rep("A2 hi", a2, ref[1])
    if prec == 1:
        rep("A2 h+l", a2 + planar_to_nhwc(bufs["A2l"], n, 8, 16), ref[1])
    rep("A3 hi", planar_to_nhwc(bufs["A3h"], n, 4, 8), ref[2])
    rep("A4", planar_to_nhwc(bufs["A4u"], n, 4, 8), ref[3])
    rep("A5", planar_to_nhwc(bufs["A5u"], n, 8, 16), ref[4])
    rep("A6", planar_to_nhwc(bufs["A6"], n, 4, 32), ref[5])
    f = feat[:n].cpu().numpy().reshape(n, 8, 8, 32)
    rep("feat", f, ref[2])
    rmse = np.mean(np.square(X - ref[6]), axis=(1, 2))
    rmae = np.mean(np.abs(X - ref[6]), axis=(1, 2))
    print("mse rel err", np.abs(mse[:n].cpu().numpy() / rmse - 1).max(), " mae rel err",
          np.abs(mae[:n].cpu().numpy() / rmae - 1).max())
    r = s.compute_anomaly_scores(list(g["crops"]))      # fp32 path
    s.engine.precision = prec
    r2 = s.compute_anomaly_scores(list(g["crops"]))
    for k in ("conservative", "moderate"):
        print(k, "max|d dec| vs golden:", np.abs(-r2[f"{k}_scores"] - g["dec_" + k[:3] if k[:3] == "con" else "dec_mod"]).max()
              if False else np.abs(r2[f"{k}_scores"] - r[f"{k}_scores"]).max(), "(vs fp32 path)")


if __name__ == "__main__":
    main()
