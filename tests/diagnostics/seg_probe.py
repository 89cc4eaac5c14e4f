"""Diagnostics and timings of the segmentation step on a B200 (prints, asserts nothing):
per-layer error against a float32 convolution, network error against the oracle, NMS / rendering
mismatches, and CUDA-event timings of normalize / U-Net / instances on a 2048 x 2048 field."""
import os
import sys
import time
import traceback

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import stardist as sd                      # noqa: E402
import test_gpu_stardist as T                          # noqa: E402
from cell_image_analysis_b200.stardist import StarDist2D   # noqa: E402
from cell_image_analysis_b200 import synth             # noqa: E402


def section(name, fn):
    print(f"--- {name}", flush=True)
    try:
        fn()
    except Exception:
        traceback.print_exc()
    sys.stdout.flush()


def ev_time(fn, reps=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    w = sd.random_model(T.CFG, seed=11)
    m = StarDist2D.from_arrays(T.CFG, w, {"prob": 0.479071, "nms": 0.3})
    m.oracle_weights = w
    eng = m.engine
    for opt in ("seg_conv_tma", "seg_conv_ws"):      # A/B runs: SEG_CONV_TMA=0 etc.
        if os.environ.get(opt.upper()):
            eng.set_option(opt, float(os.environ[opt.upper()]))

    def layers():
        for layer in range(len(m.layer_order) - 2):
            print(f"layer {layer:2d} {m.layer_order[layer]:20s} rel err {T.layer_check(m, layer, 48, 40):.3e}", flush=True)
    section("layers vs float32 conv of the same fp16 operands", layers)

    def network():
        rng = np.random.default_rng(0)
        x = rng.uniform(0, 1.5, (128, 160)).astype(np.float32)
        prob, dist = m.predict(x)
        prob, dist = prob.cpu().numpy(), dist.cpu().numpy()
        p32, d32 = sd.unet_forward(T.CFG, w, x)
        p16, d16 = sd.unet_forward(T.CFG, w, x, half_activations=True)
        print("prob range", prob.min(), prob.max(), "dist range", dist.min(), dist.max())
        print("vs f32 : prob", np.abs(prob - p32).max(), "dist rel", np.abs(dist - d32).max() / np.abs(d32).max())
        print("vs f16 : prob", np.abs(prob - p16).max(), "dist rel", np.abs(dist - d16).max() / np.abs(d16).max())
    section("network vs oracle", network)

    def norm():
        H, W, n, lo, hi, lu = synth.FIELD_CONFIGS["tiny"]
        green, _ = synth.make_field(3, H, W, n, lo, hi, lu)
        got = m.normalize_device(green).cpu().numpy()
        ref = sd.normalize(green)
        print("normalize equal:", np.array_equal(got, ref), np.abs(got - ref).max())
    section("normalize", norm)

    def inst():
        for (H, W, n_side, seed) in [(256, 320, 4, 0), (512, 512, 7, 1)]:
            cells = T._ellipse_field(H, W, n_side, seed)
            prob, dist = sd.star_maps_from_ellipses(H, W, 2, cells)
            rng = np.random.default_rng(seed)
            prob = (prob * rng.uniform(0.9, 1.0, prob.shape)).astype(np.float32)
            dist = (dist * rng.uniform(0.97, 1.03, dist.shape)).astype(np.float32)
            ref, det = sd.instances_from_prediction(prob, dist, 2, (H, W), 0.4, 0.3)
            labels, n = m.instances_from_prediction((H, W), torch.from_numpy(prob), torch.from_numpy(dist), 0.4, 0.3)
            got = labels.cpu().numpy()
            print(H, W, "n gpu", n, "n ref", len(det["prob"]), "label mismatches", int((got != ref).sum()), flush=True)
    section("instances vs oracle", inst)

    def timing():
        H = W = 2048
        green, _ = synth.make_field(0, H, W, *synth.FIELD_CONFIGS["config1"][2:])
        g = torch.from_numpy(green.view(np.int16)).cuda()
        out = torch.empty((H, W), dtype=torch.float32, device="cuda")
        import ctypes as C
        t_norm = ev_time(lambda: eng._check(eng.lib.cia_seg_normalize(eng.h, g.data_ptr(), H, W, 3.0, 99.8, out.data_ptr(),
                                                                     None, eng._stream())))
        t_net = ev_time(lambda: eng._check(eng.lib.cia_seg_predict(eng.h, out.data_ptr(), H, W, None, None, eng._stream())))
        cells = T._ellipse_field(H, W, 23, 3)
        prob, dist = sd.star_maps_from_ellipses(H, W, 2, cells)
        pd, dd = torch.from_numpy(prob).cuda(), torch.from_numpy(dist).cuda()
        labels = torch.empty((H, W), dtype=torch.int32, device="cuda")
        nn = torch.zeros(1, dtype=torch.int32, device="cuda")
        t_inst = ev_time(lambda: eng._check(eng.lib.cia_seg_instances(eng.h, pd.data_ptr(), dd.data_ptr(), H // 2, W // 2, 2, H, W,
                                                                     0.479071, 0.3, labels.data_ptr(), nn.data_ptr(), eng._stream())))
        flops = sum(2.0 * k * k * ci * co * (H >> s) * (W >> s) for (name, ci, co, k), s in
                    zip(sd.layer_plan(T.CFG), [0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 3, 3, 2, 2, 1, 1, 1, 1, 1]))
        print(f"2048x2048: normalize {t_norm:.3f} ms, U-Net {t_net:.3f} ms ({flops / t_net / 1e9:.1f} TFLOP/s of {flops / 1e9:.1f} GFLOP), "
              f"instances {t_inst:.3f} ms ({int(nn.item())} instances, {int((prob > 0.479071).sum())} candidates)")
        t0 = time.time()
        ref, det = sd.instances_from_prediction(prob, dist, 2, (H, W), 0.479071, 0.3)
        print(f"oracle post-processing {1e3 * (time.time() - t0):.0f} ms; labels equal: {np.array_equal(labels.cpu().numpy(), ref)}")
    section("timing", timing)


if __name__ == "__main__":
    main()
