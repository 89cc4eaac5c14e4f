"""GPU parity of the segmentation step (SURVEY 8f row N2; improved_detection.py:44, 62-63) against
oracle/stardist.py + oracle/stardist_post.c ("parity unpinned": restated third-party algorithms).

Gates: percentiles and normalized pixels bit-exact (integer order statistics, IEEE float32 ops); every
convolution layer within fp16 rounding of a float32 convolution of the same fp16 operands; prob / dist of the
whole network within 2e-2 of the float32 oracle and 1e-2 of its fp16-activation twin; NMS survivors and the
rendered labels bit-exact against the oracle on the same (prob, dist)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
pytestmark = pytest.mark.gpu

CFG = dict(n_channel_in=1, grid=[2, 2], n_rays=32, unet_n_depth=3, unet_n_filter_base=32,
           unet_n_conv_per_depth=2, net_conv_after_unet=128, unet_kernel_size=[3, 3], unet_pool=[2, 2],
           unet_activation="relu", unet_last_activation="relu", unet_batch_norm=False)


@pytest.fixture(scope="module")
def model():
    from cell_image_analysis_b200.stardist import StarDist2D
    from oracle import stardist as sd
    w = sd.random_model(CFG, seed=11)
    m = StarDist2D.from_arrays(CFG, w, {"prob": 0.479071, "nms": 0.3})
    m.oracle_weights = w
    return m


def planar(x):
    """NCHW-less [C, H, W] float tensor -> fp16 chunk-planar [C/8][H][W][8]"""
    Cc, H, W = x.shape
    return x.half().view(Cc // 8, 8, H, W).permute(0, 2, 3, 1).contiguous()


def unplanar(p):
    P, H, W, _ = p.shape
    return p.permute(0, 3, 1, 2).reshape(P * 8, H, W).float()


def layer_check(m, layer, Ho, Wo, seed=0):
    """max |gpu - ref| / max |ref| of one plan layer on random fp16 activations"""
    import torch
    import torch.nn.functional as F
    eng = m.engine
    info = (C.c_int32 * 6)()
    eng._check(eng.lib.cia_seg_layer_info(eng.h, layer, info))
    mode, c0, c1, cout, _shift, _n = list(info)
    g = torch.Generator(device="cpu").manual_seed(seed + layer)
    name = m.layer_order[layer]
    k, b = m.oracle_weights[name]
    kt = torch.from_numpy(np.ascontiguousarray(k.transpose(3, 2, 0, 1))).cuda()
    bt = torch.from_numpy(b).cuda()
    out = torch.zeros((cout // 8, Ho, Wo, 8), dtype=torch.float16, device="cuda")
    if mode == -1:
        img = torch.rand((Ho, Wo), generator=g).cuda()
        ref = F.relu(F.conv2d(img[None, None], kt, bt, padding=1))[0]
        eng._check(eng.lib.cia_seg_debug_layer(eng.h, layer, None, None, img.data_ptr(), Ho, Wo, out.data_ptr(), None,
                                               None, eng._stream()))
    else:
        if mode == 0:
            x0 = torch.randn((c0, Ho, Wo), generator=g).cuda().half().float()
            xin, s0, s1 = x0, planar(x0), None
        elif mode == 1:
            x0 = torch.randn((c0, 2 * Ho, 2 * Wo), generator=g).cuda().half().float()
            xin, s0, s1 = F.max_pool2d(x0[None], 2)[0], planar(x0), None
        else:
            x0 = torch.randn((c0, Ho // 2, Wo // 2), generator=g).cuda().half().float()
            x1 = torch.randn((c1, Ho, Wo), generator=g).cuda().half().float()
            xin = torch.cat([F.interpolate(x0[None], scale_factor=2, mode="nearest")[0], x1], 0)
            s0, s1 = planar(x0), planar(x1)
        ref = F.relu(F.conv2d(xin[None].double(), kt.half().double(), bt.double(), padding=1))[0].float()
        eng._check(eng.lib.cia_seg_debug_layer(eng.h, layer, s0.data_ptr(), s1.data_ptr() if s1 is not None else None,
                                               None, Ho, Wo, out.data_ptr(), None, None, eng._stream()))
    torch.cuda.synchronize()
    got = unplanar(out)
    return float((got - ref).abs().max() / ref.abs().max())


def test_normalize_bit_exact(model):
    from cell_image_analysis_b200 import synth
    from oracle import stardist as sd
    H, W, n, lo, hi, lu = synth.FIELD_CONFIGS["tiny"]
    for seed in (3, 4):
        green, _ = synth.make_field(seed, H, W, n, lo, hi, lu)
        got = model.normalize_device(green).cpu().numpy()
        ref = sd.normalize(green)
        assert np.array_equal(got, ref), np.abs(got - ref).max()
    rng = np.random.default_rng(5)     # a flat histogram and an odd size: the interpolation weights matter
    x = rng.integers(0, 65536, size=(301, 257)).astype(np.uint16)
    assert np.array_equal(model.normalize_device(x, 1, 99.8).cpu().numpy(), sd.normalize(x, 1, 99.8))


@pytest.mark.parametrize("tma,ws", [(1, 1), (0, 2), (0, 0)])
def test_every_layer_against_float32_conv(model, tma, ws):
    """(1, 1), the default: layers that read their producer directly with Cin = 32 run the TMA-fed kernel, the
    warp-specialised software-producer kernel takes the layers where it measured faster; (0, 2): every layer through
    the latter; (0, 0): the staged kernel everywhere."""
    n_layers = len(model.layer_order) - 2
    model.engine.set_option("seg_conv_tma", tma)
    model.engine.set_option("seg_conv_ws", ws)
    try:
        for layer in range(n_layers):
            # 48 x 40: edge tiles in both directions (tiles are 16 rows x 16 / 32 columns); 80 x 112: several units per CTA
            for Ho, Wo in ((48, 40), (80, 112)):
                err = layer_check(model, layer, Ho, Wo)
                print(f"tma {tma} ws {ws} layer {layer} {model.layer_order[layer]} {Ho}x{Wo}: max rel err {err:.2e}")
                assert err < 2e-3, (layer, model.layer_order[layer], err)
    finally:
        model.engine.set_option("seg_conv_tma", 1)
        model.engine.set_option("seg_conv_ws", 1)


def test_network_against_oracle(model):
    from cell_image_analysis_b200 import synth
    from oracle import stardist as sd
    H, W, n, lo, hi, lu = synth.FIELD_CONFIGS["tiny"]
    green, _ = synth.make_field(3, H, W, n, lo, hi, lu)
    x = sd.normalize(green)
    Hc, Wc = (H // 16) * 16, (W // 16) * 16
    x = np.ascontiguousarray(x[:Hc, :Wc])
    prob, dist = model.predict(x)
    prob, dist = prob.cpu().numpy(), dist.cpu().numpy()
    p32, d32 = sd.unet_forward(CFG, model.oracle_weights, x)
    p16, d16 = sd.unet_forward(CFG, model.oracle_weights, x, half_activations=True)
    e32 = (np.abs(prob - p32).max(), np.abs(dist - d32).max() / np.abs(d32).max())
    e16 = (np.abs(prob - p16).max(), np.abs(dist - d16).max() / np.abs(d16).max())
    print(f"prob/dist vs float32 oracle {e32[0]:.2e} {e32[1]:.2e}; vs fp16-activation twin {e16[0]:.2e} {e16[1]:.2e}")
    assert e32[0] < 2e-2 and e32[1] < 2e-2, e32
    assert e16[0] < 1e-2 and e16[1] < 1e-2, e16


def _ellipse_field(H, W, n_side, seed):
    from cell_image_analysis_b200 import synth
    return synth.ellipse_lattice(H, W, n_side, seed)


@pytest.mark.parametrize("H,W,n_side,seed", [(256, 320, 4, 0), (512, 512, 7, 1), (1024, 1024, 20, 2)])
def test_instances_bit_exact(model, H, W, n_side, seed):
    import torch
    from oracle import stardist as sd
    cells = _ellipse_field(H, W, n_side, seed)
    prob, dist = sd.star_maps_from_ellipses(H, W, 2, cells)
    rng = np.random.default_rng(seed)
    prob = (prob * rng.uniform(0.9, 1.0, prob.shape)).astype(np.float32)       # break ties between pixels
    dist = (dist * rng.uniform(0.97, 1.03, dist.shape)).astype(np.float32)     # ragged, overlapping polygons
    ref, det = sd.instances_from_prediction(prob, dist, 2, (H, W), 0.4, 0.3)
    labels, n = model.instances_from_prediction((H, W), torch.from_numpy(prob), torch.from_numpy(dist), 0.4, 0.3)
    got = labels.cpu().numpy()
    d = model.details(n)
    assert n == len(det["prob"]) > 0, (n, len(det["prob"]))
    assert np.array_equal(d["points"], det["points"])
    assert np.array_equal(d["prob"], det["prob"])
    assert np.array_equal(d["coord"], det["coord"])
    assert np.array_equal(got, ref), int((got != ref).sum())
    assert n >= 0.9 * len(cells)


def test_instances_of_noise(model):
    """dense random candidates (what an untrained network emits): thousands of overlapping polygons"""
    import torch
    from oracle import stardist as sd
    rng = np.random.default_rng(7)
    H = W = 256
    prob = rng.uniform(0, 1, (H // 2, W // 2)).astype(np.float32)
    dist = rng.uniform(2, 9, (H // 2, W // 2, 32)).astype(np.float32)
    ref, det = sd.instances_from_prediction(prob, dist, 2, (H, W), 0.6, 0.3)
    labels, n = model.instances_from_prediction((H, W), torch.from_numpy(prob), torch.from_numpy(dist), 0.6, 0.3)
    assert n == len(det["prob"])
    assert np.array_equal(labels.cpu().numpy(), ref)
    # nothing above the threshold: an empty label image
    labels, n = model.instances_from_prediction((H, W), torch.from_numpy(prob), torch.from_numpy(dist), 2.0, 0.3)
    assert n == 0 and int(labels.max().item()) == 0


def test_predict_instances_drop_in(model):
    """the reference's two calls end to end, labels on the device feeding the region scan"""
    from cell_image_analysis_b200 import synth
    from oracle import stardist as sd
    H, W, n, lo, hi, lu = synth.FIELD_CONFIGS["tiny"]
    green, _ = synth.make_field(3, H, W, n, lo, hi, lu)
    Hc, Wc = (H // 16) * 16, (W // 16) * 16
    green = np.ascontiguousarray(green[:Hc, :Wc])
    x = model.normalize_device(green)
    labels, details = model.predict_instances(x.cpu().numpy())
    assert labels.dtype == np.int32 and labels.shape == green.shape
    assert set(details) >= {"points", "prob", "coord"}
    # same (prob, dist) through the oracle's post-processing
    prob, dist = model.predict(x)
    ref, _ = sd.instances_from_prediction(prob.cpu().numpy(), dist.cpu().numpy(), 2, green.shape, 0.479071, 0.3)
    assert np.array_equal(labels, ref)
    dev_labels, n_inst = model.segment_device(green)
    assert np.array_equal(dev_labels.cpu().numpy(), labels) and n_inst == labels.max()


def test_reflect_padding_of_odd_sizes(model):
    from oracle import stardist as sd
    rng = np.random.default_rng(9)
    x = rng.uniform(0, 1, (70, 90)).astype(np.float32)
    prob, dist = model.predict(x)
    xp = np.pad(x, ((0, 10), (0, 6)), mode="reflect")
    p16, d16 = sd.unet_forward(CFG, model.oracle_weights, xp, half_activations=True)
    assert prob.shape == (35, 45)
    assert np.abs(prob.cpu().numpy() - p16[:35, :45]).max() < 1e-2


def test_screening_with_a_model_folder(tmp_path):
    """ProductionMutantScreening(model_dir, stardist_dir=...): imread -> segmentation on the device -> region scan,
    equal to handing the same labels over as a NumPy array (det:51-111)."""
    from cell_image_analysis_b200 import synth
    from cell_image_analysis_b200.screening import ProductionMutantScreening
    from oracle import stardist as sd
    w = sd.random_model(CFG, seed=11, dist_bias=14.0)          # polygons large enough for the area gate (>= 200 px)
    folder = tmp_path / "sd_demo"
    sd.write_model_folder(str(folder), CFG, w, prob_thresh=0.479071, nms_thresh=0.3)
    H, W, n, lo, hi, lu = synth.FIELD_CONFIGS["tiny"]
    green, _ = synth.make_field(3, H, W, n, lo, hi, lu)
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "model_dir")
    s = ProductionMutantScreening(golden, imread=lambda p: green, stardist_dir=str(folder))
    m = s.stardist_model
    assert m.layer_order == [p[0] for p in sd.layer_plan(CFG)] and m.thresholds["nms"] == 0.3
    prob, _ = m.predict(m.normalize_device(green))
    m.thresholds["prob"] = float(np.quantile(prob.cpu().numpy(), 0.7))     # an untrained network: pick a working threshold
    cells, stats = s.extract_quality_cells("field_000.tif")
    labels, _ = m.predict_instances(sd.normalize(green))
    assert labels.max() > 0
    cells2, stats2 = s.extract_quality_cells_from_labels(green, labels)
    assert len(cells) == len(cells2) and stats == stats2
    assert all(np.array_equal(a, b) for a, b in zip(cells, cells2))
    print(f"{labels.max()} instances, {len(cells)} quality cells")


def test_training_twin_with_the_gpu_model(tmp_path):
    """ImprovedAnomalyDetectionTraining.extract_quality_cells(image_path, stardist_model) (train:39-111) with the
    GPU StarDist2D as ``stardist_model``: same cells as the NumPy-label route, 'file' and 'solidity' present."""
    from cell_image_analysis_b200 import synth
    from cell_image_analysis_b200.stardist import StarDist2D
    from cell_image_analysis_b200.training import ImprovedAnomalyDetectionTraining
    from oracle import stardist as sd
    H, W, n, lo, hi, lu = synth.FIELD_CONFIGS["tiny"]
    green, _ = synth.make_field(4, H, W, n, lo, hi, lu)
    t = ImprovedAnomalyDetectionTraining(str(tmp_path), imread=lambda p: green)
    m = StarDist2D.from_arrays(CFG, sd.random_model(CFG, seed=11, dist_bias=14.0), {"prob": 0.5, "nms": 0.3},
                               engine=t.engine)
    prob, _ = m.predict(m.normalize_device(green))
    m.thresholds["prob"] = float(np.quantile(prob.cpu().numpy(), 0.7))
    cells, stats = t.extract_quality_cells("a/b/field_7.tif", m)
    labels, _ = m.predict_instances(sd.normalize(green))
    cells2, stats2 = t._x.extract_quality_cells_from_labels(green, labels)
    assert len(cells) == len(cells2) > 0
    assert all(np.array_equal(a, b) for a, b in zip(cells, cells2))
    assert all(s["file"] == "field_7.tif" and "solidity" in s for s in stats)


def test_round_trip_through_the_screen(model):
    """true labels -> star maps -> GPU instances -> region scan, gates, crops, scores: the objects come back (labels
    bit-equal to the oracle's instances, IoU > 0.9 with the truth) and the screen keeps the same cells as it does on
    the true labels."""
    import torch
    from cell_image_analysis_b200 import synth
    from cell_image_analysis_b200.screening import ProductionMutantScreening
    from oracle import stardist as sd
    H, W, n, lo, hi, lu = synth.FIELD_CONFIGS["tiny"]
    green, truth = synth.make_field(3, H, W, n, lo, hi, lu)
    prob, dist = synth.star_maps_from_labels(truth, 2)
    labels, n_inst = model.instances_from_prediction((H, W), torch.from_numpy(prob), torch.from_numpy(dist), 0.479071, 0.3)
    ref, _ = sd.instances_from_prediction(prob, dist, 2, (H, W), 0.479071, 0.3)
    got = labels.cpu().numpy()
    assert np.array_equal(got, ref) and n_inst == len(np.unique(truth)) - 1
    for i in np.unique(truth)[1:]:
        m = truth == i
        k = np.bincount(got[m]).argmax()
        assert k > 0 and (m & (got == k)).sum() / (m | (got == k)).sum() > 0.9
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "model_dir")
    s = ProductionMutantScreening(golden, segmenter=lambda ch: None)
    cells_t, stats_t = s.extract_quality_cells_from_labels(green, truth)
    cells_g, stats_g = s.extract_quality_cells_from_labels(green, labels.to(s.engine.tdev))     # device-resident labels
    assert len(cells_g) == len(cells_t) > 0
    a_t = sorted(st["area"] for st in stats_t); a_g = sorted(st["area"] for st in stats_g)
    assert np.allclose(a_t, a_g, rtol=0.12)          # polygons of 32 rays against the true ellipses



@pytest.mark.parametrize("H,W", [(16, 16), (16, 48), (64, 16), (32, 272)])
def test_small_and_oblong_fields(model, H, W):
    """fields smaller than one tile of a level (the coarsest maps are 1 x 1 ... 2 x 17 pixels; TMA boxes larger than the
    tensor) and strongly oblong ones, against the fp16-activation twin of the oracle; instances on their maps bit-equal"""
    from oracle import stardist as sd
    rng = np.random.default_rng(H * 1000 + W)
    x = rng.uniform(-0.2, 1.5, (H, W)).astype(np.float32)
    prob, dist = model.predict(x)
    p16, d16 = sd.unet_forward(CFG, model.oracle_weights, x, half_activations=True)
    assert prob.shape == p16.shape and dist.shape == d16.shape
    assert np.abs(prob.cpu().numpy() - p16).max() < 1e-2
    assert np.abs(dist.cpu().numpy() - d16).max() < 1e-2 * np.abs(d16).max()
    thr = float(np.quantile(p16, 0.6))
    labels, n = model.instances_from_prediction((H, W), prob, dist, thr, 0.3)
    ref, det = sd.instances_from_prediction(prob.cpu().numpy(), dist.cpu().numpy(), 2, (H, W), thr, 0.3)
    assert n == len(det["prob"]) and np.array_equal(labels.cpu().numpy(), ref)


def test_normalize_uint8_and_constant_fields(model):
    from oracle import stardist as sd
    rng = np.random.default_rng(21)
    x8 = rng.integers(0, 256, (96, 80)).astype(np.uint8)
    assert np.array_equal(model.normalize_device(x8).cpu().numpy(), sd.normalize(x8))
    flat = np.full((64, 64), 1234, np.uint16)                # ma == mi: division by eps, as csbdeep does
    got, ref = model.normalize_device(flat).cpu().numpy(), sd.normalize(flat)
    assert np.array_equal(got, ref)
    with pytest.raises(TypeError):
        model.normalize_device(rng.uniform(0, 1, (32, 32)).astype(np.float32))


def test_large_radii_keep_the_suppression_exact(model):
    """one candidate with a huge radius makes every candidate a neighbour of every other (reach = r + r_max): slow path,
    same result"""
    import torch
    from oracle import stardist as sd
    rng = np.random.default_rng(33)
    H = W = 128
    prob = rng.uniform(0, 1, (H // 2, W // 2)).astype(np.float32)
    dist = rng.uniform(1.5, 6, (H // 2, W // 2, 32)).astype(np.float32)
    dist[20, 20] = 90.0
    prob[20, 20] = 0.95
    ref, det = sd.instances_from_prediction(prob, dist, 2, (H, W), 0.7, 0.3)
    labels, n = model.instances_from_prediction((H, W), torch.from_numpy(prob), torch.from_numpy(dist), 0.7, 0.3)
    assert n == len(det["prob"]) and np.array_equal(labels.cpu().numpy(), ref)


def test_screen_images_equals_the_per_field_calls(tmp_path):
    """ProductionMutantScreening.screen_images (segmentation + screen, stream-ordered, labels on the device) against
    extract_quality_cells + compute_anomaly_scores field by field"""
    from cell_image_analysis_b200 import synth
    from cell_image_analysis_b200.screening import ProductionMutantScreening
    from oracle import stardist as sd
    w = sd.random_model(CFG, seed=11, dist_bias=14.0)
    folder = tmp_path / "sd_demo"
    sd.write_model_folder(str(folder), CFG, w, prob_thresh=0.479071, nms_thresh=0.3)
    H, W, n, lo, hi, lu = synth.FIELD_CONFIGS["tiny"]
    fields = np.stack([synth.make_field(s_, H, W, n, lo, hi, lu)[0] for s_ in (3, 4, 5)])
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "model_dir")
    current = {}
    s = ProductionMutantScreening(golden, imread=lambda p: current["img"], stardist_dir=str(folder))
    m = s.stardist_model
    prob, _ = m.predict(m.normalize_device(fields[0]))
    m.thresholds["prob"] = float(np.quantile(prob.cpu().numpy(), 0.7))
    res = s.screen_images(fields)
    assert len(res["n_instances"]) == 3 and res["n_instances"].min() > 0
    k = 0
    for f in range(3):
        current["img"] = fields[f]
        cells, stats = s.extract_quality_cells(f"field_{f}.tif")
        sel = res["field"] == f
        assert sel.sum() == len(cells)
        if len(cells):
            r = s.compute_anomaly_scores(cells)
            assert np.allclose(res["reconstruction_mse"][sel], r["reconstruction_mse"], rtol=1e-5)
            assert np.array_equal(res["conservative_predictions"][sel], r["conservative_predictions"])
            assert np.abs(res["moderate_scores"][sel] - r["moderate_scores"]).max() < 1e-6
        k += len(cells)
    assert k == len(res["field"]) > 0


def test_pooled_outputs_are_bit_identical(model):
    """seg_pool_out (default): TMA-fed layers write the max-pooled copy the next layer reads (the full-resolution map of
    the second layer then never exists in HBM); the maps equal those of consumer-side pooling bit for bit"""
    rng = np.random.default_rng(14)
    x = rng.uniform(-0.2, 1.6, (176, 240)).astype(np.float32)
    eng = model.engine
    p1, d1 = model.predict(x)
    eng.set_option("seg_pool_out", 0)
    try:
        p0, d0 = model.predict(x)
    finally:
        eng.set_option("seg_pool_out", 1)
    assert np.array_equal(p0.cpu().numpy(), p1.cpu().numpy()) and np.array_equal(d0.cpu().numpy(), d1.cpu().numpy())


@pytest.mark.parametrize("cfg_kw", [
    dict(grid=[1, 1], unet_n_depth=2, unet_n_filter_base=32, unet_n_conv_per_depth=2, net_conv_after_unet=64),
    dict(grid=[4, 4], unet_n_depth=1, unet_n_filter_base=32, unet_n_conv_per_depth=1, net_conv_after_unet=32),
    dict(grid=[2, 2], unet_n_depth=2, unet_n_filter_base=64, unet_n_conv_per_depth=3, net_conv_after_unet=128),
])
def test_other_stardist_configurations(cfg_kw):
    """the plan builder follows StarDist2D._build / unet_block for other grids, depths, filter counts and convolutions per
    level (first layer inside the U-Net for grid 1, a single convolution per level, three per level, 64-channel heads)"""
    from cell_image_analysis_b200.stardist import StarDist2D, layer_plan
    from oracle import stardist as sd
    cfg = dict(CFG, **cfg_kw)
    w = sd.random_model(cfg, seed=5)
    assert layer_plan(cfg) == sd.layer_plan(cfg)
    m = StarDist2D.from_arrays(cfg, w, {"prob": 0.5, "nms": 0.3})
    assert m.layer_order == [p[0] for p in sd.layer_plan(cfg)]
    g = int(cfg["grid"][0])
    rng = np.random.default_rng(3)
    x = rng.uniform(-0.2, 1.5, (64, 96)).astype(np.float32)
    prob, dist = m.predict(x)
    p16, d16 = sd.unet_forward(cfg, w, x, half_activations=True)
    assert prob.shape == (64 // g, 96 // g) == p16.shape
    assert np.abs(prob.cpu().numpy() - p16).max() < 1e-2
    assert np.abs(dist.cpu().numpy() - d16).max() < 1e-2 * np.abs(d16).max()
    thr = float(np.quantile(p16, 0.6))
    labels, n = m.instances_from_prediction((64, 96), prob, dist, thr, 0.3)
    ref, det = sd.instances_from_prediction(prob.cpu().numpy(), dist.cpu().numpy(), g, (64, 96), thr, 0.3)
    assert n == len(det["prob"]) and np.array_equal(labels.cpu().numpy(), ref)
