"""Batched segmentation (F equally sized fields per launch sequence) and the images-in, scores-out call
cia_screen_images.  The contract is bit-equality per field with the single-field calls, which tests/test_gpu_stardist.py
pins against the oracle: normalized pixels, prob / dist, labels and counts, cell records, scores and strain
accumulators."""
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
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "model_dir")


@pytest.fixture(scope="module")
def model():
    from cell_image_analysis_b200.stardist import StarDist2D
    from oracle import stardist as sd
    w = sd.random_model(CFG, seed=11)
    return StarDist2D.from_arrays(CFG, w, {"prob": 0.479071, "nms": 0.3})


@pytest.fixture(scope="module")
def screener(tmp_path_factory):
    """ProductionMutantScreening with the golden artifacts and a GPU StarDist model whose polygons pass the area gate"""
    from cell_image_analysis_b200.screening import ProductionMutantScreening
    from oracle import stardist as sd
    folder = tmp_path_factory.mktemp("sd") / "sd_demo"
    sd.write_model_folder(str(folder), CFG, sd.random_model(CFG, seed=11, dist_bias=14.0), prob_thresh=0.479071,
                          nms_thresh=0.3)
    s = ProductionMutantScreening(GOLDEN, segmenter=None, stardist_dir=str(folder))
    m = s.stardist_model
    green = _tiny_fields((3,))[0]
    prob, _ = m.predict(m.normalize_device(green))
    m.thresholds["prob"] = float(np.quantile(prob.cpu().numpy(), 0.7))     # an untrained network: a working threshold
    s.sd_folder = str(folder)
    return s


def _tiny_fields(seeds, H=None, W=None):
    from cell_image_analysis_b200 import synth
    h, w, n, lo, hi, lu = synth.FIELD_CONFIGS["tiny"]
    f = np.stack([synth.make_field(s, h, w, n, lo, hi, lu)[0] for s in seeds])
    return np.ascontiguousarray(f[:, :H or h, :W or w])


def _dev16(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int16)).cuda()


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


# ---- 1. normalisation ------------------------------------------------------------------------------------------
def test_normalize_fields_equal_single_field_and_reflect_pad(model):
    import torch
    eng = model.engine
    H, W = 70, 90                                   # pads to 80 x 96 (multiples of grid * 2^depth = 16)
    green = _tiny_fields((3,), H, W)[0]
    flat = np.full((H, W), 1234, np.uint16)
    widened = np.random.default_rng(21).integers(0, 256, (H, W)).astype(np.uint8).astype(np.uint16)
    fields = np.stack([green, flat, widened])
    Hp, Wp = 80, 96
    out = torch.full((3, Hp, Wp), float("nan"), dtype=torch.float32, device="cuda")
    eng._check(eng.lib.cia_seg_normalize_fields(eng.h, _ptr(_dev16(fields)), 3, H, W, 3.0, 99.8, _ptr(out), eng._stream()))
    got = out.cpu().numpy()
    for f in range(3):
        one = torch.empty((H, W), dtype=torch.float32, device="cuda")
        eng._check(eng.lib.cia_seg_normalize(eng.h, _ptr(_dev16(fields[f])), H, W, 3.0, 99.8, _ptr(one), None,
                                             eng._stream()))
        ref = np.pad(one.cpu().numpy(), ((0, Hp - H), (0, Wp - W)), mode="reflect")
        assert np.array_equal(got[f], ref), (f, np.nanmax(np.abs(got[f] - ref)))


# ---- 2. U-Net ----------------------------------------------------------------------------------------------------
def _predict_fields(model, x, F, Hp, Wp):
    import torch
    eng = model.engine
    g = model.grid
    prob = torch.empty((F, Hp // g, Wp // g), dtype=torch.float32, device="cuda")
    dist = torch.empty((F, Hp // g, Wp // g, 32), dtype=torch.float32, device="cuda")
    eng._check(eng.lib.cia_seg_predict_fields(eng.h, _ptr(x), F, Hp, Wp, _ptr(prob), _ptr(dist), eng._stream()))
    return prob, dist


def _predict_one(model, x, Hp, Wp):
    import torch
    eng = model.engine
    g = model.grid
    prob = torch.empty((Hp // g, Wp // g), dtype=torch.float32, device="cuda")
    dist = torch.empty((Hp // g, Wp // g, 32), dtype=torch.float32, device="cuda")
    eng._check(eng.lib.cia_seg_predict(eng.h, _ptr(x), Hp, Wp, _ptr(prob), _ptr(dist), eng._stream()))
    return prob, dist


# option settings that route every layer through each kernel form: TMA-fed (+ pooled output), software-producer,
# staged, consumer-side pooling
SETTINGS = {
    "default": {},
    "ws_everywhere": dict(seg_conv_tma=0, seg_conv_ws=2),
    "staged": dict(seg_conv_tma=0, seg_conv_ws=0),
    "no_pool_out": dict(seg_pool_out=0),
}
DEFAULTS = dict(seg_conv_tma=1, seg_conv_ws=1, seg_pool_out=1)


@pytest.mark.parametrize("setting", list(SETTINGS))
@pytest.mark.parametrize("H,W", [(16, 48), (32, 272), (144, 208)])
def test_predict_fields_bit_equal_per_field(model, setting, H, W):
    import torch
    eng = model.engine
    for k, v in SETTINGS[setting].items():
        eng.set_option(k, v)
    try:
        rng = np.random.default_rng(H * 7 + W)
        x = torch.from_numpy(rng.uniform(-0.2, 1.6, (5, H, W)).astype(np.float32)).cuda()
        singles = [_predict_one(model, x[f].contiguous(), H, W) for f in range(5)]
        for F in (1, 2, 5):
            prob, dist = _predict_fields(model, x[:F].contiguous(), F, H, W)
            for f in range(F):
                assert torch.equal(prob[f], singles[f][0]), (setting, F, f)
                assert torch.equal(dist[f], singles[f][1]), (setting, F, f)
    finally:
        for k, v in DEFAULTS.items():
            eng.set_option(k, v)


def test_predict_fields_two_full_size_fields(model):
    import torch
    rng = np.random.default_rng(2048)
    x = torch.from_numpy(rng.uniform(-0.2, 1.6, (2, 2048, 2048)).astype(np.float32)).cuda()
    prob, dist = _predict_fields(model, x, 2, 2048, 2048)
    for f in range(2):
        p1, d1 = _predict_one(model, x[f].contiguous(), 2048, 2048)
        assert torch.equal(prob[f], p1) and torch.equal(dist[f], d1), f


# ---- 3. instances ------------------------------------------------------------------------------------------------
def _instances_fields(model, prob, dist, H, W, pt, nt=0.3):
    import torch
    eng = model.engine
    F, Hgp, Wgp = prob.shape
    labels = torch.full((F, H, W), -7, dtype=torch.int32, device="cuda")
    n = torch.full((F,), -1, dtype=torch.int32, device="cuda")
    eng._check(eng.lib.cia_seg_instances_fields(eng.h, _ptr(prob), _ptr(dist), F, Hgp, Wgp, 2, H, W, float(pt), float(nt),
                                                _ptr(labels), _ptr(n), eng._stream()))
    return labels.cpu().numpy(), n.cpu().numpy()


def _instances_one(model, prob, dist, H, W, pt, nt=0.3):
    import torch
    labels, n = model.instances_from_prediction((H, W), torch.as_tensor(prob).contiguous(), torch.as_tensor(dist).contiguous(),
                                                pt, nt)
    return labels.cpu().numpy(), n


def _check_instances(model, prob, dist, H, W, pt):
    """maps [F][Hgp][Wgp] (padded): per field equal to the single-field call on the logical part"""
    import torch
    hg, wg = -(-H // 2), -(-W // 2)
    labels, n = _instances_fields(model, torch.from_numpy(prob).cuda(), torch.from_numpy(dist).cuda(), H, W, pt)
    for f in range(prob.shape[0]):
        ref, n1 = _instances_one(model, prob[f, :hg, :wg], dist[f, :hg, :wg], H, W, pt)
        assert n[f] == n1, (f, n[f], n1)
        assert np.array_equal(labels[f], ref), (f, int((labels[f] != ref).sum()))
    return labels, n


def _noise_maps(rng, Hg, Wg, lo=1.5, hi=6.0):
    return rng.uniform(0, 1, (Hg, Wg)).astype(np.float32), rng.uniform(lo, hi, (Hg, Wg, 32)).astype(np.float32)


def test_instances_fields_mixed_batch(model):
    """a field with no candidates, the huge-radius field of test_large_radii_keep_the_suppression_exact, noise, and
    star maps of real objects, in one call"""
    from cell_image_analysis_b200 import synth
    from oracle import stardist as sd
    H = W = 128
    rng = np.random.default_rng(33)
    p_big, d_big = _noise_maps(rng, 64, 64)
    d_big[20, 20] = 90.0
    p_big[20, 20] = 0.95
    p_none = np.zeros((64, 64), np.float32)
    d_none = np.full((64, 64, 32), 3.0, np.float32)
    p_noise, d_noise = _noise_maps(np.random.default_rng(7), 64, 64, 2, 9)
    cells = synth.ellipse_lattice(H, W, 3, 4)
    p_obj, d_obj = sd.star_maps_from_ellipses(H, W, 2, cells)
    prob = np.stack([p_big, p_none, p_noise, p_obj.astype(np.float32)])
    dist = np.stack([d_big, d_none, d_noise, d_obj.astype(np.float32)])
    _, n = _check_instances(model, prob, dist, H, W, 0.7)
    assert n[1] == 0 and n[0] > 0 and n[2] > 0 and n[3] > 0


@pytest.mark.parametrize("H,W", [(70, 90), (250, 250)])
def test_instances_fields_of_padded_maps(model, H, W):
    """candidates only inside each field's logical ceil(H/2) x ceil(W/2) part: the padding holds high probabilities"""
    Hp, Wp = H + (-H % 16), W + (-W % 16)
    rng = np.random.default_rng(H)
    prob = np.empty((3, Hp // 2, Wp // 2), np.float32)
    dist = np.empty((3, Hp // 2, Wp // 2, 32), np.float32)
    for f in range(3):
        prob[f], dist[f] = _noise_maps(rng, Hp // 2, Wp // 2, 2, 8)
        prob[f, -(-H // 2):, :] = 0.99
        prob[f, :, -(-W // 2):] = 0.99
    _check_instances(model, prob, dist, H, W, 0.8)


def test_instances_fields_do_not_cross_fields(model):
    """the same polygon at the same place in two fields is kept in both; a large candidate on field 0's last rows
    leaves field 1 (empty) untouched"""
    H = W = 96
    prob = np.zeros((3, 48, 48), np.float32)
    dist = np.full((3, 48, 48, 32), 4.0, np.float32)
    prob[0, 10, 20] = prob[1, 10, 20] = 0.9
    prob[0, 45, 24] = 0.95                    # last logical row the 2-pixel border allows; reaches 40 px past it
    dist[0, 45, 24] = 40.0
    labels, n = _check_instances(model, prob, dist, H, W, 0.5)
    assert n[0] == 2 and n[1] == 1 and n[2] == 0
    assert labels[2].max() == 0
    small = labels[0][20, 40]
    assert small > 0 and np.array_equal(labels[1] > 0, labels[0] == small)


# ---- 4-6. the fused call -----------------------------------------------------------------------------------------
def _chain_per_field(s, seg, img, max_label, cap, field_strain, n_strains):
    """normalize -> predict -> instances per field, then one cia_screen_fields on the stacked labels"""
    import torch
    eng, m = s.engine, s.stardist_model
    F, H, W = img.shape
    labels = torch.empty((F, H, W), dtype=torch.int32, device="cuda")
    n_inst = np.zeros(F, np.int64)
    for f in range(F):
        x = m.normalize_device(seg[f])
        prob, dist = m.predict(x)
        lab, n = m.instances_from_prediction((H, W), prob, dist)
        labels[f] = lab
        n_inst[f] = n
    out = eng.alloc_outputs(cap, F, keep_crops=True, keep_features=True)
    acc = torch.zeros((n_strains, 8), dtype=torch.float64, device="cuda")
    eng.screen_fields(_dev16(img), labels, max_label, out, field_strain=field_strain, acc=acc)
    eng.check_status()
    return out, acc, labels, n_inst


def _fused(s, seg, img, max_label, cap, field_strain, n_strains, keep_labels=True):
    import torch
    eng, m = s.engine, s.stardist_model
    F, H, W = img.shape
    out = eng.alloc_outputs(cap, F, keep_crops=True, keep_features=True)
    acc = torch.zeros((n_strains, 8), dtype=torch.float64, device="cuda")
    n = torch.full((F,), -1, dtype=torch.int32, device="cuda")
    labels = torch.full((F, H, W), -7, dtype=torch.int32, device="cuda") if keep_labels else None
    sd = _dev16(seg)
    eng.screen_images(sd, _dev16(img) if img is not seg else sd, max_label, out, m.thresholds["prob"], m.thresholds["nms"],
                      n_instances=n, labels_out=labels, field_strain=field_strain, acc=acc)
    return out, acc, labels, n


def _assert_acc(a1, a2):
    """strain accumulators: the counts exactly; the sums to rounding (cia_strain_accumulate adds with fp64 atomics,
    whose order varies from run to run even for one and the same call)"""
    import torch
    assert torch.equal(a1[:, :3], a2[:, :3])
    assert torch.allclose(a1, a2, rtol=1e-12, atol=0)


def _assert_same(o1, a1, o2, a2):
    import torch
    n = int(o1["counts"][0].item())
    assert torch.equal(o1["counts"], o2["counts"])
    assert n > 0
    assert torch.equal(o1["cells"][:n], o2["cells"][:n])
    for k in ("mse", "mae", "dec_cons", "dec_mod", "pred_cons", "pred_mod", "crops", "features"):
        assert torch.equal(o1[k][:n], o2[k][:n]), k
    _assert_acc(a1, a2)


@pytest.mark.parametrize("F", [1, 3, 16])
def test_screen_images_equals_the_chain(screener, F):
    import torch
    fields = _tiny_fields(range(3, 3 + F))
    strain = torch.tensor([f % 2 for f in range(F)], dtype=torch.int32, device="cuda")
    cap = 1024 * F
    o1, a1, l1, n1 = _chain_per_field(screener, fields, fields, 4096, cap, strain, 2)
    o2, a2, l2, n2 = _fused(screener, fields, fields, 4096, cap, strain, 2)
    screener.engine.check_status()
    _assert_same(o1, a1, o2, a2)
    assert torch.equal(l1, l2)
    assert np.array_equal(n1, n2.cpu().numpy())


def test_screen_images_three_channel_fields(screener):
    """segmentation on one channel, analysis on another (det:54-59)"""
    import torch
    seg = _tiny_fields((5, 6))
    img = _tiny_fields((8, 9))
    strain = torch.zeros(2, dtype=torch.int32, device="cuda")
    o1, a1, l1, _ = _chain_per_field(screener, seg, img, 4096, 2048, strain, 1)
    o2, a2, l2, _ = _fused(screener, seg, img, 4096, 2048, strain, 1)
    screener.engine.check_status()
    _assert_same(o1, a1, o2, a2)
    assert torch.equal(l1, l2)


def test_screen_images_two_full_size_fields(screener):
    import torch
    from cell_image_analysis_b200 import synth
    fields = np.stack([f for f, _ in synth.make_fields([1, 2], "config1")])
    strain = torch.tensor([0, 1], dtype=torch.int32, device="cuda")
    o1, a1, l1, n1 = _chain_per_field(screener, fields, fields, 65536, 65536, strain, 2)
    o2, a2, l2, n2 = _fused(screener, fields, fields, 65536, 65536, strain, 2)
    screener.engine.check_status()
    _assert_same(o1, a1, o2, a2)
    assert torch.equal(l1, l2) and np.array_equal(n1, n2.cpu().numpy())


def test_screen_images_launch_count_does_not_depend_on_F(screener):
    import torch
    eng = screener.engine
    counts = {}
    for F in (1, 16):
        fields = _tiny_fields(range(10, 10 + F))
        strain = torch.zeros(F, dtype=torch.int32, device="cuda")
        _fused(screener, fields, fields, 4096, 4096, strain, 1)   # warm-up: workspaces, first-use attributes
        eng.check_status()
        before = eng.launch_count
        _fused(screener, fields, fields, 4096, 4096, strain, 1, keep_labels=False)
        counts[F] = eng.launch_count - before
        eng.check_status()
    assert counts[1] == counts[16], counts


def test_screen_images_reports_too_many_instances(screener):
    import torch
    from cell_image_analysis_b200._lib import CIA_E_LABEL, CiaError
    fields = _tiny_fields((3, 4))
    strain = torch.zeros(2, dtype=torch.int32, device="cuda")
    _, _, _, n = _fused(screener, fields, fields, 4096, 2048, strain, 1)
    screener.engine.check_status()
    n = n.cpu().numpy()
    assert n.max() > 2
    _fused(screener, fields, fields, int(n.max()) - 1, 2048, strain, 1)
    with pytest.raises(CiaError) as e:
        screener.engine.check_status()
    assert e.value.code == CIA_E_LABEL


def test_segment_fields_equals_segment_device(screener):
    m = screener.stardist_model
    fields = _tiny_fields((3, 4, 5), 120, 200)                # reflect padding on the device
    labels, n = m.segment_fields(fields)
    for f in range(3):
        l1, n1 = m.segment_device(fields[f])
        assert np.array_equal(labels[f].cpu().numpy(), l1.cpu().numpy()) and int(n[f]) == n1, f


# ---- 7. BatchScreen images-only passes ---------------------------------------------------------------------------
def test_batch_screen_images_host_equals_device_and_the_chain(screener):
    """5 fields in chunks of 2 (a short last chunk): run_images_host == run_images_device == the per-field chain"""
    import torch
    from cell_image_analysis_b200.batch import BatchScreen
    eng, m = screener.engine, screener.stardist_model
    fields = _tiny_fields(range(20, 26))
    F = 5
    strain = torch.tensor([0, 1, 0, 1, 1], dtype=torch.int32, device="cuda")
    pt, nt = m.thresholds["prob"], m.thresholds["nms"]
    dev = _dev16(fields)                                     # pool of 6 (multiple of the chunk)
    bs_d = BatchScreen(eng, 256, 256, 4096, chunk_fields=2, n_strains=2, cells_per_field_cap=512)
    bs_d.run_images_device(dev, dev, F, pt, nt, strain_of_visit=strain)
    bs_d.sync()
    acc_d = bs_d.acc.clone()
    pinned = torch.from_numpy(fields.view(np.int16)).pin_memory()
    bs_h = BatchScreen(eng, 256, 256, 4096, chunk_fields=2, n_strains=2, cells_per_field_cap=512)
    bs_h.run_images_host(pinned, pinned, F, pt, nt, strain_of_visit=strain)
    r = bs_h.collect_host()
    _assert_acc(bs_h.acc, acc_d)
    # the per-field chain over the same 5 fields, one screen_fields call per chunk of 2 (the accumulation order)
    acc_c = torch.zeros((2, 8), dtype=torch.float64, device="cuda")
    cells, counts = [], []
    for c0 in range(0, F, 2):
        sl = slice(c0, min(F, c0 + 2))
        o, a, _, _ = _chain_per_field(screener, fields[sl], fields[sl], 4096, 1024, strain[sl], 2)
        acc_c += a
        n = int(o["counts"][0].item())
        rec = o["cells"][:n].cpu().numpy().view(np.dtype(r["cells"].dtype)).reshape(-1).copy()
        rec["field"] += c0
        cells.append(rec)
        counts.append(o["counts"][1:1 + sl.stop - sl.start].cpu().numpy())
        assert np.array_equal(r["mse"][sum(len(x) for x in cells[:-1]):][:n], o["mse"][:n].cpu().numpy())
    cells = np.concatenate(cells)
    assert r["n_cells"] == len(cells) > 0
    assert np.array_equal(r["cells"], cells)
    assert np.array_equal(r["field_counts"], np.concatenate(counts))
    assert bs_h.h2d_bytes == F * 256 * 256 * 2                 # only the images crossed PCIe
    # the chain sums each chunk into its own accumulator (the exact accumulator contract is
    # test_screen_images_equals_the_chain); here the totals must agree to rounding
    assert torch.allclose(acc_c, bs_h.acc, rtol=1e-12, atol=0)


# ---- 8. the sharded screen with a GPU StarDist model ---------------------------------------------------------------
def _npload(path):
    return np.load(path)


def _sample_folders(root):
    """three strains of two files each (arrays saved under *.tif names, read back by _npload); strain 'mutB' holds
    three-channel images: segmentation channel 2, analysis channel 1 (det:54-59).  Six files in chunks of four: a short
    last chunk."""
    fields = _tiny_fields(range(30, 37))
    folders = {}
    for s, name in enumerate(("wt", "mutA", "mutB")):
        d = os.path.join(str(root), name)
        os.makedirs(d, exist_ok=True)
        folders[name] = d
        for k in range(2):
            f = fields[2 * s + k]
            img = np.stack([np.zeros_like(f), fields[6 - k], f], -1) if name == "mutB" else f
            with open(os.path.join(d, f"field_{k}.tif"), "wb") as fh:
                np.save(fh, img)
    return folders


def _compare_sharded(res1, det1, res2, det2):
    assert list(res1) == list(res2) and len(res1) == 3
    for name in res1:
        a, b = res1[name], res2[name]
        for k in ("sample_name", "total_cells", "files_processed", "conservative_anomaly_rate", "moderate_anomaly_rate"):
            assert a[k] == b[k], (name, k)
        mse = np.array([r["mse"] for r in det1 if r["sample_name"] == name], np.float64)
        assert abs(b["mean_mse"] - np.mean(mse)) <= 1e-12 and abs(b["std_mse"] - np.std(mse)) <= 1e-9
    assert len(det1) == len(det2) > 0
    for r1, r2 in zip(det1, det2):
        assert r1 == r2, (r1, r2)


def test_sharded_screen_with_a_gpu_model_equals_the_per_file_loop(screener, tmp_path):
    """screen_mutant_samples_sharded with stardist_dir= (world size 1): the loaders only read files, each chunk is
    segmented and screened in cia_screen_images; results and rows equal the reference-shaped per-file loop"""
    folders = _sample_folders(tmp_path)
    old = screener.imread
    screener.imread = _npload
    try:
        res1, det1 = screener.screen_mutant_samples(folders)
        res2, det2 = screener.screen_mutant_samples_sharded(folders, chunk_fields=4)
    finally:
        screener.imread = old
    _compare_sharded(res1, det1, res2, det2)


def _sharded_worker(rank, world, port, sd_folder, prob_thresh, root, q):
    import torch
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from cell_image_analysis_b200.screening import ProductionMutantScreening
    s = ProductionMutantScreening(GOLDEN, imread=_npload, device=rank, precision=1, stardist_dir=sd_folder)
    s.stardist_model.thresholds["prob"] = prob_thresh
    q.put((rank,) + s.screen_mutant_samples_sharded(_sample_folders(root), chunk_fields=4))
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_screen_with_a_gpu_model_two_gpus(screener, tmp_path):
    import socket
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    folders = _sample_folders(tmp_path)
    old = screener.imread
    screener.imread = _npload
    try:
        res1, det1 = screener.screen_mutant_samples(folders)
    finally:
        screener.imread = old
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    args = (screener.sd_folder, screener.stardist_model.thresholds["prob"], str(tmp_path), q)
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, port) + args) for r in range(2)]
    for p in procs:
        p.start()
    got = sorted([q.get(timeout=600) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    _compare_sharded(res1, det1, got[0][1], got[0][2])
    assert got[1][1] == {} and got[1][2] == []
