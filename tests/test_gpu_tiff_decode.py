"""Device decode of compressed TIFF fields (cia_tiff_decode_fields, tiff_device.py): bit-equal to read_tiff in every
combination of compression, predictor, strips / tiles, chunky / planar, 1 / 3 samples, 8 / 16 bit and byte order,
with field sides that are not multiples of the strip or tile size; a corrupted segment flags only its own field; the
sharded screen over compressed files equals the same screen over the uncompressed files."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

import tiff_fixtures  # noqa: E402
from test_gpu_screen_images import CFG, GOLDEN, _tiny_fields  # noqa: E402


@pytest.fixture(scope="module")
def screener(tmp_path_factory):
    from cell_image_analysis_b200.screening import ProductionMutantScreening
    from oracle import stardist as sd
    folder = tmp_path_factory.mktemp("sd") / "sd_demo"
    sd.write_model_folder(str(folder), CFG, sd.random_model(CFG, seed=11, dist_bias=14.0), prob_thresh=0.479071,
                          nms_thresh=0.3)
    s = ProductionMutantScreening(GOLDEN, segmenter=None, stardist_dir=str(folder))
    m = s.stardist_model
    green = _tiny_fields((3,))[0]
    prob, _ = m.predict(m.normalize_device(green))
    m.thresholds["prob"] = float(np.quantile(prob.cpu().numpy(), 0.7))
    return s


def _image(rng, H, W, spp, dtype):
    hi = 255 if dtype == np.uint8 else 65535
    a = np.cumsum(rng.integers(-60, 61, (H, W, spp)), axis=1) + rng.integers(0, hi, (1, 1, spp))
    a = np.mod(a, hi + 1).astype(dtype)
    return a[..., 0] if spp == 1 else a


def test_device_decode_equals_read_tiff_in_every_combination(screener, tmp_path):
    from cell_image_analysis_b200.tiff_device import decode_tiff_files
    from cell_image_analysis_b200.tiff_min import read_tiff
    rng = np.random.default_rng(5)
    H, W = 45, 70                                  # neither a multiple of 16-row strips nor of 32 x 48 tiles
    paths = []
    for comp in (1, 5, 8, 32773):
        for pred in (1, 2):
            for tile in (None, (32, 48)):
                for spp, planar in ((1, 1), (3, 1), (3, 2)):
                    for dtype in (np.uint8, np.uint16):
                        for bo in ("<", ">"):
                            p = str(tmp_path / f"f{len(paths):03d}.tif")
                            tiff_fixtures.write(p, _image(rng, H, W, spp, dtype), bo=bo, planar=planar,
                                                compression=comp, predictor=pred, rows_per_strip=16, tile=tile)
                            paths.append(p)
    order = rng.permutation(len(paths))            # chunks of 16 mixing compressions and layouts
    for c0 in range(0, len(paths), 16):
        chunk = [paths[i] for i in order[c0:c0 + 16]]
        seg, green, status = decode_tiff_files(screener.engine, chunk)
        assert not status.any()
        seg, green = seg.cpu().numpy(), green.cpu().numpy()
        for k, p in enumerate(chunk):
            ws, wg = tiff_fixtures.channels(read_tiff(p))
            np.testing.assert_array_equal(green[k], wg, err_msg=p)
            np.testing.assert_array_equal(seg[k], ws, err_msg=p)


def test_one_corrupted_segment_flags_only_its_field(screener, tmp_path):
    from cell_image_analysis_b200.tiff_device import decode_tiff_files
    from cell_image_analysis_b200.tiff_min import page_layout, read_tiff
    rng = np.random.default_rng(6)
    paths = []
    for k in range(16):
        p = str(tmp_path / f"c{k:02d}.tif")
        tiff_fixtures.write(p, _image(rng, 200, 260, 1, np.uint16), compression=(8, 5, 32773)[k % 3], predictor=2,
                            rows_per_strip=16)
        paths.append(p)
    bad = 6                                        # Deflate: a flipped bit inside its fourth strip
    buf = bytearray(open(paths[bad], "rb").read())
    off, cnt = page_layout(bytes(buf)).segments[3]
    buf[off + cnt // 2] ^= 0x10
    open(paths[bad], "wb").write(bytes(buf))
    seg, green, status = decode_tiff_files(screener.engine, paths)
    assert status[bad] != 0
    assert not np.delete(status, bad).any()
    green = green.cpu().numpy()
    for k, p in enumerate(paths):
        if k != bad:
            np.testing.assert_array_equal(green[k], read_tiff(p))


def _folders(tmp_path, compressed, bad=None):
    from cell_image_analysis_b200.tiff_min import write_tiff
    fields = _tiny_fields(tuple(range(20, 30)))
    folders = {}
    for s, name in enumerate(("strain_a", "strain_b")):
        d = tmp_path / (name + ("_z" if compressed else "_raw"))
        d.mkdir()
        for k in range(5):
            i = 5 * s + k
            p = str(d / f"field_{k}.tif")
            if compressed:
                tiff_fixtures.write(p, fields[i], compression=(5, 8)[i % 2], predictor=2, rows_per_strip=16)
            else:
                write_tiff(p, fields[i])
            if i == bad:
                buf = bytearray(open(p, "rb").read())
                if compressed:
                    buf[len(buf) // 3] ^= 0xFF
                else:
                    buf = buf[:8] + b"\xff" * 64         # neither read_tiff nor OpenCV reads it
                open(p, "wb").write(bytes(buf))
        folders[name] = str(d)
    return folders


def test_sharded_screen_over_compressed_files_equals_uncompressed(screener, tmp_path):
    import cell_image_analysis_b200.tiff_device as td
    calls = []
    orig = td.TiffChunk.decode
    td.TiffChunk.decode = lambda self, *a: (calls.append(self.n_segs), orig(self, *a))[1]
    try:
        res_z, det_z = screener.screen_mutant_samples_sharded(_folders(tmp_path, True), chunk_fields=4)
    finally:
        td.TiffChunk.decode = orig
    assert len(calls) == 3                         # 10 files in chunks of 4: every one decoded on the device
    res_r, det_r = screener.screen_mutant_samples_sharded(_folders(tmp_path, False), chunk_fields=4)
    assert det_z == det_r and len(det_r) > 0
    _same_results(res_z, res_r)


def _same_results(res_z, res_r):
    """counts exact; the strain means within fp64 rounding (the device accumulator sums in arrival order)"""
    assert res_z.keys() == res_r.keys()
    for k in res_r:
        for key, v in res_r[k].items():
            assert res_z[k][key] == pytest.approx(v, rel=1e-12, abs=1e-15), (k, key)


def test_a_corrupt_compressed_file_is_reported_and_skipped(screener, tmp_path, capsys):
    bad = 7                                        # a Deflate file: its Adler-32 catches any flip
    res_z, det_z = screener.screen_mutant_samples_sharded(_folders(tmp_path, True, bad=bad), chunk_fields=4)
    out_z = capsys.readouterr().out
    res_r, det_r = screener.screen_mutant_samples_sharded(_folders(tmp_path, False, bad=bad), chunk_fields=4)
    out_r = capsys.readouterr().out
    name = os.path.join("strain_b_z", "field_2.tif")
    assert f"Error processing {tmp_path / name}" in out_z
    assert f"Error processing {tmp_path / os.path.join('strain_b_raw', 'field_2.tif')}" in out_r
    assert det_z == det_r
    _same_results(res_z, res_r)


def test_run_images_host_keeps_each_chunks_decode_status(screener, tmp_path):
    """three chunks in one run_images_host call on two buffer sets: chunk 2 decodes into the buffers of chunk 0, whose
    flags must have been read back first; the flagged field stays out of the strain totals without strain ids, and
    every other field screens exactly as when its image is copied from pinned memory"""
    import torch
    from cell_image_analysis_b200.batch import BatchScreen
    from cell_image_analysis_b200.tiff_device import TiffChunk, parse_field
    from cell_image_analysis_b200.tiff_min import page_layout
    fields = _tiny_fields(tuple(range(40, 52)))
    Fc, n, bad = 4, len(fields), 1
    paths = []
    for k, f in enumerate(fields):
        p = str(tmp_path / f"m{k:02d}.tif")
        tiff_fixtures.write(p, f, compression=8, predictor=2, rows_per_strip=16)
        paths.append(p)
    buf = bytearray(open(paths[bad], "rb").read())
    off, cnt = page_layout(bytes(buf)).segments[1]
    buf[off + cnt // 2] ^= 0x10
    open(paths[bad], "wb").write(bytes(buf))
    H, W = fields.shape[1:]
    m = screener.stardist_model
    pt, nt = m.thresholds["prob"], m.thresholds["nms"]
    bs = BatchScreen(screener.engine, H, W, 4096, chunk_fields=Fc)
    unused = torch.zeros((n, H, W), dtype=torch.int16).pin_memory()      # every field is decoded on the device
    chunks = [TiffChunk([parse_field(p) for p in paths[c:c + Fc]], range(Fc)) for c in range(0, n, Fc)]
    bs.run_images_host(unused, unused, n, pt, nt, tiff=chunks)
    r = bs.collect_host()
    st = bs.tiff_status[:3].numpy().reshape(-1)
    assert st[bad] != 0 and not np.delete(st, bad).any()
    ref = BatchScreen(screener.engine, H, W, 4096, chunk_fields=Fc)
    pool = torch.from_numpy(np.ascontiguousarray(fields).view(np.int16)).pin_memory()
    ref.run_images_host(pool, pool, n, pt, nt)
    r2 = ref.collect_host()
    good = np.delete(np.arange(n), bad)
    np.testing.assert_array_equal(r["field_counts"][good], r2["field_counts"][good])
    keep, keep2 = r["cells"]["field"] != bad, r2["cells"]["field"] != bad
    assert keep2.sum() > 0
    for k in ("mse", "mae", "dec_cons", "dec_mod", "pred_cons", "pred_mod"):
        np.testing.assert_array_equal(r[k][keep], r2[k][keep2], err_msg=k)
    assert bs.acc[0, 0].item() == keep2.sum()
