"""Device decode of Zstandard TIFF fields (cia_tiff_decode_fields, compression 50000 and 34926): bit-equal to read_tiff in
every combination of code, predictor, strips / tiles, chunky / planar, 1 / 3 samples, 8 / 16 bit and byte order; zstd,
Deflate, LZW and PackBits files in one launch; a corrupt zstd field flags only itself; the sharded screen over zstd
files equals the same screen over the uncompressed files."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
pytestmark = [pytest.mark.gpu]

import tiff_fixtures  # noqa: E402
import zstd_fixtures as zf  # noqa: E402
from test_gpu_screen_images import _tiny_fields  # noqa: E402
from test_gpu_tiff_decode import _image, _same_results, screener  # noqa: E402,F401

if zf.ZSTD is None:
    pytestmark.append(pytest.mark.skip(reason=zf.SKIP_REASON))


def _check_chunk(engine, chunk):
    from cell_image_analysis_b200.tiff_device import decode_tiff_files
    from cell_image_analysis_b200.tiff_min import read_tiff
    seg, green, status = decode_tiff_files(engine, chunk)
    assert not status.any()
    seg, green = seg.cpu().numpy(), green.cpu().numpy()
    for k, p in enumerate(chunk):
        ws, wg = tiff_fixtures.channels(read_tiff(p))
        np.testing.assert_array_equal(green[k], wg, err_msg=p)
        np.testing.assert_array_equal(seg[k], ws, err_msg=p)


def test_device_decode_of_zstd_equals_read_tiff_in_every_combination(screener, tmp_path, monkeypatch):
    zf.patch_encode(monkeypatch, level=5, checksum=1)
    rng = np.random.default_rng(15)
    H, W = 45, 70                                  # neither a multiple of 16-row strips nor of 32 x 48 tiles
    paths = []
    for comp in zf.CODES:
        for pred in (1, 2):
            for tile in (None, (32, 48)):
                for spp, planar in ((1, 1), (3, 1), (3, 2)):
                    for dtype in (np.uint8, np.uint16):
                        for bo in ("<", ">"):
                            p = str(tmp_path / f"z{len(paths):03d}.tif")
                            tiff_fixtures.write(p, _image(rng, H, W, spp, dtype), bo=bo, planar=planar,
                                                compression=comp, predictor=pred, rows_per_strip=16, tile=tile)
                            paths.append(p)
    order = rng.permutation(len(paths))
    for c0 in range(0, len(paths), 16):
        _check_chunk(screener.engine, [paths[i] for i in order[c0:c0 + 16]])


def test_zstd_deflate_lzw_and_packbits_in_one_launch(screener, tmp_path, monkeypatch):
    zf.patch_encode(monkeypatch, level=19, checksum=1)
    rng = np.random.default_rng(16)
    paths = []
    for k in range(16):
        comp = (50000, 8, 5, 32773, 34926, 32946)[k % 6]
        p = str(tmp_path / f"m{k:02d}.tif")
        tiff_fixtures.write(p, _image(rng, 300, 260, 1 + 2 * (k % 2), np.uint16), compression=comp,
                            predictor=1 + k % 2, rows_per_strip=(16, 64, 300)[k % 3])
        paths.append(p)
    _check_chunk(screener.engine, paths)


def test_a_corrupt_zstd_field_flags_only_itself(screener, tmp_path, monkeypatch):
    from cell_image_analysis_b200.tiff_device import decode_tiff_files
    from cell_image_analysis_b200.tiff_min import page_layout, read_tiff
    zf.patch_encode(monkeypatch, checksum=1)
    rng = np.random.default_rng(17)
    paths = []
    for k in range(16):
        p = str(tmp_path / f"c{k:02d}.tif")
        tiff_fixtures.write(p, _image(rng, 200, 260, 1, np.uint16), compression=(50000, 8, 5, 32773)[k % 4],
                            predictor=2, rows_per_strip=16)
        paths.append(p)
    clean = {k: decode_tiff_files(screener.engine, [p])[1][0].cpu().numpy() for k, p in enumerate(paths)}
    for bad, how in ((4, "checksum"), (8, "truncated"), (12, "magic")):
        bad_path = str(tmp_path / f"bad{bad}.tif")
        if how == "truncated":                     # the fourth strip's frame cut in half, inside its one block
            strips = []

            def cut_fourth(raw, c):
                strips.append(zf.compress(raw, 3, checksum=1))
                return strips[-1][:len(strips[-1]) // 2] if len(strips) == 4 else strips[-1]
            monkeypatch.setattr(tiff_fixtures, "encode", cut_fourth)
            tiff_fixtures.write(bad_path, read_tiff(paths[bad]), compression=50000, predictor=1, rows_per_strip=16)
            zf.patch_encode(monkeypatch, checksum=1)
        else:
            buf = bytearray(open(paths[bad], "rb").read())
            off, cnt = page_layout(bytes(buf)).segments[3]
            buf[off + cnt - 1 if how == "checksum" else off] ^= 0x20
            open(bad_path, "wb").write(bytes(buf))
        chunk = list(paths)
        chunk[bad] = bad_path
        seg, green, status = decode_tiff_files(screener.engine, chunk)
        assert status[bad] & 1, how
        assert not np.delete(status, bad).any(), how
        green = green.cpu().numpy()
        for k, p in enumerate(paths):
            if k != bad:
                np.testing.assert_array_equal(green[k], clean[k])
                np.testing.assert_array_equal(green[k], read_tiff(p))


def test_sharded_screen_over_zstd_files_equals_uncompressed(screener, tmp_path, monkeypatch):
    import cell_image_analysis_b200.tiff_device as td
    from cell_image_analysis_b200.tiff_min import write_tiff
    zf.patch_encode(monkeypatch, checksum=1)
    fields = _tiny_fields(tuple(range(20, 30)))
    folders = {"z": {}, "raw": {}}
    for s, name in enumerate(("strain_a", "strain_b")):
        for kind in folders:
            d = tmp_path / f"{name}_{kind}"
            d.mkdir()
            folders[kind][name] = str(d)
            for k in range(5):
                p = str(d / f"field_{k}.tif")
                img = fields[5 * s + k]
                if kind == "z":
                    tiff_fixtures.write(p, img, compression=zf.CODES[k % 2], predictor=2, rows_per_strip=16)
                else:
                    write_tiff(p, img)
    calls = []
    orig = td.TiffChunk.decode
    monkeypatch.setattr(td.TiffChunk, "decode", lambda self, *a: (calls.append(self.n_segs), orig(self, *a))[1])
    res_z, det_z = screener.screen_mutant_samples_sharded(folders["z"], chunk_fields=4)
    assert len(calls) == 3                         # 10 files in chunks of 4: every one decoded on the device
    monkeypatch.setattr(td.TiffChunk, "decode", orig)
    res_r, det_r = screener.screen_mutant_samples_sharded(folders["raw"], chunk_fields=4)
    assert det_z == det_r and len(det_r) > 0
    _same_results(res_z, res_r)
