"""Zstandard TIFF fields on the host: ``read_tiff`` of zstd files (compression 50000 and 34926) equals the array they
were written from in every layout the reader reads; without libcia a zstd file raises ``TiffError`` naming the
library; the device qualification and routing take zstd files."""
import numpy as np
import pytest

from cell_image_analysis_b200 import tiff_device as td
from cell_image_analysis_b200 import tiff_min

import tiff_fixtures
import zstd_fixtures as zf

pytestmark = pytest.mark.skipif(zf.ZSTD is None, reason=zf.SKIP_REASON or "")


def _image(rng, H, W, spp, dtype):
    hi = 255 if dtype == np.uint8 else 65535
    a = np.cumsum(rng.integers(-60, 61, (H, W, spp)), axis=1) + rng.integers(0, hi, (1, 1, spp))
    a = np.mod(a, hi + 1).astype(dtype)
    return a[..., 0] if spp == 1 else a


def test_read_tiff_of_zstd_files_in_every_layout(tmp_path, monkeypatch):
    zf.patch_encode(monkeypatch, level=5, checksum=1)
    rng = np.random.default_rng(11)
    H, W = 45, 70                                  # neither a multiple of 16-row strips nor of 32 x 48 tiles
    n = 0
    for comp in zf.CODES:
        for pred in (1, 2):
            for tile in (None, (32, 48)):
                for spp, planar in ((1, 1), (3, 1), (3, 2)):
                    for dtype in (np.uint8, np.uint16):
                        for bo in ("<", ">"):
                            img = _image(rng, H, W, spp, dtype)
                            p = str(tmp_path / f"z{n:03d}.tif")
                            tiff_fixtures.write(p, img, bo=bo, planar=planar, compression=comp, predictor=pred,
                                                rows_per_strip=16, tile=tile)
                            got = tiff_min.read_tiff(p)
                            assert got.dtype == img.dtype, p
                            np.testing.assert_array_equal(got, img, err_msg=p)
                            lay = tiff_min.page_layout(open(p, "rb").read())
                            assert lay.compression == comp and lay.device_decodable()
                            n += 1
    assert n == 2 * 2 * 2 * 3 * 2 * 2


def test_corrupt_and_truncated_zstd_strips_raise(tmp_path, monkeypatch):
    zf.patch_encode(monkeypatch, checksum=1)
    img = _image(np.random.default_rng(12), 64, 80, 1, np.uint16)
    p = str(tmp_path / "z.tif")
    tiff_fixtures.write(p, img, compression=50000, predictor=2, rows_per_strip=16)
    buf = bytearray(open(p, "rb").read())
    off, cnt = tiff_min.page_layout(bytes(buf)).segments[2]
    flipped = bytearray(buf)
    flipped[off + cnt - 2] ^= 0x01                 # inside the content checksum
    with pytest.raises(tiff_min.TiffError, match="corrupt Zstandard"):
        tiff_min.read_tiff(bytes(flipped))
    # a strip whose frame holds fewer bytes than the strip: the reader's "truncated" error
    short = zf.compress(img[32:40].astype("<u2").tobytes(), 3)
    monkeypatch.setattr(tiff_fixtures, "encode", lambda raw, c: short)
    tiff_fixtures.write(p, img, compression=50000, predictor=1, rows_per_strip=16)
    with pytest.raises(tiff_min.TiffError, match="truncated"):
        tiff_min.read_tiff(p)


def test_zstd_without_libcia_names_the_library(tmp_path, monkeypatch):
    zf.patch_encode(monkeypatch)
    p = str(tmp_path / "z.tif")
    tiff_fixtures.write(p, np.arange(400, dtype=np.uint16).reshape(20, 20), compression=34926)
    monkeypatch.setattr(tiff_min, "_native", lambda: None)
    with pytest.raises(tiff_min.TiffError, match="libcia"):
        tiff_min.read_tiff(p)


def test_device_route_takes_zstd_files_up_to_the_zstd_limit(tmp_path, monkeypatch):
    zf.patch_encode(monkeypatch)
    img = _image(np.random.default_rng(13), 96, 128, 1, np.uint16)
    for comp in zf.CODES:
        p = str(tmp_path / f"r{comp}.tif")
        tiff_fixtures.write(p, img, compression=comp, predictor=2, rows_per_strip=16)
        buf = open(p, "rb").read()
        assert td.device_route(p, buf) is not None
        assert td.device_route(p, buf, dtype=np.uint8) is None
        monkeypatch.setattr(td, "MAX_DEVICE_ZSTD_SEGMENT_BYTES", 16 * 128 * 2 - 1)
        assert td.device_route(p, buf) is None     # one byte above the limit: the host reader
        monkeypatch.setattr(td, "MAX_DEVICE_SEGMENT_BYTES", 0)
        monkeypatch.setattr(td, "MAX_DEVICE_ZSTD_SEGMENT_BYTES", 16 * 128 * 2)
        assert td.device_route(p, buf) is not None  # zstd takes its own limit, not Deflate's
        monkeypatch.undo()
        zf.patch_encode(monkeypatch)
    assert td.max_device_segment_bytes(50000) == td.max_device_segment_bytes(34926) == td.MAX_DEVICE_ZSTD_SEGMENT_BYTES
    assert td.max_device_segment_bytes(8) == td.MAX_DEVICE_SEGMENT_BYTES
