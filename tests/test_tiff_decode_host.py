"""The device TIFF decoders (csrc/tiff_decode.h) compiled for the host under AddressSanitizer + UBSan
(tests/host_fuzz/fuzz_tiff_decode.cpp): Deflate byte-exact against Python's zlib over levels, strategies, window
sizes and memory levels, with the same accept / refuse decision on truncated, bit-flipped and random streams; LZW and
PackBits equal to the host decoders of csrc/host_tiff.cpp.  Then the page layout and segment table the device gets,
decoded segment by segment with the same decoders and assembled like the kernel does, against ``read_tiff`` on
files from write_tiff, OpenCV, PIL and a byte-by-byte writer (big endian, planar)."""
import os
import random
import shutil
import struct
import subprocess
import zlib

import numpy as np
import pytest

from cell_image_analysis_b200 import tiff_min
from cell_image_analysis_b200.tiff_device import TiffField, pack_fields

import tiff_fixtures

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "cell-image-analysis_b200", "csrc")
ENV = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    exe = str(tmp_path_factory.mktemp("tdfuzz") / "fuzz_tiff_decode")
    cmd = [gxx, "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
           os.path.join(ROOT, "tests", "host_fuzz", "fuzz_tiff_decode.cpp"), os.path.join(CSRC, "host_tiff.cpp"),
           "-o", exe]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0 and ("asan" in r.stdout or "ubsan" in r.stdout):
        pytest.skip("sanitizer runtimes not installed")
    assert r.returncode == 0, r.stdout
    return exe


def decode(exe, tmp_path, records):
    """records: (kind 0 Deflate / 1 LZW / 2 PackBits, bytes, cap) -> list of bytes or None (refused)"""
    inp, out = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as f:
        for kind, data, cap in records:
            f.write(struct.pack("<BQI", kind, cap, len(data)) + data)
    r = subprocess.run([exe, "records", str(inp), str(out)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, env=ENV, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("ok:"), r.stdout[-3000:]
    buf, pos, res = out.read_bytes(), 0, []
    for _ in records:
        (n,) = struct.unpack_from("<q", buf, pos)
        pos += 8
        res.append(None if n < 0 else buf[pos:pos + n])
        pos += max(n, 0)
    assert pos == len(buf)
    return res


def _payloads(rng):
    img = (np.cumsum(rng.integers(-40, 41, (48, 96)), axis=1) + 30000).astype("<u2").tobytes()
    return [img, rng.integers(0, 256, 5000, dtype=np.uint8).tobytes(), b"abcab" * 3000 + bytes(range(256)) * 40,
            b"", b"x"]


def _zlib_or_none(data):
    try:
        return zlib.decompress(data)
    except zlib.error:
        return None


def test_deflate_round_trips_match_zlib(harness, tmp_path):
    rng = np.random.default_rng(0)
    streams = []
    strategies = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]
    for data in _payloads(rng):
        for level in range(10):
            streams.append(zlib.compress(data, level))
        for strategy in strategies:
            for wbits in range(9, 16):
                for mem in (1, 9):
                    c = zlib.compressobj(6, zlib.DEFLATED, wbits, mem, strategy)
                    streams.append(c.compress(data) + c.flush())
    recs = [(0, s, 1 << 20) for s in streams]
    got = decode(harness, tmp_path, recs)
    for s, g in zip(streams, got):
        assert g == zlib.decompress(s)
    # clipped capacities: zlib.decompress(data)[:cap], the whole stream still checked
    recs = [(0, s, len(zlib.decompress(s)) // 3) for s in streams[:40]]
    for (_, s, cap), g in zip(recs, decode(harness, tmp_path, recs)):
        assert g == zlib.decompress(s)[:cap]


def test_deflate_refusals_match_zlib(harness, tmp_path):
    rng = random.Random(1)
    base = []
    for data in _payloads(np.random.default_rng(1)):
        for level in (0, 1, 6, 9):
            base.append(zlib.compress(data, level))
        c = zlib.compressobj(6, zlib.DEFLATED, 15, 9, zlib.Z_FIXED)
        base.append(c.compress(data) + c.flush())
    streams = []
    for s in base:
        streams.append(s + b"trailing bytes are ignored")
        for _ in range(6):
            streams.append(s[:rng.randrange(len(s))])                       # truncated
        for _ in range(25):
            b = bytearray(s)
            for _ in range(rng.choice((1, 1, 2, 4))):
                i = rng.randrange(len(b))
                b[i] ^= 1 << rng.randrange(8)                               # bit flips
            streams.append(bytes(b))
    for _ in range(300):
        n = rng.randrange(2, 600)
        streams.append(b"\x78\x9c" + bytes(rng.randrange(256) for _ in range(n)))   # random blocks, valid header
        streams.append(bytes(rng.randrange(256) for _ in range(n)))
    recs = [(0, s, 1 << 20) for s in streams]
    got = decode(harness, tmp_path, recs)
    refused = 0
    for s, g in zip(streams, got):
        want = _zlib_or_none(s)
        assert g == want, (s[:32], g is None, want is None)
        refused += want is None
    assert refused > 500 and refused < len(streams)


def _strips(path):
    buf = open(path, "rb").read()
    lay = tiff_min.page_layout(buf)
    cs = 1 if lay.planar == 2 else lay.spp
    return lay, [(buf[o:o + c], rows * cols * cs * lay.dtype.itemsize)
                 for (o, c), (_, _, _, rows, cols) in zip(lay.segments, lay.segment_rects())]


def test_lzw_and_packbits_equal_the_host_decoders(harness, tmp_path):
    import cv2
    rng = np.random.default_rng(2)
    img = (np.cumsum(rng.integers(-3, 4, (70, 90)), axis=1) + 500).astype(np.uint16)
    recs = []
    for kind, comp in ((1, cv2.IMWRITE_TIFF_COMPRESSION_LZW), (2, cv2.IMWRITE_TIFF_COMPRESSION_PACKBITS)):
        for pred in (1, 2):
            for a in (img, (img % 256).astype(np.uint8), np.dstack([img, img // 2, img // 3])):
                p = str(tmp_path / f"cv_{kind}_{pred}_{a.ndim}_{a.dtype}.tif")
                assert cv2.imwrite(p, a, [cv2.IMWRITE_TIFF_COMPRESSION, comp, cv2.IMWRITE_TIFF_PREDICTOR, pred])
                lay, strips = _strips(p)
                assert lay.compression == (5 if kind == 1 else 32773)
                for data, need in strips:
                    recs += [(kind, data, need), (kind, data, need // 2), (kind, data, need + 7), (kind, data, 0)]
                    b = bytearray(data)
                    for _ in range(3):
                        b[rng.integers(len(b))] ^= 1 << int(rng.integers(8))
                    recs += [(kind, bytes(b), need), (kind, data[:len(data) // 2], need)]
    for kind in (1, 2):
        for _ in range(200):
            recs.append((kind, rng.integers(0, 256, int(rng.integers(0, 800)), dtype=np.uint8).tobytes(),
                         int(rng.integers(0, 3000))))
    decode(harness, tmp_path, recs)             # the harness fails on any difference from csrc/host_tiff.cpp


def test_random_streams_stay_in_bounds(harness):
    r = subprocess.run([harness, "random", "3000"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                       env=ENV, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("ok:"), r.stdout[-3000:]


def assemble(harness, tmp_path, fields):
    """The device path on the host: pack_fields' table, each segment decoded by tiff_decode.h, then the kernel's
    per-segment step (zero fill, byte order, predictor, crop, channel planes) in NumPy"""
    src, segs, _ = pack_fields(fields)
    kinds = {1: None, 5: 1, 8: 0, 32946: 0, 32773: 2}
    recs, order = [], []
    for s in segs:
        need = int(s["rows"] * s["cols"] * s["samples"] * s["bytes_per_sample"])
        data = src[s["src_off"]:s["src_off"] + s["src_len"]].tobytes()
        k = kinds[int(s["compression"])]
        if k is None:
            order.append(data[:need])
        else:
            order.append(len(recs))
            recs.append((k, data, need))
    dec = decode(harness, tmp_path, recs) if recs else []
    F = len(fields)
    H, W = fields[0].shape
    seg_p, img_p = np.zeros((F, H, W), np.uint16), np.zeros((F, H, W), np.uint16)
    status = np.zeros(F, np.int32)
    for s, o in zip(segs, order):
        raw = o if isinstance(o, bytes) else dec[o]
        need = int(s["rows"] * s["cols"] * s["samples"] * s["bytes_per_sample"])
        if raw is None or len(raw) < need:
            status[s["field"]] |= 1 if raw is None else 2
            raw = (raw or b"").ljust(need, b"\0")
        dt = np.dtype(("<" if not s["big_endian"] else ">") + ("u1" if s["bytes_per_sample"] == 1 else "u2"))
        a = np.frombuffer(raw[:need], dt).reshape(s["rows"], s["cols"], s["samples"]).astype(dt.newbyteorder("="))
        if s["predictor"] == 2:
            a = np.cumsum(a, axis=1, dtype=a.dtype)
        y0, x0 = int(s["y0"]), int(s["x0"])
        hh, ww = min(int(s["rows"]), H - y0), min(int(s["cols"]), W - x0)
        for plane, k in ((seg_p, s["seg_sample"]), (img_p, s["img_sample"])):
            if k >= 0:
                plane[s["field"], y0:y0 + hh, x0:x0 + ww] = a[:hh, :ww, k]
    return seg_p, img_p, status


def _fixture_files(tmp_path):
    import cv2
    from PIL import Image
    rng = np.random.default_rng(3)
    H, W = 75, 101
    g16 = (np.cumsum(rng.integers(-50, 51, (H, W)), axis=1) + 20000).astype(np.uint16)
    rgb16 = np.dstack([g16, g16 // 3 + 7, g16 * np.uint16(5)]).astype(np.uint16)
    files = []
    for name, kw in (("wt_strips", dict(rows_per_strip=16, compression=8)), ("wt_tiles", dict(tile=(32, 48), compression=8)),
                     ("wt_big", dict(bigtiff=True, compression=1, rows_per_strip=7))):
        p = str(tmp_path / f"{name}.tif")
        tiff_min.write_tiff(p, g16, **kw)
        files.append(p)
    p = str(tmp_path / "wt_rgb.tif")
    tiff_min.write_tiff(p, rgb16, compression=8, rows_per_strip=10)
    files.append(p)
    for comp in (cv2.IMWRITE_TIFF_COMPRESSION_LZW, cv2.IMWRITE_TIFF_COMPRESSION_ADOBE_DEFLATE,
                 cv2.IMWRITE_TIFF_COMPRESSION_PACKBITS):
        for pred in (1, 2):
            for a in (g16, (g16 % 256).astype(np.uint8), rgb16[..., ::-1]):
                p = str(tmp_path / f"cv_{comp}_{pred}_{a.ndim}_{a.dtype}.tif")
                assert cv2.imwrite(p, a, [cv2.IMWRITE_TIFF_COMPRESSION, comp, cv2.IMWRITE_TIFF_PREDICTOR, pred])
                files.append(p)
    for comp in ("tiff_lzw", "tiff_adobe_deflate", "packbits", None):
        for img in (Image.fromarray((g16 % 256).astype(np.uint8)), Image.fromarray((rgb16 % 256).astype(np.uint8)),
                    Image.fromarray(g16)):
            p = str(tmp_path / f"pil_{comp}_{img.mode}.tif")
            img.save(p, compression=comp) if comp else img.save(p)
            files.append(p)
    for bo in ("<", ">"):
        for planar in (1, 2):
            for comp in (1, 5, 8, 32773):
                for pred in (1, 2):
                    for tile in (None, (32, 48)):
                        p = str(tmp_path / f"bb_{bo == '>'}_{planar}_{comp}_{pred}_{tile is None}.tif")
                        tiff_fixtures.write(p, rgb16 if planar == 2 or comp == 8 else g16, bo=bo, planar=planar,
                                            compression=comp, predictor=pred, rows_per_strip=16, tile=tile)
                        files.append(p)
    return files


def test_layout_and_segment_table_reproduce_read_tiff(harness, tmp_path):
    files = _fixture_files(tmp_path)
    assert len(files) > 60
    seen = set()
    for p in files:
        buf = open(p, "rb").read()
        lay = tiff_min.page_layout(buf)
        want = tiff_min.read_tiff(p)
        assert (lay.H, lay.W) == want.shape[:2] and lay.dtype.newbyteorder("=") == want.dtype
        assert lay.spp == (1 if want.ndim == 2 else want.shape[2])
        seen.add((lay.dtype.byteorder == ">", lay.planar, lay.compression, lay.predictor, lay.tiled))
        if lay.spp == 2 or not lay.device_decodable():
            continue
        seg, img, status = assemble(harness, tmp_path, [TiffField(p, buf, lay)])
        ws, wg = tiff_fixtures.channels(want)
        assert not status.any(), p
        np.testing.assert_array_equal(seg[0], ws, err_msg=p)
        np.testing.assert_array_equal(img[0], wg, err_msg=p)
    assert {(True, 2, 5, 2, True), (False, 1, 5, 2, False), (False, 1, 32773, 2, False), (False, 1, 8, 1, True),
            (False, 1, 8, 2, False)} <= seen


def test_qualification():
    lay = tiff_min.PageLayout(H=4, W=4, dtype=np.dtype("<u2"), spp=1, planar=1, compression=5, predictor=2,
                              tiled=False, tw=4, th=4, segments=[(8, 10)], next_ifd=0)
    assert lay.device_decodable()
    for k, v in (("next_ifd", 100), ("dtype", np.dtype("<i2")), ("dtype", np.dtype("<u4")), ("dtype", np.dtype("<f4")),
                 ("compression", 7), ("predictor", 3)):
        bad = tiff_min.PageLayout(**{**{s: getattr(lay, s) for s in tiff_min.PageLayout.__slots__}, k: v})
        assert not bad.device_decodable(), (k, v)
