"""Zstandard fixtures for the TIFF decoder tests: libzstd (``libzstd.so.1``) through ctypes as encoder and oracle, a
frame walker that names the block, literals and sequence types a frame uses, the ASan + UBSan harness of
tests/host_fuzz/fuzz_tiff_zstd.cpp, and a ``tiff_fixtures.encode`` that writes zstd strips (compression 50000 or
34926)."""
import ctypes as C
import os
import shutil
import struct
import subprocess

import pytest

import tiff_fixtures

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "cell-image-analysis_b200", "csrc")
ENV = dict(os.environ, ASAN_OPTIONS="detect_leaks=0")
CODES = (50000, 34926)

# ZSTD_cParameter values of the stable API (zstd.h)
PARAMS = {"level": 100, "window_log": 101, "strategy": 107, "ldm": 160, "content_size": 200, "checksum": 201}


def _load():
    try:
        z = C.CDLL("libzstd.so.1")
    except OSError as e:
        return None, f"libzstd.so.1 cannot be loaded: {e}"
    z.ZSTD_compressBound.restype, z.ZSTD_compressBound.argtypes = C.c_size_t, [C.c_size_t]
    z.ZSTD_createCCtx.restype, z.ZSTD_createCCtx.argtypes = C.c_void_p, []
    z.ZSTD_freeCCtx.restype, z.ZSTD_freeCCtx.argtypes = C.c_size_t, [C.c_void_p]
    z.ZSTD_CCtx_setParameter.restype, z.ZSTD_CCtx_setParameter.argtypes = C.c_size_t, [C.c_void_p, C.c_int, C.c_int]
    z.ZSTD_compress2.restype = C.c_size_t
    z.ZSTD_compress2.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    z.ZSTD_compress.restype = C.c_size_t
    z.ZSTD_compress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int]
    z.ZSTD_decompress.restype = C.c_size_t
    z.ZSTD_decompress.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
    z.ZSTD_isError.restype, z.ZSTD_isError.argtypes = C.c_uint, [C.c_size_t]
    return z, None


ZSTD, SKIP_REASON = _load()


def compress(data: bytes, level: int = 3, **params) -> bytes:
    """one frame; ``params``: names of PARAMS.  Plain ZSTD_compress when none is given"""
    cap = ZSTD.ZSTD_compressBound(len(data))
    out = C.create_string_buffer(max(cap, 1))
    if not params:
        n = ZSTD.ZSTD_compress(out, cap, data, len(data), level)
    else:
        cc = ZSTD.ZSTD_createCCtx()
        try:
            for k, v in {"level": level, **params}.items():
                r = ZSTD.ZSTD_CCtx_setParameter(cc, PARAMS[k], int(v))
                assert not ZSTD.ZSTD_isError(r), (k, v)
            n = ZSTD.ZSTD_compress2(cc, out, cap, data, len(data))
        finally:
            ZSTD.ZSTD_freeCCtx(cc)
    assert not ZSTD.ZSTD_isError(n)
    return out.raw[:n]


def decompress(frames: bytes, cap: int):
    """ZSTD_decompress into ``cap`` bytes; None when libzstd refuses"""
    out = C.create_string_buffer(max(cap, 1))
    n = ZSTD.ZSTD_decompress(out, cap, frames, len(frames))
    return None if ZSTD.ZSTD_isError(n) else out.raw[:n]


def walk(buf: bytes, seen: set) -> set:
    """adds to ``seen`` what the frames in ``buf`` use: ("block", raw | rle | compressed), ("literals", raw | rle),
    ("literals", compressed | treeless, streams), ("sequences", ll | of | ml, predefined | rle | fse | repeat)"""
    modes = ("predefined", "rle", "fse", "repeat")
    i = 0
    while i < len(buf):
        (magic,) = struct.unpack_from("<I", buf, i)
        if magic & 0xFFFFFFF0 == 0x184D2A50:
            i += 8 + struct.unpack_from("<I", buf, i + 4)[0]
            continue
        fhd = buf[i + 4]
        single = fhd >> 5 & 1
        i += 5 + (1 - single) + (0, 1, 2, 4)[fhd & 3] + (single, 2, 4, 8)[fhd >> 6]
        while True:
            bh = int.from_bytes(buf[i:i + 3], "little")
            i += 3
            btype, bsize = bh >> 1 & 3, bh >> 3
            seen.add(("block", ("raw", "rle", "compressed")[btype]))
            if btype == 2:
                b = buf[i:i + bsize]
                lt, sf = b[0] & 3, b[0] >> 2 & 3
                if lt < 2:
                    seen.add(("literals", ("raw", "rle")[lt]))
                    size = b[0] >> 3 if sf in (0, 2) else (b[0] >> 4) | (b[1] << 4) | ((b[2] << 12) if sf == 3 else 0)
                    p = (1, 2, 1, 3)[sf] + (size if lt == 0 else 1)
                else:
                    hl, bits = (3, 3, 4, 5)[sf], (10, 10, 14, 18)[sf]
                    p = hl + (int.from_bytes(b[:hl], "little") >> (4 + bits) & ((1 << bits) - 1))
                    seen.add(("literals", ("compressed", "treeless")[lt - 2], 1 if sf == 0 else 4))
                nseq = b[p]
                p += 1 + (0 if nseq < 128 else 2 if nseq == 255 else 1)
                if nseq:
                    for name, shift in (("ll", 6), ("of", 4), ("ml", 2)):
                        seen.add(("sequences", name, modes[b[p] >> shift & 3]))
            i += 1 if btype == 1 else bsize
            if bh & 1:
                break
        i += 4 if fhd >> 2 & 1 else 0
    return seen


def build_harness(tmp_dir) -> str:
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("no g++")
    exe = os.path.join(str(tmp_dir), "fuzz_tiff_zstd")
    cmd = [gxx, "-O1", "-g", "-std=c++17", "-fsanitize=address,undefined", "-fno-sanitize-recover=all",
           os.path.join(ROOT, "tests", "host_fuzz", "fuzz_tiff_zstd.cpp"), os.path.join(CSRC, "host_tiff.cpp"),
           "-o", exe]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0 and ("asan" in r.stdout or "ubsan" in r.stdout):
        pytest.skip("sanitizer runtimes not installed")
    assert r.returncode == 0, r.stdout
    return exe


def decode(exe, tmp_path, records):
    """records: (bytes, cap) -> list of bytes, or None where the decoder refuses the stream"""
    inp, out = tmp_path / "zin.bin", tmp_path / "zout.bin"
    with open(inp, "wb") as f:
        for data, cap in records:
            f.write(struct.pack("<QI", cap, len(data)) + data)
    r = subprocess.run([exe, "records", str(inp), str(out)], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, env=ENV, timeout=900)
    assert r.returncode == 0 and r.stdout.startswith("ok:"), r.stdout[-3000:]
    buf, pos, res = out.read_bytes(), 0, []
    for _ in records:
        (n,) = struct.unpack_from("<q", buf, pos)
        pos += 8
        res.append(None if n < 0 else buf[pos:pos + n])
        pos += max(n, 0)
    assert pos == len(buf)
    return res


def patch_encode(monkeypatch, level=3, **params):
    """``tiff_fixtures.write`` then compresses strips / tiles of codes 50000 and 34926 with libzstd"""
    orig = tiff_fixtures.encode
    monkeypatch.setattr(tiff_fixtures, "encode",
                        lambda raw, c: compress(raw, level, **params) if c in CODES else orig(raw, c))
