"""The Zstandard decoder (td_zstd of csrc/tiff_decode.h, the code the device runs) compiled for the host under
AddressSanitizer + UBSan (tests/host_fuzz/fuzz_tiff_zstd.cpp), against libzstd: byte-exact over levels, strategies,
window logs, long-distance matching, checksum and content-size flags and inputs at the 128 KB block edge, with a frame
walker proving every block, literals and sequence type was decoded; concatenated and skippable frames; refusal of
dictionaries; and truncated, bit-flipped and checksum-flipped frames, which come back corrupt or short and never
read or write out of bounds."""
import random
import subprocess

import numpy as np
import pytest

import zstd_fixtures as zf

pytestmark = pytest.mark.skipif(zf.ZSTD is None, reason=zf.SKIP_REASON or "")


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    return zf.build_harness(tmp_path_factory.mktemp("zfuzz"))


def _inputs():
    rng = np.random.default_rng(7)
    words = [bytes(rng.integers(97, 123, int(rng.integers(2, 9)), dtype=np.uint8)) for _ in range(400)]
    text = b" ".join(words[int(k)] for k in rng.zipf(1.3, 60000) % 400)
    rand = rng.integers(0, 256, 131072, dtype=np.uint8).tobytes()

    def patched(ch):                               # rand with every 16th byte ch
        p = bytearray(rand)
        p[::16] = ch * len(p[::16])
        return bytes(p)
    # blocks 2 and 3 copy the block before them in 15-byte matches at one offset, with one literal ("Z", "Y") between
    # them: RLE literals and RLE tables for all three codes
    field = (np.cumsum(rng.integers(-40, 41, (256, 512)), axis=1) + 30000).astype("<u2").tobytes()
    return {
        "empty": b"", "one": b"x", "constant": b"\7" * 200000, "random": rand[:50000],
        "ramp16": (np.arange(150000) % 65536).astype("<u2").tobytes(), "ramp8": bytes(range(256)) * 600,
        "field16": field, "text": text, "short_text": text[:200], "repeat_patched": rand + patched(b"Z") + patched(b"Y"),
        "edge-1": field[:131071], "edge": field[:131072], "edge+1": field[:131073],
    }


def test_round_trips_match_libzstd_and_reach_every_type(harness, tmp_path):
    ins = _inputs()
    frames = []                                    # (frame, content)
    for name, data in ins.items():
        for level in (-5, 1, 3, 9, 19, 22):
            frames.append((zf.compress(data, level, checksum=1), data))
        for checksum in (0, 1):
            for content_size in (0, 1):
                frames.append((zf.compress(data, 3, checksum=checksum, content_size=content_size), data))
    for strategy in range(1, 10):                  # ZSTD_fast .. ZSTD_btultra2
        for name in ("text", "field16", "repeat_patched"):
            frames.append((zf.compress(ins[name], 6, strategy=strategy, checksum=1), ins[name]))
    big = ins["field16"] + ins["text"] + ins["field16"]
    for wlog in range(10, 28):
        for ldm in (0, 1):
            frames.append((zf.compress(big, 5, window_log=wlog, ldm=ldm, checksum=wlog % 2), big))
    seen = set()
    for f, _ in frames:
        zf.walk(f, seen)
        assert zf.decompress(f, 1 << 20) is not None
    recs = [(f, len(d) + 64) for f, d in frames]    # room to spare: the whole frame is decoded
    for (f, d), got in zip(frames, zf.decode(harness, tmp_path, recs)):
        assert got == zf.decompress(f, len(d)) == d
    recs = [(f, len(d) // 3) for f, d in frames if len(d) > 3]      # clipped: the first cap bytes
    for (f, cap), got in zip(recs, zf.decode(harness, tmp_path, recs)):
        assert got == zf.decompress(f, 1 << 20)[:cap]
    want = {("block", t) for t in ("raw", "rle", "compressed")}
    want |= {("literals", t) for t in ("raw", "rle")}
    want |= {("literals", t, s) for t in ("compressed", "treeless") for s in (1, 4)}
    want |= {("sequences", c, m) for c in ("ll", "of", "ml") for m in ("predefined", "rle", "fse", "repeat")}
    assert want <= seen, want - seen


def _dict_id(frame: bytes, did: int) -> bytes:
    """the frame with a one-byte dictionary ID field holding ``did`` (the frame must have none)"""
    fhd = frame[4]
    assert fhd & 3 == 0
    at = 5 + (0 if fhd & 0x20 else 1)
    return frame[:4] + bytes([fhd | 1]) + frame[5:at] + bytes([did]) + frame[at:]


def test_concatenated_skippable_and_dictionary_frames(harness, tmp_path):
    ins = _inputs()
    a, b, c = ins["text"][:30000], ins["field16"][:40000], ins["short_text"]
    fa, fb, fc = (zf.compress(x, 3, checksum=1) for x in (a, b, c))
    skip = (0x184D2A5A).to_bytes(4, "little") + (5).to_bytes(4, "little") + b"12345"
    empty_skip = (0x184D2A50).to_bytes(4, "little") + bytes(4)
    cases = [
        (fa + fb + fc, a + b + c),
        (skip + fa + empty_skip + fb + skip, a + b),
        (fa + zf.compress(b"", 3) + fc, a + c),
        (_dict_id(fa, 0), a),                       # a dictionary ID field holding 0: no dictionary
    ]
    recs = [(f, len(want) + 10) for f, want in cases]
    for (f, want), got in zip(cases, zf.decode(harness, tmp_path, recs)):
        assert got == want == zf.decompress(f, len(want) + 10)
    refused = [
        _dict_id(fa, 9),                            # a dictionary is needed
        fa + b"\x01\x02\x03",                       # trailing bytes that are no frame
        fa + skip[:-1],                             # truncated skippable frame
        fa + (0xFD2FB527).to_bytes(4, "little") + fb,   # unknown magic
    ]
    for f, got in zip(refused, zf.decode(harness, tmp_path, [(f, 1 << 20) for f in refused])):
        assert got is None and zf.decompress(f, 1 << 20) is None
    # a frame whose content exceeds the capacity is cut there, and what follows it is not read
    got = zf.decode(harness, tmp_path, [(fa + fb, len(a) + 100), (fa + b"junk", len(a))])
    assert got == [(a + b)[:len(a) + 100], a]


def test_truncated_and_flipped_frames_are_corrupt_or_short(harness, tmp_path):
    rng = random.Random(3)
    ins = _inputs()
    base = [(zf.compress(ins["text"][:3000], 3, checksum=1), ins["text"][:3000]),
            (zf.compress(ins["field16"][:6000], 19, checksum=1), ins["field16"][:6000]),
            (zf.compress(ins["repeat_patched"][:1500], 1, checksum=0), ins["repeat_patched"][:1500]),
            (zf.compress(ins["text"][:20000], -5, checksum=1, content_size=0), ins["text"][:20000])]
    recs, kinds = [], []
    for f, d in base:
        for k in range(len(f)):                    # every truncation
            recs.append((f[:k], len(d)))
            kinds.append(("trunc", d))
        for _ in range(300):                       # bit flips
            b = bytearray(f)
            for _ in range(rng.choice((1, 1, 2, 3))):
                b[rng.randrange(len(b))] ^= 1 << rng.randrange(8)
            recs.append((bytes(b), len(d)))
            kinds.append(("flip", d, f[4] >> 2 & 1))
        if f[4] >> 2 & 1:
            for bit in range(32):                  # the content checksum
                b = bytearray(f)
                b[len(b) - 4 + bit // 8] ^= 1 << (bit % 8)
                recs.append((bytes(b), len(d)))
                kinds.append(("checksum", d))
    got = zf.decode(harness, tmp_path, recs)
    refused = 0
    for g, kind in zip(got, kinds):
        d = kind[1]
        if kind[0] == "checksum":
            assert g is None
        elif kind[0] == "trunc":
            assert g is None or len(g) < len(d)
        elif kind[2]:                              # flipped with a checksum: refused, short or intact
            assert g is None or len(g) < len(d) or g == d
        refused += g is None
    assert refused > len(recs) // 2


def _header_bytes(frame: bytes) -> int:
    """magic + frame header"""
    fhd = frame[4]
    single = fhd >> 5 & 1
    return 5 + (1 - single) + (0, 1, 2, 4)[fhd & 3] + (single, 2, 4, 8)[fhd >> 6]


def test_a_declared_content_size_bounds_the_frame(harness, tmp_path):
    """a frame that declares its content size and fits the capacity is decoded and checked completely: one that writes
    past the size is refused, not cut at the capacity; a mutated frame comes back refused or intact"""
    rng = random.Random(5)
    ins = _inputs()
    d = ins["text"][:3000]
    f = zf.compress(d, 3, checksum=1)
    fhd = f[4]
    assert fhd >> 6 == 1                           # a 2-byte content size field (value - 256)
    at = _header_bytes(f) - 2
    lying = f[:at] + (len(d) - 100 - 256).to_bytes(2, "little") + f[at + 2:]
    no_checksum = zf.compress(d, 3, checksum=0)
    at2 = _header_bytes(no_checksum) - 2
    lying2 = no_checksum[:at2] + (len(d) - 100 - 256).to_bytes(2, "little") + no_checksum[at2 + 2:]
    recs = [(lying, len(d) - 100), (lying2, len(d) - 100), (lying2, len(d) - 200)]
    got = zf.decode(harness, tmp_path, recs)
    assert got[0] is None and got[1] is None       # past the declared size: refused at exactly that capacity
    assert got[2] == d[:len(d) - 200]              # a capacity below the declared size: cut there, unchecked
    assert all(zf.decompress(x, 1 << 20) is None for x in (lying, lying2))
    base = [(zf.compress(ins["field16"][:8000], lvl, checksum=1), ins["field16"][:8000]) for lvl in (1, 19)]
    base.append((zf.compress(ins["repeat_patched"][:5000], 3, checksum=1), ins["repeat_patched"][:5000]))
    recs, want = [], []
    for f, d in base:
        h = _header_bytes(f)
        for _ in range(400):                       # flips past the frame header, capacity = the content size
            b = bytearray(f)
            for _ in range(rng.choice((1, 2, 3))):
                b[rng.randrange(h, len(b))] ^= 1 << rng.randrange(8)
            recs.append((bytes(b), len(d)))
            want.append(d)
    got = zf.decode(harness, tmp_path, recs)
    assert all(g is None or g == d for g, d in zip(got, want))
    assert sum(g is None for g in got) > len(got) // 2


def test_random_frames_stay_in_bounds(harness):
    r = subprocess.run([harness, "random", "20000"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                       env=zf.ENV, timeout=600)
    assert r.returncode == 0 and r.stdout.startswith("ok:"), r.stdout[-3000:]
