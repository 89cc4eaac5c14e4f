"""TIFF reader/writer for microscopy fields (SURVEY.md §8f row N1): the stand-in for
``tiff.imread`` (improved_detection.py:51) -- tifffile is not installable here.

Reads what acquisition software and ImageJ write for 8/16/32-bit fields: classic TIFF and BigTIFF,
little or big endian, strips or tiles, chunky or planar samples, integer and IEEE float samples,
compression none / LZW / Deflate (zlib, both tag values) / PackBits / Zstandard (50000 and the older 34926),
horizontal differencing (Predictor 2), and multi-page files (pages of one shape come back stacked
``[pages, H, W(, S)]`` like ``tifffile.imread``).  LZW and PackBits are decoded natively (libcia:
csrc/host_tiff.cpp) with a pure-Python fallback when the library has not been built; Zstandard is decoded
only by libcia, with the decoder the device runs.  JPEG / JPEG-XR / LERC etc. raise
``TiffError`` -- ``_default_imread`` then tries tifffile / OpenCV when they are present.
"""
from __future__ import annotations

import struct
import zlib

import numpy as np

_TYPES = {1: ("B", 1), 2: ("c", 1), 3: ("H", 2), 4: ("I", 4), 5: ("II", 8), 6: ("b", 1),
          8: ("h", 2), 9: ("i", 4), 16: ("Q", 8), 17: ("q", 8), 18: ("Q", 8)}


class TiffError(ValueError):
    pass


def _ifd_values(buf, bo, typ, count, value_field, pos):
    if typ not in _TYPES:
        return None
    fmt, size = _TYPES[typ]
    n = count * size
    data = value_field[:n] if n <= len(value_field) else buf[pos:pos + n]
    if len(data) < n:
        raise TiffError("truncated IFD value")
    if typ == 5:
        v = struct.unpack(bo + "II" * count, data)
        return [v[2 * i] / max(v[2 * i + 1], 1) for i in range(count)]
    if typ == 2:
        return [bytes(data)]
    return list(struct.unpack(bo + fmt * count, data))


def _lzw_python(src: bytes, cap: int) -> bytes:
    """TIFF 6.0 LZW (MSB-first codes, early change).  Fallback for hosts without libcia."""
    table = [bytes([i]) for i in range(256)] + [b"", b""]
    out = bytearray()
    bits, acc, have, old = 9, 0, 0, None
    for byte in src:
        acc = (acc << 8) | byte
        have += 8
        if have < bits:
            continue
        code = (acc >> (have - bits)) & ((1 << bits) - 1)
        have -= bits
        acc &= (1 << have) - 1
        if code == 257:
            break
        if code == 256:
            table = table[:258]
            bits, old = 9, None
            continue
        if old is None:
            entry = table[code]
        elif code < len(table):
            entry = table[code]
            table.append(old + entry[:1])
        elif code == len(table):
            entry = old + old[:1]
            table.append(entry)
        else:
            raise TiffError("corrupt LZW stream")
        out += entry
        old = entry
        if len(table) + 1 >= (1 << bits) and bits < 12:
            bits += 1
        if len(out) >= cap:
            break
    return bytes(out[:cap])


def _packbits_python(src: bytes, cap: int) -> bytes:
    out, i = bytearray(), 0
    while i < len(src) and len(out) < cap:
        h = src[i] - 256 if src[i] > 127 else src[i]
        i += 1
        if h >= 0:
            out += src[i:i + h + 1]
            i += h + 1
        elif h != -128:
            out += src[i:i + 1] * (1 - h)
            i += 1
    return bytes(out[:cap])


def _native():
    try:
        from . import _lib
        return _lib.load()
    except Exception:
        return None


def _decompress(data: bytes, compression: int, cap: int) -> bytes:
    if compression == 1:
        return data[:cap]
    if compression in (8, 32946):
        try:
            return zlib.decompress(data)[:cap]
        except zlib.error as e:
            raise TiffError(f"corrupt Deflate data: {e}") from e
    if compression in (5, 32773):
        lib = _native()
        if lib is not None:
            import ctypes as C
            dst = C.create_string_buffer(cap)
            fn = lib.cia_tiff_lzw_decode if compression == 5 else lib.cia_tiff_packbits_decode
            n = fn(data, len(data), dst, cap)
            if n < 0:
                raise TiffError("corrupt LZW / PackBits stream")
            return dst.raw[:n]
        return _lzw_python(data, cap) if compression == 5 else _packbits_python(data, cap)
    if compression in ZSTD_COMPRESSIONS:
        lib = _native()
        if lib is None:
            raise TiffError("Zstandard TIFF data needs libcia.so: build it with `python __graft_entry__.py build`")
        import ctypes as C
        dst = C.create_string_buffer(cap)
        n = lib.cia_tiff_zstd_decode(data, len(data), dst, cap)
        if n < 0:
            raise TiffError("corrupt Zstandard stream")
        return dst.raw[:n]
    raise TiffError(f"TIFF compression {compression} is not supported")


class PageLayout:
    """One IFD, parsed: what decoding the page needs, on the host or on the device (``cia_tiff_decode_fields``).
    ``segments`` lists (file offset, byte count) of each strip / tile in decode order (plane, row, column), the
    count clipped to the file's end as the reader slices it; ``rows`` is the decoded rows of each (tiles are always
    full size, the last strip is not)."""
    __slots__ = ("H", "W", "dtype", "spp", "planar", "compression", "predictor", "tiled", "tw", "th", "segments",
                 "next_ifd")

    def __init__(self, **kw):
        for k, v in kw.items():
            setattr(self, k, v)

    def segment_rects(self):
        """(plane, y0, x0, rows, cols) of each segment, in the order of ``segments``."""
        planes = self.spp if self.planar == 2 else 1
        across, down = -(-self.W // self.tw), -(-self.H // self.th)
        return [(p, ty * self.th, tx * self.tw, self.th if self.tiled else min(self.th, self.H - ty * self.th),
                 self.tw) for p in range(planes) for ty in range(down) for tx in range(across)]

    def device_decodable(self) -> bool:
        """Single-page file of 8- or 16-bit unsigned samples, compression none / LZW / Deflate / PackBits / Zstandard,
        predictor 1 or 2: what ``cia_tiff_decode_fields`` decodes bit for bit like ``read_tiff``."""
        return (self.next_ifd == 0 and self.dtype.kind == "u" and self.dtype.itemsize in (1, 2)
                and self.compression in DEVICE_COMPRESSIONS and self.predictor in (1, 2))


ZSTD_COMPRESSIONS = (50000, 34926)      # libtiff's COMPRESSION_ZSTD, and the code older tifffile versions wrote
DEVICE_COMPRESSIONS = (1, 5, 8, 32946, 32773) + ZSTD_COMPRESSIONS


def _parse_page(buf, bo, big, ifd) -> PageLayout:
    """One IFD -> its layout (no pixel data is read)."""
    if big:
        (n_entries,) = struct.unpack(bo + "Q", buf[ifd:ifd + 8])
        base, esz, vsz, ofmt = ifd + 8, 20, 8, "Q"
    else:
        (n_entries,) = struct.unpack(bo + "H", buf[ifd:ifd + 2])
        base, esz, vsz, ofmt = ifd + 2, 12, 4, "I"
    tags = {}
    for i in range(n_entries):
        e = buf[base + esz * i: base + esz * (i + 1)]
        if len(e) < esz:
            raise TiffError("truncated IFD")
        tag, typ = struct.unpack(bo + "HH", e[:4])
        (count,) = struct.unpack(bo + ofmt, e[4:4 + vsz])
        (off,) = struct.unpack(bo + ofmt, e[4 + vsz:4 + 2 * vsz])
        tags[tag] = _ifd_values(buf, bo, typ, count, e[4 + vsz:4 + 2 * vsz], off)
    (next_ifd,) = struct.unpack(bo + ofmt, buf[base + esz * n_entries: base + esz * n_entries + vsz])

    def tag1(t, default=None):
        v = tags.get(t)
        return default if not v else v[0]
    W, H = tag1(256), tag1(257)
    if not W or not H:
        raise TiffError("missing image dimensions")
    compression = tag1(259, 1)
    spp = tag1(277, 1)
    bits = tags.get(258, [1])
    if len(set(bits)) != 1 or bits[0] not in (8, 16, 32, 64):
        raise TiffError(f"unsupported BitsPerSample {bits}")
    fmt = tag1(339, 1)
    if fmt not in (1, 2, 3):
        raise TiffError(f"unsupported SampleFormat {fmt}")
    dt = np.dtype(f"{bo}{'u' if fmt == 1 else 'i' if fmt == 2 else 'f'}{bits[0] // 8}")
    if fmt == 3 and bits[0] not in (32, 64):
        raise TiffError("float samples must be 32 or 64 bit")
    planar = tag1(284, 1)
    predictor = tag1(317, 1)
    if predictor not in (1, 2) or (predictor == 2 and fmt == 3):
        raise TiffError(f"unsupported Predictor {predictor}")
    planes = spp if planar == 2 else 1              # separately stored sample planes
    tiled = 322 in tags or 324 in tags
    if tiled:
        tw, th = tag1(322), tag1(323)
        offsets, counts = tags.get(324), tags.get(325)
        if not tw or not th:
            raise TiffError("missing tile dimensions")
    else:
        tw, th = W, min(tag1(278, H) or H, H)
        offsets, counts = tags.get(273), tags.get(279)
    if not offsets:
        raise TiffError("missing strip / tile offsets")
    across, down = -(-W // tw), -(-H // th)
    if not counts:
        if compression != 1 or len(offsets) != 1:
            raise TiffError("missing strip byte counts")
        counts = [H * W * spp * dt.itemsize]
    if len(counts) != len(offsets) or len(offsets) < across * down * planes:
        raise TiffError("inconsistent strip / tile tables")
    n = len(buf)
    segments = [(o, max(0, min(c, n - o))) for o, c in zip(offsets[:across * down * planes], counts)]
    return PageLayout(H=H, W=W, dtype=dt, spp=spp, planar=planar, compression=compression, predictor=predictor,
                      tiled=tiled, tw=tw, th=th, segments=segments, next_ifd=next_ifd)


def _decode_page(buf, lay: PageLayout) -> np.ndarray:
    """The pixels of a parsed page, decoded on the host."""
    dt, H, W, spp = lay.dtype, lay.H, lay.W, lay.spp
    planes = spp if lay.planar == 2 else 1
    cs = 1 if lay.planar == 2 else spp              # samples per pixel inside one segment
    out = np.zeros((planes, H, W, cs), dt.newbyteorder("="))
    for (off, cnt), (p, y0, x0, rows, tw) in zip(lay.segments, lay.segment_rects()):
        need = rows * tw * cs * dt.itemsize
        raw = _decompress(bytes(buf[off:off + cnt]), lay.compression, need)
        if len(raw) < need:
            raise TiffError("truncated strip / tile data")
        seg = np.frombuffer(raw, dt, rows * tw * cs).reshape(rows, tw, cs).astype(dt.newbyteorder("="))
        if lay.predictor == 2:
            seg = np.cumsum(seg, axis=1, dtype=seg.dtype)   # horizontal differencing, wraps like the writer
        hh, ww = min(rows, H - y0), min(tw, W - x0)
        out[p, y0:y0 + hh, x0:x0 + ww] = seg[:hh, :ww]
    if lay.planar == 2:
        img = out[..., 0].transpose(1, 2, 0) if spp > 1 else out[0, ..., 0]
    else:
        img = out[0] if spp > 1 else out[0, ..., 0]
    return np.ascontiguousarray(img)


def _read_page(buf, bo, big, ifd):
    """One IFD -> (array, offset of the next IFD)."""
    lay = _parse_page(buf, bo, big, ifd)
    return _decode_page(buf, lay), lay.next_ifd


def _header(buf):
    """(byte order, BigTIFF?, offset of the first IFD)"""
    if len(buf) < 8:
        raise TiffError("not a TIFF file")
    if buf[:2] == b"II":
        bo = "<"
    elif buf[:2] == b"MM":
        bo = ">"
    else:
        raise TiffError("not a TIFF file")
    (magic,) = struct.unpack(bo + "H", buf[2:4])
    if magic == 42:
        big = False
        (ifd,) = struct.unpack(bo + "I", buf[4:8])
    elif magic == 43:
        big = True
        if len(buf) < 16 or struct.unpack(bo + "HH", buf[4:8]) != (8, 0):
            raise TiffError("malformed BigTIFF header")
        (ifd,) = struct.unpack(bo + "Q", buf[8:16])
    else:
        raise TiffError("not a TIFF file")
    return bo, big, ifd


def page_layout(buf) -> PageLayout:
    """Layout of the first page of the TIFF file held in ``buf`` (bytes), parsed exactly as ``read_tiff`` parses it;
    raises ``TiffError`` where ``read_tiff`` would on the directory."""
    bo, big, ifd = _header(buf)
    if not ifd or ifd >= len(buf):
        raise TiffError("no image in file")
    try:
        return _parse_page(buf, bo, big, ifd)
    except TiffError:
        raise
    except (struct.error, TypeError, IndexError, ValueError, OverflowError, MemoryError) as e:
        raise TiffError(f"malformed TIFF directory: {type(e).__name__}: {e}") from e


def read_tiff(path) -> np.ndarray:
    """The image of a TIFF file; ``path`` may also be the file's bytes, already read."""
    if isinstance(path, (bytes, bytearray, memoryview)):
        buf = bytes(path)
    else:
        with open(path, "rb") as f:
            buf = f.read()
    bo, big, ifd = _header(buf)
    pages, seen = [], set()
    while ifd and ifd not in seen and ifd < len(buf):
        seen.add(ifd)
        try:
            page, ifd = _read_page(buf, bo, big, ifd)
        except TiffError:
            raise
        except (struct.error, TypeError, IndexError, ValueError, OverflowError, MemoryError) as e:
            raise TiffError(f"malformed TIFF directory: {type(e).__name__}: {e}") from e   # corrupted tag values
        if pages and (page.shape != pages[0].shape or page.dtype != pages[0].dtype):
            break                                   # thumbnails / pyramids: keep the first series, like tifffile
        pages.append(page)
    if not pages:
        raise TiffError("no image in file")
    return pages[0] if len(pages) == 1 else np.stack(pages)


def write_tiff(path: str, img: np.ndarray, rows_per_strip: int = 64, compression: int = 1, tile=None,
               bigtiff: bool = False) -> None:
    """Little-endian TIFF writer (fixtures for tests and examples): strips or ``tile=(th, tw)``
    tiles (multiples of 16), uncompressed or Deflate (``compression=8``), classic or BigTIFF."""
    img = np.ascontiguousarray(img)
    if img.dtype not in (np.uint8, np.uint16, np.uint32):
        raise TiffError("write_tiff: uint8/16/32 only")
    if compression not in (1, 8):
        raise TiffError("write_tiff: compression 1 (none) or 8 (Deflate)")
    H, W = img.shape[:2]
    spp = 1 if img.ndim == 2 else img.shape[2]
    a = img.astype(img.dtype.newbyteorder("<")).reshape(H, W, spp)
    segs = []
    if tile:
        th, tw = tile
        if th % 16 or tw % 16:
            raise TiffError("tile sides must be multiples of 16")
        for y in range(0, H, th):
            for x in range(0, W, tw):
                t = np.zeros((th, tw, spp), a.dtype)
                t[:min(th, H - y), :min(tw, W - x)] = a[y:y + th, x:x + tw]
                segs.append(t.tobytes())
    else:
        segs = [a[r:r + rows_per_strip].tobytes() for r in range(0, H, rows_per_strip)]
    if compression == 8:
        segs = [zlib.compress(b) for b in segs]
    data = b"".join(b + (b"\0" if len(b) % 2 else b"") for b in segs)
    sizes = [len(b) for b in segs]
    padded = [len(b) + len(b) % 2 for b in segs]
    bits = img.itemsize * 8
    header = 16 if bigtiff else 8
    ifd_off = header + len(data)
    offs = [header + sum(padded[:k]) for k in range(len(segs))]
    osz, ofmt, otyp = (8, "Q", 16) if bigtiff else (4, "I", 4)
    esz = 20 if bigtiff else 12
    extra = bytearray()
    entries = []
    tags = [(256, 4, [W]), (257, 4, [H]), (258, 3, [bits] * spp), (259, 3, [compression]),
            (262, 3, [1 if spp == 1 else 2]), (277, 3, [spp]), (284, 3, [1]), (339, 3, [1] * spp)]
    if tile:
        tags += [(322, 4, [tile[1]]), (323, 4, [tile[0]]), (324, otyp, offs), (325, otyp, sizes)]
    else:
        tags += [(273, otyp, offs), (278, 4, [rows_per_strip]), (279, otyp, sizes)]
    tags.sort()
    n_entries = len(tags)
    extra_base = ifd_off + (8 if bigtiff else 2) + esz * n_entries + osz
    for tag, typ, values in tags:
        fmt, _size = _TYPES[typ]
        payload = struct.pack("<" + fmt * len(values), *values)
        if len(payload) <= osz:
            field = payload.ljust(osz, b"\0")
        else:
            field = struct.pack("<" + ofmt, extra_base + len(extra))
            extra.extend(payload + (b"\0" if len(payload) % 2 else b""))
        entries.append(struct.pack("<HH" + ofmt, tag, typ, len(values)) + field)
    with open(path, "wb") as f:
        if bigtiff:
            f.write(b"II" + struct.pack("<HHHQ", 43, 8, 0, ifd_off))
            f.write(data)
            f.write(struct.pack("<Q", n_entries) + b"".join(entries) + struct.pack("<Q", 0) + bytes(extra))
        else:
            f.write(b"II" + struct.pack("<HI", 42, ifd_off))
            f.write(data)
            f.write(struct.pack("<H", n_entries) + b"".join(entries) + struct.pack("<I", 0) + bytes(extra))
