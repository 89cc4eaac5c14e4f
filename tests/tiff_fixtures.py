"""TIFF files built byte by byte for the decoder tests: either byte order, strips or tiles, chunky or planar samples,
compression none / LZW / Deflate / PackBits, predictor 1 or 2 -- combinations no single writer here produces."""
import struct
import zlib

import numpy as np


def lzw_encode(data: bytes) -> bytes:
    """TIFF LZW (MSB-first codes, early change), libtiff's code-width schedule"""
    out, acc, have = bytearray(), 0, 0

    def put(code, bits):
        nonlocal acc, have
        acc = (acc << bits) | code
        have += bits
        while have >= 8:
            out.append((acc >> (have - 8)) & 0xFF)
            have -= 8
        acc &= (1 << have) - 1
    table, nxt, bits = {}, 258, 9
    put(256, bits)
    cur = None
    for c in data:
        if cur is None:
            cur = (c,)
            code_cur = c
            continue
        key = (code_cur, c)
        if key in table:
            code_cur = table[key]
            continue
        put(code_cur, bits)
        table[key] = nxt
        nxt += 1
        if nxt >= (1 << bits) and bits < 12:
            bits += 1
        if nxt >= 4094:
            put(256, bits)
            table, nxt, bits = {}, 258, 9
        code_cur = c
    if cur is not None:
        put(code_cur, bits)
    put(257, bits)
    if have:
        out.append((acc << (8 - have)) & 0xFF)
    return bytes(out)


def packbits_encode(data: bytes) -> bytes:
    out, i = bytearray(), 0
    while i < len(data):
        j = i
        while j + 1 < len(data) and data[j + 1] == data[i] and j - i < 127:
            j += 1
        if j > i:
            out += bytes([(257 - (j - i + 1)) & 0xFF, data[i]])
            i = j + 1
        else:
            k = min(128, len(data) - i)
            out += bytes([k - 1]) + data[i:i + k]
            i += k
    return bytes(out)


def encode(raw: bytes, compression: int) -> bytes:
    if compression == 1:
        return raw
    if compression in (8, 32946):
        return zlib.compress(raw)
    if compression == 5:
        return lzw_encode(raw)
    if compression == 32773:
        return packbits_encode(raw)
    raise ValueError(compression)


def write(path, img, bo="<", planar=1, compression=8, predictor=1, rows_per_strip=16, tile=None):
    """``img`` uint8 / uint16 [H, W] or [H, W, S]; ``tile=(th, tw)`` writes tiles (multiples of 16)."""
    img = np.ascontiguousarray(img)
    H, W = img.shape[:2]
    spp = 1 if img.ndim == 2 else img.shape[2]
    a = img.reshape(H, W, spp)
    planes = [a[..., p:p + 1] for p in range(spp)] if planar == 2 else [a]
    dt = img.dtype.newbyteorder(bo)
    segs = []
    for pl in planes:
        if tile:
            th, tw = tile
            blocks = []
            for y in range(0, H, th):
                for x in range(0, W, tw):
                    t = np.zeros((th, tw, pl.shape[2]), img.dtype)
                    t[:min(th, H - y), :min(tw, W - x)] = pl[y:y + th, x:x + tw]
                    blocks.append(t)
        else:
            blocks = [pl[r:r + rows_per_strip] for r in range(0, H, rows_per_strip)]
        for b in blocks:
            if predictor == 2:
                b = b.copy()
                b[:, 1:] = b[:, 1:] - b[:, :-1]          # wraps in the sample type
            segs.append(encode(np.ascontiguousarray(b).astype(dt).tobytes(), compression))
    data = b"".join(s + (b"\0" if len(s) % 2 else b"") for s in segs)
    offs, pos = [], 8
    for s in segs:
        offs.append(pos)
        pos += len(s) + len(s) % 2
    ifd_off = 8 + len(data)
    tags = [(256, 4, [W]), (257, 4, [H]), (258, 3, [img.itemsize * 8] * spp), (259, 3, [compression]),
            (262, 3, [1 if spp == 1 else 2]), (277, 3, [spp]), (284, 3, [planar]), (317, 3, [predictor]),
            (339, 3, [1] * spp)]
    if tile:
        tags += [(322, 4, [tile[1]]), (323, 4, [tile[0]]), (324, 4, offs), (325, 4, [len(s) for s in segs])]
    else:
        tags += [(273, 4, offs), (278, 4, [rows_per_strip]), (279, 4, [len(s) for s in segs])]
    tags.sort()
    extra_base = ifd_off + 2 + 12 * len(tags) + 4
    extra, entries = bytearray(), []
    for tag, typ, vals in tags:
        fmt = "H" if typ == 3 else "I"
        payload = struct.pack(bo + fmt * len(vals), *vals)
        if len(payload) <= 4:
            field = payload.ljust(4, b"\0")
        else:
            field = struct.pack(bo + "I", extra_base + len(extra))
            extra += payload
        entries.append(struct.pack(bo + "HHI", tag, typ, len(vals)) + field)
    with open(path, "wb") as f:
        f.write((b"II" if bo == "<" else b"MM") + struct.pack(bo + "HI", 42, ifd_off))
        f.write(data)
        f.write(struct.pack(bo + "H", len(tags)) + b"".join(entries) + struct.pack(bo + "I", 0) + bytes(extra))


def channels(img):
    """(seg, green) of a read_tiff result as the screen splits it (det:54-59), widened to uint16"""
    if img.ndim == 3 and img.shape[-1] >= 3:
        return img[..., 2].astype(np.uint16), img[..., 1].astype(np.uint16)
    return img.astype(np.uint16), img.astype(np.uint16)
