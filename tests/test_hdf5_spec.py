"""hdf5_min against files that were NOT produced by this repository's own writer.

1. A file written by the real libhdf5: ``tests/golden/testhdf5_7.4_GLNX86.mat``, a copy of the
   4 KB file of SciPy's test data (scipy/io/matlab/tests/data, BSD-3-Clause) -- a MATLAB 7.3
   file = HDF5 1.6/1.8 behind a 512-byte user block: superblock v0, symbol-table root group, B-tree
   v1 + SNOD + local heap, v1 object headers, contiguous IEEE dataset.
2. Files assembled byte by byte in this test from the HDF5 File Format Specification 3.0 (section
   numbers in the comments) -- independent of ``oracle/h5write.py`` -- covering what h5py emits and
   the in-tree writer does not: a v1 object header whose symbol-table message sits in a
   *continuation block* behind NIL / modification-time / attribute messages, a two-level group
   B-tree over several SNODs, a *chunked* dataset (layout v3 class 2, chunk B-tree with partial edge
   chunks), a big-endian dataset, a compact dataset, and a superblock-v2 / OHDR file with compact
   link messages and Jenkins lookup3 checksums.
"""
import os
import struct

import numpy as np
import pytest

from cell_image_analysis_b200 import hdf5_min

UNDEF = 0xFFFFFFFFFFFFFFFF
SIG = b"\x89HDF\r\n\x1a\n"


def test_reads_a_file_written_by_the_real_libhdf5():
    p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "testhdf5_7.4_GLNX86.mat")
    f = hdf5_min.H5File(open(p, "rb").read())
    assert f.sb_version == 0 and f.base_addr == 512          # superblock found behind the user block
    ds = f.datasets()
    assert list(ds) == ["testdouble"]
    assert ds["testdouble"].dtype == np.float64 and ds["testdouble"].shape == (9, 1)
    # scipy/io/matlab/tests/gen_mat*.m: testdouble = 0:pi/4:2*pi
    np.testing.assert_array_equal(ds["testdouble"].ravel(), np.arange(9) * (np.pi / 4))


# ---------------------------------------------------------------------------------------------
# byte-level builder (spec sections in brackets)
# ---------------------------------------------------------------------------------------------
class Img:
    def __init__(self, size):
        self.b = bytearray(size)
        self.top = 0

    def at(self, off, data):
        assert off + len(data) <= len(self.b)
        self.b[off:off + len(data)] = data
        self.top = max(self.top, off + len(data))


def msg_v1(mtype, data, flags=0):
    """[IV.A.1.a] v1 header message: type u16, size u16, flags u8, 3 reserved, data padded to 8."""
    data = data + b"\0" * ((-len(data)) % 8)
    return struct.pack("<HHB3x", mtype, len(data), flags) + data


def ohdr_v1(messages, n_messages=None, size=None):
    """[IV.A.1.a] version 1 prefix: version, reserved, #messages u16, ref count u32, header size u32, pad to 8."""
    body = b"".join(messages)
    return struct.pack("<BxHII4x", 1, n_messages if n_messages is not None else len(messages), 1,
                       size if size is not None else len(body)) + body


def dataspace_v1(shape):
    """[IV.A.2.b] version 1: version, rank, flags, 5 reserved, dims u64."""
    return struct.pack("<BBB5x", 1, len(shape), 0) + b"".join(struct.pack("<Q", d) for d in shape)


def dtype_float(size, big_endian=False):
    """[IV.A.2.d] class 1 (floating point) version 1; bit field 0: byte order | mantissa normalisation 2 << 4."""
    exp_bits, mant = {4: (8, 23), 8: (11, 52)}[size]
    return struct.pack("<BBBBI", 0x11, 0x20 | (1 if big_endian else 0), size * 8 - 1, 0, size) + \
        struct.pack("<HHBBBBI", 0, size * 8, mant, exp_bits, 0, mant, (1 << (exp_bits - 1)) - 1)


def dtype_int(size, signed=True):
    """[IV.A.2.d] class 0 (fixed point): bit 3 = signed."""
    return struct.pack("<BBBBI", 0x10, 0x08 if signed else 0, 0, 0, size) + struct.pack("<HH", 0, size * 8)


def layout_v3_contiguous(addr, nbytes):
    return struct.pack("<BBQQ", 3, 1, addr, nbytes)                     # [IV.A.2.i] class 1


def layout_v3_compact(raw):
    return struct.pack("<BBH", 3, 0, len(raw)) + raw                    # [IV.A.2.i] class 0


def layout_v3_chunked(btree, chunk_dims, itemsize):
    dims = list(chunk_dims) + [itemsize]                                # dimensionality = rank + 1
    return struct.pack("<BBBQ", 3, 2, len(dims), btree) + b"".join(struct.pack("<I", d) for d in dims)


def fill_value_v2():
    return struct.pack("<BBBB", 2, 2, 2, 0)                             # [IV.A.2.f] undefined fill value


def mtime_msg():
    return struct.pack("<B3xI", 1, 1700000000)                          # [IV.A.2.s] modification time


def attribute_v1(name, value_f64):
    """[IV.A.2.m] version 1 attribute "name" = scalar float64 (h5py / Keras attach several of these)."""
    nm = name.encode() + b"\0"
    dt, ds = dtype_float(8), struct.pack("<BBB5x", 1, 0, 0)
    pad = lambda x: x + b"\0" * ((-len(x)) % 8)                          # noqa: E731
    return struct.pack("<BxHHH", 1, len(nm), len(dt), len(ds)) + pad(nm) + pad(dt) + pad(ds) + \
        struct.pack("<d", value_f64)


def symbol_entry(name_off, header, cache=0, btree=0, heap=0):
    """[III.C] symbol table entry, 40 bytes."""
    return struct.pack("<QQII", name_off, header, cache, 0) + struct.pack("<QQ", btree, heap)


def build_v0_file():
    """Superblock v0 [II.A]; root group -> continuation block -> symbol table message [IV.A.2.r];
    level-1 group B-tree [III.A.1] over two SNODs [III.B]; four datasets."""
    img = Img(8192)
    rng = np.random.default_rng(5)
    data = {
        "alpha": rng.standard_normal((3, 4)).astype("<f4"),             # contiguous
        "beta_be": rng.standard_normal((6,)).astype(">f8"),             # big-endian
        "chunked": rng.standard_normal((5, 7)).astype("<f4"),           # chunk (2, 4): partial edge chunks
        "tiny": np.array([1, -2, 3], "<i2"),                            # compact
        "zeta": np.arange(10, dtype="<u8").reshape(2, 5),
    }
    names = sorted(data)                                                # a B-tree orders its keys by name
    # ---- local heap [III.D]: "" at offset 0, then the link names
    heap_data = bytearray(b"\0" * 8)
    name_off = {}
    for n in names:
        name_off[n] = len(heap_data)
        heap_data += n.encode() + b"\0"
        heap_data += b"\0" * ((-len(heap_data)) % 8)
    HEAP, HEAP_DATA = 0x300, 0x340
    free_off = len(heap_data)
    heap_data += struct.pack("<QQ", 1, 32) + b"\0" * 16                 # one free block (next = 1: last)
    img.at(HEAP, b"HEAP" + struct.pack("<B3xQQQ", 0, len(heap_data), free_off, HEAP_DATA))
    img.at(HEAP_DATA, bytes(heap_data))

    # ---- raw data + dataset object headers (each with fill-value and mtime messages in front)
    cursor = [0x800]

    def put_raw(raw, align=8):
        cursor[0] = (cursor[0] + align - 1) // align * align
        off = cursor[0]
        img.at(off, raw)
        cursor[0] += len(raw)
        return off

    headers = {}
    for n in names:
        a = data[n]
        dt = dtype_float(a.dtype.itemsize, a.dtype.byteorder == ">") if a.dtype.kind == "f" else \
            dtype_int(a.dtype.itemsize, a.dtype.kind == "i")
        if n == "tiny":
            layout = layout_v3_compact(a.tobytes())
        elif n == "chunked":
            cd = (2, 4)
            keys = []
            for r0 in range(0, a.shape[0], cd[0]):
                for c0 in range(0, a.shape[1], cd[1]):
                    blk = np.zeros(cd, a.dtype)
                    sub = a[r0:r0 + cd[0], c0:c0 + cd[1]]
                    blk[:sub.shape[0], :sub.shape[1]] = sub
                    keys.append(((r0, c0), put_raw(blk.tobytes())))
            # [III.A.1] node type 1 (raw data chunks), level 0: key = chunk size u32, filter mask u32, offsets u64 x (rank + 1)
            node = b"TREE" + struct.pack("<BBHQQ", 1, 0, len(keys), UNDEF, UNDEF)
            for (r0, c0), addr in keys:
                node += struct.pack("<IIQQQ", cd[0] * cd[1] * 4, 0, r0, c0, 0) + struct.pack("<Q", addr)
            node += struct.pack("<IIQQQ", 0, 0, a.shape[0] + 1, a.shape[1] + 1, 0)     # closing key
            layout = layout_v3_chunked(put_raw(node), cd, 4)
        else:
            layout = layout_v3_contiguous(put_raw(a.tobytes()), a.nbytes)
        msgs = [msg_v1(0x0005, fill_value_v2()), msg_v1(0x0001, dataspace_v1(a.shape)), msg_v1(0x0003, dt, flags=1),
                msg_v1(0x0012, mtime_msg()), msg_v1(0x0008, layout), msg_v1(0x000C, attribute_v1("scale", 0.5))]
        headers[n] = put_raw(ohdr_v1(msgs))

    # ---- two symbol-table nodes [III.B] under a level-1 B-tree node
    SNOD0, SNOD1, TREE = 0x400, 0x540, 0x680
    split = 3
    for addr, part in ((SNOD0, names[:split]), (SNOD1, names[split:])):
        body = b"SNOD" + struct.pack("<BxH", 1, len(part))
        for n in part:
            body += symbol_entry(name_off[n], headers[n])
        img.at(addr, body + b"\0" * (8 + 8 * 40 - len(body)))           # 2K = 8 entry slots
    tree = b"TREE" + struct.pack("<BBHQQ", 0, 1, 2, UNDEF, UNDEF)       # type 0, level 1, two children
    tree += struct.pack("<QQ", 0, SNOD0) + struct.pack("<QQ", name_off[names[split - 1]], SNOD1)
    tree += struct.pack("<Q", name_off[names[-1]])
    img.at(TREE, tree)

    # ---- root object header: NIL + mtime + continuation [IV.A.2.q]; the symbol table message lives in the block
    ROOT, CONT = 0x100, 0x200
    cont = msg_v1(0x0000, b"\0" * 8) + msg_v1(0x0011, struct.pack("<QQ", TREE, HEAP))
    img.at(CONT, cont)
    first = [msg_v1(0x0000, b"\0" * 16), msg_v1(0x0012, mtime_msg()),
             msg_v1(0x0010, struct.pack("<QQ", CONT, len(cont)))]
    img.at(ROOT, ohdr_v1(first, n_messages=len(first) + 2))

    # ---- superblock v0 [II.A] + root symbol table entry (cache type 1: B-tree / heap in the scratch pad)
    eof = (cursor[0] + 7) // 8 * 8
    sb = SIG + struct.pack("<BBBBBBBBHHI", 0, 0, 0, 0, 0, 8, 8, 0, 4, 16, 0)
    sb += struct.pack("<QQQQ", 0, UNDEF, eof, UNDEF) + symbol_entry(0, ROOT, cache=1, btree=TREE, heap=HEAP)
    img.at(0, sb)
    return bytes(img.b[:eof]), data


def test_spec_built_v0_file_continuation_two_level_btree_chunked_bigendian():
    raw, data = build_v0_file()
    f = hdf5_min.H5File(raw)
    assert f.sb_version == 0
    ds = f.datasets()
    assert sorted(ds) == sorted(data)
    for name, want in data.items():
        got = ds[name]
        assert got.shape == want.shape and got.dtype.itemsize == want.dtype.itemsize, name
        assert got.dtype.byteorder == want.dtype.byteorder or want.dtype.itemsize == 1, name
        np.testing.assert_array_equal(got, want, err_msg=name)


def test_spec_built_file_behind_a_user_block():
    """[II.A] the superblock may sit at 512, 1024, ...; addresses are relative to the base address."""
    raw, data = build_v0_file()
    b = bytearray(b"U" * 1024 + raw)
    b[1024 + 24:1024 + 32] = struct.pack("<Q", 1024)                    # base address field of the superblock
    ds = hdf5_min.H5File(bytes(b)).datasets()
    np.testing.assert_array_equal(ds["chunked"], data["chunked"])
    np.testing.assert_array_equal(ds["beta_be"], data["beta_be"])


# ---- superblock v2 + version 2 object headers ------------------------------------------------
def lookup3(data: bytes, init: int = 0) -> int:
    """Bob Jenkins' lookup3 ``hashlittle`` -- the checksum of every v2 structure [II.A, IV.A.1.b]."""
    M = 0xFFFFFFFF
    rot = lambda x, k: ((x << k) | (x >> (32 - k))) & M                 # noqa: E731
    a = b = c = (0xDEADBEEF + len(data) + init) & M
    i, n = 0, len(data)
    while n > 12:
        a = (a + int.from_bytes(data[i:i + 4], "little")) & M
        b = (b + int.from_bytes(data[i + 4:i + 8], "little")) & M
        c = (c + int.from_bytes(data[i + 8:i + 12], "little")) & M
        a = (a - c) & M; a ^= rot(c, 4); c = (c + b) & M
        b = (b - a) & M; b ^= rot(a, 6); a = (a + c) & M
        c = (c - b) & M; c ^= rot(b, 8); b = (b + a) & M
        a = (a - c) & M; a ^= rot(c, 16); c = (c + b) & M
        b = (b - a) & M; b ^= rot(a, 19); a = (a + c) & M
        c = (c - b) & M; c ^= rot(b, 4); b = (b + a) & M
        i += 12; n -= 12
    if n == 0:
        return c
    tail = data[i:] + b"\0" * (12 - n)
    a = (a + int.from_bytes(tail[0:4], "little")) & M
    b = (b + int.from_bytes(tail[4:8], "little")) & M
    c = (c + int.from_bytes(tail[8:12], "little")) & M
    c ^= b; c = (c - rot(b, 14)) & M
    a ^= c; a = (a - rot(c, 11)) & M
    b ^= a; b = (b - rot(a, 25)) & M
    c ^= b; c = (c - rot(b, 16)) & M
    a ^= c; a = (a - rot(c, 4)) & M
    b ^= a; b = (b - rot(a, 14)) & M
    c ^= b; c = (c - rot(b, 24)) & M
    return c


def test_lookup3_known_answers():
    # the self-test vectors of lookup3.c (driver5): hashlittle("", 0) and the "Four score" string
    assert lookup3(b"", 0) == 0xDEADBEEF
    assert lookup3(b"", 0xDEADBEEF) == 0xBD5B7DDE
    assert lookup3(b"Four score and seven years ago", 0) == 0x17770551
    assert lookup3(b"Four score and seven years ago", 1) == 0xCD628161


def msg_v2(mtype, data, flags=0):
    return struct.pack("<BHB", mtype, len(data), flags) + data          # [IV.A.1.b] no padding, no creation order


def ohdr_v2(messages, continuation=None):
    """[IV.A.1.b] "OHDR", version 2, flags (bits 0-1: size of the chunk-0 length field = 2 bytes)."""
    body = b"".join(messages)
    if continuation is not None:
        body += msg_v2(0x10, struct.pack("<QQ", *continuation))
    h = b"OHDR" + struct.pack("<BBH", 2, 0x01, len(body)) + body
    return h + struct.pack("<I", lookup3(h))


def link_msg(name, addr):
    nm = name.encode()
    return struct.pack("<BBB", 1, 0x00, len(nm)) + nm + struct.pack("<Q", addr)   # [IV.A.2.g] hard link


def test_spec_built_v2_file_compact_links_and_ochk():
    img = Img(4096)
    a = np.linspace(-1, 1, 12, dtype="<f4").reshape(3, 4)
    b = np.arange(5, dtype="<i8")
    A_RAW, B_RAW, A_HDR, B_HDR, GRP, ROOT, OCHK = 0x400, 0x440, 0x200, 0x280, 0x300, 0x80, 0x380
    img.at(A_RAW, a.tobytes()); img.at(B_RAW, b.tobytes())
    ds2 = lambda shape: struct.pack("<BBBB", 2, len(shape), 0, 1) + b"".join(struct.pack("<Q", d) for d in shape)  # noqa: E731
    img.at(A_HDR, ohdr_v2([msg_v2(0x01, ds2(a.shape)), msg_v2(0x03, dtype_float(4)), msg_v2(0x05, fill_value_v2()),
                           msg_v2(0x08, layout_v3_contiguous(A_RAW, a.nbytes))]))
    img.at(B_HDR, ohdr_v2([msg_v2(0x01, ds2(b.shape)), msg_v2(0x03, dtype_int(8)),
                           msg_v2(0x08, layout_v3_contiguous(B_RAW, b.nbytes))]))
    # link info message [IV.A.2.c]: version 0, flags 0, fractal heap / name index addresses undefined = compact links
    link_info = struct.pack("<BBQQ", 0, 0, UNDEF, UNDEF)
    # the sub-group keeps its second link in a continuation chunk "OCHK" [IV.A.1.b]
    ochk_body = msg_v2(0x06, link_msg("b", B_HDR))
    ochk = b"OCHK" + ochk_body
    ochk += struct.pack("<I", lookup3(ochk))
    img.at(OCHK, ochk)
    img.at(GRP, ohdr_v2([msg_v2(0x02, link_info), msg_v2(0x06, link_msg("a", A_HDR))], continuation=(OCHK, len(ochk))))
    img.at(ROOT, ohdr_v2([msg_v2(0x02, link_info), msg_v2(0x06, link_msg("vars", GRP))]))
    eof = 0x440 + b.nbytes
    sb = SIG + struct.pack("<BBBB", 2, 8, 8, 0) + struct.pack("<QQQQ", 0, UNDEF, eof, ROOT)   # [II.A] version 2
    img.at(0, sb + struct.pack("<I", lookup3(sb)))
    f = hdf5_min.H5File(bytes(img.b[:eof]))
    assert f.sb_version == 2
    ds = f.datasets()
    assert sorted(ds) == ["vars/a", "vars/b"]
    np.testing.assert_array_equal(ds["vars/a"], a)
    np.testing.assert_array_equal(ds["vars/b"], b)


def test_dense_links_and_filters_are_refused_not_guessed():
    img = Img(1024)
    ROOT = 0x80
    link_info = struct.pack("<BBQQ", 0, 0, 0x300, UNDEF)                # fractal heap address set = dense storage
    img.at(ROOT, ohdr_v2([msg_v2(0x02, link_info)]))
    sb = SIG + struct.pack("<BBBB", 2, 8, 8, 0) + struct.pack("<QQQQ", 0, UNDEF, 1024, ROOT)
    img.at(0, sb + struct.pack("<I", lookup3(sb)))
    with pytest.raises(hdf5_min.H5FormatError):
        hdf5_min.H5File(bytes(img.b)).datasets()
