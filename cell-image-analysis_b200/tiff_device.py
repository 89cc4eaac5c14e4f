"""Device decode of compressed TIFF fields (SURVEY.md §8f row N1): the host parses the directory and packs the
compressed strips / tiles of a chunk of fields into one buffer; ``cia_tiff_decode_fields`` (csrc/tiff_dev.cu)
decodes every segment of the chunk in one launch into the uint16 (segmentation, analysis) planes that
``cia_screen_images`` takes (det:54-59), bit for bit what ``tiff_min.read_tiff`` returns.  Only the compressed
bytes cross PCIe.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .tiff_min import ZSTD_COMPRESSIONS, PageLayout, TiffError, page_layout

# A field whose largest strip / tile decodes to more bytes than this goes through the host reader: one segment is
# one serial stream on the device (tools/tiff_decode_probe.py, DESIGN §6 "TIFF decode on the device").
MAX_DEVICE_SEGMENT_BYTES = 1 << 20
# The same limit for Zstandard, set end to end: one warp decodes a zstd segment at about 5 MB/s, and the host route
# decodes on all loader threads while the device screens, so the sharded screen is faster with the device route up
# to 512 KB segments (128 rows of a 2048-wide uint16 field) and slower from 1 MB on (tools/tiff_zstd_probe.py,
# DESIGN §6).
MAX_DEVICE_ZSTD_SEGMENT_BYTES = 1 << 19


def max_device_segment_bytes(compression: int) -> int:
    """The largest decoded strip / tile of a field ``device_route`` sends to the device, by codec"""
    return MAX_DEVICE_ZSTD_SEGMENT_BYTES if compression in ZSTD_COMPRESSIONS else MAX_DEVICE_SEGMENT_BYTES


class TiffField:
    """A TIFF file's bytes with the layout of its (only) page."""
    __slots__ = ("path", "buf", "layout")

    def __init__(self, path: str, buf: bytes, layout: PageLayout):
        self.path, self.buf, self.layout = path, buf, layout

    @property
    def shape(self):
        return self.layout.H, self.layout.W

    @property
    def channels(self):
        """1: the one plane serves segmentation and analysis; 3: channel 2 segments, channel 1 is analysed"""
        return 1 if self.layout.spp == 1 else 3


def parse_field(path: str, buf: bytes = None) -> TiffField:
    """Reads ``path`` (unless its bytes ``buf`` are given) and parses its directory; raises ``TiffError`` for a file
    ``cia_tiff_decode_fields`` does not decode (multi-page, float / signed / 32-bit samples, other codecs, two-sample
    pixels)."""
    if buf is None:
        with open(path, "rb") as f:
            buf = f.read()
    lay = page_layout(buf)
    if not lay.device_decodable() or lay.spp == 2:
        raise TiffError("not decodable on the device")
    return TiffField(path, buf, lay)


def device_route(path: str, buf: bytes, dtype=np.uint16):
    """The parsed field when the product path should decode the file ``path`` (its bytes ``buf``) on the device -- a
    qualifying compressed file of ``dtype`` samples whose segments are small enough to decode in parallel -- else
    None."""
    try:
        f = parse_field(path, buf)
    except TiffError:
        return None
    lay = f.layout
    cs = 1 if lay.planar == 2 else lay.spp
    seg_bytes = lay.th * lay.tw * cs * lay.dtype.itemsize
    if (lay.compression == 1 or lay.dtype.newbyteorder("=") != np.dtype(dtype)
            or seg_bytes > max_device_segment_bytes(lay.compression)):
        return None
    return f


def pack_fields(fields, slots=None):
    """(src uint8 [n], segment table TIFF_SEGMENT_DTYPE [k], scratch bytes) of ``fields`` placed at ``slots``
    (default 0..len-1) of a chunk."""
    slots = range(len(fields)) if slots is None else slots
    parts, recs, src_off, dst_off = [], [], 0, 0
    for slot, f in zip(slots, fields):
        lay = f.layout
        cs = 1 if lay.planar == 2 else lay.spp
        bps = lay.dtype.itemsize
        for (off, cnt), (p, y0, x0, rows, cols) in zip(lay.segments, lay.segment_rects()):
            if lay.spp == 1:
                seg_s = img_s = 0
            elif lay.planar == 2:
                seg_s, img_s = (0 if p == 2 else -1), (0 if p == 1 else -1)
            else:
                seg_s, img_s = 2, 1
            recs.append((src_off, cnt, dst_off, slot, lay.compression, lay.predictor, bps,
                         int(lay.dtype.byteorder == ">"), cs, y0, x0, rows, cols, seg_s, img_s))
            parts.append(f.buf[off:off + cnt])
            src_off += cnt
            dst_off += rows * cols * cs * bps
    src = np.frombuffer(b"".join(parts), np.uint8) if parts else np.zeros(0, np.uint8)
    return src, np.array(recs, dtype=_lib.TIFF_SEGMENT_DTYPE), dst_off


class TiffChunk:
    """The device-decoded fields of one chunk: their compressed segments and the segment table packed into one pinned
    staging buffer (the table 8-byte aligned after the bytes), so that one copy moves the chunk."""

    def __init__(self, fields, slots, pinned: torch.Tensor = None):
        src, segs, self.scratch_bytes = pack_fields(fields, slots)
        self.n_segs, self.src_bytes = len(segs), len(src)
        self.table_off = -(-len(src) // 8) * 8
        self.total = self.table_off + segs.nbytes
        if pinned is None or pinned.numel() < self.total:
            pinned = torch.empty(max(self.total, 1), dtype=torch.uint8, pin_memory=True)
        self.pinned = pinned
        a = pinned.numpy()
        a[:len(src)] = src
        a[self.table_off:self.total] = segs.view(np.uint8)
        self.paths, self.slots = [f.path for f in fields], list(slots)

    def upload(self, dev: torch.Tensor):
        """One asynchronous H2D copy on the current stream into ``dev`` (uint8, at least ``total`` bytes)."""
        dev[:self.total].copy_(self.pinned[:self.total], non_blocking=True)

    def decode(self, engine, dev: torch.Tensor, scratch: torch.Tensor, seg_out, img_out, status):
        """Enqueues the decode of the uploaded chunk on the current stream."""
        decode_packed(engine, dev[:self.src_bytes], dev[self.table_off:self.total], self.n_segs,
                      scratch[:max(self.scratch_bytes, 1)], seg_out, img_out, status)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def decode_packed(engine, src_dev: torch.Tensor, segs_dev: torch.Tensor, n_segs: int, scratch: torch.Tensor,
                  seg_out, img_out: torch.Tensor, status: torch.Tensor, stream=None):
    """Enqueues ``cia_tiff_decode_fields`` on ``stream`` (default: the current stream): device buffers in, the
    planes ``seg_out`` (may be None or ``img_out``) / ``img_out`` [F, H, W] and ``status`` int32 [F] out."""
    F, H, W = img_out.shape
    s = stream if stream is not None else torch.cuda.current_stream(engine.tdev)
    engine._check(engine.lib.cia_tiff_decode_fields(
        engine.h, _ptr(src_dev), src_dev.numel(), _ptr(segs_dev), n_segs, F, H, W, _ptr(scratch), scratch.numel(),
        None if seg_out is None or seg_out is img_out else _ptr(seg_out), _ptr(img_out), _ptr(status),
        C.c_void_p(s.cuda_stream)))


def decode_tiff_files(engine, paths):
    """Decodes equally sized TIFF files on ``engine``'s GPU.  Returns ``(seg, green, status)``: uint16 cuda tensors
    [F, H, W] -- the segmentation and analysis channels, both the one plane of a single-channel file, 8-bit samples
    widened -- and a numpy int32 status per file, 0 when the planes equal ``read_tiff``'s channels bit for bit,
    nonzero for a corrupt or truncated file (its planes are then meaningless).  Raises ``TiffError`` for a file the
    device does not decode and ``ValueError`` when the files differ in size."""
    fields = [parse_field(p) for p in paths]
    if not fields:
        raise ValueError("no files")
    H, W = fields[0].shape
    if any(f.shape != (H, W) for f in fields):
        raise ValueError("decode_tiff_files needs equally sized fields")
    dev = engine.tdev
    src, segs, scratch_bytes = pack_fields(fields)
    F = len(fields)
    green = torch.empty((F, H, W), dtype=torch.int16, device=dev)
    seg = green if all(f.channels == 1 for f in fields) else torch.empty_like(green)
    status = torch.empty(F, dtype=torch.int32, device=dev)
    src_dev = torch.from_numpy(src.copy()).to(dev)
    segs_dev = torch.from_numpy(segs.view(np.uint8)).to(dev)
    scratch = torch.empty(max(scratch_bytes, 1), dtype=torch.uint8, device=dev)
    decode_packed(engine, src_dev, segs_dev, len(segs), scratch, seg, green, status)
    st = status.cpu().numpy()
    return seg.view(torch.uint16), green.view(torch.uint16), st
