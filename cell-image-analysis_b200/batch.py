"""Chunked, stream-pipelined screening of many equally sized fields -- the
throughput form of the ``screen_mutant_samples`` loop (improved_detection.py:164-199):
fields -> cells -> scores -> per-strain accumulators, with no host synchronisation
inside a pass.

Two entry points:
  * ``run_device``: fields already resident in HBM (a pool tensor indexed by chunk);
  * ``run_host``: fields in pinned host memory; H2D copies run on a copy stream into
    double-buffered device chunks while the previous chunk is being scored, and the
    per-cell results are copied back D2H inside the pass.
and their images-only forms ``run_images_device`` / ``run_images_host``, which segment every chunk on the
device (``cia_screen_images``, a StarDist model loaded on the engine): no labels exist outside HBM.
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np
import torch

from . import _lib

STAGES = ("scan", "gates", "crop", "cae", "svm", "accumulate")


class BatchScreen:
    def __init__(self, engine, H: int, W: int, max_label: int, chunk_fields: int = 16,
                 n_strains: int = 1, cells_per_field_cap: int | None = None,
                 label_transport: str = "rle", host_threads: int = 0, rle_fraction: float = 1.0,
                 scan_runs: bool = True, host_buffers: int = 2, image_transport: str = "dense"):
        """``label_transport``: "rle" run-length encodes the int32 label fields on the host
        cores (csrc/transport.cu) so that only the runs cross PCIe; "raw" copies them as is.
        ``rle_fraction`` < 1 sends only that share of the chunks as runs and the rest raw (several
        ranks sharing the host cores: the encoder and the PCIe link then work side by side).
        ``scan_runs``: build the region table from the runs themselves (``cia_screen_fields_rle``);
        False expands them to the dense field first (``cia_rle_expand``)."""
        """``image_transport``: "dense" copies whole images; "patches" (with run-length labels scanned from the
        runs) sends only the bbox rectangles of the labelled regions -- all the device ever reads of an image --
        packed by the encoder threads and scattered into a dense device buffer after the region scan.  It cuts
        the H2D bytes 5x (8.9 -> 1.65 GB per 1024 fields) but costs host time: on the benchmark host (16-24
        vCPUs) the end-to-end rate is no better with it (one GPU: 172-186 vs 170 ms, two: 324-409 vs 276-289
        ms per step), so "dense" is the default; it is the better choice where PCIe, not the host cores, is
        the scarce resource."""
        assert label_transport in ("rle", "raw") and image_transport in ("patches", "dense")
        self.image_transport = image_transport
        self.label_transport, self.host_threads = label_transport, host_threads
        self.rle_fraction = 1.0 if label_transport == "rle" and rle_fraction >= 1.0 else \
            (0.0 if label_transport == "raw" else max(0.0, float(rle_fraction)))
        self.scan_runs = scan_runs
        self.eng = engine
        self.H, self.W, self.max_label = H, W, max_label
        self.Fc = chunk_fields
        self.cap = chunk_fields * (cells_per_field_cap or max_label)
        self.n_strains = n_strains
        d = engine.tdev
        # device-side chunk buffers of the host pass (2 = double buffering; a third was measured and buys
        # nothing: the pass is paced by the PCIe link, not by buffer turnover)
        self.NB = max(2, int(host_buffers))
        self.out = [engine.alloc_outputs(self.cap, chunk_fields) for _ in range(self.NB)]
        self.acc = torch.zeros((n_strains, 8), dtype=torch.float64, device=d)
        self.compute = torch.cuda.Stream(device=d)
        self.copy = torch.cuda.Stream(device=d)
        self.d2h = torch.cuda.Stream(device=d)       # result read-back, off the compute stream
        self._stage = None

    # ---- profiling ----
    def profile_begin(self, n_calls: int):
        self.eng._check(self.eng.lib.cia_profile_begin(self.eng.h, n_calls))

    def profile_layers(self):
        """CAE stage split by conv layer (ms summed over the recorded calls); before ``profile_end``."""
        ms = (C.c_double * 7)()
        self.eng._check(self.eng.lib.cia_profile_layers(self.eng.h, ms))
        return [float(v) for v in ms]

    def profile_end(self):
        ms = (C.c_double * 6)()
        n = C.c_int(0)
        self.eng._check(self.eng.lib.cia_profile_end(self.eng.h, ms, C.byref(n)))
        return dict(zip(STAGES, [float(v) for v in ms])), int(n.value)

    # ---- device-resident pass ----
    def run_device(self, images: torch.Tensor, labels: torch.Tensor, n_fields: int,
                   strain_of_visit: torch.Tensor | None = None):
        """One pass over ``n_fields`` field visits, cycling the resident pool
        ``images``/``labels`` [P,H,W] chunk by chunk.  Enqueues only; returns nothing.
        Per-strain accumulators (column 0 = cell count) land in ``self.acc``."""
        P = images.shape[0]
        assert P % self.Fc == 0 and n_fields % self.Fc == 0
        eng = self.eng
        with torch.cuda.stream(self.compute):
            if self._stage is not None:                  # a host pass may still be reading self.out back
                for e in self._stage["out_free"]:
                    self.compute.wait_event(e)
            for i in range(n_fields // self.Fc):
                p0 = (i * self.Fc) % P
                o = self.out[i & 1]
                st = None if strain_of_visit is None else strain_of_visit[i * self.Fc:(i + 1) * self.Fc]
                eng.screen_fields(images[p0:p0 + self.Fc], labels[p0:p0 + self.Fc], self.max_label, o,
                                  field_strain=st, acc=self.acc)

    def run_images_device(self, seg: torch.Tensor, images: torch.Tensor, n_fields: int, prob_thresh: float,
                          nms_thresh: float, strain_of_visit: torch.Tensor | None = None):
        """``run_device`` with the labels made on the device: each chunk is segmented from ``seg`` (uint16 viewed
        as int16 [P,H,W]; may be ``images``) and screened on ``images`` in one ``cia_screen_images`` call."""
        P = images.shape[0]
        assert P % self.Fc == 0 and seg.shape == images.shape
        eng = self.eng
        with torch.cuda.stream(self.compute):
            if self._stage is not None:
                for e in self._stage["out_free"]:
                    self.compute.wait_event(e)
            for i in range(-(-n_fields // self.Fc)):        # the last chunk may be short
                p0 = (i * self.Fc) % P
                nf = min(self.Fc, n_fields - i * self.Fc)
                o = self.out[i & 1]
                st = None if strain_of_visit is None else strain_of_visit[i * self.Fc:i * self.Fc + nf]
                eng.screen_images(seg[p0:p0 + nf], images[p0:p0 + nf], self.max_label, o, prob_thresh,
                                  nms_thresh, field_strain=st, acc=self.acc)

    # ---- host-resident pass (H2D + D2H inside) ----
    def _ensure_stage(self, n_chunks):
        d = self.eng.tdev
        if self._stage is None:
            self._stage = dict(
                img=[torch.empty((self.Fc, self.H, self.W), dtype=torch.int16, device=d) for _ in range(self.NB)],
                lab=[torch.empty((self.Fc, self.H, self.W), dtype=torch.int32, device=d) for _ in range(self.NB)],
                ready=[torch.cuda.Event() for _ in range(self.NB)],
                done=[torch.cuda.Event() for _ in range(self.NB)],
                out_ready=[torch.cuda.Event() for _ in range(self.NB)],
                out_free=[torch.cuda.Event() for _ in range(self.NB)])
            if self.label_transport == "rle":
                sw = self.eng.rle_slot_words(self.H, self.W)
                self._stage.update(
                    h_rle=[torch.empty((self.Fc, sw), dtype=torch.int32, pin_memory=True) for _ in range(self.NB)],
                    d_rle=[torch.empty((self.Fc, sw), dtype=torch.int32, device=d) for _ in range(self.NB)],
                    words=[np.zeros(self.Fc, np.uint32) for _ in range(self.NB)])
                if self.image_transport == "patches" and self.scan_runs:
                    cap_px = self.H * self.W // 2          # a field whose bbox rectangles exceed half its pixels goes densely
                    self._stage.update(
                        h_patch=[torch.empty((self.Fc, cap_px), dtype=torch.int16, pin_memory=True) for _ in range(self.NB)],
                        d_patch=[torch.empty((self.Fc, cap_px), dtype=torch.int16, device=d) for _ in range(self.NB)],
                        patch_px=[np.zeros(self.Fc, np.uint32) for _ in range(self.NB)])
        if getattr(self, "_host_chunks", 0) < n_chunks:
            cap = self.cap
            pin = dict(pin_memory=True)
            self.h_cells = torch.empty((n_chunks, cap, 56), dtype=torch.uint8, **pin)
            self.h_counts = torch.empty((n_chunks, 1 + self.Fc), dtype=torch.int32, **pin)
            self.h_mse = torch.empty((n_chunks, cap), dtype=torch.float32, **pin)
            self.h_mae = torch.empty((n_chunks, cap), dtype=torch.float32, **pin)
            self.h_dc = torch.empty((n_chunks, cap), dtype=torch.float64, **pin)
            self.h_dm = torch.empty((n_chunks, cap), dtype=torch.float64, **pin)
            self.h_pc = torch.empty((n_chunks, cap), dtype=torch.int8, **pin)
            self.h_pm = torch.empty((n_chunks, cap), dtype=torch.int8, **pin)
            self._host_chunks = n_chunks

    def host_bytes_per_pass(self, n_fields):
        """(H2D, D2H) bytes of one ``run_host`` pass; H2D is what the last pass actually sent."""
        n_chunks = n_fields // self.Fc
        h2d = getattr(self, "h2d_bytes", 0) or n_fields * self.H * self.W * 6
        per_chunk = self.cap * (56 + 4 + 4 + 8 + 8 + 1 + 1) + 4 * (1 + self.Fc)
        return h2d, n_chunks * per_chunk + self.n_strains * 64

    def run_host(self, images_pinned: torch.Tensor, labels_pinned: torch.Tensor, n_fields: int,
                 strain_of_visit: torch.Tensor | None = None):
        """One pass over ``n_fields`` field visits read from pinned host pools [P,H,W]
        (int16-viewed uint16 image, int32 labels).  Enqueues copies + compute; call
        ``collect_host`` (after a stream sync) for the results."""
        P = images_pinned.shape[0]
        assert P % self.Fc == 0 and n_fields % self.Fc == 0
        n_chunks = n_fields // self.Fc
        self._ensure_stage(n_chunks)
        S, eng = self._stage, self.eng
        px = self.Fc * self.H * self.W
        self.h2d_bytes = 0
        self.encode_seconds = 0.0          # host time spent inside the run-length encoder this pass
        n_rle = 0
        for i in range(n_chunks):
            b = i % self.NB
            p0 = (i * self.Fc) % P
            f = self.rle_fraction
            rle = self.label_transport == "rle" and int((i + 1) * f) > int(i * f)
            use_patches = rle and "h_patch" in S
            patches_ok = False
            if not use_patches:
                with torch.cuda.stream(self.copy):
                    self.copy.wait_event(S["done"][b])
                    S["img"][b].copy_(images_pinned[p0:p0 + self.Fc], non_blocking=True)
            if rle:
                # the host encodes chunk i while the device works on chunk i-1; the staging buffers are reused
                # only after their previous upload (chunk i-NB)
                S["ready"][b].synchronize()
                t0 = time.perf_counter()
                if use_patches:
                    rle, patches_ok = eng.rle_encode_pack(labels_pinned[p0:p0 + self.Fc], images_pinned[p0:p0 + self.Fc],
                                                          S["h_rle"][b], S["words"][b], self.max_label, S["h_patch"][b],
                                                          S["patch_px"][b], self.host_threads)
                else:
                    rle = eng.rle_encode(labels_pinned[p0:p0 + self.Fc], S["h_rle"][b], S["words"][b],
                                         self.host_threads)
                self.encode_seconds += time.perf_counter() - t0
            with torch.cuda.stream(self.copy):
                if use_patches:
                    self.copy.wait_event(S["done"][b])
                    if rle and patches_ok:
                        eng.patch_upload(S["h_patch"][b], S["patch_px"][b], S["d_patch"][b])
                        self.h2d_bytes += 2 * int(S["patch_px"][b].sum())
                    else:
                        patches_ok = False
                        S["img"][b].copy_(images_pinned[p0:p0 + self.Fc], non_blocking=True)
                        self.h2d_bytes += 2 * px
                else:
                    self.h2d_bytes += 2 * px
                if rle:
                    n_rle += 1
                    if self.scan_runs:
                        eng.rle_upload(S["h_rle"][b], S["words"][b], S["d_rle"][b])
                    else:
                        eng.rle_upload_expand(S["h_rle"][b], S["words"][b], S["d_rle"][b], S["lab"][b])
                    self.h2d_bytes += 4 * int(S["words"][b].sum())
                else:
                    S["lab"][b].copy_(labels_pinned[p0:p0 + self.Fc], non_blocking=True)
                    self.h2d_bytes += 4 * px
                S["ready"][b].record(self.copy)
            with torch.cuda.stream(self.compute):
                self.compute.wait_event(S["ready"][b])
                self.compute.wait_event(S["out_free"][b])       # chunk i-2's results have been read back
                o = self.out[b]
                st = None if strain_of_visit is None else strain_of_visit[i * self.Fc:(i + 1) * self.Fc]
                eng.screen_fields(S["img"][b], S["lab"][b], self.max_label, o, field_strain=st, acc=self.acc,
                                  rle_slots=S["d_rle"][b] if rle and self.scan_runs else None,
                                  patches=S["d_patch"][b] if use_patches and patches_ok else None)
                S["done"][b].record(self.compute)
                S["out_ready"][b].record(self.compute)
            self._read_back(i, b, o)
        self._last_chunks = n_chunks
        self._last_fields = n_fields
        self.last_rle_share = n_rle / max(n_chunks, 1)        # share of the chunks that crossed PCIe as runs

    def _read_back(self, i, b, o):
        """D2H of chunk i's results (device buffer set b) on the read-back stream"""
        S = self._stage
        with torch.cuda.stream(self.d2h):
            self.d2h.wait_event(S["out_ready"][b])
            self.h_counts[i].copy_(o["counts"], non_blocking=True)
            self.h_cells[i].copy_(o["cells"], non_blocking=True)
            self.h_mse[i].copy_(o["mse"], non_blocking=True)
            self.h_mae[i].copy_(o["mae"], non_blocking=True)
            self.h_dc[i].copy_(o["dec_cons"], non_blocking=True)
            self.h_dm[i].copy_(o["dec_mod"], non_blocking=True)
            self.h_pc[i].copy_(o["pred_cons"], non_blocking=True)
            self.h_pm[i].copy_(o["pred_mod"], non_blocking=True)
            S["out_free"][b].record(self.d2h)

    def run_images_host(self, seg_pinned: torch.Tensor, images_pinned: torch.Tensor, n_fields: int, prob_thresh: float,
                        nms_thresh: float, strain_of_visit: torch.Tensor | None = None):
        """``run_host`` with the labels made on the device: only images cross PCIe -- one buffer per chunk when
        ``seg_pinned`` is ``images_pinned`` (single-channel fields), two when the segmentation channel differs.
        Same chunking, double buffering, read-back and ``collect_host`` as ``run_host``."""
        P = images_pinned.shape[0]
        assert P % self.Fc == 0 and seg_pinned.shape == images_pinned.shape
        n_chunks = -(-n_fields // self.Fc)          # the last chunk may be short
        self._ensure_stage(n_chunks)
        S, eng = self._stage, self.eng
        same = seg_pinned is images_pinned
        if not same and "seg" not in S:
            S["seg"] = [torch.empty((self.Fc, self.H, self.W), dtype=torch.int16, device=eng.tdev) for _ in range(self.NB)]
        self.h2d_bytes = 0
        for i in range(n_chunks):
            b = i % self.NB
            p0 = (i * self.Fc) % P
            nf = min(self.Fc, n_fields - i * self.Fc)
            with torch.cuda.stream(self.copy):
                self.copy.wait_event(S["done"][b])
                S["img"][b][:nf].copy_(images_pinned[p0:p0 + nf], non_blocking=True)
                if not same:
                    S["seg"][b][:nf].copy_(seg_pinned[p0:p0 + nf], non_blocking=True)
                self.h2d_bytes += (1 if same else 2) * 2 * nf * self.H * self.W
                S["ready"][b].record(self.copy)
            with torch.cuda.stream(self.compute):
                self.compute.wait_event(S["ready"][b])
                self.compute.wait_event(S["out_free"][b])
                o = self.out[b]
                o["counts"][1 + nf:].zero_()            # per-field counts of the fields a short chunk does not have
                st = None if strain_of_visit is None else strain_of_visit[i * self.Fc:i * self.Fc + nf]
                eng.screen_images((S["img"][b] if same else S["seg"][b])[:nf], S["img"][b][:nf], self.max_label, o,
                                  prob_thresh, nms_thresh, field_strain=st, acc=self.acc)
                S["done"][b].record(self.compute)
                S["out_ready"][b].record(self.compute)
            self._read_back(i, b, o)
        self._last_chunks = n_chunks
        self._last_fields = n_fields

    def collect_host(self):
        """Compact the per-chunk host buffers of the last ``run_host`` into flat arrays.  Raises if
        a kernel of the pass reported a capacity overflow, an out-of-range label or an unsupported
        bbox (nothing is truncated silently)."""
        self.sync()
        n_chunks = self._last_chunks
        counts = self.h_counts[:n_chunks].numpy()
        if (counts[:, 0] > self.cap).any():
            raise _lib.CiaError(_lib.CIA_E_CAPACITY, f"a chunk produced {int(counts[:, 0].max())} cells, capacity "
                                f"{self.cap} (raise cells_per_field_cap)")
        ks = counts[:, 0]
        cat = lambda t: np.concatenate([t[i, :ks[i]].numpy() for i in range(n_chunks)])
        cells = np.concatenate([self.h_cells[i, :ks[i]].numpy().view(_lib.CELL_DTYPE).reshape(-1)
                                for i in range(n_chunks)])
        chunk_of = np.repeat(np.arange(n_chunks), ks)
        cells = cells.copy()
        cells["field"] += chunk_of.astype(np.int32) * self.Fc      # visit index within the pass
        return dict(n_cells=int(ks.sum()), field_counts=counts[:, 1:].reshape(-1)[:self._last_fields], cells=cells,
                    mse=cat(self.h_mse), mae=cat(self.h_mae), dec_cons=cat(self.h_dc),
                    dec_mod=cat(self.h_dm), pred_cons=cat(self.h_pc), pred_mod=cat(self.h_pm))

    def sync(self):
        """Wait for every stream of the pass and raise on a device-side status (CIA_E_CAPACITY /
        _LABEL / _UNSUPPORTED) raised by any of its kernels."""
        self.copy.synchronize()
        self.d2h.synchronize()
        self.eng.check_status(self.compute)
