"""Host side of the drop-in: mirrors ``ProductionMutantScreening``
(improved_detection.py:18-244) method for method, with every computation of the hot
path done by libcia.so on the GPU.  PyTorch is used only for device buffers, streams
and (in ``distributed.py``) the process group.

There is no CPU fallback: constructing ``Engine`` without a CUDA device or without
the built library raises.
"""
from __future__ import annotations

import ctypes as C
import os
from glob import glob

import numpy as np
import torch

from . import _lib
from .artifacts import load_model_dir

PRECISION_FP32 = 0
PRECISION_TC = 1


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _np_ptr(a):
    return C.c_void_p(a.ctypes.data) if a is not None else C.c_void_p(0)


class Engine:
    """Owns a libcia handle on one GPU and the uploaded artifacts."""

    def __init__(self, device: int = 0, precision: int = PRECISION_TC):
        if not torch.cuda.is_available():
            raise RuntimeError("cell_image_analysis_b200 needs a CUDA device (sm_100a); no CPU fallback")
        self.lib = _lib.load()
        self.device = int(device)
        self.tdev = torch.device("cuda", self.device)
        torch.cuda.set_device(self.device)
        torch.zeros(1, device=self.tdev)          # make sure the primary context exists
        h = C.c_void_p()
        rc = self.lib.cia_create(self.device, C.byref(h))
        if rc != 0:
            raise _lib.CiaError(rc, "cia_create failed")
        self.h = h
        self.params = _lib.default_params()
        self.precision = precision
        self._options = {}                        # cia_set_option values set through this object
        self.n_features = 2048
        self.n_components = None

    def close(self):
        if getattr(self, "h", None):
            self.lib.cia_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- helpers ----
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.tdev).cuda_stream)

    def _check(self, rc):
        _lib.check(self.h, rc)

    def check_status(self, stream=None):
        """Raise if a kernel reported CIA_E_CAPACITY / _LABEL / _UNSUPPORTED since the last check
        (synchronises ``stream``, default torch's current stream)."""
        s = self._stream() if stream is None else C.c_void_p(stream.cuda_stream)
        self._check(self.lib.cia_check_status(self.h, s))

    def set_option(self, name: str, value: float):
        self._check(self.lib.cia_set_option(self.h, name.encode(), float(value)))
        self._options[name] = value

    @property
    def launch_count(self) -> int:
        return int(self.lib.cia_launch_count(self.h))

    # ---- artifacts ----
    def load_artifacts(self, arts: dict):
        def cae(which, w):
            n = w["n_conv"]
            ks = [np.ascontiguousarray(k, np.float32) for k in w["kernels"]]
            bs = [np.ascontiguousarray(b, np.float32) for b in w["biases"]]
            bn = [np.ascontiguousarray(a, np.float32) for t in w["bns"] for a in t]
            K = (C.c_void_p * n)(*[k.ctypes.data for k in ks])
            B = (C.c_void_p * n)(*[b.ctypes.data for b in bs])
            N = (C.c_void_p * max(len(bn), 1))(*[a.ctypes.data for a in bn])
            self._check(self.lib.cia_load_cae(self.h, which, n, K, B, N, C.c_float(w["bn_eps"])))
        cae(0, arts["autoencoder"])
        self.encoder_separate = not arts.get("encoder_same", True)
        if self.encoder_separate:
            cae(1, arts["encoder"])
        sp = arts["scaler_pca"]
        self._check(self.lib.cia_load_scaler_pca(
            self.h, sp["F"], sp["C"], _np_ptr(sp["center"]), _np_ptr(sp["scale"]),
            int(sp["center_is_f32"]), _np_ptr(sp["components"]), _np_ptr(sp["offset"]),
            int(sp["f32_flow"])))
        self.n_features, self.n_components = sp["F"], sp["C"]
        for which, key in ((0, "svm_conservative"), (1, "svm_moderate")):
            m = arts[key]
            self._check(self.lib.cia_load_svm(self.h, which, m["sv"].shape[0], m["sv"].shape[1],
                                              _np_ptr(m["sv"]), _np_ptr(m["coef"]),
                                              C.c_double(m["gamma"]), C.c_double(m["rho"])))

    # ---- stages (device tensors in / out) ----
    def label_scan(self, labels: torch.Tensor, max_label: int) -> torch.Tensor:
        """labels int32 [F,H,W] (cuda) -> uint8 tensor viewable as REGION_DTYPE [F, max_label]."""
        F, H, W = labels.shape
        regions = torch.empty((F, max_label, 64), dtype=torch.uint8, device=self.tdev)
        self._check(self.lib.cia_label_scan(self.h, _ptr(labels), F, H, W, max_label, _ptr(regions),
                                            self._stream()))
        return regions

    def filter(self, images: torch.Tensor, regions: torch.Tensor, cells_cap: int):
        F, H, W = images.shape
        max_label = regions.shape[1]
        cells = torch.empty((max(cells_cap, 1), 56), dtype=torch.uint8, device=self.tdev)
        counts = torch.zeros(1 + F, dtype=torch.int32, device=self.tdev)
        self._check(self.lib.cia_filter(self.h, _ptr(images), F, H, W, max_label, _ptr(regions),
                                        C.byref(self.params), _ptr(cells), cells_cap, _ptr(counts),
                                        C.c_void_p(counts.data_ptr() + 4), self._stream()))
        return cells, counts

    def solidity(self, labels: torch.Tensor, cells: torch.Tensor, n: int) -> torch.Tensor:
        """prop.solidity (det:106) of the first ``n`` cells; labels int32 [F,H,W] (cuda)."""
        F, H, W = labels.shape
        out = torch.empty(max(n, 1), dtype=torch.float64, device=self.tdev)
        self._check(self.lib.cia_solidity(self.h, _ptr(labels), H, W, _ptr(cells), n, None, _ptr(out), self._stream()))
        return out

    def crop_resize(self, images: torch.Tensor, cells: torch.Tensor, n: int, n_dev=None,
                    want64: bool = False, params=None):
        F, H, W = images.shape
        c32 = torch.empty((max(n, 1), 64, 64), dtype=torch.float32, device=self.tdev)
        c64 = torch.empty((max(n, 1), 64, 64), dtype=torch.float64, device=self.tdev) if want64 else None
        self._check(self.lib.cia_crop_resize(self.h, _ptr(images), H, W, _ptr(cells), n, _ptr(n_dev),
                                             C.byref(params or self.params), _ptr(c32), _ptr(c64), self._stream()))
        return c32, c64

    def debug_clahe_levels(self, images: torch.Tensor, cells: torch.Tensor, n: int, sizes):
        """Test tap: uint16 CLAHE levels (before the [0,1] rescale) of each cell, flattened."""
        F, H, W = images.shape
        offs = np.concatenate([[0], np.cumsum(np.asarray(sizes, np.int64))])
        off_t = torch.from_numpy(offs[:-1].copy()).to(self.tdev)
        lv = torch.zeros(int(offs[-1]) + 1, dtype=torch.int16, device=self.tdev)
        c32 = torch.empty((max(n, 1), 64, 64), dtype=torch.float32, device=self.tdev)
        self._check(self.lib.cia_debug_clahe_levels(self.h, _ptr(images), H, W, _ptr(cells), n,
                                                    C.byref(self.params), _ptr(c32), _ptr(lv),
                                                    _ptr(off_t), self._stream()))
        self.check_status()
        return lv[:-1].cpu().numpy().view(np.uint16), offs

    def cae_forward(self, crops32: torch.Tensor, n: int, n_dev=None, precision=None):
        mse = torch.empty(max(n, 1), dtype=torch.float32, device=self.tdev)
        mae = torch.empty(max(n, 1), dtype=torch.float32, device=self.tdev)
        feat = torch.empty((max(n, 1), 2048), dtype=torch.float32, device=self.tdev)
        prec = self.precision if precision is None else precision
        self._check(self.lib.cia_cae_forward(self.h, _ptr(crops32), n, _ptr(n_dev), _ptr(mse), _ptr(mae),
                                             _ptr(feat), prec, self._stream()))
        return mse, mae, feat

    def svm_decision(self, feat: torch.Tensor, n: int, n_dev=None, want_pca: bool = False, precision=None):
        """Scaler -> PCA -> both detectors.  ``precision`` 0 (the exact anchor, like ``cae_forward``'s) runs the
        fp64 DMMA kernels whatever the ``svm_kernel`` / ``pca_kernel`` options say; anything else follows them
        (default: the tcgen05 kernels)."""
        prec = self.precision if precision is None else precision
        if prec == 0:
            saved = {k: self._options.get(k, 1) for k in ("svm_kernel", "pca_kernel")}
            for k in saved:
                self._check(self.lib.cia_set_option(self.h, k.encode(), 0.0))
            try:
                return self._svm_decision(feat, n, n_dev, want_pca)
            finally:
                for k, v in saved.items():
                    self._check(self.lib.cia_set_option(self.h, k.encode(), float(v)))
        return self._svm_decision(feat, n, n_dev, want_pca)

    def _svm_decision(self, feat: torch.Tensor, n: int, n_dev=None, want_pca: bool = False):
        dc = torch.empty(max(n, 1), dtype=torch.float64, device=self.tdev)
        dm = torch.empty(max(n, 1), dtype=torch.float64, device=self.tdev)
        pc = torch.empty(max(n, 1), dtype=torch.int8, device=self.tdev)
        pm = torch.empty(max(n, 1), dtype=torch.int8, device=self.tdev)
        z = torch.empty((max(n, 1), self.n_components), dtype=torch.float64, device=self.tdev) if want_pca else None
        self._check(self.lib.cia_svm_decision(self.h, _ptr(feat), n, _ptr(n_dev), _ptr(dc), _ptr(dm),
                                              _ptr(pc), _ptr(pm), _ptr(z), self._stream()))
        return dc, dm, pc, pm, z

    # ---- run-length label transport (csrc/transport.cu) ----
    def rle_slot_words(self, H: int, W: int) -> int:
        return int(self.lib.cia_rle_slot_words(H, W))

    def rle_encode(self, labels_host: torch.Tensor, slots_host: torch.Tensor, field_words: np.ndarray,
                   threads: int = 0) -> bool:
        """Encode int32 host labels [F,H,W] into ``slots_host`` [F, slot_words] (int32-viewed
        words).  Returns False if a field does not fit its slot (caller sends raw labels)."""
        F, H, W = labels_host.shape
        rc = self.lib.cia_rle_encode_fields(labels_host.data_ptr(), F, H, W, slots_host.data_ptr(),
                                            slots_host.shape[1], field_words.ctypes.data, None, threads)
        if rc == _lib.CIA_E_CAPACITY:
            return False
        if rc != 0:
            raise _lib.CiaError(rc, "cia_rle_encode_fields failed")
        return True

    def rle_encode_pack(self, labels_host: torch.Tensor, images_host: torch.Tensor, slots_host: torch.Tensor,
                        field_words: np.ndarray, label_cap: int, patches_host: torch.Tensor, patch_px: np.ndarray,
                        threads: int = 0):
        """``rle_encode`` + the patch transport of the image: the thread that encoded a field also packs the
        bbox rectangles of its labels from ``images_host`` [F,H,W] (int16-viewed uint16) into ``patches_host``
        [F, patch_cap_px].  Returns (labels_ok, patches_ok): False where a field did not fit its slot."""
        F, H, W = labels_host.shape
        rc = self.lib.cia_rle_encode_pack_fields(labels_host.data_ptr(), images_host.data_ptr(), F, H, W,
                                                 slots_host.data_ptr(), slots_host.shape[1], field_words.ctypes.data,
                                                 None, int(label_cap), patches_host.data_ptr(), patches_host.shape[1],
                                                 patch_px.ctypes.data, threads)
        if rc == _lib.CIA_E_CAPACITY:
            return False, False
        if rc != 0:
            raise _lib.CiaError(rc, "cia_rle_encode_pack_fields failed")
        return True, bool((patch_px != 0xFFFFFFFF).all())

    def patch_upload(self, patches_host: torch.Tensor, patch_px: np.ndarray, patches_dev: torch.Tensor):
        """Async: copy the used pixels of every field's patch slot."""
        F, cap = patches_host.shape
        self._check(self.lib.cia_patch_upload(self.h, patches_host.data_ptr(), F, cap, patch_px.ctypes.data,
                                              patches_dev.data_ptr(), self._stream()))

    def rle_upload_expand(self, slots_host: torch.Tensor, field_words: np.ndarray, slots_dev: torch.Tensor,
                          labels_dev: torch.Tensor):
        """Async: copy the used words of every slot and expand to dense int32 labels [F,H,W]."""
        F, H, W = labels_dev.shape
        sw = slots_host.shape[1]
        self._check(self.lib.cia_rle_upload(self.h, slots_host.data_ptr(), F, sw, field_words.ctypes.data,
                                            slots_dev.data_ptr(), self._stream()))
        self._check(self.lib.cia_rle_expand(self.h, slots_dev.data_ptr(), F, sw, H, W, labels_dev.data_ptr(),
                                            self._stream()))

    def rle_upload(self, slots_host: torch.Tensor, field_words: np.ndarray, slots_dev: torch.Tensor):
        """Async: copy the used words of every slot (no expansion: ``label_scan_rle`` /
        ``screen_fields(rle_slots=...)`` read the runs themselves)."""
        F, sw = slots_host.shape
        self._check(self.lib.cia_rle_upload(self.h, slots_host.data_ptr(), F, sw, field_words.ctypes.data,
                                            slots_dev.data_ptr(), self._stream()))

    def label_scan_rle(self, slots_dev: torch.Tensor, H: int, W: int, max_label: int) -> torch.Tensor:
        """``label_scan`` from run-length encoded fields [F, slot_words] (int32-viewed words)."""
        F, sw = slots_dev.shape
        regions = torch.empty((F, max_label, 64), dtype=torch.uint8, device=self.tdev)
        self._check(self.lib.cia_label_scan_rle(self.h, _ptr(slots_dev), sw, F, H, W, max_label, _ptr(regions),
                                                self._stream()))
        return regions

    # ---- fused path ----
    def alloc_outputs(self, cells_cap: int, n_fields: int, keep_crops=False, keep_features=False):
        d = self.tdev
        out = dict(
            cells=torch.empty((cells_cap, 56), dtype=torch.uint8, device=d),
            counts=torch.zeros(1 + n_fields, dtype=torch.int32, device=d),
            mse=torch.empty(cells_cap, dtype=torch.float32, device=d),
            mae=torch.empty(cells_cap, dtype=torch.float32, device=d),
            dec_cons=torch.empty(cells_cap, dtype=torch.float64, device=d),
            dec_mod=torch.empty(cells_cap, dtype=torch.float64, device=d),
            pred_cons=torch.empty(cells_cap, dtype=torch.int8, device=d),
            pred_mod=torch.empty(cells_cap, dtype=torch.int8, device=d),
            crops=torch.empty((cells_cap, 64, 64), dtype=torch.float32, device=d) if keep_crops else None,
            features=torch.empty((cells_cap, 2048), dtype=torch.float32, device=d) if keep_features else None,
        )
        out["cap"] = cells_cap
        return out

    def _scores(self, out):
        return _lib.Scores(out["mse"].data_ptr(), out["mae"].data_ptr(), out["dec_cons"].data_ptr(),
                           out["dec_mod"].data_ptr(), out["pred_cons"].data_ptr(),
                           out["pred_mod"].data_ptr())

    def screen_fields(self, images: torch.Tensor, labels: torch.Tensor, max_label: int, out: dict,
                      field_strain: torch.Tensor = None, acc: torch.Tensor = None, precision=None,
                      rle_slots: torch.Tensor = None, patches: torch.Tensor = None):
        """Enqueue the whole path for device-resident fields (no host sync).  With ``rle_slots``
        ([F, slot_words] device words of the run-length transport) ``labels`` is ignored and the
        region scan runs on the runs themselves.  With ``patches`` as well ([F, patch_cap_px] device pixels of
        the patch transport) ``images`` is a dense SCRATCH buffer the bbox rectangles are scattered into."""
        F, H, W = images.shape
        sc = self._scores(out)
        prec = self.precision if precision is None else precision
        ns = 0 if acc is None else acc.shape[0]
        if rle_slots is not None and patches is not None:
            self._check(self.lib.cia_screen_fields_rle_patches(
                self.h, _ptr(images), _ptr(patches), patches.shape[1], _ptr(rle_slots), rle_slots.shape[1], F, H, W,
                max_label, C.byref(self.params), prec, _ptr(out["cells"]), out["cap"], _ptr(out["counts"]),
                C.c_void_p(out["counts"].data_ptr() + 4), C.byref(sc), _ptr(out["crops"]),
                _ptr(out["features"]), _ptr(field_strain), _ptr(acc), ns, self._stream()))
            return
        if rle_slots is not None:
            self._check(self.lib.cia_screen_fields_rle(
                self.h, _ptr(images), _ptr(rle_slots), rle_slots.shape[1], F, H, W, max_label,
                C.byref(self.params), prec, _ptr(out["cells"]), out["cap"], _ptr(out["counts"]),
                C.c_void_p(out["counts"].data_ptr() + 4), C.byref(sc), _ptr(out["crops"]),
                _ptr(out["features"]), _ptr(field_strain), _ptr(acc), ns, self._stream()))
            return
        self._check(self.lib.cia_screen_fields(
            self.h, _ptr(images), _ptr(labels), F, H, W, max_label, C.byref(self.params), prec,
            _ptr(out["cells"]), out["cap"], _ptr(out["counts"]), C.c_void_p(out["counts"].data_ptr() + 4),
            C.byref(sc), _ptr(out["crops"]), _ptr(out["features"]), _ptr(field_strain), _ptr(acc), ns,
            self._stream()))

    def screen_images(self, seg_images: torch.Tensor, images: torch.Tensor, max_label: int, out: dict,
                      prob_thresh: float, nms_thresh: float, n_instances: torch.Tensor = None,
                      labels_out: torch.Tensor = None, field_strain: torch.Tensor = None, acc: torch.Tensor = None,
                      precision=None):
        """``screen_fields`` with the labels made on the device from ``seg_images`` (uint16 [F, H, W], may be
        ``images`` itself): batched StarDist segmentation (needs ``cia_seg_load``) then the fused path, no host
        sync.  ``n_instances`` int32 [F] and ``labels_out`` int32 [F, H, W] are optional device outputs."""
        F, H, W = images.shape
        if tuple(seg_images.shape) != (F, H, W):
            raise ValueError(f"seg_images {tuple(seg_images.shape)} and images {(F, H, W)} differ in shape")
        sc = self._scores(out)
        prec = self.precision if precision is None else precision
        ns = 0 if acc is None else acc.shape[0]
        self._check(self.lib.cia_screen_images(
            self.h, _ptr(seg_images), _ptr(images), F, H, W, float(prob_thresh), float(nms_thresh), max_label,
            C.byref(self.params), prec, _ptr(out["cells"]), out["cap"], _ptr(out["counts"]),
            C.c_void_p(out["counts"].data_ptr() + 4), C.byref(sc), _ptr(out["crops"]), _ptr(out["features"]),
            _ptr(field_strain), _ptr(acc), ns, _ptr(n_instances), _ptr(labels_out), self._stream()))

    def screen_fields_host(self, images: np.ndarray, labels: np.ndarray, max_label: int,
                           cells_cap: int, precision=None):
        """Host buffers in, host results out (H2D + D2H inside the call; synchronises)."""
        F, H, W = images.shape
        assert images.dtype == np.uint16 and labels.dtype == np.int32
        assert images.flags.c_contiguous and labels.flags.c_contiguous
        cells = np.empty(cells_cap, _lib.CELL_DTYPE)
        n = np.zeros(1, np.int32)
        fc = np.zeros(F, np.int32)
        res = dict(mse=np.empty(cells_cap, np.float32), mae=np.empty(cells_cap, np.float32),
                   dec_cons=np.empty(cells_cap, np.float64), dec_mod=np.empty(cells_cap, np.float64),
                   pred_cons=np.empty(cells_cap, np.int8), pred_mod=np.empty(cells_cap, np.int8))
        sc = _lib.Scores(res["mse"].ctypes.data, res["mae"].ctypes.data, res["dec_cons"].ctypes.data,
                         res["dec_mod"].ctypes.data, res["pred_cons"].ctypes.data,
                         res["pred_mod"].ctypes.data)
        prec = self.precision if precision is None else precision
        self._check(self.lib.cia_screen_fields_host(
            self.h, _np_ptr(images), _np_ptr(labels), F, H, W, max_label, C.byref(self.params), prec,
            _np_ptr(cells), cells_cap, _np_ptr(n), _np_ptr(fc), C.byref(sc), self._stream()))
        k = int(n[0])
        res = {key: v[:k] for key, v in res.items()}
        res.update(cells=cells[:k], n_cells=k, field_counts=fc)
        return res


def _default_imread(path):
    """tiff.imread (det:51): tifffile when installed, else the in-tree baseline-TIFF reader
    (uncompressed strips), else OpenCV's decoder with the file's channel order restored.
    Upstream of the hot path (SURVEY N1)."""
    try:
        import tifffile
        return tifffile.imread(path)
    except ImportError:
        pass
    from .tiff_min import TiffError, read_tiff
    try:
        return read_tiff(path)
    except TiffError:
        import cv2
        img = cv2.imread(path, cv2.IMREAD_UNCHANGED)
        if img is None:
            raise IOError(f"cannot read {path}")
        if img.ndim == 3 and img.shape[-1] >= 3:
            img = img[..., ::-1] if img.shape[-1] == 3 else img[..., [2, 1, 0, 3]]
        return img


class UnsupportedImageError(TypeError):
    """The analysis channel has a dtype the CUDA path does not take (anything but 8- / 16-bit
    unsigned).  Raised THROUGH the catch-all of ``extract_quality_cells`` (det:113-115) so that
    such a file is not silently counted as "0 cells"."""


class ProductionMutantScreening:
    """Drop-in for the reference class of the same name (improved_detection.py:18).

    Differences, all at the edge of the hot path:
      * ``segmenter``: callable ``seg_channel -> int32 labels`` standing in for
        csbdeep ``normalize`` + ``StarDist2D.predict_instances`` (det:44, 62-63), which
        need a network download and are out of scope (SURVEY C9).  When omitted,
        StarDist is imported lazily on the first ``extract_quality_cells`` call.
      * ``extract_quality_cells_from_labels(green, labels)`` is the seam the CUDA path
        implements (det:66-111).
    """

    def __init__(self, model_dir, segmenter=None, imread=None, device: int = 0,
                 precision: int = PRECISION_TC, stardist_dir=None):
        self.model_dir = model_dir
        self.segmenter = segmenter
        self.imread = imread or _default_imread
        self.engine = Engine(device=device, precision=precision)
        self.stardist_model = None
        self.load_trained_models()
        if stardist_dir is not None and segmenter is None:
            # det:44 on the GPU (csrc/segment.cu): a StarDist model folder instead of the download; the labels of
            # det:62-63 stay on the device and feed the region scan without crossing PCIe
            from .stardist import StarDist2D
            self.stardist_model = StarDist2D(None, name=os.path.basename(os.path.normpath(stardist_dir)),
                                             basedir=os.path.dirname(os.path.normpath(stardist_dir)) or ".",
                                             engine=self.engine)
            self.segmenter = lambda ch: self.stardist_model.segment_device(ch)[0]

    # det:23-46
    def load_trained_models(self):
        print("Loading trained models...")
        self.artifacts = load_model_dir(self.model_dir)
        self.engine.load_artifacts(self.artifacts)
        sk = self.artifacts["sklearn"]
        self.scaler, self.pca = sk["scaler"], sk["pca"]
        self.detector_conservative = sk["detector_conservative"]
        self.detector_moderate = sk["detector_moderate"]
        print("All models loaded successfully!")

    def _segment(self, seg_channel):
        if self.segmenter is None:
            from csbdeep.utils import normalize                 # det:7
            from stardist.models import StarDist2D              # det:6
            model = StarDist2D.from_pretrained("2D_versatile_fluo")   # det:44
            self.segmenter = lambda ch: model.predict_instances(normalize(ch))[0]   # det:62-63
        return self.segmenter(seg_channel)

    # det:48-115
    def extract_quality_cells(self, image_path):
        try:
            image = self.imread(image_path)
            if image.ndim == 3 and image.shape[-1] >= 3:        # det:54-59
                seg_channel = image[..., 2]
                green_channel = image[..., 1]
            else:
                seg_channel = image
                green_channel = image
            labels = self._segment(seg_channel)
            return self.extract_quality_cells_from_labels(green_channel, labels)
        except UnsupportedImageError:
            raise
        except Exception as e:                                   # det:113-115
            print(f"Error processing {image_path}: {e}")
            return [], []

    # det:66-111
    def extract_quality_cells_from_labels(self, green_channel, labels, return_regions=False):
        eng = self.engine
        green = np.ascontiguousarray(green_channel)
        params = self.engine.params
        if green.dtype == np.uint8:
            # 8-bit fields: same arithmetic on the widened values; only img_as_float's factor inside
            # equalize_adapthist (det:98) differs (1/255 instead of 1/65535)
            green = green.astype(np.uint16)
            params = _lib.default_params()
            C.memmove(C.byref(params), C.byref(self.engine.params), C.sizeof(params))
            params.intensity_inv = 1.0 / 255.0
        elif green.dtype != np.uint16:
            raise UnsupportedImageError(
                f"analysis channel dtype {green.dtype}: the CUDA path takes uint16 (16-bit TIFF fields) and "
                "uint8 images; convert float / signed images before screening")
        if isinstance(labels, torch.Tensor):          # device-resident labels (stardist.StarDist2D.segment_device)
            lab = labels.to(device=eng.tdev, dtype=torch.int32).contiguous()
            if tuple(lab.shape) != green.shape or lab.ndim != 2:
                raise ValueError("labels and image must be 2-D arrays of the same shape")
            max_label = int(lab.max().item()) if lab.numel() else 0
            l = lab[None]
        else:
            lab = np.ascontiguousarray(labels, dtype=np.int32)
            if lab.shape != green.shape or lab.ndim != 2:
                raise ValueError("labels and image must be 2-D arrays of the same shape")
            max_label = int(lab.max()) if lab.size else 0
            l = None
        if max_label <= 0:
            return ([], [], None) if return_regions else ([], [])
        g = torch.from_numpy(green.view(np.int16)).to(eng.tdev)[None]   # uint16 bytes; only the pointer is used
        if l is None:
            l = torch.from_numpy(lab).to(eng.tdev)[None]
        regions = eng.label_scan(l, max_label)
        cells, counts = eng.filter(g, regions, max_label)
        n = int(counts[0].item())
        eng.check_status()
        if n == 0:
            return ([], [], regions) if return_regions else ([], [])
        _c32, c64 = eng.crop_resize(g, cells, n, want64=True, params=params)
        sol = eng.solidity(l, cells, n)
        eng.check_status()
        crops = c64[:n].cpu().numpy()
        sol = sol[:n].cpu().numpy()
        rec = cells[:n].cpu().numpy().view(_lib.CELL_DTYPE).reshape(-1)
        quality_cells = [crops[i] for i in range(n)]
        cell_stats = [{"area": float(r["area"]), "eccentricity": float(r["eccentricity"]),
                       "solidity": float(sol[i]), "mean_intensity": float(r["mean_intensity"]),
                       "std_intensity": float(r["std_intensity"])} for i, r in enumerate(rec)]   # det:103-109
        if return_regions:
            return quality_cells, cell_stats, rec
        return quality_cells, cell_stats

    # det:117-153
    def compute_anomaly_scores(self, cell_images):
        if len(cell_images) == 0:
            return {}
        eng = self.engine
        X = np.expand_dims(np.array(cell_images), axis=-1).astype("float32")       # det:122
        n = X.shape[0]
        x = torch.from_numpy(np.ascontiguousarray(X[..., 0])).to(eng.tdev)
        mse, mae, feat = eng.cae_forward(x, n)
        dc, dm, pc, pm, _ = eng.svm_decision(feat, n)
        eng.check_status()
        cp = pc[:n].cpu().numpy().astype(np.intp)
        mp = pm[:n].cpu().numpy().astype(np.intp)
        return {
            "reconstruction_mse": mse[:n].cpu().numpy(),
            "reconstruction_mae": mae[:n].cpu().numpy(),
            "conservative_predictions": cp,
            "moderate_predictions": mp,
            "conservative_scores": -dc[:n].cpu().numpy(),        # det:149
            "moderate_scores": -dm[:n].cpu().numpy(),
            "conservative_anomaly_rate": np.sum(cp == -1) / len(cp),
            "moderate_anomaly_rate": np.sum(mp == -1) / len(mp),
        }

    # train:328-339 (the arithmetic; plots stay with the caller)
    def evaluate_reconstruction_quality(self, cell_images):
        r = self.compute_anomaly_scores(cell_images)
        return r["reconstruction_mse"], r["reconstruction_mae"]

    # train:398-402: encoder.predict + flatten, the features create_anomaly_detector fits on
    def encode_features(self, cell_images):
        if len(cell_images) == 0:
            return np.zeros((0, 2048), np.float32)
        eng = self.engine
        X = np.expand_dims(np.array(cell_images), axis=-1).astype("float32")
        x = torch.from_numpy(np.ascontiguousarray(X[..., 0])).to(eng.tdev)
        _mse, _mae, feat = eng.cae_forward(x, X.shape[0])
        eng.check_status()
        return feat[:X.shape[0]].cpu().numpy()

    # det:246-261: CSV files + text report (figures are presentation only and not produced)
    def save_and_visualize_results(self, results, detailed_results, output_dir):
        from .reporting import save_and_report
        return save_and_report(results, detailed_results, output_dir)

    # det:155-244
    def screen_mutant_samples(self, test_folders_dict, output_dir=None):
        if output_dir:
            os.makedirs(output_dir, exist_ok=True)
        print("=== Starting Mutant Screening with Improved Model ===")
        results, detailed_results = {}, []
        for sample_name, folder_path in test_folders_dict.items():
            print(f"\nProcessing {sample_name}...")
            tif_files = sorted(glob(os.path.join(folder_path, "*.tif")))
            if not tif_files:
                print(f"  No .tif files found in {folder_path}")
                continue
            sample_cells = []
            for file_path in tif_files:
                cells, _stats = self.extract_quality_cells(file_path)
                sample_cells.extend(cells)
                print(f"  {os.path.basename(file_path)}: {len(cells)} cells")
            print(f"  Total {sample_name} cells: {len(sample_cells)}")
            if len(sample_cells) == 0:
                print(f"  No quality cells extracted from {sample_name}")
                continue
            s = self.compute_anomaly_scores(sample_cells)
            results[sample_name] = summarize_sample(sample_name, len(tif_files), s)
            detailed_results.extend(detail_rows(sample_name, s))
        if output_dir:
            self.save_and_visualize_results(results, detailed_results, output_dir)      # det:242
        return results, detailed_results


    # det:155-244 over the ranks of a torch.distributed process group (one process per GPU)
    def screen_mutant_samples_sharded(self, test_folders_dict, output_dir=None, chunk_fields: int = 16):
        from .distributed import screen_mutant_samples_sharded
        return screen_mutant_samples_sharded(self, test_folders_dict, output_dir, chunk_fields)

    def screen_images(self, images, cells_cap_per_field: int = 4096, prob_thresh=None, nms_thresh=None,
                      seg_images=None, chunk_fields: int = 16):
        """det:51-153 for a batch of uint16 fields with NOTHING but the images given: normalize -> U-Net -> instances
        (csrc/segment.cu) -> region scan -> gates -> crops -> autoencoder -> SVMs through ``cia_screen_images``, up to
        ``chunk_fields`` fields per call, all enqueued on one stream (the labels never leave the device; one host
        synchronisation at the end).  ``seg_images`` (same shape) is the segmentation channel when it differs from the
        analysis channel (det:54-59); default: ``images`` itself.  Needs ``stardist_dir=`` (or ``self.stardist_model``).
        At most ``cells_cap_per_field`` instances per field.  Returns per-cell arrays in (field, ascending label) order:
        ``field``, ``label``, ``reconstruction_mse`` / ``_mae``, ``conservative_scores`` / ``moderate_scores`` (negated
        decisions, det:149-150), ``*_predictions``, and ``n_instances`` per field."""
        m = self.stardist_model
        if m is None:
            raise RuntimeError("screen_images needs the GPU segmentation: construct with stardist_dir=<model folder>")
        eng = self.engine
        imgs = np.ascontiguousarray(images)
        if imgs.dtype != np.uint16 or imgs.ndim != 3:
            raise UnsupportedImageError(f"screen_images takes uint16 [F, H, W] fields, got {imgs.dtype} {imgs.shape}")
        segs = imgs if seg_images is None else np.ascontiguousarray(seg_images)
        if segs.dtype != np.uint16 or segs.shape != imgs.shape:
            raise UnsupportedImageError(f"seg_images must be uint16 {imgs.shape}, got {segs.dtype} {segs.shape}")
        F, H, W = imgs.shape
        cap = int(cells_cap_per_field)
        pt = m.thresholds["prob"] if prob_thresh is None else prob_thresh
        nt = m.thresholds["nms"] if nms_thresh is None else nms_thresh
        dev = torch.from_numpy(imgs.view(np.int16)).to(eng.tdev)
        sdev = dev if segs is imgs else torch.from_numpy(segs.view(np.int16)).to(eng.tdev)
        n_inst = torch.zeros(F, dtype=torch.int32, device=eng.tdev)
        outs = []
        for f0 in range(0, F, chunk_fields):
            nf = min(chunk_fields, F - f0)
            o = eng.alloc_outputs(cap * nf, nf)
            eng.screen_images(sdev[f0:f0 + nf], dev[f0:f0 + nf], cap, o, pt, nt, n_instances=n_inst[f0:f0 + nf])
            outs.append((f0, o))
        eng.check_status()                   # synchronises; raises on capacity / label overflow
        cols = {k: [] for k in ("field", "label", "mse", "mae", "dec_cons", "dec_mod", "pred_cons", "pred_mod")}
        for f0, o in outs:
            n = int(o["counts"][0].item())
            rec = o["cells"][:n].cpu().numpy().view(_lib.CELL_DTYPE).reshape(-1)
            cols["field"].append(f0 + rec["field"].astype(np.int64))
            cols["label"].append(rec["label"].astype(np.int64))
            for k in ("mse", "mae", "dec_cons", "dec_mod", "pred_cons", "pred_mod"):
                cols[k].append(o[k][:n].cpu().numpy())
        cat = {k: np.concatenate(v) if v else np.zeros(0) for k, v in cols.items()}
        return {"field": cat["field"], "label": cat["label"],
                "reconstruction_mse": cat["mse"], "reconstruction_mae": cat["mae"],
                "conservative_scores": -cat["dec_cons"], "moderate_scores": -cat["dec_mod"],      # det:149-150
                "conservative_predictions": cat["pred_cons"].astype(np.intp),
                "moderate_predictions": cat["pred_mod"].astype(np.intp),
                "n_instances": n_inst.cpu().numpy()}

    def screen_fields_sharded(self, fields, field_strain, n_strains: int, chunk_fields: int = 16):
        """``fields``: sequence of (green uint16 [H,W], labels int32 [H,W]) of one size, ``field_strain``
        their strain ids.  Every rank scores fields[rank::world]; returns the all-reduced per-strain
        accumulator [S,8] and (rank 0) the per-cell rows in reference order (distributed.ShardedScreen)."""
        from .distributed import GpuFieldScorer, ShardedScreen
        sh = ShardedScreen(GpuFieldScorer(self.engine, chunk_fields=chunk_fields))
        return sh.screen(lambda i: fields[i], len(fields), field_strain, n_strains)


def summarize_sample(sample_name, files_processed, s):
    """det:202-212."""
    return {
        "sample_name": sample_name,
        "total_cells": len(s["reconstruction_mse"]),
        "files_processed": files_processed,
        "conservative_anomaly_rate": s["conservative_anomaly_rate"],
        "moderate_anomaly_rate": s["moderate_anomaly_rate"],
        "mean_mse": np.mean(s["reconstruction_mse"]),
        "std_mse": np.std(s["reconstruction_mse"]),
        "mean_mae": np.mean(s["reconstruction_mae"]),
        "std_mae": np.std(s["reconstruction_mae"]),
    }


def detail_rows(sample_name, s):
    """det:217-234."""
    rows = []
    for i, (mse, mae, cp, mp, cs, ms) in enumerate(zip(
            s["reconstruction_mse"], s["reconstruction_mae"], s["conservative_predictions"],
            s["moderate_predictions"], s["conservative_scores"], s["moderate_scores"])):
        rows.append({"sample_name": sample_name, "cell_id": i, "mse": mse, "mae": mae,
                     "conservative_anomaly": cp == -1, "moderate_anomaly": mp == -1,
                     "conservative_score": cs, "moderate_score": ms})
    return rows
