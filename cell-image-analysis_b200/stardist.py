"""Host side of the segmentation step: mirrors the two calls the reference makes,

    normalized_seg = normalize(seg_channel)                                     # improved_detection.py:62
    labels, details = self.stardist_model.predict_instances(normalized_seg)     # improved_detection.py:63

(``StarDist2D.from_pretrained('2D_versatile_fluo')`` at improved_detection.py:44; the training twin at
CAE_improved_modeltrain.py:54-55) with csbdeep's ``normalize`` and stardist's ``StarDist2D`` names, argument
meaning and return types, every computation done by libcia.so on the GPU (csrc/segment.cu): percentile
normalisation, the U-Net on tcgen05, candidate selection, polygon NMS and label rendering.  The labels can stay
on the device and feed ``extract_quality_cells_from_labels`` without crossing PCIe.

A model is a StarDist model folder (``config.json``, ``thresholds.json``, ``weights_best.h5`` /
``weights_last.h5``) read without h5py / Keras.  ``from_pretrained`` needs such a folder on disk (there is no
download): ``$CIA_STARDIST_MODELS/<name>``.  No CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import re

import numpy as np
import torch

from .hdf5_min import H5File


class SegConfig(C.Structure):
    _fields_ = [("n_channel_in", C.c_int32), ("grid", C.c_int32), ("n_rays", C.c_int32),
                ("unet_n_depth", C.c_int32), ("unet_n_filter_base", C.c_int32),
                ("unet_n_conv_per_depth", C.c_int32), ("net_conv_after_unet", C.c_int32),
                ("reserved", C.c_int32)]


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _layer_key(name: str):
    """Application order of the convolution layers of StarDist2D._build + csbdeep unet_block."""
    m = re.fullmatch(r"conv2d(?:_(\d+))?", name)
    if m:
        return (0, int(m.group(1) or 0), 0)
    m = re.fullmatch(r"(?:.*?)down_level_(\d+)_no_(\d+)", name)
    if m:
        return (1, int(m.group(1)), int(m.group(2)))
    m = re.fullmatch(r"(?:.*?)middle_(\d+)", name)
    if m:
        return (2, int(m.group(1)), 0)
    m = re.fullmatch(r"(?:.*?)up_level_(\d+)_no_(\d+)", name)
    if m:
        return (3, -int(m.group(1)), int(m.group(2)))
    return {"features": (4, 0, 0), "prob": (5, 0, 0), "dist": (6, 0, 0)}.get(name)


def load_weights_h5(path: str) -> dict:
    """{layer name: (kernel HWIO float32, bias float32)} from a Keras H5 weights file
    (``/<layer>/<layer>/kernel:0``; also the ``/layers/<layer>/vars/0|1`` layout of ``*.weights.h5``)."""
    with open(path, "rb") as f:
        ds = H5File(f.read()).datasets()
    out = {}
    for key, arr in ds.items():
        parts = key.split("/")
        leaf = parts[-1]
        if leaf in ("kernel:0", "bias:0", "kernel", "bias") and len(parts) >= 2:
            layer, which = parts[-2], leaf.split(":")[0]
        elif len(parts) >= 3 and parts[-2] == "vars" and leaf in ("0", "1"):
            layer, which = parts[-3], "kernel" if leaf == "0" else "bias"
        else:
            continue
        out.setdefault(layer, {})[which] = np.ascontiguousarray(arr, np.float32)
    return {k: (v["kernel"], v["bias"]) for k, v in out.items() if "kernel" in v and "bias" in v}


def layer_plan(config: dict):
    """[(layer name, cin, cout, kernel side)] in application order: StarDist2D._build (grid blocks, `features`,
    `prob`, `dist`) around csbdeep's unet_block (down levels, middle, up levels with skip concatenation)."""
    grid, depth = int(config["grid"][0]), int(config["unet_n_depth"])
    nconv, base = int(config["unet_n_conv_per_depth"]), int(config["unet_n_filter_base"])
    plan, cin, k = [], int(config.get("n_channel_in", 1)), 0
    pooled = 1
    while pooled < grid:
        for _ in range(nconv):
            plan.append(("conv2d" if k == 0 else f"conv2d_{k}", cin, base, 3))
            cin, k = base, k + 1
        pooled *= 2
    skips = []
    for n in range(depth):
        for i in range(nconv):
            plan.append((f"down_level_{n}_no_{i}", cin, base << n, 3))
            cin = base << n
        skips.append(cin)
    for i in range(nconv - 1):
        plan.append((f"middle_{i}", cin, base << depth, 3))
        cin = base << depth
    plan.append((f"middle_{nconv}", cin, base << max(0, depth - 1), 3))
    cin = base << max(0, depth - 1)
    for n in reversed(range(depth)):
        cin += skips[n]
        for i in range(nconv - 1):
            plan.append((f"up_level_{n}_no_{i}", cin, base << n, 3))
            cin = base << n
        plan.append((f"up_level_{n}_no_{nconv}", cin, base << max(0, n - 1), 3))
        cin = base << max(0, n - 1)
    after = int(config["net_conv_after_unet"])
    return plan + [("features", cin, after, 3), ("prob", after, 1, 1), ("dist", after, int(config["n_rays"]), 1)]


def network_flops(config: dict, H: int, W: int) -> float:
    """multiply-adds x 2 of one forward pass over an H x W field"""
    grid, depth, nconv = int(config["grid"][0]), int(config["unet_n_depth"]), int(config["unet_n_conv_per_depth"])
    shifts, s = [], 0
    pooled = 1
    while pooled < grid:
        shifts += [s] * nconv
        s, pooled = s + 1, pooled * 2
    for _ in range(depth):
        shifts += [s] * nconv
        s += 1
    shifts += [s] * nconv
    for _ in range(depth):
        s -= 1
        shifts += [s] * nconv
    shifts += [s, s, s]
    return float(sum(2.0 * k * k * ci * co * (H >> sh) * (W >> sh) for (_, ci, co, k), sh in zip(layer_plan(config), shifts)))


def random_weights(config: dict, seed: int = 11) -> dict:
    """Synthetic He-normal weights {layer: (kernel HWIO, bias)} (the pretrained models are not available offline):
    the arithmetic and the memory traffic of the network do not depend on the weight values."""
    rng = np.random.default_rng(seed)
    out = {}
    for name, cin, cout, k in layer_plan(config):
        kern = (rng.standard_normal((k, k, cin, cout)) * np.sqrt(2.0 / (k * k * cin))).astype(np.float32)
        bias = (rng.standard_normal(cout) * 0.05).astype(np.float32)
        if name == "dist":
            bias[:] = 6.0
        out[name] = (kern, bias)
    return out


CONFIG_2D_VERSATILE_FLUO = dict(n_channel_in=1, grid=[2, 2], n_rays=32, unet_n_depth=3, unet_n_filter_base=32,
                                unet_n_conv_per_depth=2, net_conv_after_unet=128, unet_kernel_size=[3, 3],
                                unet_pool=[2, 2], unet_activation="relu", unet_last_activation="relu",
                                unet_batch_norm=False)


def ray_angles(n_rays=32):
    return np.linspace(0, 2 * np.pi, n_rays, endpoint=False)


class StarDist2D:
    """Drop-in for ``stardist.models.StarDist2D`` as the reference uses it (det:44, 63)."""

    def __init__(self, config=None, name=None, basedir=".", engine=None, device: int = 0):
        from .screening import Engine
        self.engine = engine if engine is not None else Engine(device=device)
        self.name, self.basedir = name, basedir
        self.thresholds = {"prob": 0.5, "nms": 0.4}       # stardist's defaults when thresholds.json is absent
        if config is None:
            folder = os.path.join(basedir, name)
            with open(os.path.join(folder, "config.json")) as f:
                config = json.load(f)
            tj = os.path.join(folder, "thresholds.json")
            if os.path.exists(tj):
                with open(tj) as f:
                    self.thresholds = json.load(f)
            wfile = next((os.path.join(folder, w) for w in ("weights_best.h5", "weights_last.h5", "weights_now.h5")
                          if os.path.exists(os.path.join(folder, w))), None)
            if wfile is None:
                raise FileNotFoundError(f"no weights_best.h5 / weights_last.h5 in {folder}")
            self.config = config
            self.load_weights(load_weights_h5(wfile))
        else:
            self.config = config

    @classmethod
    def from_pretrained(cls, name_or_alias, engine=None, device: int = 0):
        """The reference downloads '2D_versatile_fluo' (det:44); here the model folder must already be on disk
        under ``$CIA_STARDIST_MODELS`` (no network)."""
        root = os.environ.get("CIA_STARDIST_MODELS", "")
        if not root or not os.path.isdir(os.path.join(root, name_or_alias)):
            raise FileNotFoundError(
                f"pretrained StarDist model '{name_or_alias}' is not on disk: put its folder (config.json, "
                "thresholds.json, weights_best.h5) under $CIA_STARDIST_MODELS; nothing is downloaded")
        return cls(None, name=name_or_alias, basedir=root, engine=engine, device=device)

    @classmethod
    def from_arrays(cls, config: dict, weights: dict, thresholds=None, engine=None, device: int = 0):
        m = cls(config, engine=engine, device=device)
        if thresholds:
            m.thresholds = dict(thresholds)
        m.load_weights(weights)
        return m

    # ---- StarDist2D._build: upload the layers in application order ----
    def load_weights(self, weights: dict):
        cfg = self.config
        grid = tuple(cfg.get("grid", (1, 1)))
        if len(grid) != 2 or grid[0] != grid[1]:
            raise ValueError(f"grid {grid}: only square grids are supported")
        if cfg.get("unet_batch_norm", False):
            raise ValueError("unet_batch_norm=True is not supported")
        if tuple(cfg.get("unet_kernel_size", (3, 3))) != (3, 3) or tuple(cfg.get("unet_pool", (2, 2))) != (2, 2):
            raise ValueError("only 3x3 kernels with 2x2 pooling are supported")
        for act in ("unet_activation", "unet_last_activation"):
            if cfg.get(act, "relu") != "relu":
                raise ValueError(f"{act}={cfg[act]!r}: only relu is supported")
        named = [(k, _layer_key(k)) for k in weights]
        unknown = [k for k, key in named if key is None]
        if unknown:
            raise ValueError(f"unrecognised layers in the weights file: {unknown}")
        order = [k for k, _ in sorted(named, key=lambda kv: kv[1])]
        ks = [np.ascontiguousarray(weights[k][0], np.float32) for k in order]
        bs = [np.ascontiguousarray(weights[k][1], np.float32) for k in order]
        n = len(order)
        shapes = np.array([k.shape for k in ks], np.int64).reshape(n, 4)
        sc = SegConfig(int(cfg.get("n_channel_in", 1)), int(grid[0]), int(cfg.get("n_rays", 32)),
                       int(cfg.get("unet_n_depth", 3)), int(cfg.get("unet_n_filter_base", 32)),
                       int(cfg.get("unet_n_conv_per_depth", 2)), int(cfg.get("net_conv_after_unet", 128)), 0)
        K = (C.c_void_p * n)(*[k.ctypes.data for k in ks])
        B = (C.c_void_p * n)(*[b.ctypes.data for b in bs])
        phis = ray_angles(sc.n_rays)
        rs, rc = np.ascontiguousarray(np.sin(phis)), np.ascontiguousarray(np.cos(phis))
        eng = self.engine
        eng._check(eng.lib.cia_seg_load(eng.h, C.byref(sc), n, K, B, C.c_void_p(shapes.ctypes.data),
                                        C.c_void_p(rs.ctypes.data), C.c_void_p(rc.ctypes.data)))
        self.layer_order = order
        self.grid = int(grid[0])
        self.n_rays = sc.n_rays
        self.div_by = self.grid << sc.unet_n_depth

    # ---- device-side pieces ----
    def normalize_device(self, seg_channel, pmin=3, pmax=99.8):
        """csbdeep ``normalize`` of a uint16 / uint8 field on the GPU -> float32 cuda tensor [H, W]."""
        eng = self.engine
        x = np.ascontiguousarray(seg_channel)
        if x.dtype == np.uint8:
            x = x.astype(np.uint16)
        if x.dtype != np.uint16 or x.ndim != 2:
            raise TypeError(f"normalize: the CUDA path takes 2-D uint16 / uint8 fields, got {x.dtype} {x.shape}")
        d = torch.from_numpy(x.view(np.int16)).to(eng.tdev)
        out = torch.empty(x.shape, dtype=torch.float32, device=eng.tdev)
        eng._check(eng.lib.cia_seg_normalize(eng.h, _ptr(d), x.shape[0], x.shape[1], float(pmin), float(pmax),
                                             _ptr(out), C.c_void_p(0), eng._stream()))
        return out

    def _as_device_image(self, img):
        eng = self.engine
        if isinstance(img, torch.Tensor):
            t = img.to(device=eng.tdev, dtype=torch.float32).contiguous()
        else:
            a = np.asarray(img)
            if a.ndim == 3 and a.shape[-1] == 1:
                a = a[..., 0]
            t = torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(eng.tdev)
        if t.ndim != 2:
            raise ValueError(f"expected a 2-D single-channel image, got shape {tuple(t.shape)}")
        H, W = t.shape
        pad = (-H % self.div_by, -W % self.div_by)
        if pad != (0, 0):     # StarDist pads to a multiple of grid * 2^depth with np.pad(mode='reflect')
            t = torch.nn.functional.pad(t[None, None], (0, pad[1], 0, pad[0]), mode="reflect")[0, 0].contiguous()
        return t, (H, W)

    def predict(self, img):
        """-> prob [H/g, W/g], dist [H/g, W/g, n_rays] as float32 cuda tensors (StarDist2D.predict)."""
        eng = self.engine
        t, (H, W) = self._as_device_image(img)
        Hp, Wp = t.shape
        prob = torch.empty((Hp // self.grid, Wp // self.grid), dtype=torch.float32, device=eng.tdev)
        dist = torch.empty((Hp // self.grid, Wp // self.grid, self.n_rays), dtype=torch.float32, device=eng.tdev)
        eng._check(eng.lib.cia_seg_predict(eng.h, _ptr(t), Hp, Wp, _ptr(prob), _ptr(dist), eng._stream()))
        hg, wg = -(-H // self.grid), -(-W // self.grid)
        return prob[:hg, :wg].contiguous(), dist[:hg, :wg].contiguous()

    def instances_from_prediction(self, img_shape, prob, dist, prob_thresh=None, nms_thresh=None, sync=True):
        """prob / dist cuda tensors -> (labels int32 cuda tensor [H, W], n_instances).  ``sync=False`` returns the
        count as a one-element cuda tensor instead of reading it back (a stream-ordered pipeline stage)."""
        eng = self.engine
        pt = self.thresholds["prob"] if prob_thresh is None else prob_thresh
        nt = self.thresholds["nms"] if nms_thresh is None else nms_thresh
        H, W = img_shape
        prob = prob.to(eng.tdev, torch.float32).contiguous()
        dist = dist.to(eng.tdev, torch.float32).contiguous()
        Hg, Wg = prob.shape
        labels = torch.empty((H, W), dtype=torch.int32, device=eng.tdev)
        n = torch.zeros(1, dtype=torch.int32, device=eng.tdev)
        eng._check(eng.lib.cia_seg_instances(eng.h, _ptr(prob), _ptr(dist), Hg, Wg, self.grid, H, W, float(pt),
                                             float(nt), _ptr(labels), _ptr(n), eng._stream()))
        return labels, (int(n.item()) if sync else n)

    def details(self, n):
        eng = self.engine
        pts = torch.empty((max(n, 1), 2), dtype=torch.int32, device=eng.tdev)
        pr = torch.empty(max(n, 1), dtype=torch.float32, device=eng.tdev)
        co = torch.empty((max(n, 1), 2, self.n_rays), dtype=torch.float32, device=eng.tdev)
        eng._check(eng.lib.cia_seg_details(eng.h, n, _ptr(pts), _ptr(pr), _ptr(co), eng._stream()))
        return {"points": pts[:n].cpu().numpy(), "prob": pr[:n].cpu().numpy(), "coord": co[:n].cpu().numpy()}

    # ---- the reference's call (det:63) ----
    def predict_instances(self, img, prob_thresh=None, nms_thresh=None, return_device=False, **unused):
        """``labels, details = model.predict_instances(normalize(x))``: labels int32 [H, W] (NumPy, or a cuda
        tensor with ``return_device=True``), details with 'points', 'prob', 'coord' of the kept polygons."""
        prob, dist = self.predict(img)
        shape = tuple(img.shape[:2])
        labels, n = self.instances_from_prediction(shape, prob, dist, prob_thresh, nms_thresh)
        details = self.details(n)
        return (labels if return_device else labels.cpu().numpy()), details

    def segment_fields(self, seg_images, prob_thresh=None, nms_thresh=None):
        """normalize + predict_instances of F equally sized fields in one launch sequence per stage: uint16 [F, H, W]
        (NumPy or a cuda tensor; uint8 is widened) -> (labels int32 cuda [F, H, W], n_instances int32 cuda [F]), each
        field equal bit for bit to ``segment_device`` of that field (reflect padding is done on the device)."""
        eng = self.engine
        if isinstance(seg_images, torch.Tensor):
            t = seg_images
            if t.dtype == torch.uint8:
                t = t.to(torch.int16)
            elif t.dtype == torch.uint16:
                t = t.view(torch.int16)
            elif t.dtype != torch.int16:       # int16: raw uint16 bits, as the rest of this package passes them
                raise TypeError(f"segment_fields takes uint16 / uint8 fields, got {t.dtype}")
            d = t.to(eng.tdev).contiguous()
        else:
            x = np.ascontiguousarray(seg_images)
            if x.dtype == np.uint8:
                x = x.astype(np.uint16)
            if x.dtype != np.uint16:
                raise TypeError(f"segment_fields takes uint16 / uint8 fields, got {x.dtype}")
            d = torch.from_numpy(x.view(np.int16)).to(eng.tdev)
        if d.ndim != 3:
            raise ValueError(f"segment_fields takes [F, H, W] fields, got shape {tuple(d.shape)}")
        F, H, W = d.shape
        pt = self.thresholds["prob"] if prob_thresh is None else prob_thresh
        nt = self.thresholds["nms"] if nms_thresh is None else nms_thresh
        Hp, Wp = H + (-H % self.div_by), W + (-W % self.div_by)
        x = torch.empty((F, Hp, Wp), dtype=torch.float32, device=eng.tdev)
        labels = torch.empty((F, H, W), dtype=torch.int32, device=eng.tdev)
        n = torch.zeros(F, dtype=torch.int32, device=eng.tdev)
        s = eng._stream()
        eng._check(eng.lib.cia_seg_normalize_fields(eng.h, _ptr(d), F, H, W, 3.0, 99.8, _ptr(x), s))
        eng._check(eng.lib.cia_seg_predict_fields(eng.h, _ptr(x), F, Hp, Wp, None, None, s))
        eng._check(eng.lib.cia_seg_instances_fields(eng.h, None, None, F, Hp // self.grid, Wp // self.grid, self.grid, H, W,
                                                    float(pt), float(nt), _ptr(labels), _ptr(n), s))
        return labels, n

    def segment_device(self, seg_channel):
        """normalize + predict_instances with everything resident: uint16 field -> int32 cuda labels, n."""
        x = self.normalize_device(seg_channel)
        prob, dist = self.predict(x)
        return self.instances_from_prediction(tuple(np.shape(seg_channel)[:2]), prob, dist)


def normalize(x, pmin=3, pmax=99.8, engine=None, device: int = 0):
    """csbdeep.utils.normalize for 16-bit fields on the GPU (det:62) -> float32 ndarray."""
    from .screening import Engine
    eng = engine if engine is not None else Engine(device=device)
    m = StarDist2D.__new__(StarDist2D)
    m.engine = eng
    return m.normalize_device(x, pmin, pmax).cpu().numpy()
