"""ctypes binding of libcia.so (include/cia.h).  No fallback: if the CUDA library is
missing or a call fails, this module raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcia.so")


CIA_E_CUDA, CIA_E_ARG, CIA_E_STATE, CIA_E_CAPACITY, CIA_E_LABEL, CIA_E_UNSUPPORTED = -1, -2, -3, -4, -5, -6


class CiaError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libcia error {code}: {msg}")
        self.code = code


class Region(C.Structure):
    _fields_ = [("area", C.c_uint32), ("minr", C.c_int32), ("minc", C.c_int32),
                ("maxr", C.c_int32), ("maxc", C.c_int32), ("flags", C.c_int32),
                ("m10", C.c_uint64), ("m01", C.c_uint64), ("m20", C.c_uint64),
                ("m02", C.c_uint64), ("m11", C.c_uint64)]


class Cell(C.Structure):
    _fields_ = [("field", C.c_int32), ("label", C.c_int32), ("minr", C.c_int32),
                ("minc", C.c_int32), ("maxr", C.c_int32), ("maxc", C.c_int32),
                ("area", C.c_int32), ("pad_", C.c_int32), ("eccentricity", C.c_double),
                ("mean_intensity", C.c_double), ("std_intensity", C.c_double)]


class Params(C.Structure):
    _fields_ = [("border_margin", C.c_int32), ("area_min", C.c_int32), ("area_max", C.c_int32),
                ("ecc_max", C.c_double), ("mean_min", C.c_double), ("std_min", C.c_double),
                ("clip_limit", C.c_double), ("intensity_inv", C.c_double)]


class Scores(C.Structure):
    _fields_ = [("mse", C.c_void_p), ("mae", C.c_void_p), ("dec_conservative", C.c_void_p),
                ("dec_moderate", C.c_void_p), ("pred_conservative", C.c_void_p),
                ("pred_moderate", C.c_void_p)]


REGION_DTYPE = np.dtype([("area", "<u4"), ("minr", "<i4"), ("minc", "<i4"), ("maxr", "<i4"),
                         ("maxc", "<i4"), ("flags", "<i4"), ("m10", "<u8"), ("m01", "<u8"),
                         ("m20", "<u8"), ("m02", "<u8"), ("m11", "<u8")])
CELL_DTYPE = np.dtype([("field", "<i4"), ("label", "<i4"), ("minr", "<i4"), ("minc", "<i4"),
                       ("maxr", "<i4"), ("maxc", "<i4"), ("area", "<i4"), ("pad_", "<i4"),
                       ("eccentricity", "<f8"), ("mean_intensity", "<f8"), ("std_intensity", "<f8")])
# cia_tiff_segment: one compressed strip / tile of a field (cia_tiff_decode_fields)
TIFF_SEGMENT_DTYPE = np.dtype([("src_off", "<u8"), ("src_len", "<u8"), ("dst_off", "<u8"), ("field", "<i4"),
                               ("compression", "<i4"), ("predictor", "<i4"), ("bytes_per_sample", "<i4"),
                               ("big_endian", "<i4"), ("samples", "<i4"), ("y0", "<i4"), ("x0", "<i4"),
                               ("rows", "<i4"), ("cols", "<i4"), ("seg_sample", "<i4"), ("img_sample", "<i4")])
assert TIFF_SEGMENT_DTYPE.itemsize == 72
assert REGION_DTYPE.itemsize == C.sizeof(Region) == 64
assert CELL_DTYPE.itemsize == C.sizeof(Cell) == 56

# name -> (restype, argtypes); every symbol include/cia.h declares
_P = C.c_void_p
_I = C.c_int
SIGNATURES = {
    "cia_version": (_I, []),
    "cia_create": (_I, [_I, C.POINTER(_P)]),
    "cia_destroy": (_I, [_P]),
    "cia_last_error": (C.c_char_p, [_P]),
    "cia_default_params": (None, [C.POINTER(Params)]),
    "cia_check_status": (_I, [_P, _P]),
    "cia_set_option": (_I, [_P, C.c_char_p, C.c_double]),
    "cia_load_cae": (_I, [_P, _I, _I, C.POINTER(_P), C.POINTER(_P), C.POINTER(_P), C.c_float]),
    "cia_load_scaler_pca": (_I, [_P, _I, _I, _P, _P, _I, _P, _P, _I]),
    "cia_load_svm": (_I, [_P, _I, _I, _I, _P, _P, C.c_double, C.c_double]),
    "cia_label_scan": (_I, [_P, _P, _I, _I, _I, _I, _P, _P]),
    "cia_filter": (_I, [_P, _P, _I, _I, _I, _I, _P, C.POINTER(Params), _P, _I, _P, _P, _P]),
    "cia_solidity": (_I, [_P, _P, _I, _I, _P, _I, _P, _P, _P]),
    "cia_crop_resize": (_I, [_P, _P, _I, _I, _P, _I, _P, C.POINTER(Params), _P, _P, _P]),
    "cia_debug_clahe_levels": (_I, [_P, _P, _I, _I, _P, _I, C.POINTER(Params), _P, _P, _P, _P]),
    "cia_cae_forward": (_I, [_P, _P, _I, _P, _P, _P, _P, _I, _P]),
    "cia_svm_decision": (_I, [_P, _P, _I, _P, _P, _P, _P, _P, _P, _P]),
    "cia_strain_accumulate": (_I, [_P, _P, _I, _P, C.POINTER(Scores), _P, _P, _I, _P]),
    "cia_screen_fields": (_I, [_P, _P, _P, _I, _I, _I, _I, C.POINTER(Params), _I, _P, _I, _P, _P,
                               C.POINTER(Scores), _P, _P, _P, _P, _I, _P]),
    "cia_screen_fields_host": (_I, [_P, _P, _P, _I, _I, _I, _I, C.POINTER(Params), _I, _P, _I, _P,
                                    _P, C.POINTER(Scores), _P]),
    "cia_rle_slot_words": (C.c_size_t, [_I, _I]),
    "cia_rle_encode_fields": (_I, [_P, _I, _I, _I, _P, C.c_size_t, _P, _P, _I]),
    "cia_host_read_probe": (C.c_double, [_P, C.c_size_t, _I, _I]),
    "cia_rle_upload": (_I, [_P, _P, _I, C.c_size_t, _P, _P, _P]),
    "cia_rle_expand": (_I, [_P, _P, _I, C.c_size_t, _I, _I, _P, _P]),
    "cia_label_scan_rle": (_I, [_P, _P, C.c_size_t, _I, _I, _I, _I, _P, _P]),
    "cia_screen_fields_rle": (_I, [_P, _P, _P, C.c_size_t, _I, _I, _I, _I, C.POINTER(Params), _I, _P, _I, _P, _P,
                                   C.POINTER(Scores), _P, _P, _P, _P, _I, _P]),
    "cia_rle_encode_pack_fields": (_I, [_P, _P, _I, _I, _I, _P, C.c_size_t, _P, _P, _I, _P, C.c_size_t, _P, _I]),
    "cia_patch_upload": (_I, [_P, _P, _I, C.c_size_t, _P, _P, _P]),
    "cia_screen_fields_rle_patches": (_I, [_P, _P, _P, C.c_size_t, _P, C.c_size_t, _I, _I, _I, _I, C.POINTER(Params), _I,
                                           _P, _I, _P, _P, C.POINTER(Scores), _P, _P, _P, _P, _I, _P]),
    "cia_tiff_lzw_decode": (C.c_longlong, [_P, C.c_size_t, _P, C.c_size_t]),
    "cia_tiff_packbits_decode": (C.c_longlong, [_P, C.c_size_t, _P, C.c_size_t]),
    "cia_tiff_zstd_decode": (C.c_longlong, [_P, C.c_size_t, _P, C.c_size_t]),
    "cia_tiff_decode_fields": (_I, [_P, _P, C.c_size_t, _P, _I, _I, _I, _I, _P, C.c_size_t, _P, _P, _P, _P]),
    "cia_profile_begin": (_I, [_P, _I]),
    "cia_profile_end": (_I, [_P, C.POINTER(C.c_double), C.POINTER(_I)]),
    "cia_profile_layers": (_I, [_P, C.POINTER(C.c_double)]),
    "cia_debug_copy_workspace": (_I, [_P, _I, C.c_size_t, _P, C.c_size_t]),
    "cia_launch_count": (C.c_int64, [_P]),
    # fits of create_anomaly_detector (csrc/fit.cu)
    "cia_fit_robust_scaler": (_I, [_P, _P, _I, _I, _P, _P, _P, _P]),
    "cia_fit_pca_gram": (_I, [_P, _P, _I, _I, _P, _P, _P]),
    "cia_ocsvm_fit": (_I, [_P, _P, _I, _I, C.c_double, C.c_double, C.c_double, _I, _P, _P, _P]),
    # segmentation (csrc/segment.cu)
    "cia_seg_load": (_I, [_P, _P, _I, C.POINTER(_P), C.POINTER(_P), _P, _P, _P]),
    "cia_seg_normalize": (_I, [_P, _P, _I, _I, C.c_double, C.c_double, _P, _P, _P]),
    "cia_seg_predict": (_I, [_P, _P, _I, _I, _P, _P, _P]),
    "cia_seg_instances": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, C.c_double, C.c_double, _P, _P, _P]),
    "cia_seg_details": (_I, [_P, _I, _P, _P, _P, _P]),
    "cia_seg_layer_info": (_I, [_P, _I, _P]),
    "cia_seg_debug_layer": (_I, [_P, _I, _P, _P, _P, _I, _I, _P, _P, _P, _P]),
    "cia_seg_normalize_fields": (_I, [_P, _P, _I, _I, _I, C.c_double, C.c_double, _P, _P]),
    "cia_seg_predict_fields": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "cia_seg_instances_fields": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, C.c_double, C.c_double, _P, _P, _P]),
    "cia_screen_images": (_I, [_P, _P, _P, _I, _I, _I, C.c_double, C.c_double, _I, C.POINTER(Params), _I, _P, _I, _P, _P,
                               C.POINTER(Scores), _P, _P, _P, _P, _I, _P, _P, _P]),
}

_lib = None


def load():
    """dlopen libcia.so and set the prototypes.  Raises if the library is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python __graft_entry__.py build` "
                "(nvcc, sm_100a).  There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(handle, rc):
    if rc != 0:
        msg = load().cia_last_error(handle)
        raise CiaError(rc, msg.decode() if msg else "?")


def default_params() -> Params:
    p = Params()
    load().cia_default_params(C.byref(p))
    return p
