"""Device against host decode of compressed TIFF fields, and the sharded screen over compressed files.

  decode   F = 16 fields of 2048 x 2048 uint16 per compression x predictor x layout (64-row strips, 16-row strips, one
           strip per field, 256-row strips = 1 MB segments, 256 x 256 tiles): cia_tiff_decode_fields on the packed
           chunk (CUDA events, best of 5 after a warm-up; the chunk's compressed bytes are already on the device)
           against tiff_min.read_tiff on one core (best of 2 per file over 4 files).  Rates are GB/s of decoded output.
  screen   screen_mutant_samples_sharded(stardist_dir=...) on one GPU over a folder of Deflate + predictor-2 files
           (64-row strips: decoded on the device; one strip per field: above MAX_DEVICE_SEGMENT_BYTES, read on the
           host) against the same images uncompressed, read with the default reader and with a caller's reader (the
           route to the device is then off: the loader path as it was before the device decode); fields/s and the
           seconds the loader threads spend reading, parsing and decoding files.

Writes <out>/tiff_decode_probe.json with the card name and power limit.
  python tools/tiff_decode_probe.py --out /tmp/tiff_probe
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import tiff_fixtures  # noqa: E402
from cell_image_analysis_b200 import stardist as sdp, synth, tiff_device as td  # noqa: E402
from cell_image_analysis_b200.tiff_min import read_tiff, write_tiff  # noqa: E402

# 256-row strips decode to 1 MB per segment: the size of MAX_DEVICE_SEGMENT_BYTES
LAYOUTS = {"strips64": dict(rows_per_strip=64), "strips16": dict(rows_per_strip=16),
           "strips256": dict(rows_per_strip=256), "one_strip": dict(rows_per_strip=2048),
           "tiles256": dict(tile=(256, 256))}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True,
                           text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        q = f"unavailable: {e}"
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q}


def fields(n, H=2048, W=2048):
    h, w, nc, lo, hi, lu = synth.FIELD_CONFIGS["tiny"]
    out = []
    for s in range(n):
        f, _ = synth.make_field(100 + s, h, w, nc, lo, hi, lu)
        noise = np.random.default_rng(s).integers(0, 96, (H, W))            # sensor noise: realistic Deflate ratios
        out.append((np.tile(f, (-(-H // h), -(-W // w)))[:H, :W] + noise).astype(np.uint16))
    return out


def write_set(d, imgs, comp, pred, layout):
    """16 files of one compression x predictor x layout; OpenCV writes LZW / PackBits strips, the in-repo writer
    Deflate and LZW / PackBits tiles (4 distinct fields encoded in Python, each file copied 4 times)"""
    import cv2
    paths = []
    for k, a in enumerate(imgs):
        p = os.path.join(d, f"{comp}_{pred}_{layout}_{k:02d}.tif")
        if comp == 8:
            tiff_fixtures.write(p, a, compression=8, predictor=pred, **LAYOUTS[layout])
        elif layout == "tiles256":
            if k < 4:
                tiff_fixtures.write(p, a, compression=comp, predictor=pred, **LAYOUTS[layout])
            else:
                shutil.copy(paths[k % 4], p)
        else:
            flag = cv2.IMWRITE_TIFF_COMPRESSION_LZW if comp == 5 else cv2.IMWRITE_TIFF_COMPRESSION_PACKBITS
            cv2.imwrite(p, a, [cv2.IMWRITE_TIFF_COMPRESSION, flag, cv2.IMWRITE_TIFF_PREDICTOR, pred,
                               cv2.IMWRITE_TIFF_ROWSPERSTRIP, LAYOUTS[layout]["rows_per_strip"]])
        paths.append(p)
    return paths


def device_rate(eng, paths):
    fs = [td.parse_field(p) for p in paths]
    chunk = td.TiffChunk(fs, range(len(fs)))
    dev = torch.empty(chunk.total, dtype=torch.uint8, device=eng.tdev)
    scratch = torch.empty(chunk.scratch_bytes, dtype=torch.uint8, device=eng.tdev)
    H, W = fs[0].shape
    img = torch.empty((len(fs), H, W), dtype=torch.int16, device=eng.tdev)
    status = torch.empty(len(fs), dtype=torch.int32, device=eng.tdev)
    chunk.upload(dev)
    torch.cuda.synchronize()
    best = 1e9
    for r in range(6):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        chunk.decode(eng, dev, scratch, None, img, status)
        b.record()
        b.synchronize()
        if r:
            best = min(best, a.elapsed_time(b) / 1e3)
    assert not status.cpu().numpy().any()
    want = read_tiff(paths[0])
    assert np.array_equal(img[0].cpu().numpy().view(np.uint16), want)
    out_bytes = len(fs) * H * W * 2
    segs = len(fs[0].layout.segments)
    return dict(seconds=best, gbps=out_bytes / best / 1e9, segments_per_field=segs,
                compressed_mb=chunk.src_bytes / 1e6, decoded_mb=out_bytes / 1e6)


def host_rate(paths):
    ts = []
    for p in paths[:4]:
        t = []
        for _ in range(2):
            t0 = time.perf_counter()
            a = read_tiff(p)
            t.append(time.perf_counter() - t0)
        ts.append(min(t))
    return dict(seconds_per_field=float(np.mean(ts)), gbps_per_core=a.nbytes / float(np.mean(ts)) / 1e9)


def screen(screener, folders, label, default_reader=True):
    """wall time of the sharded screen and the loader threads' time (file read, parse, host decode)"""
    from cell_image_analysis_b200 import distributed, screening
    spent, lock = [0.0], threading.Lock()

    def timed(fn):
        def w(*a):
            t0 = time.perf_counter()
            try:
                return fn(*a)
            finally:
                with lock:
                    spent[0] += time.perf_counter() - t0
        return w
    orig = td.device_route, screening._default_imread, distributed._read_file
    td.device_route, screening._default_imread, distributed._read_file = (timed(f) for f in orig)
    # a caller's reader (any other callable) turns the device route off
    screener.imread = screening._default_imread if default_reader else timed(lambda p: orig[1](p))
    try:
        screener.screen_mutant_samples_sharded(folders, chunk_fields=16)      # warm-up
        spent[0] = 0.0
        t0 = time.perf_counter()
        res, _ = screener.screen_mutant_samples_sharded(folders, chunk_fields=16)
        wall = time.perf_counter() - t0
    finally:
        td.device_route, screening._default_imread, distributed._read_file = orig
        screener.imread = orig[1]
    n = sum(len(os.listdir(f)) for f in folders.values())
    return dict(workload=label, default_reader=default_reader, fields=n, seconds=wall, fields_per_s=n / wall,
                loader_thread_seconds=spent[0], cells=sum(r["total_cells"] for r in res.values()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--screen-fields", type=int, default=64)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    from cell_image_analysis_b200.screening import ProductionMutantScreening
    res = {"card": card(), "decode": [], "screen": []}
    tmp = tempfile.mkdtemp()
    cfg = dict(n_channel_in=1, grid=[2, 2], n_rays=32, unet_n_depth=3, unet_n_filter_base=32, unet_n_conv_per_depth=2,
               net_conv_after_unet=128, unet_kernel_size=[3, 3], unet_pool=[2, 2], unet_activation="relu",
               unet_last_activation="relu", unet_batch_norm=False)
    screener = ProductionMutantScreening(os.path.join(ROOT, "tests", "golden", "model_dir"))
    screener.stardist_model = sdp.StarDist2D.from_arrays(cfg, sdp.random_weights(cfg), {"prob": 0.5, "nms": 0.3},
                                                         engine=screener.engine)    # synthetic weights
    eng = screener.engine
    imgs = fields(16)
    for comp in (8, 5, 32773):
        for pred in (1, 2):
            for layout in LAYOUTS:
                d = tempfile.mkdtemp(dir=tmp)
                paths = write_set(d, imgs, comp, pred, layout)
                row = dict(compression=comp, predictor=pred, layout=layout, device=device_rate(eng, paths),
                           host=host_rate(paths))
                row["device_over_host_core"] = row["device"]["gbps"] / row["host"]["gbps_per_core"]
                print(json.dumps(row), flush=True)
                res["decode"].append(row)
                for p in paths:
                    os.remove(p)
    m = screener.stardist_model                   # synthetic weights: the lowest probability quantile that keeps a
    prob, _ = m.predict(m.normalize_device(imgs[0]))  # field under the screen's 4096 instances
    for q in (0.9, 0.97, 0.99, 0.995, 0.999):
        m.thresholds["prob"] = float(np.quantile(prob.cpu().numpy(), q))
        if int(m.segment_device(imgs[0])[0].max()) <= 2048:
            break
    res["screen_prob_quantile"] = q
    many = [imgs[k % 16] for k in range(a.screen_fields)]
    for label, kw in (("uncompressed", None), ("deflate_pred2_strips64", dict(rows_per_strip=64)),
                      ("deflate_pred2_one_strip", dict(rows_per_strip=2048))):
        d = os.path.join(tmp, label)
        os.makedirs(d)
        for k, img in enumerate(many):
            p = os.path.join(d, f"f{k:03d}.tif")
            write_tiff(p, img) if kw is None else tiff_fixtures.write(p, img, compression=8, predictor=2, **kw)
        # uncompressed: the default reader (route decided per file) and a caller's reader (the loader path before
        # the device decode), alternated three times to show the spread between runs of one workload
        for rnd in range(3 if kw is None else 1):
            for default_reader in ((True, False) if kw is None else (True,)):
                r = dict(screen(screener, {"s": d}, label, default_reader), round=rnd)
                print(json.dumps(r), flush=True)
                res["screen"].append(r)
    res["max_device_segment_bytes"] = td.MAX_DEVICE_SEGMENT_BYTES
    with open(os.path.join(a.out, "tiff_decode_probe.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
