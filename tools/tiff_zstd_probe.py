"""Zstandard TIFF fields: device against host decode rates, and the sharded screen over zstd files against Deflate.

  decode   16 fields of 2048 x 2048 uint16 (4 distinct fields, each file copied 4 times) per level (3, 19) x predictor x
           layout (16- to 1024-row strips, one strip per field): cia_tiff_decode_fields on the packed chunk (CUDA
           events, best of 5 after a warm-up; the compressed bytes already on the device) against the in-tree decoder
           (cia_tiff_zstd_decode) and libzstd (ZSTD_decompress) on one host core, each timed over every segment of 4
           files, best of 2.  Rates are GB/s of decoded output.  Level 19 is measured with predictor 2 only.
  screen   screen_mutant_samples_sharded(stardist_dir=...) on one GPU over 64 fields written with zstd (level 3) and
           with Deflate, predictor 2, in 64-row strips (both decoded on the device) and in one strip per field (8 MB
           segments, above both routing limits: decoded by the loader threads), alternated twice; fields/s and the seconds the
           loader threads spend reading, parsing and decoding files.
  route    the same screen over 64 zstd fields (level 3, predictor 2) in 32- to 512-row strips, each once with the device
           route and once with every file sent to the host reader (up to 8 loader threads decoding in parallel, while
           the device screens the previous chunk), alternated twice.

The routing limit (tiff_device.MAX_DEVICE_ZSTD_SEGMENT_BYTES) is the largest segment size at which the device route
runs the screen at least as fast as the host route in every round.  Writes <out>/tiff_zstd_probe.json with the card name and power limit.
  python tools/tiff_zstd_probe.py --out /tmp/zstd_probe
"""
import argparse
import ctypes as C
import json
import os
import shutil
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import tiff_fixtures  # noqa: E402
import zstd_fixtures as zf  # noqa: E402
from tiff_decode_probe import card, device_rate, fields, screen  # noqa: E402
from cell_image_analysis_b200 import _lib, stardist as sdp, tiff_device as td, tiff_min  # noqa: E402

LAYOUTS = {"strips16": 16, "strips64": 64, "strips256": 256, "strips512": 512, "strips1024": 1024, "one_strip": 2048}
LEVEL = [3]                                       # the zstd level tiff_fixtures.write uses


def _install_encoder():
    orig = tiff_fixtures.encode
    tiff_fixtures.encode = lambda raw, c: zf.compress(raw, LEVEL[0]) if c in zf.CODES else orig(raw, c)


def write_set(d, imgs, level, pred, rows, copies=4):
    """the 4 distinct fields of ``imgs`` written with zstd at ``level`` in ``rows``-row strips, each copied"""
    LEVEL[0] = level

    def one(k):
        p = os.path.join(d, f"z{level}_{pred}_{rows}_{k:02d}.tif")
        tiff_fixtures.write(p, imgs[k], compression=50000, predictor=pred, rows_per_strip=rows)
        return p
    with ThreadPoolExecutor(4) as ex:
        base = list(ex.map(one, range(4)))
    paths = list(base)
    for k in range(4, 4 * copies):
        p = os.path.join(d, f"z{level}_{pred}_{rows}_{k:02d}.tif")
        shutil.copy(base[k % 4], p)
        paths.append(p)
    return paths


def host_rates(paths):
    """in-tree decoder and libzstd on one core over every segment of 4 files (best of 2)"""
    lib = _lib.load()
    segs = []
    for p in paths[:4]:
        buf = open(p, "rb").read()
        lay = tiff_min.page_layout(buf)
        for (o, c), (_, _, _, rows, cols) in zip(lay.segments, lay.segment_rects()):
            segs.append((buf[o:o + c], rows * cols * 2))
    cap = max(n for _, n in segs)
    dst = C.create_string_buffer(cap)
    total = sum(n for _, n in segs)
    out = {}
    for name, fn in (("in_tree", lambda s, n: lib.cia_tiff_zstd_decode(s, len(s), dst, n)),
                     ("libzstd", lambda s, n: zf.ZSTD.ZSTD_decompress(dst, n, s, len(s)))):
        best = 1e9
        for _ in range(2):
            t0 = time.perf_counter()
            for s, n in segs:
                assert fn(s, n) == n
            best = min(best, time.perf_counter() - t0)
        out[name] = dict(seconds=best, gbps_per_core=total / best / 1e9)
    return out


def zstd_folder(tmp, imgs, rows, n):
    """n fields (the 16 distinct ones of ``imgs`` repeated) as zstd level 3, predictor 2, ``rows``-row strips"""
    d = os.path.join(tmp, f"route_{rows}")
    os.makedirs(d)
    LEVEL[0] = 3
    for k in range(n):
        p = os.path.join(d, f"f{k:03d}.tif")
        if k < 16:
            tiff_fixtures.write(p, imgs[k], compression=50000, predictor=2, rows_per_strip=rows)
        else:
            shutil.copy(os.path.join(d, f"f{k % 16:03d}.tif"), p)
    return d


def route(screener, folders):
    """fields/s of each folder with the zstd route forced to the device and to the host reader"""
    rows_out = []
    limit = td.MAX_DEVICE_ZSTD_SEGMENT_BYTES
    try:
        for rnd in range(2):
            for rows, d in folders.items():
                for where, lim in (("device", 1 << 40), ("host", 0)):
                    td.MAX_DEVICE_ZSTD_SEGMENT_BYTES = lim
                    r = dict(screen(screener, {"s": d}, f"zstd3_pred2_strips{rows}"), route=where, round=rnd,
                             segment_bytes=rows * 2048 * 2)
                    print(json.dumps(r), flush=True)
                    rows_out.append(r)
    finally:
        td.MAX_DEVICE_ZSTD_SEGMENT_BYTES = limit
    return rows_out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--screen-fields", type=int, default=64)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    if zf.ZSTD is None:
        raise SystemExit(zf.SKIP_REASON)
    from cell_image_analysis_b200.screening import ProductionMutantScreening
    _install_encoder()
    res = {"card": card(), "decode": [], "screen": [], "route": []}
    tmp = tempfile.mkdtemp()
    cfg = dict(n_channel_in=1, grid=[2, 2], n_rays=32, unet_n_depth=3, unet_n_filter_base=32, unet_n_conv_per_depth=2,
               net_conv_after_unet=128, unet_kernel_size=[3, 3], unet_pool=[2, 2], unet_activation="relu",
               unet_last_activation="relu", unet_batch_norm=False)
    screener = ProductionMutantScreening(os.path.join(ROOT, "tests", "golden", "model_dir"))
    screener.stardist_model = sdp.StarDist2D.from_arrays(cfg, sdp.random_weights(cfg), {"prob": 0.5, "nms": 0.3},
                                                         engine=screener.engine)    # synthetic weights
    eng = screener.engine
    imgs = fields(16)
    for level, preds in ((3, (1, 2)), (19, (2,))):
        for pred in preds:
            for layout, rows in LAYOUTS.items():
                d = tempfile.mkdtemp(dir=tmp)
                paths = write_set(d, imgs, level, pred, rows)
                row = dict(level=level, predictor=pred, layout=layout, segment_bytes=rows * 2048 * 2,
                           device=device_rate(eng, paths), host=host_rates(paths))
                row["device_over_in_tree_core"] = row["device"]["gbps"] / row["host"]["in_tree"]["gbps_per_core"]
                row["device_over_libzstd_core"] = row["device"]["gbps"] / row["host"]["libzstd"]["gbps_per_core"]
                print(json.dumps(row), flush=True)
                res["decode"].append(row)
                shutil.rmtree(d)
    m = screener.stardist_model                   # synthetic weights: as tools/tiff_decode_probe.py
    prob, _ = m.predict(m.normalize_device(imgs[0]))
    for q in (0.9, 0.97, 0.99, 0.995, 0.999):
        m.thresholds["prob"] = float(np.quantile(prob.cpu().numpy(), q))
        if int(m.segment_device(imgs[0])[0].max()) <= 2048:
            break
    res["screen_prob_quantile"] = q
    many = [imgs[k % 16] for k in range(a.screen_fields)]
    folders = {}
    LEVEL[0] = 3
    for comp in (50000, 8):
        for rows in (64, 2048):
            label = f"{'zstd3' if comp == 50000 else 'deflate'}_pred2_{'strips64' if rows == 64 else 'one_strip'}"
            d = os.path.join(tmp, label)
            os.makedirs(d)
            distinct = {}
            for k, img in enumerate(many):
                p = os.path.join(d, f"f{k:03d}.tif")
                if k % 16 in distinct:
                    shutil.copy(distinct[k % 16], p)
                    continue
                tiff_fixtures.write(p, img, compression=comp, predictor=2, rows_per_strip=rows)
                distinct[k % 16] = p
            folders[label] = d
    for rnd in range(2):
        for label, d in folders.items():
            r = dict(screen(screener, {"s": d}, label), round=rnd)
            print(json.dumps(r), flush=True)
            res["screen"].append(r)
    res["route"] = route(screener, {rows: zstd_folder(tmp, imgs, rows, a.screen_fields) for rows in (32, 64, 128, 256, 512)})
    wins = {}                                     # segment size -> the device route won every round
    for r in res["route"]:
        if r["route"] == "device":
            host = next(h for h in res["route"] if h["route"] == "host" and h["round"] == r["round"]
                        and h["segment_bytes"] == r["segment_bytes"])
            wins[r["segment_bytes"]] = wins.get(r["segment_bytes"], True) and r["fields_per_s"] >= host["fields_per_s"]
    won = [b for b in sorted(wins) if all(wins[c] for c in sorted(wins) if c <= b)]
    res["route_limit_bytes"] = won[-1] if won else 0
    res["max_device_zstd_segment_bytes_during_run"] = td.MAX_DEVICE_ZSTD_SEGMENT_BYTES
    with open(os.path.join(a.out, "tiff_zstd_probe.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
