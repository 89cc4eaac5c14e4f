#!/usr/bin/env python
"""bench.py -- cells scored/sec through the per-cell screening hot path
(label scan -> gates -> crop + CLAHE + resize -> CAE recon error -> scaler/PCA -> 2x RBF
one-class SVM -> per-strain accumulators), BASELINE.json's metric.

  python bench.py --gpus N --steps K --warmup W           # CUDA path (this repo)
  python bench.py --impl reference --gpus N --steps K ...  # reference CPU path (oracle port)
  python bench.py ... --dump-outputs DIR                   # + the last timed step's outputs as DIR/*.npy

A step is one pass over ``--fields`` synthetic 2048x2048 fields (config 2 of
BASELINE.json: 1000 fields, ~500k cells) per GPU, visiting a resident pool of
``--pool`` distinct seeded fields chunk by chunk (the pool, 25 MB per field, is far
larger than the 126 MB L2).  ``value`` is timed with the pool resident in HBM; ``e2e``
runs the same pass from pinned HOST memory with the H2D copies and the D2H read of the
per-cell results inside the timed region.  Multi-GPU: one process per GPU, fields
sharded (each rank its own 1000 visits, weak scaling), one NCCL all-reduce of the
per-strain accumulator per step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "cells scored/sec (crop+resize+CAE+SVM)"
UNIT = "cells/s"
MODEL_DIR = os.path.join(ROOT, "tests", "golden", "model_dir")
FLOP_PER_CELL = 100.27e6          # SURVEY 8d: L1..L7 conv MACs*2
CAE_PASS_CELLS = 18944            # cells per pass over the seven layers (cae_tc.cu)
LAYER_MFLOP = [2.359, 37.749, 9.437, 1.180, 9.437, 37.749, 2.359]   # SURVEY 8d, L1..L7
ISSUED_FLOP_RATIO = (3 * (2.359 + 37.749 + 9.437) + (1.180 + 9.437 + 37.749 + 2.359)) / 100.27   # split-precision encoder
H = W = 2048
N_CELLS_PER_FIELD = 520


def _gen_field(seed):
    from cell_image_analysis_b200 import synth
    return synth.make_field(int(seed))


def make_pool(seeds):
    import multiprocessing as mp
    with mp.get_context("fork").Pool(min(len(seeds), os.cpu_count() or 1)) as pool:
        fields = pool.map(_gen_field, list(seeds))
    greens = np.stack([f[0] for f in fields])
    labels = np.stack([f[1] for f in fields])
    return greens, labels


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.proc, self.lines = gpu, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------
# reference CPU path (oracle port), used by cpu_baseline and --impl reference
# ---------------------------------------------------------------------------
_REF = {}


def _ref_init(threads):
    import torch
    torch.set_num_threads(threads)
    from cell_image_analysis_b200.artifacts import load_model_dir
    a = load_model_dir(MODEL_DIR)
    ae = a["autoencoder"]
    _REF["w"] = {"kernels": ae["kernels"], "biases": ae["biases"], "bns": ae["bns"]}
    _REF["sk"] = a["sklearn"]


def _ref_field(idx):
    """One field through the restated reference path: per-cell Python loop
    (improved_detection.py:72-111) then one compute_anomaly_scores call (det:117-153)."""
    from oracle import extraction, scoring
    green, labels = _REF["fields"][idx]
    t0 = time.perf_counter()
    cells, stats, kept, tab = extraction.extract_quality_cells_from_labels(green, labels)
    t1 = time.perf_counter()
    sk = _REF["sk"]
    s = scoring.compute_anomaly_scores(cells, _REF["w"], _REF["w"], sk["scaler"], sk["pca"],
                                       sk["detector_conservative"], sk["detector_moderate"], exact=False)
    t2 = time.perf_counter()
    return len(cells), t1 - t0, t2 - t1


def cpu_baseline_inline(n_fields=2):
    """Single process, as the reference runs: Python per-cell loop, BLAS/conv threads =
    all cores, libsvm serial.  Bounded sample; field synthesis is outside the timing."""
    cores = os.cpu_count() or 1
    _ref_init(cores)
    _REF["fields"] = [_gen_field(s) for s in range(n_fields)]
    n, te, ts = 0, 0.0, 0.0
    for i in range(n_fields):
        k, a, b = _ref_field(i)
        n += k; te += a; ts += b
    return {"value": n / (te + ts), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n_fields} config-1 fields (seeds 0..{n_fields - 1}, {n} cells), restated reference "
                      f"CPU path (oracle; scipy/sklearn real, skimage/Keras restated), single process, "
                      f"{cores} BLAS/conv threads; extraction {te:.1f}s, scoring {ts:.1f}s"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (the oracle port;
    the reference itself is two Python scripts whose skimage/TensorFlow imports are not
    installable here) on all host cores: one worker process per core, each running the
    reference's single-threaded per-cell loop on its own field."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = os.cpu_count() or 1
    per_step = cores
    _REF["fields"] = [_gen_field(s) for s in range(per_step)]      # inherited by the forked workers
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_ref_init, initargs=(1,)) as pool:
        for _ in range(args.warmup):
            pool.map(_ref_field, range(per_step), chunksize=1)
        n, dt = 0, 0.0
        for _ in range(args.steps):
            t_s = time.perf_counter()
            res = pool.map(_ref_field, range(per_step), chunksize=1)
            dt += time.perf_counter() - t_s
            n += sum(r[0] for r in res)
    val = n / dt
    sample = (f"{per_step} config-1 fields per step ({n // max(args.steps, 1)} cells), one worker process per "
              f"core ({cores}) running the reference's per-cell Python loop + one scoring call per field")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64/f32 (CPU)",
            "data": "synthetic",
            "config": {"workload": "config 2 sample: 2048x2048 uint16 fields + int32 labels, ~475 scored cells/field",
                       "fields_per_step": per_step},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def host_probe(eng, bs, g_pin, l_pin, host_threads, world, dev, barrier):
    """Host-memory side of the end-to-end pass, measured on every rank at the same time: streaming
    reads of the pinned label pool with the encoder's thread count, alone and next to back-to-back
    H2D copies of the image pool (what the DMA engine does during a pass).  Sums over ranks."""
    import torch
    import torch.distributed as dist
    lib = eng.lib
    threads = host_threads if host_threads > 0 else (os.cpu_count() or 1)
    nbytes = l_pin.numel() * 4
    stage = torch.empty_like(g_pin, device=dev)
    barrier()
    alone = lib.cia_host_read_probe(l_pin.data_ptr(), nbytes, threads, 2)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 12
    with torch.cuda.stream(bs.copy):
        e0.record(bs.copy)
        for _ in range(reps):
            stage.copy_(g_pin, non_blocking=True)
        e1.record(bs.copy)
    busy = lib.cia_host_read_probe(l_pin.data_ptr(), nbytes, threads, 2)
    still_copying = not e1.query()
    bs.copy.synchronize()
    h2d_gbs = reps * g_pin.numel() * 2 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    v = torch.tensor([alone, busy, h2d_gbs], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(v, op=dist.ReduceOp.SUM)
    return {"read_gbs_alone": float(v[0]), "read_gbs_next_to_h2d": float(v[1]), "h2d_gbs_next_to_reads": float(v[2]),
            "threads_per_rank": threads, "copies_outlasted_probe": bool(still_copying)}


def svm_extras():
    """Scaler/PCA + both detectors timed at detector sizes the golden artifacts do not have:
    'realistic' (2 x 5000 SVs, 100-d: nu * N_train for a ~50k-100k cell training set) and BASELINE
    config 4 (2 x 20000 SVs, 256-d).  Synthetic detectors (random SVs), real kernels: the default
    tcgen05 GEMM-form kernels (score_tc.cu) and the fp64 DMMA anchor (svm_kernel = pca_kernel = 0)."""
    import torch
    from cell_image_analysis_b200.artifacts import load_model_dir
    from cell_image_analysis_b200.screening import Engine
    arts = load_model_dir(MODEL_DIR)
    pk = peaks()
    out = {}
    for tag, nsv, dim, n in (("realistic_5k_sv_100d", 5000, 100, 30400), ("config4_20k_sv_256d", 20000, 256, 30400)):
        rng = np.random.default_rng(1)
        q, _ = np.linalg.qr(rng.standard_normal((2048, dim)))
        a = dict(arts)
        a["scaler_pca"] = dict(arts["scaler_pca"], C=dim, center=None, scale=None, components=np.ascontiguousarray(q.T),
                               offset=np.zeros(dim), f32_flow=True)
        for k in ("svm_conservative", "svm_moderate"):
            a[k] = dict(sv=rng.standard_normal((nsv, dim)) * 3.0, coef=rng.uniform(0, 1, nsv), gamma=1.0 / (dim * 9.0), rho=1.0)
        eng = Engine(device=0, precision=1)
        eng.load_artifacts(a)
        feat = torch.from_numpy((rng.standard_normal((n, 2048)) * 3.0).astype(np.float32)).to(eng.tdev)
        flop = (2.0 * dim * 2 * nsv + 2.0 * 2048 * dim) * n
        res = {"cells": n}
        for name, kern in (("tcgen05", 1), ("dmma_fp64", 0)):
            eng.set_option("svm_kernel", kern)
            eng.set_option("pca_kernel", kern)
            for _ in range(3):
                eng.svm_decision(feat, n)
            torch.cuda.synchronize()
            best = 1e9
            for _ in range(3):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(5):
                    eng.svm_decision(feat, n)
                e1.record()
                torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1) / 5)
            tf = flop / (best * 1e-3) / 1e12
            res[name] = {"ms": best, "cells_per_s": n / (best * 1e-3), "algorithmic_tflops": tf}
            if kern == 1:
                res[name].update(issued_tflops=3 * tf, issued_frac_of_bf16_peak=3 * tf / pk["tf_burst"])
            else:
                res[name].update(frac_of_dmma_peak=tf / 37.0)
        res["speedup"] = res["dmma_fp64"]["ms"] / res["tcgen05"]["ms"]
        out[tag] = res
        eng.close()
    out["note"] = ("scaler/PCA + 2 detectors per call; tcgen05: fp16 hi/lo operands, 3 MMAs per product (issued = 3 x algorithmic), "
                   f"peak = bf16 dense burst {pk['tf_burst']:.0f} TFLOP/s ({pk['source']}); dmma_fp64: mma.sync.m8n8k4.f64, measured "
                   "DMMA peak 37 TFLOP/s (profiles/fp64_peak_test.cu); best of 3 rounds of 5 calls")
    return out


def segmentation_extras(with_cpu: bool):
    """The producer of the label field (SURVEY 8f N2: csbdeep normalize + StarDist2D.predict_instances,
    improved_detection.py:62-63) timed on one 2048 x 2048 field: percentile normalisation, the 2D_versatile_fluo
    U-Net topology with synthetic weights (the pretrained weights are not available offline; the arithmetic does
    not depend on their values), and candidates + polygon NMS + label rendering on the (prob, dist) maps a trained
    network emits for a field of ~530 ellipses; then the same labels through the screening path."""
    import torch
    from cell_image_analysis_b200 import stardist as sdp, synth
    from cell_image_analysis_b200.artifacts import load_model_dir
    from cell_image_analysis_b200.screening import Engine
    pk = peaks()
    H = W = 2048
    cfg = sdp.CONFIG_2D_VERSATILE_FLUO
    eng = Engine(device=0, precision=1)
    m = sdp.StarDist2D.from_arrays(cfg, sdp.random_weights(cfg), {"prob": 0.479071, "nms": 0.3}, engine=eng)
    green, _ = _gen_field(0)
    g = torch.from_numpy(green.view(np.int16)).to(eng.tdev)
    x = torch.empty((H, W), dtype=torch.float32, device=eng.tdev)
    prob, dist = synth.star_maps_from_ellipses(H, W, 2, synth.ellipse_lattice(H, W, 23, 3))
    pd, dd = torch.from_numpy(prob).to(eng.tdev), torch.from_numpy(dist).to(eng.tdev)
    labels = torch.empty((H, W), dtype=torch.int32, device=eng.tdev)
    n_inst = torch.zeros(1, dtype=torch.int32, device=eng.tdev)
    st = eng._stream

    def f_norm():
        eng._check(eng.lib.cia_seg_normalize(eng.h, g.data_ptr(), H, W, 3.0, 99.8, x.data_ptr(), None, st()))

    def f_net():
        eng._check(eng.lib.cia_seg_predict(eng.h, x.data_ptr(), H, W, None, None, st()))

    def f_inst():
        eng._check(eng.lib.cia_seg_instances(eng.h, pd.data_ptr(), dd.data_ptr(), H // 2, W // 2, 2, H, W, 0.479071, 0.3,
                                             labels.data_ptr(), n_inst.data_ptr(), st()))

    def timed(fn, reps=5):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / reps)
        return best

    t_norm, t_net, t_inst = timed(f_norm), timed(f_net), timed(f_inst)
    l0 = eng.launch_count
    f_norm(); f_net(); f_inst()
    launches = eng.launch_count - l0
    flops = sdp.network_flops(cfg, H, W)
    total = t_norm + t_net + t_inst
    # the whole chain of det:51-153 for one field with nothing but the uint16 image given: normalize, U-Net,
    # instances (on the star maps of THIS field's true labels: what a trained network emits; the synthetic-weight
    # network's own maps are computed and discarded), region scan, gates, crops, autoencoder, SVMs
    _, truth = _gen_field(0)
    pt, dt = synth.star_maps_from_labels(truth, 2)
    ptd, dtd = torch.from_numpy(pt).to(eng.tdev), torch.from_numpy(dt).to(eng.tdev)
    eng.load_artifacts(load_model_dir(MODEL_DIR))
    out = eng.alloc_outputs(4096, 1)
    img3 = g.view(1, H, W)

    def f_chain():
        f_norm()
        f_net()
        eng._check(eng.lib.cia_seg_instances(eng.h, ptd.data_ptr(), dtd.data_ptr(), H // 2, W // 2, 2, H, W, 0.479071, 0.3,
                                             labels.data_ptr(), n_inst.data_ptr(), st()))
        eng.screen_fields(img3, labels.view(1, H, W), 1024, out)

    t_chain = timed(f_chain)
    eng.check_status()
    chain_cells = int(out["counts"][0].item())
    chain_inst = int(n_inst.item())
    f_inst()
    out = {
        "field": [H, W], "model": "2D_versatile_fluo topology (grid 2, depth 3, 32 filters, 128 features, 32 rays), synthetic weights",
        "normalize_ms": t_norm, "unet_ms": t_net, "instances_ms": t_inst, "ms_per_field": total, "fields_per_s": 1e3 / total,
        "unet_gflop": flops / 1e9, "unet_tflops": flops / (t_net * 1e-3) / 1e12,
        "unet_frac_of_bf16_peak": flops / (t_net * 1e-3) / 1e12 / pk["tf_burst"],
        "candidates": int((prob > np.float32(0.479071)).sum()), "instances": int(n_inst.item()),
        "dtype": "f16 tensor core U-Net (fp32 accumulate), f64 polygon overlap",
        "gpu_launches_per_field": int(launches),
        "chain": {"what": "uint16 image -> normalize -> U-Net -> instances -> region scan -> gates -> crops -> autoencoder -> SVMs, "
                          "one field per call, labels never leave the device",
                  "ms_per_field": t_chain, "fields_per_s": 1e3 / t_chain, "instances": chain_inst, "scored_cells": chain_cells,
                  "cells_per_s": chain_cells * 1e3 / t_chain},
        "note": "CUDA events, best of 3 rounds of 5 calls per stage; one field per call",
    }
    if with_cpu:
        # restated CPU path of the same step (oracle: torch-CPU float32 U-Net, C post-processing), one field
        from oracle import stardist as sdo
        t0 = time.perf_counter()
        xn = sdo.normalize(green)
        t1 = time.perf_counter()
        sdo.unet_forward(cfg, sdp.random_weights(cfg), xn)
        t2 = time.perf_counter()
        ref, _ = sdo.instances_from_prediction(prob, dist, 2, (H, W), 0.479071, 0.3)
        t3 = time.perf_counter()
        out["cpu_port"] = {"normalize_ms": 1e3 * (t1 - t0), "unet_ms": 1e3 * (t2 - t1), "instances_ms": 1e3 * (t3 - t2),
                           "cores": os.cpu_count(), "kind": "port",
                           "labels_equal_gpu": bool(np.array_equal(ref, labels.cpu().numpy())),
                           "sample": "one 2048 x 2048 field; the oracle's suppression is a plain O(kept x candidates) loop"}
    eng.close()
    return out


# ---------------------------------------------------------------------------
SCORE_KEYS = ("mse", "mae", "dec_cons", "dec_mod", "pred_cons", "pred_mod")
# --dump-outputs: two row sets (device pass, end-to-end pass) of 16 columns x 8 bytes stay near 32 MB, within 64 MB
MAX_DUMP_ROWS = 1 << 17


def per_cell_rows(cells, scores, max_rows):
    """Per-cell results as named columns, rows in (field, label) order so that two builds compare row by
    row whatever order the device compacted them in; more than ``max_rows`` rows: a fixed seeded sample."""
    order = np.lexsort((cells["label"], cells["field"]))
    if len(order) > max_rows:
        order = order[np.sort(np.random.default_rng(0).choice(len(order), max_rows, replace=False))]
    cols = {f"cell_{k}": cells[k][order] for k in cells.dtype.names if k != "pad_"}
    cols.update({k: scores[k][order] for k in SCORE_KEYS})
    return cols


def device_pass_outputs(bs, n_chunks):
    """What a device-resident pass leaves its caller: the per-strain accumulators and the per-cell
    results of its last chunk (``run_device`` writes chunk i into ``bs.out[i & 1]``)."""
    from cell_image_analysis_b200 import _lib
    o = bs.out[(n_chunks - 1) & 1]
    n = min(int(o["counts"][0].item()), o["cap"])
    cells = o["cells"][:n].cpu().numpy().view(_lib.CELL_DTYPE).reshape(-1)
    rows = per_cell_rows(cells, {k: o[k][:n].cpu().numpy() for k in SCORE_KEYS}, MAX_DUMP_ROWS)
    return dict(strain_acc=bs.acc.cpu().numpy(), field_counts=o["counts"][1:].cpu().numpy(), **rows)


def write_outputs(path, arrays):
    """``<path>/<name>.npy``: float32 arrays as they are, everything else as float64 (exact for the
    integer columns)."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


def run_native(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from cell_image_analysis_b200.artifacts import load_model_dir
    from cell_image_analysis_b200.batch import BatchScreen
    from cell_image_analysis_b200.distributed import allreduce_strain_acc
    from cell_image_analysis_b200.screening import Engine

    eng = Engine(device=local, precision=args.precision)
    eng.load_artifacts(load_model_dir(MODEL_DIR))
    dev = eng.tdev

    Fc, P, NF = args.chunk, args.pool, args.fields
    assert P % Fc == 0 and NF % Fc == 0
    greens, labels = make_pool([rank * 100003 + i for i in range(P)])
    max_label = int(labels.max())
    g_pin = torch.from_numpy(greens.view(np.int16)).pin_memory()
    l_pin = torch.from_numpy(labels).pin_memory()
    g_dev, l_dev = g_pin.to(dev), l_pin.to(dev)
    n_strains = args.strains if args.strains > 0 else (100 if world > 1 else 4)
    visit_strain = (torch.arange(NF, dtype=torch.int32) * n_strains // NF).to(dev)   # contiguous blocks
    rle_fraction = args.rle_fraction
    if args.label_transport == "auto":
        # Every chunk crosses PCIe as runs.  One GPU: the 16 host cores encode faster than the device
        # screens.  Several ranks share the host cores AND the host DRAM: two ranks reach 3.3M
        # cells/s end to end whether all chunks or 85 % of them are encoded (raw copies: 2.1M), i.e.
        # the hosts memory bandwidth, read once by the encoder or by the DMA engine, is the limit.
        args.label_transport = "rle"
        if world > 1 and args.host_threads <= 0:
            args.host_threads = max(1, (os.cpu_count() or 1) // world)
    if rle_fraction < 0:
        rle_fraction = 1.0
    bs = BatchScreen(eng, H, W, max_label, chunk_fields=Fc, n_strains=n_strains,
                     label_transport=args.label_transport, host_threads=args.host_threads,
                     rle_fraction=rle_fraction, host_buffers=args.host_buffers,
                     image_transport="dense" if args.image_transport == "auto" else args.image_transport)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        with torch.cuda.stream(bs.compute):
            bs.acc.zero_()
        bs.run_device(g_dev, l_dev, NF, visit_strain)
        if world > 1:
            with torch.cuda.stream(bs.compute):
                allreduce_strain_acc(bs.acc)        # the path's only collective (SURVEY 8e)

    def step_host():
        with torch.cuda.stream(bs.compute):
            bs.acc.zero_()
        bs.run_host(g_pin, l_pin, NF, visit_strain)
        if world > 1:
            with torch.cuda.stream(bs.compute):
                allreduce_strain_acc(bs.acc)

    # ---- device-resident: warmup, then K timed steps ----
    for _ in range(args.warmup):
        step_device()
    barrier()
    eng.check_status()
    chunks_per_step = NF // Fc
    bs.profile_begin(args.steps * chunks_per_step)
    l0 = eng.launch_count
    sampler = ClockSampler(local)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(bs.compute)
    for _ in range(args.steps):
        step_device()
    e1.record(bs.compute)
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    clocks = sampler.stop()
    launches = eng.launch_count - l0
    layer_ms = None
    if args.precision != 0:
        try:
            layer_ms = bs.profile_layers()        # CAE stage split by conv layer
        except Exception:
            layer_ms = None
    stage_ms, nrec = bs.profile_end()
    eng.check_status()
    dump = device_pass_outputs(bs, chunks_per_step) if args.dump_outputs and rank == 0 else None
    # cells per step on this rank: one extra untimed pass without the all-reduce
    cells_local = torch.tensor([0.0], dtype=torch.float64, device=dev)
    bs.sync(); bs.acc.zero_(); bs.run_device(g_dev, l_dev, NF, visit_strain); bs.sync()
    cells_local[0] = bs.acc[:, 0].sum()
    cells_per_step_local = float(cells_local.item())
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(cells_local, op=dist.ReduceOp.SUM)
    cells_per_step = float(cells_local.item())
    t_ms = float(ms.item())
    value = cells_per_step * args.steps / (t_ms * 1e-3)

    # ---- end to end from pinned host memory ----
    step_host(); bs.sync()
    res = bs.collect_host()
    assert res["n_cells"] == int(round(cells_per_step_local)), (res["n_cells"], cells_per_step_local)
    sum_hw = int(((res["cells"]["maxr"] - res["cells"]["minr"]).astype(np.int64) *
                  (res["cells"]["maxc"] - res["cells"]["minc"])).sum())
    barrier()
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0.record(bs.compute)
    t_wall = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    h1.record(bs.compute)
    bs.sync()
    t_wall = time.perf_counter() - t_wall
    barrier()
    ems = torch.tensor([max(h0.elapsed_time(h1), 0.0)], dtype=torch.float64, device=dev)
    ems[0] = max(float(ems.item()), t_wall * 1e3)       # copy-stream time before the first compute
    if world > 1:
        dist.all_reduce(ems, op=dist.ReduceOp.MAX)
    e2e_value = cells_per_step * args.steps / (float(ems.item()) * 1e-3)
    if dump is not None:
        last = bs.collect_host()
        dump.update(e2e_field_counts=last["field_counts"],
                    **{f"e2e_{k}": v for k, v in per_cell_rows(last["cells"], last, MAX_DUMP_ROWS).items()})
        write_outputs(args.dump_outputs, dump)
    h2d, d2h = bs.host_bytes_per_pass(NF)
    eng.check_status()
    enc_s = getattr(bs, "encode_seconds", 0.0)          # host time inside the encoder during the LAST timed pass
    host = host_probe(eng, bs, g_pin, l_pin, args.host_threads, world, dev, barrier)
    enc_gbs = torch.tensor([4.0 * NF * H * W / enc_s / 1e9 if enc_s > 0 else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(enc_gbs, op=dist.ReduceOp.SUM)

    if rank == 0:
        pk = peaks()
        cae_ms = stage_ms["cae"] / args.steps
        crop_ms = stage_ms["crop"] / args.steps
        scan_ms = stage_ms["scan"] / args.steps
        svm_ms = stage_ms["svm"] / args.steps
        tf = FLOP_PER_CELL * cells_per_step_local / (cae_ms * 1e-3) / 1e12
        crop_gbs = (2.0 * sum_hw + 16384.0 * cells_per_step_local) / (crop_ms * 1e-3) / 1e9
        scan_gbs = 4.0 * H * W * NF / (scan_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("cae_stage_dram_bytes_per_cell")
            traffic = None if traffic is None else traffic * cells_per_step_local
        split = 3.0 if args.precision == 1 else 1.0       # fp16 MMAs per encoder product (hi*lo, lo*hi, hi*hi)
        stage_roofline = {"kernel": "CAE forward stage (7 conv layers + error reduction)", "bound": "tensor",
                          "achieved": tf, "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": tf / pk["tf_sust"],
                          "traffic": traffic, "peak_source": pk["source"] + ", bf16 dense sustained",
                          # what the tensor pipe executes: the encoder (49.55 of the 100.27 MFLOP) runs three
                          # fp16 MMAs per product to deliver fp32-grade features
                          "issued_tflops": tf * ISSUED_FLOP_RATIO if args.precision == 1 else tf,
                          "issued_frac": (tf * ISSUED_FLOP_RATIO if args.precision == 1 else tf) / pk["tf_sust"],
                          "share_of_step": cae_ms / (t_ms / args.steps)}
        roofline = stage_roofline
        layers = None
        if layer_ms is not None and layer_ms[1] > 0:
            # the dominant kernel: layer 2 (conv_tc_acc2_kernel, 32 -> 64 channels at 32x32, one launch per
            # chunk); its time comes from CUDA events recorded in-stream around that launch
            l2_ms = layer_ms[1] / args.steps
            l2_launches = chunks_per_step * -(-bs.cap // CAE_PASS_CELLS)      # passes per call (cae_tc.cu CH_MAX)
            l2_tf = LAYER_MFLOP[1] * 1e6 * cells_per_step_local / (l2_ms * 1e-3) / 1e12
            l2_traffic = None
            if os.path.exists(tp):
                l2_traffic = json.load(open(tp)).get("l2_kernel_dram_bytes_per_cell")
                l2_traffic = None if l2_traffic is None else l2_traffic * cells_per_step_local / l2_launches
            roofline = {"kernel": "conv_tc_acc2_kernel<32,64,32,3> (CAE layer 2, tcgen05 implicit GEMM, split-precision)",
                        "bound": "tensor", "achieved": l2_tf, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                        "frac": l2_tf / pk["tf_sust"], "traffic": l2_traffic,
                        "peak_source": pk["source"] + ", bf16 dense sustained",
                        "algorithmic_mflop_per_cell": LAYER_MFLOP[1], "launches_per_step": l2_launches,
                        "avg_launch_ms": l2_ms / l2_launches,
                        "issued_tflops": l2_tf * split, "issued_frac": l2_tf * split / pk["tf_sust"],
                        "note": "achieved = algorithmic FLOPs (37.749 MFLOP per cell x cells per launch) / launch "
                                "time; the kernel issues 3 fp16 MMAs per product for fp32-grade features "
                                "(issued_*: the algorithmic ceiling of this split is 1/3 of the issued rate), and ncu "
                                "shows its tensor-core pipe > 90 % busy, bound by operand reads from shared memory at "
                                "N = 64 (profiles/r2k_l2_full.txt); traffic per launch",
                        "share_of_step": l2_ms / (t_ms / args.steps)}
            layers = {f"L{i + 1}": {"ms_per_step": layer_ms[i] / args.steps,
                                    "tflops": LAYER_MFLOP[i] * 1e6 * cells_per_step_local / (layer_ms[i] / args.steps * 1e-3) / 1e12}
                      for i in range(7) if layer_ms[i] > 0}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (CAE fp32 FMA, fp64 flush) / f64 (CLAHE+resize, PCA, SVM) / int (scan)"
                     if args.precision == 0 else "f16 tensor cores (CAE, PCA, SVM cross term: fp16 hi+lo operands, fp32 accumulate) / f64 norms and sums",
            "data": "synthetic",
            "config": {"workload": ("config 2" if world == 1 else f"config 5 (multi-strain screen, {n_strains} strains, fields "
                                    f"sharded over {world} GPUs, one all-reduce of the [S,8] accumulator per step)") +
                                   f": {NF} visits/GPU/step of 2048x2048 uint16 fields + int32 labels "
                                   f"(~{cells_per_step_local / NF:.0f} scored cells/field), resident pool of {P} "
                                   f"distinct seeded fields ({P * 25.2:.0f} MB > 126 MB L2) cycled in chunks of {Fc}",
                       "fields_per_step_per_gpu": NF, "cells_per_step": cells_per_step, "strains": n_strains,
                       "artifacts": "tests/golden/model_dir (synthetic CAE weights; scaler/PCA(100)/2 SVMs fit with sklearn)",
                       "precision": args.precision, "l2_policy": "inputs larger than L2"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": float(ems.item()) / args.steps,
                    "label_transport": args.label_transport, "image_transport": bs.image_transport, "rle_fraction": round(getattr(bs, "last_rle_share", bs.rle_fraction), 3),
                    "host_threads": args.host_threads or (os.cpu_count() or 1),
                    "host": dict(host, encoder_gbs=float(enc_gbs.item()),
                                 host_dram_traffic_gbs=(4.0 + 2.0) * H * W * (e2e_value / (cells_per_step_local / NF)) / 1e9,
                                 pcie_floor_ms=h2d / (host["h2d_gbs_next_to_reads"] / world * 1e9) * 1e3,   # this rank's bytes over its link
                                 bound=("gpu" if e2e_value > 0.9 * value else
                                        "pcie" if float(ems.item()) / args.steps < 1.2 * h2d / (host["h2d_gbs_next_to_reads"] / world * 1e9) * 1e3 else
                                        ("host-dram" if (4.0 + 2.0) * H * W * (e2e_value / (cells_per_step_local / NF)) / 1e9
                                         > 0.7 * (host["read_gbs_next_to_h2d"] + host["h2d_gbs_next_to_reads"]) else "host-cores")),
                                 note="per field the encoder reads 16.8 MB of labels and the DMA engine 8.4 MB of image from "
                                      "host DRAM; read_gbs_*: cia_host_read_probe on the pinned label pool on all ranks at "
                                      "once; encoder_gbs: label bytes / host time inside cia_rle_encode_fields"),
                    "api": "BatchScreen.run_host -> cia_screen_fields_rle / cia_screen_fields (pinned host pool of "
                           "uint16 images + int32 labels; with label_transport=rle the share rle_fraction of the "
                           "chunks is run-length encoded by the host cores inside the timed region and scanned "
                           "from the runs on the device, the rest crosses PCIe raw; double-buffered H2D)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
            "stages_ms_per_step": {k: v / args.steps for k, v in stage_ms.items()},
            "cae_layers": layers,
            "stage_rooflines": {
                "cae_stage": stage_roofline,
                "label_scan": {"bound": "hbm", "achieved": scan_gbs, "peak": pk["hbm"], "unit": "GB/s",
                               "frac": scan_gbs / pk["hbm"]},
                "crop_clahe_resize": {"bound": "hbm", "achieved": crop_gbs, "peak": pk["hbm"], "unit": "GB/s",
                                      "frac": crop_gbs / pk["hbm"]},
                "svm_ms": svm_ms},
        }
        if world == 1 and not args.no_svm_extras:
            line["extra"] = {"svm": svm_extras()}
        if world == 1 and not args.no_seg_extras:
            line.setdefault("extra", {})["segmentation"] = segmentation_extras(not args.no_cpu_baseline)
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_inline(args.cpu_fields)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--fields", type=int, default=1024, help="field visits per GPU per step (config 2: ~1000)")
    ap.add_argument("--pool", type=int, default=64, help="distinct resident fields per GPU")
    ap.add_argument("--chunk", type=int, default=64, help="fields per fused call (measured: 32 -> 2.45M, 64 -> 2.49M cells/s)")
    ap.add_argument("--strains", type=int, default=0,
                    help="strains the field visits are spread over (0 = 4 on one GPU; 100 on several: BASELINE config 5)")
    ap.add_argument("--precision", type=int, default=1,
                    help="CAE path: 0 exact fp32 CUDA cores, 1 tcgen05 (split-precision encoder), 2 tcgen05 + fp32 encoder")
    ap.add_argument("--label-transport", default="auto", choices=["auto", "rle", "raw"],
                    help="e2e arm: how the int32 label fields cross PCIe (rle = lossless host run-length encode; "
                         "auto = rle, with cores/ranks encoder threads per rank)")
    ap.add_argument("--host-threads", type=int, default=0, help="host threads of the RLE encoder (0 = all cores / ranks)")
    ap.add_argument("--rle-fraction", type=float, default=-1.0,
                    help="share of the chunks sent as runs (rest raw); < 0 = all of them")
    ap.add_argument("--cpu-fields", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-svm-extras", action="store_true")
    ap.add_argument("--no-seg-extras", action="store_true")
    ap.add_argument("--host-buffers", type=int, default=2, help="device chunk buffers of the host pass (A/B)")
    ap.add_argument("--image-transport", default="auto", choices=["auto", "patches", "dense"],
                    help="e2e pass: send whole images or only the bbox rectangles of the labelled regions "
                         "(auto = dense: measured faster on this host at 1 and 2 GPUs, DESIGN.md section 6)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last step computed as DIR/<name>.npy (float32 / float64): "
                         "strain_acc and field_counts plus the per-cell rows of the device pass's last chunk, and "
                         "e2e_* for the end-to-end pass (at most 2^17 rows each, a seeded sample beyond that)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native path")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
