"""Per-field against batched segmentation + screen on 2048 x 2048 fields (2D_versatile_fluo topology, synthetic
weights, as bench.py's extra.segmentation), for F in {1, 4, 16}:

  chain      normalize -> predict -> instances -> screen_fields, once per field (the composition before the batched
             calls) against cia_seg_*_fields -> one screen_fields over the F fields; instances run on the star maps of
             the fields' true labels (what a trained network emits), so candidate counts are realistic.  The two forms
             alternate in one process; best of several rounds, CUDA events.
  screen_images  cia_screen_images as one call, with a quantile threshold on the synthetic network's own maps.

Writes <out>/images_probe.json with the card name and power limit.
  python tools/images_probe.py --out /tmp/images_probe
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cell_image_analysis_b200 import stardist as sdp, synth  # noqa: E402
from cell_image_analysis_b200.artifacts import load_model_dir  # noqa: E402
from cell_image_analysis_b200.screening import Engine  # noqa: E402


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True,
                           timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired) as e:
        q = f"unavailable: {e}"
    return {"device": name, "nvidia_smi": q}


def best_of(fn, rounds, reps):
    best = 1e9
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / reps)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--fields", default="1,4,16")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--distinct", type=int, default=4, help="distinct seeded fields (repeated up to F)")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    H = W = 2048
    cfg = sdp.CONFIG_2D_VERSATILE_FLUO
    eng = Engine(device=0, precision=1)
    m = sdp.StarDist2D.from_arrays(cfg, sdp.random_weights(cfg), {"prob": 0.479071, "nms": 0.3}, engine=eng)
    eng.load_artifacts(load_model_dir(os.path.join(ROOT, "tests", "golden", "model_dir")))
    cfg1 = synth.FIELD_CONFIGS["config1"]
    base = [synth.make_field(s, *cfg1) for s in range(args.distinct)]
    maps = [synth.star_maps_from_labels(t, 2) for _, t in base]
    Fs = [int(v) for v in args.fields.split(",")]
    Fmax = max(Fs)
    greens = np.stack([base[f % args.distinct][0] for f in range(Fmax)])
    g_all = torch.from_numpy(greens.view(np.int16)).cuda()
    p_all = torch.stack([torch.from_numpy(maps[f % args.distinct][0]) for f in range(Fmax)]).cuda()
    d_all = torch.stack([torch.from_numpy(maps[f % args.distinct][1]) for f in range(Fmax)]).cuda()
    st = eng._stream
    lib, h = eng.lib, eng.h
    res = {"card": card(), "field": [H, W], "distinct_fields": args.distinct, "rounds": args.rounds, "per_F": {}}

    # a working threshold for the synthetic network's own maps (cia_screen_images)
    x1 = m.normalize_device(greens[0])
    prob1, _ = m.predict(x1)
    q_thr = float(torch.quantile(prob1.flatten()[::7].float(), 0.995).item())
    res["screen_images_prob_thresh"] = q_thr

    for F in Fs:
        g = g_all[:F]
        pmap, dmap = p_all[:F].contiguous(), d_all[:F].contiguous()
        x = torch.empty((F, H, W), dtype=torch.float32, device="cuda")
        labels = torch.empty((F, H, W), dtype=torch.int32, device="cuda")
        n_inst = torch.zeros(F, dtype=torch.int32, device="cuda")
        out_pf = [eng.alloc_outputs(1024, 1) for _ in range(F)]
        out_b = eng.alloc_outputs(1024 * F, F)
        out_si = eng.alloc_outputs(8192 * F, F)

        def per_field():
            for f in range(F):
                eng._check(lib.cia_seg_normalize(h, g[f].data_ptr(), H, W, 3.0, 99.8, x[f].data_ptr(), None, st()))
                eng._check(lib.cia_seg_predict(h, x[f].data_ptr(), H, W, None, None, st()))
                eng._check(lib.cia_seg_instances(h, pmap[f].data_ptr(), dmap[f].data_ptr(), H // 2, W // 2, 2, H, W, 0.479071,
                                                 0.3, labels[f].data_ptr(), n_inst[f:f + 1].data_ptr(), st()))
                eng.screen_fields(g[f:f + 1], labels[f:f + 1], 1024, out_pf[f])

        def batched():
            eng._check(lib.cia_seg_normalize_fields(h, g.data_ptr(), F, H, W, 3.0, 99.8, x.data_ptr(), st()))
            eng._check(lib.cia_seg_predict_fields(h, x.data_ptr(), F, H, W, None, None, st()))
            eng._check(lib.cia_seg_instances_fields(h, pmap.data_ptr(), dmap.data_ptr(), F, H // 2, W // 2, 2, H, W, 0.479071,
                                                    0.3, labels.data_ptr(), n_inst.data_ptr(), st()))
            eng.screen_fields(g, labels, 1024, out_b)

        def fused():
            eng.screen_images(g, g, 65536, out_si, q_thr, 0.3, n_instances=n_inst)

        for fn in (per_field, batched, fused):
            fn()
        torch.cuda.synchronize()
        eng.check_status()
        counts = {}
        for name, fn in (("per_field", per_field), ("batched", batched), ("screen_images", fused)):
            l0 = eng.launch_count
            fn()
            torch.cuda.synchronize()
            counts[name] = eng.launch_count - l0
        eng.check_status()
        cells_b = int(out_b["counts"][0].item())
        cells_pf = sum(int(o["counts"][0].item()) for o in out_pf)
        t = {"per_field": 1e9, "batched": 1e9, "screen_images": 1e9}
        for _ in range(args.rounds):         # alternate the forms in the same process
            t["per_field"] = min(t["per_field"], best_of(per_field, 1, 2))
            t["batched"] = min(t["batched"], best_of(batched, 1, 2))
            t["screen_images"] = min(t["screen_images"], best_of(fused, 1, 2))
        eng.check_status()
        si_cells = int(out_si["counts"][0].item())
        si_inst = n_inst.cpu().numpy().tolist()
        # candidates of the synthetic network's maps at that threshold (the same maps the fused call made)
        eng._check(lib.cia_seg_normalize_fields(h, g.data_ptr(), F, H, W, 3.0, 99.8, x.data_ptr(), st()))
        pr = torch.empty((F, H // 2, W // 2), dtype=torch.float32, device="cuda")
        eng._check(lib.cia_seg_predict_fields(h, x.data_ptr(), F, H, W, pr.data_ptr(), None, st()))
        cand = int((pr[:, 2:-2, 2:-2] > q_thr).sum().item())
        r = {
            "per_field_chain": {"ms_per_field": t["per_field"] / F, "cells_per_s": cells_pf / (t["per_field"] * 1e-3),
                                "launches_per_call": counts["per_field"], "cells": cells_pf},
            "batched_chain": {"ms_per_field": t["batched"] / F, "cells_per_s": cells_b / (t["batched"] * 1e-3),
                              "launches_per_call": counts["batched"], "cells": cells_b},
            "screen_images": {"ms_per_field": t["screen_images"] / F, "cells_per_s": si_cells / (t["screen_images"] * 1e-3),
                              "launches_per_call": counts["screen_images"], "cells": si_cells, "candidates": cand,
                              "instances_per_field": si_inst},
            "speedup_batched_over_per_field": t["per_field"] / t["batched"],
        }
        res["per_F"][str(F)] = r
        print(F, json.dumps(r), flush=True)
        del x, labels, out_pf, out_b, out_si, pr
        torch.cuda.empty_cache()
    with open(os.path.join(args.out, "images_probe.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
