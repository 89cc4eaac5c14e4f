"""Multi-GPU screening (SURVEY.md §8e): the strain / file loops of ``screen_mutant_samples``
(improved_detection.py:164-234) sharded over one process per GPU.

Fields are independent, so they shard by index (field i -> rank i mod R) with NO data-path
collective: every rank holds a full replica of the artifacts and screens its own fields through
the fused CUDA path.  Two exchanges finish a screen:

* one ``all_reduce(sum)`` of the per-strain accumulator ``[S, 8]`` float64 -- the reductions behind
  det:151-152 and det:202-211 (NCCL on GPUs, gloo in the CPU tests).  Row: {n_cells,
  n_conservative_anomalies, n_moderate_anomalies, sum mse, sum mse^2, sum mae, sum mae^2, 0};
* the per-cell rows of ``detailed_cell_results.csv`` (det:217-234) stay rank-local on the device
  side and are concatenated on the HOST in reference order (strain order, sorted file, ascending
  label) -- an object gather, no GPU collective, as north_star restricts NCCL to the count reduce.

``ShardedScreen`` is the engine-agnostic driver (the per-rank scorer is injected: ``GpuFieldScorer``
in production, a NumPy stand-in in the gloo tests); ``screen_mutant_samples_sharded`` is the
drop-in twin of det:155-244 built on it.
"""
from __future__ import annotations

import math
import os
from glob import glob

import numpy as np
import torch
import torch.distributed as dist

ACC_COLS = 8
ROW_KEYS = ("mse", "mae", "dec_cons", "dec_mod", "pred_cons", "pred_mod")


def _world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_fields(n_fields: int, rank: int, world: int):
    """Field i -> rank i mod world (round robin keeps per-strain load even)."""
    return list(range(rank, n_fields, world))


def allreduce_strain_acc(acc: torch.Tensor) -> torch.Tensor:
    """Sum the [S, 8] float64 accumulator over ranks (no-op without a process group)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(acc, op=dist.ReduceOp.SUM)
    return acc


def strain_summary(acc_row, sample_name=None, files_processed=None):
    """Per-strain result dict (det:202-212) from an accumulator row.  std is the
    population std (ddof=0) via sqrt(E[x^2] - E[x]^2) in float64."""
    n, nc, nm, s1, s2, a1, a2 = [float(v) for v in acc_row[:7]]
    if n <= 0:
        return None
    mean_mse, mean_mae = s1 / n, a1 / n
    out = {
        "total_cells": int(round(n)),
        "conservative_anomaly_rate": nc / n,
        "moderate_anomaly_rate": nm / n,
        "mean_mse": mean_mse,
        "std_mse": math.sqrt(max(s2 / n - mean_mse * mean_mse, 0.0)),
        "mean_mae": mean_mae,
        "std_mae": math.sqrt(max(a2 / n - mean_mae * mean_mae, 0.0)),
    }
    if sample_name is not None:
        out = {"sample_name": sample_name, **out}
    if files_processed is not None:
        out["files_processed"] = files_processed
    return out


def accumulate_rows(acc: np.ndarray, strain: int, rows: dict):
    """Host restatement of ``cia_strain_accumulate`` for one field's rows (used by scorers that
    do not accumulate on the device)."""
    a = acc[strain]
    m, e = rows["mse"].astype(np.float64), rows["mae"].astype(np.float64)
    a[0] += len(m)
    a[1] += int((rows["pred_cons"] == -1).sum())
    a[2] += int((rows["pred_mod"] == -1).sum())
    a[3] += m.sum(); a[4] += (m * m).sum(); a[5] += e.sum(); a[6] += (e * e).sum()


class GpuFieldScorer:
    """Per-rank scorer on one GPU: chunks of equally sized fields through ``BatchScreen.run_host``
    (pinned staging, run-length label transport, fused ``cia_screen_fields*`` call, device-side
    per-strain accumulation)."""

    def __init__(self, engine, chunk_fields: int = 16, label_transport: str = "rle", host_threads: int = 0):
        self.eng, self.Fc = engine, chunk_fields
        self.label_transport, self.host_threads = label_transport, host_threads
        self._bs = None

    def _batch(self, H, W, max_label, n_strains):
        from .batch import BatchScreen
        bs = self._bs
        if bs is None or (bs.H, bs.W, bs.n_strains) != (H, W, n_strains) or bs.max_label < max_label:
            bs = BatchScreen(self.eng, H, W, max(max_label, 1), chunk_fields=self.Fc, n_strains=n_strains,
                             label_transport=self.label_transport, host_threads=self.host_threads)
            self._g = torch.zeros((self.Fc, H, W), dtype=torch.int16).pin_memory()
            self._l = torch.zeros((self.Fc, H, W), dtype=torch.int32).pin_memory()
            self._bs = bs
        return bs

    def score(self, fields, strains, n_strains):
        """fields: list of (green uint16 [H,W], labels int32 [H,W]) pairs OR of zero-argument callables
        returning such a pair (file decode + segmentation); callables of chunk k+1 are resolved by a
        thread pool while the device scores chunk k, so at most two chunks of fields are alive.
        strains: strain id per field.  Returns (acc [S,8] float64 tensor on this rank's device, list
        of per-field row dicts)."""
        from concurrent.futures import ThreadPoolExecutor
        dev = self.eng.tdev
        total = torch.zeros((n_strains, ACC_COLS), dtype=torch.float64, device=dev)
        if not fields:
            return total, []
        out = []
        chunks = [list(range(c0, min(c0 + self.Fc, len(fields)))) for c0 in range(0, len(fields), self.Fc)]
        resolve = lambda f: f() if callable(f) else f
        with ThreadPoolExecutor(max_workers=min(8, self.Fc)) as pool:
            pending = [pool.submit(resolve, fields[i]) for i in chunks[0]]
            for ci, idx in enumerate(chunks):
                chunk = [p.result() for p in pending]
                pending = [pool.submit(resolve, fields[i]) for i in chunks[ci + 1]] if ci + 1 < len(chunks) else []
                ok = [f for f in chunk if f is not None]       # None: the loader gave up on this file (det:113-115)
                if not ok:
                    out.extend({**{k: np.zeros(0) for k in ROW_KEYS}, "label": np.zeros(0, np.int32)} for _ in chunk)
                    continue
                H, W = ok[0][0].shape
                blank = (np.zeros((H, W), np.uint16), np.zeros((H, W), np.int32))
                chunk = [f if f is not None else blank for f in chunk]
                max_label = max(int(l.max()) if l.size else 0 for _, l in chunk)
                old = self._bs
                bs = self._batch(H, W, max_label, n_strains)
                if bs is not old:                              # first chunk, or a larger label range / field size
                    bs.sync()
                    bs.acc.zero_()
                self._l.zero_()                                # a short last chunk is padded with empty fields
                for j, (g, l) in enumerate(chunk):
                    if g.shape != (H, W) or l.shape != (H, W):
                        raise ValueError("a chunk needs equally sized fields (pad or group by size)")
                    if g.dtype != np.uint16:
                        raise TypeError("fields must be uint16 (widen 8-bit fields before screening)")
                    self._g[j].copy_(torch.from_numpy(np.ascontiguousarray(g).view(np.int16)))
                    self._l[j].copy_(torch.from_numpy(np.ascontiguousarray(l, np.int32)))
                st = torch.zeros(self.Fc, dtype=torch.int32)
                st[:len(chunk)] = torch.tensor([strains[i] for i in idx], dtype=torch.int32)
                bs.run_host(self._g, self._l, self.Fc, st.to(dev))
                r = bs.collect_host()                          # synchronises, raises on a device-side status
                total += bs.acc
                bs.acc.zero_()
                starts = np.concatenate([[0], np.cumsum(r["field_counts"])])
                for j in range(len(chunk)):
                    s0, s1 = int(starts[j]), int(starts[j + 1])
                    rows = {k: r[k][s0:s1].copy() for k in ROW_KEYS}
                    rows["label"] = r["cells"]["label"][s0:s1].copy()
                    out.append(rows)
        return total, out


    def score_images(self, fields, strains, n_strains, prob_thresh: float, nms_thresh: float, max_label: int = 4096):
        """``score`` for fields given as (seg channel, green channel) uint16 [H,W] pairs (or zero-argument callables
        returning one; None = the loader gave up on the file): each chunk is segmented AND screened on the device
        through ``BatchScreen.run_images_host`` (StarDist model loaded on the engine), so only the images cross PCIe
        and the loader threads make no GPU calls.  ``max_label`` bounds the instances of one field (CIA_E_LABEL
        beyond).  Returns what ``score`` returns."""
        from concurrent.futures import ThreadPoolExecutor
        from .batch import BatchScreen
        dev = self.eng.tdev
        total = torch.zeros((n_strains, ACC_COLS), dtype=torch.float64, device=dev)
        if not fields:
            return total, []
        empty = lambda: {**{k: np.zeros(0) for k in ROW_KEYS}, "label": np.zeros(0, np.int32)}
        out = []
        chunks = [list(range(c0, min(c0 + self.Fc, len(fields)))) for c0 in range(0, len(fields), self.Fc)]
        resolve = lambda f: f() if callable(f) else f
        with ThreadPoolExecutor(max_workers=min(8, self.Fc)) as pool:
            pending = [pool.submit(resolve, fields[i]) for i in chunks[0]]
            for ci, idx in enumerate(chunks):
                chunk = [p.result() for p in pending]
                pending = [pool.submit(resolve, fields[i]) for i in chunks[ci + 1]] if ci + 1 < len(chunks) else []
                ok = [j for j, f in enumerate(chunk) if f is not None]
                if not ok:
                    out.extend(empty() for _ in chunk)
                    continue
                H, W = chunk[ok[0]][1].shape
                bs = self._bs
                if bs is None or (bs.H, bs.W, bs.n_strains, bs.max_label) != (H, W, n_strains, max_label):
                    if bs is not None:
                        bs.sync()
                    bs = BatchScreen(self.eng, H, W, max_label, chunk_fields=self.Fc, n_strains=n_strains)
                    self._g = torch.zeros((self.Fc, H, W), dtype=torch.int16).pin_memory()
                    self._s = torch.zeros((self.Fc, H, W), dtype=torch.int16).pin_memory()
                    self._bs = bs
                bs.acc.zero_()
                same = all(chunk[j][0] is chunk[j][1] for j in ok)     # single-channel fields: one upload
                for k, j in enumerate(ok):
                    seg, g = chunk[j]
                    if seg.shape != (H, W) or g.shape != (H, W):
                        raise ValueError("a chunk needs equally sized fields (pad or group by size)")
                    if g.dtype != np.uint16 or seg.dtype not in (np.uint16, np.uint8):
                        raise TypeError("fields must be uint16 (widen 8-bit fields before screening)")
                    self._g[k].copy_(torch.from_numpy(np.ascontiguousarray(g).view(np.int16)))
                    if not same:
                        self._s[k].copy_(torch.from_numpy(np.ascontiguousarray(seg, np.uint16).view(np.int16)))
                st = torch.tensor([strains[idx[j]] for j in ok], dtype=torch.int32)
                bs.run_images_host(self._g if same else self._s, self._g, len(ok), prob_thresh, nms_thresh, st.to(dev))
                r = bs.collect_host()                          # synchronises, raises on a device-side status
                total += bs.acc
                starts = np.concatenate([[0], np.cumsum(r["field_counts"])])
                rows = {}
                for k, j in enumerate(ok):
                    s0, s1 = int(starts[k]), int(starts[k + 1])
                    rows[j] = {kk: r[kk][s0:s1].copy() for kk in ROW_KEYS}
                    rows[j]["label"] = r["cells"]["label"][s0:s1].copy()
                out.extend(rows.get(j) or empty() for j in range(len(chunk)))
        return total, out


class ShardedScreen:
    """Shards a list of fields over the ranks of the current process group, scores each rank's share
    and assembles the global result.  ``scorer.score(fields, strains, n_strains) -> (acc, rows)``."""

    def __init__(self, scorer, score=None):
        """``score``: the scorer's method to call (default ``scorer.score``; e.g. a bound ``score_images``)."""
        self.scorer = scorer
        self.score = score or scorer.score
        self.rank, self.world = _world()

    def screen(self, load_field, n_fields: int, field_strain, n_strains: int):
        """``load_field(i) -> (green, labels)`` is called only for this rank's fields (so decoding and
        segmentation shard too).  Returns ``(acc, rows)``: the all-reduced [S,8] accumulator (numpy,
        identical on every rank) and, on rank 0, the per-cell rows of all fields in reference order
        as a dict of arrays with ``field`` (global index), ``strain`` and ``label`` columns
        (``None`` on the other ranks)."""
        mine = shard_fields(n_fields, self.rank, self.world)
        fields = [(lambda i=i: load_field(i)) for i in mine]       # resolved chunk by chunk by the scorer
        acc, rows = self.score(fields, [int(field_strain[i]) for i in mine], n_strains)
        acc = allreduce_strain_acc(acc)                       # the path's only collective
        local = [(i, r) for i, r in zip(mine, rows)]
        if self.world > 1:
            gathered = [None] * self.world if self.rank == 0 else None
            dist.gather_object(local, gathered, dst=0)
        else:
            gathered = [local]
        acc_np = acc.detach().cpu().numpy()
        if self.rank != 0:
            return acc_np, None
        by_field = {i: r for part in gathered for i, r in part}
        assert sorted(by_field) == list(range(n_fields)), "every field must be scored by exactly one rank"
        cols = {k: [] for k in ROW_KEYS + ("label", "field", "strain")}
        for i in range(n_fields):                             # reference order: field order, ascending label
            r = by_field[i]
            n = len(r["label"])
            for k in ROW_KEYS + ("label",):
                cols[k].append(r[k])
            cols["field"].append(np.full(n, i, np.int64))
            cols["strain"].append(np.full(n, int(field_strain[i]), np.int64))
        return acc_np, {k: (np.concatenate(v) if v else np.zeros(0)) for k, v in cols.items()}


def screen_mutant_samples_sharded(screener, test_folders_dict, output_dir=None, chunk_fields: int = 16):
    """Sharded twin of ``ProductionMutantScreening.screen_mutant_samples`` (det:155-244): call it
    from every rank of an initialised process group (one process per GPU; ``screener`` built on that
    rank's device).  Files are enumerated like the reference (strains in dict order, ``sorted(glob)``),
    sharded round robin, read and segmented on their rank, scored through the fused path; the
    per-strain numbers come from the all-reduced accumulator.  With a GPU StarDist model (``stardist_dir=``)
    the loader threads only read files and split channels; segmentation and screening run per chunk in
    ``cia_screen_images`` on the rank's stream (no labels through the host).  A caller's own ``segmenter``
    keeps the (green, labels) route.  Returns ``(results, detailed_results)``
    on rank 0 -- same keys as det:202-212 / 225-234 -- and ``({}, [])`` elsewhere."""
    rank, world = _world()
    names, files, strain_of = [], [], []
    for sample_name, folder in test_folders_dict.items():
        tif = sorted(glob(os.path.join(folder, "*.tif")))              # det:167
        if not tif:
            if rank == 0:
                print(f"  No .tif files found in {folder}")
            continue
        names.append(sample_name)
        files.extend(tif)
        strain_of.extend([len(names) - 1] * len(tif))
    if not files:
        return {}, []

    sd_model = screener.stardist_model

    def load_images(i):
        try:
            image = screener.imread(files[i])
            if image.ndim == 3 and image.shape[-1] >= 3:                  # det:54-59
                return np.ascontiguousarray(image[..., 2]), np.ascontiguousarray(image[..., 1])
            return image, image
        except Exception as e:                                            # det:113-115: the file contributes no cells
            print(f"Error processing {files[i]}: {e}")
            return None

    def load(i):
        try:
            image = screener.imread(files[i])
            if image.ndim == 3 and image.shape[-1] >= 3:                  # det:54-59
                seg, green = image[..., 2], image[..., 1]
            else:
                seg = green = image
            labels = screener._segment(seg)
            if hasattr(labels, "cpu"):        # stardist_dir=...: the GPU segmentation returns a device tensor
                labels = labels.cpu().numpy()
            return np.ascontiguousarray(green), np.ascontiguousarray(labels, np.int32)
        except Exception as e:                                            # det:113-115: the file contributes no cells
            print(f"Error processing {files[i]}: {e}")
            return None

    scorer = GpuFieldScorer(screener.engine, chunk_fields=chunk_fields)
    if sd_model is not None:
        th = sd_model.thresholds
        sh = ShardedScreen(scorer, lambda f, st, ns: scorer.score_images(f, st, ns, th["prob"], th["nms"]))
        acc, rows = sh.screen(load_images, len(files), strain_of, len(names))
    else:
        sh = ShardedScreen(scorer)
        acc, rows = sh.screen(load, len(files), strain_of, len(names))
    if rank != 0:
        return {}, []
    results, detailed = {}, []
    for s, name in enumerate(names):
        r = strain_summary(acc[s], sample_name=name, files_processed=strain_of.count(s))
        if r is None:
            print(f"  No quality cells extracted from {name}")
            continue
        # key order of det:202-212
        results[name] = {k: r[k] for k in ("sample_name", "total_cells", "files_processed",
                                           "conservative_anomaly_rate", "moderate_anomaly_rate",
                                           "mean_mse", "std_mse", "mean_mae", "std_mae")}
        sel = np.nonzero(rows["strain"] == s)[0]
        for cid, j in enumerate(sel):                                     # det:217-234, cell_id = enumeration order
            detailed.append({"sample_name": name, "cell_id": cid, "mse": rows["mse"][j], "mae": rows["mae"][j],
                             "conservative_anomaly": rows["pred_cons"][j] == -1,
                             "moderate_anomaly": rows["pred_mod"][j] == -1,
                             "conservative_score": -rows["dec_cons"][j],       # det:149-150: scores are negated
                             "moderate_score": -rows["dec_mod"][j]})
    if output_dir:
        screener.save_and_visualize_results(results, detailed, output_dir)   # det:242
    return results, detailed
