"""bench.py's output contract, checked on the committed bench lines (profiles/*.json are the driver-format
lines of real B200 runs) and on the argument parser -- no GPU needed -- and, on a GPU, on a tiny run of --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"}


def _line(name):
    for raw in open(os.path.join(ROOT, "profiles", name)):
        if raw.startswith("{"):
            return json.loads(raw)
    raise AssertionError(name)


def test_native_line_carries_the_contract_keys():
    d = _line("r2k_bench_default.json")
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["metric"] in base["metric"] and d["unit"] == "cells/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["warmup"] >= 3 and d["gpu_launches"] > 0
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] > 0
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    c = d["cpu_baseline"]
    assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["sample"]
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_final_line_carries_the_segmentation_extras():
    """the last bench line of the round: the contract keys plus extra.segmentation (SURVEY 8f N2)"""
    d = _line("r2u_bench_default.json")
    assert BASE_KEYS <= set(d), BASE_KEYS - set(d)
    sg = d["extra"]["segmentation"]
    assert abs(sg["ms_per_field"] - (sg["normalize_ms"] + sg["unet_ms"] + sg["instances_ms"])) < 1e-6
    assert sg["instances"] > 0 and sg["candidates"] > sg["instances"] and sg["gpu_launches_per_field"] > 0
    assert abs(sg["unet_tflops"] - sg["unet_gflop"] / sg["unet_ms"]) < 1e-6 * sg["unet_tflops"] + 1e-9
    assert sg["cpu_port"]["kind"] == "port" and sg["cpu_port"]["labels_equal_gpu"] is True
    ch = sg["chain"]
    assert ch["scored_cells"] > 0 and abs(ch["cells_per_s"] - ch["scored_cells"] * 1e3 / ch["ms_per_field"]) < 1e-3


def test_reference_line():
    d = _line("r2k_bench_reference.json")
    assert d["impl"] == "reference" and d["unit"] == "cells/s" and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_multi_gpu_line_is_weak_scaling_with_config5_strains():
    d = _line("r2f_bench_2gpu.json")
    assert d["n_gpus"] == 2 and d["scaling"] == "weak" and d["config"]["strains"] == 100


def test_cli_defaults():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dump-outputs"):
        assert flag in out.stdout


def test_dumped_rows_do_not_depend_on_the_device_order():
    """per-cell rows come out in (field, label) order whatever order they went in, and a pass with more rows than
    the cap is cut to the same seeded sample every time"""
    import bench
    from cell_image_analysis_b200 import _lib
    rng = np.random.default_rng(5)
    n = 1000
    cells = np.zeros(n, _lib.CELL_DTYPE)
    cells["field"], cells["label"] = rng.integers(0, 8, n), rng.permutation(n) + 1
    scores = {k: rng.standard_normal(n) for k in bench.SCORE_KEYS}
    a = bench.per_cell_rows(cells, scores, 300)
    p = rng.permutation(n)
    b = bench.per_cell_rows(cells[p], {k: v[p] for k, v in scores.items()}, 300)
    assert all(np.array_equal(a[k], b[k]) for k in a) and len(a["mse"]) == 300
    key = a["cell_field"].astype(np.int64) * n + a["cell_label"]
    assert np.all(np.diff(key) > 0)


@pytest.mark.gpu
def test_steps_and_dumped_outputs(tmp_path):
    """--steps sets the timed steps, and the last step's outputs do not depend on how many steps ran before it"""
    dumps, launches = {}, {}
    for steps in (1, 2):
        d = tmp_path / f"steps{steps}"
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                              "--fields", "4", "--pool", "2", "--chunk", "2", "--no-cpu-baseline", "--no-svm-extras",
                              "--no-seg-extras", "--dump-outputs", str(d)], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps
        launches[steps] = line["gpu_launches"]            # kernels launched inside the timed window
        dumps[steps] = {f.stem: np.load(f) for f in d.glob("*.npy")}
    assert launches[1] > 0 and launches[2] == 2 * launches[1], launches
    a, b = dumps[1], dumps[2]
    assert set(a) == set(b) and {"strain_acc", "field_counts", "mse", "e2e_mse", "e2e_field_counts"} <= set(a)
    assert a["strain_acc"][:, 0].sum() > 0 and len(a["mse"]) == a["field_counts"].sum()
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        np.testing.assert_allclose(a[k], b[k], rtol=1e-6 if a[k].dtype == np.float32 else 1e-12, err_msg=k)
