"""bench.py keeps the driver's JSON contract: the reference (CPU) arm is exercised here on a small workload; the B200
arm under -m gpu.  Sizes are chosen so that both finish in seconds - they check the line's shape, not its numbers."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"}


def _run(args, timeout=600):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_reference_arm_prints_the_contract_line():
    line = _run(["--impl", "reference", "--workload", "C1", "--steps", "1", "--warmup", "0", "--cpu-sample-rows", "512"])
    assert BASE_KEYS <= set(line) and line["impl"] == "reference"
    assert line["metric"] == "finch_full_hierarchy_embeddings_per_s" and line["unit"] == "embeddings/s"
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["data"] == "synthetic"
    assert "workload" in line["config"] and "model" not in line["config"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and "sample" in cb
    # (the timing arm feeds approximate level-0 neighbours as initial_rank - no min_sim cut - so only the first levels
    # coincide with the reference's [1170, 101, 25, 8, 5] for BASELINE configs[0])
    assert line["cpu_baseline"]["detail"]["num_clust"][:2] == [1170, 101]
    # one full pass of the level-0 stage sits next to the extrapolated figure
    assert line["cpu_baseline"]["detail"]["nn_stage_full_s"] > 0


def test_reference_arm_uses_all_cores_under_torchrun_environment():
    """torch.distributed.run exports OMP_NUM_THREADS=1; the CPU arm must still time the reference on every core."""
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "C1", "--steps", "1",
                        "--warmup", "0", "--cpu-sample-rows", "256", "--no-full-nn"], capture_output=True, text=True,
                       timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["cpu_baseline"]["cores"] == (os.cpu_count() or 1)


@pytest.mark.gpu
def test_b200_arm_prints_the_contract_line(tmp_path, golden_dir):
    line = _run(["--workload", "C1", "--steps", "2", "--warmup", "3", "--cpu-sample-rows", "512",
                 "--dump-outputs", str(tmp_path)])
    assert BASE_KEYS <= set(line) and "impl" not in line
    assert len(line["step_host_ms_rank0"]) == 2
    # the outputs of the last timed call: the label matrix of the unmodified reference on every row but ties (C1 has one)
    c, num_clust = np.load(tmp_path / "c.npy"), np.load(tmp_path / "num_clust.npy")
    assert c.dtype == num_clust.dtype == np.float64 and not (tmp_path / "c_rows.npy").exists()
    g = np.load(os.path.join(golden_dir, "c1_9537x512.npz"))
    assert num_clust.tolist() == [1170, 101, 25, 8, 5] and c.shape == (9537, 5)
    assert (c != g["c"]).any(axis=1).sum() <= 2
    assert {"gpu_launches", "clocks", "roofline", "nn_stage", "finch_seconds", "parity", "e2e_pageable", "retrieval"} <= set(line)
    assert line["gpu_launches"] > 0 and line["n_gpus"] == 1 and line["steps"] == 2 and line["warmup"] >= 3
    rf = line["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(rf) and rf["bound"] == "tensor"
    assert abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9 and rf["frac"] <= 1.0      # a hardware rate
    assert "traffic_source" in rf and "algorithmic_tflops" in rf
    e2e = line["e2e"]
    assert e2e["h2d_bytes_per_step"] == 9537 * 512 * 4 and e2e["d2h_bytes_per_step"] > 0 and e2e["value"] > 0
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(line["clocks"])
    assert line["config"]["partitions"] == [1170, 101, 25, 8, 5]
    par = line["parity"]
    assert par["levels_ge1_equal_oracle_given_gpu_nn0"] is True
    assert par["first_neighbors_tc_equals_exact_kernel"]["equal"] and par["first_neighbors_tc_equals_exact_kernel"]["rows_checked"] == 9537
    assert par["first_neighbors_equal_oracle"]["equal_outside_ties"] and par["first_neighbors_equal_oracle"]["rows_checked"] == 9537
    assert line["e2e_pageable"]["h2d_bytes_per_step"] == e2e["h2d_bytes_per_step"] and line["e2e_pageable"]["value"] > 0
    assert line["retrieval"]["C2_top50"]["indices_equal_exact_kernels"] is True
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["unit"] == line["unit"]


def test_dumped_outputs_stay_within_their_budget(tmp_path):
    """bench.dump_outputs: a label matrix too large for the budget is written as the same seeded row sample every time."""
    import bench
    c = np.arange(3000 * 4, dtype=np.int32).reshape(3000, 4)
    bench.dump_outputs(tmp_path / "full", c, [3000, 40, 5, 2])
    assert np.array_equal(np.load(tmp_path / "full" / "c.npy"), c) and not (tmp_path / "full" / "c_rows.npy").exists()
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, c, [3000, 40, 5, 2], max_bytes=20000)
        assert sum(f.stat().st_size for f in (tmp_path / run).iterdir()) <= 20000 + 3 * 128      # (+ .npy headers)
    rows = np.load(tmp_path / "a" / "c_rows.npy")
    assert np.array_equal(rows, np.load(tmp_path / "b" / "c_rows.npy")) and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "c.npy"), c[rows.astype(np.int64)])
    assert np.load(tmp_path / "a" / "num_clust.npy").tolist() == [3000, 40, 5, 2]


def test_stall_rule_of_the_timed_loops():
    """bench.has_stalled_call: a loop is measured again only when a single call stands out (the stalls seen on the GPU
    boxes: 55 ms and 149 ms calls among 15-19 ms ones), never for ordinary jitter or for uniformly slow calls."""
    import bench
    assert bench.has_stalled_call([55.808, 14.104, 14.167, 14.156, 14.568, 14.579, 14.595, 14.975, 15.322, 14.985])
    assert bench.has_stalled_call([19.078, 19.157, 19.148, 149.498, 77.455, 19.001, 18.962, 18.966, 19.831, 23.916])
    assert not bench.has_stalled_call([26.677, 25.38, 26.022, 26.867, 26.174, 26.672, 27.257, 27.216, 27.129, 26.526])
    assert not bench.has_stalled_call([37.8] * 10)          # a slow box is not a stall
    assert not bench.has_stalled_call([30.0, 90.0])          # too few calls to tell
