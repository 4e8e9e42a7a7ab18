"""bench.py's JSON contract.  CPU: the --impl reference arm (the oracle on host cores).  GPU: the product arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}
DUMPED = ("status", "best_rank", "basis", "x_B", "objective", "counts")


def run_bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def load_dump(d):
    got = {name: np.load(os.path.join(d, name + ".npy")) for name in DUMPED}
    assert all(v.dtype == np.float64 for v in got.values())
    return got


def assert_dump_is_record(got, i, res, m):
    """Row i of a --dump-outputs directory against a result struct, bit for bit."""
    assert got["status"][i] == res.status and got["best_rank"][i] == res.best_rank
    assert got["counts"][i].tolist() == [res.n_bases, res.n_singular, res.n_infeasible, res.n_feasible]
    assert got["basis"][i].tolist() == list(res.basis)[:m]
    assert got["x_B"][i].tolist() == list(res.x_B)[:m] and got["objective"][i] == res.objective


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_reference_arm_dump_outputs_cpu(oracle, tmp_path):
    """--dump-outputs plumbing on the CPU arm: the last step's records as float64, identical from run to run and
    equal, field for field, to the record the oracle returns.  The arm IS the oracle, so this checks the dump and
    its determinism, not the answer; test_product_arm_dump_outputs_gpu compares two implementations."""
    from simplexmethod_b200 import lpgen
    dumps = []
    for k in range(2):
        d = tmp_path / f"run{k}"
        run_bench("--impl", "reference", "--m", "6", "--n", "16", "--seed", "3", "--steps", "2", "--warmup", "0",
                  "--dump-outputs", str(d))
        dumps.append(load_dump(d))
    assert all(np.array_equal(dumps[0][name], dumps[1][name]) for name in DUMPED)
    A, b, c, mx = lpgen.dense_lp(6, 16, 3)
    res, _ = oracle.solve(A, b, c, mx)
    assert dumps[0]["basis"].shape == (1, 6) and dumps[0]["counts"][0, 0] == 8008     # C(16, 6): one full window
    assert_dump_is_record(dumps[0], 0, res, 6)


def test_reference_arm_json_cpu():
    d = run_bench("--impl", "reference", "--m", "8", "--n", "24", "--steps", "1", "--warmup", "1")
    assert BASE_KEYS <= set(d)
    assert d["impl"] == "reference" and d["unit"] == "bases/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] > 1e5
    assert d["e2e"] == {"value": d["value"], "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0
    rc = d["reference_code"]            # side figure: the reference's own per-basis code (oracle/_ref), when built
    assert rc is None or rc.get("value", 0) > 1e3 or "unavailable" in rc


@pytest.mark.gpu
def test_product_arm_json_gpu(gpu_lib):
    d = run_bench("--m", "10", "--n", "30", "--steps", "3", "--warmup", "3", "--cpu-ranks", "3000000")
    assert BASE_KEYS | {"clocks", "roofline", "cpu_baseline"} <= set(d)
    assert "impl" not in d and d["n_gpus"] == 1 and d["scaling"] == "strong" and d["vs_baseline"] is None
    assert d["gpu_launches"] == d["steps"]           # ONE kernel per enumeration (fused finalize, no memset)
    assert d["ms_per_step_best"] <= d["ms_per_step_median"] and d["roofline"]["launch_ms_best"] <= d["roofline"]["launch_ms_median"]
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] == 256 and d["e2e"]["value"] > 1e8
    r = d["roofline"]
    assert r["bound"] == "fp64" and r["unit"] == "TFLOP/s" and r["peak"] > 10 and r["frac"] == pytest.approx(r["achieved"] / r["peak"])
    assert r["per_basis_lu_kernel"]["frac"] < 1.0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 1e5
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    assert d["result"]["best_rank"] == 1579911 and d["result"]["n_feasible"] == 66804      # the oracle's answer for this LP


@pytest.mark.gpu
def test_product_arm_dump_outputs_gpu(gpu_lib, oracle, tmp_path):
    """--dump-outputs on the GPU arm: the merged record of the last timed step, bit for bit the oracle's."""
    from simplexmethod_b200 import lpgen
    d = run_bench("--m", "8", "--n", "24", "--seed", "2", "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
                  "--dump-outputs", str(tmp_path))
    assert d["steps"] == 2 and d["gpu_launches"] == 2
    got = load_dump(tmp_path)
    assert got["basis"].shape == (1, 8)
    A, b, c, mx = lpgen.dense_lp(8, 24, 2)
    res, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count())
    assert_dump_is_record(got, 0, res, 8)
    assert got["basis"][0].tolist() == d["result"]["basis"] and got["objective"][0] == d["result"]["objective"]
