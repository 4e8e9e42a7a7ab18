"""Times enumgpu_solve_objectives (many cost vectors over one feasible set) on one GPU and prints one JSON line.

For dense (12, 40) seed 1 (the headline LP, 5.59 G bases) and dense (10, 30) seed 1 (30.0 M bases), and K in
{1, 16, 256, 4096} cost vectors drawn from a normal distribution with a fixed seed:
  wall_ms       host clock around the call (it ends in a stream synchronisation)
  kernel_ms     the call's own CUDA-event span (listing + objective passes)
  k_objectives_ms, k_obj_values_ms
                device time of those kernels alone, from a separate torch.profiler run with CUDA activities
and, per LP, one enumgpu_solve with the LP's own c for comparison (wall and kernel_ms).
Each entry is warmed up once and then timed `--reps` times; medians and spreads are printed next to the device name,
its power limit and its maximum SM clock, read in the same run.
Usage: python scripts/bench_objectives.py [--reps 5] [--ks 1,16,256,4096]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import simplexmethod_b200 as sm  # noqa: E402
from simplexmethod_b200 import _abi, lpgen  # noqa: E402


def device_facts():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [v.strip() for v in q.split(",")]
        return {"device": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:            # the numbers are still reported, marked as lacking the card's facts
        return {"device": "unknown", "error": str(e)}


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def kernel_times(fn):
    """Device time (ms) per kernel family of one call of fn, from torch.profiler; None if the profiler is unavailable."""
    try:
        import torch  # noqa: F401
        from torch.profiler import ProfilerActivity, profile
    except Exception:
        return None
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    out = {"k_objectives_ms": 0.0, "k_obj_values_ms": 0.0, "k_obj_finish_ms": 0.0, "enumeration_ms": 0.0}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        name = e.key
        if "k_objectives" in name:
            out["k_objectives_ms"] += us * 1e-3
        elif "k_obj_values" in name:
            out["k_obj_values_ms"] += us * 1e-3
        elif "k_obj_finish" in name:
            out["k_obj_finish_ms"] += us * 1e-3
        elif "k_shared" in name or "k_independent" in name:
            out["enumeration_ms"] += us * 1e-3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--ks", default="1,16,256,4096")
    args = ap.parse_args()
    L = sm.lib()
    if L.enumgpu_device_count() < 1:
        raise SystemExit("bench_objectives needs a CUDA device (libenumgpu has no CPU fallback)")
    out = device_facts()
    o = _abi.Options(-1.0, -1.0, 0, 0, 0, 0, None, None, 0, 0, 0, 0)
    for m, n in [(12, 40), (10, 30)]:
        A, b, c, mx = lpgen.dense_lp(m, n, 1)
        A = np.asfortranarray(A, dtype=float)
        b = np.ascontiguousarray(b, dtype=float)
        c = np.ascontiguousarray(c, dtype=float)
        p = _abi.Problem(m, n, m, int(bool(mx)), A.ctypes.data, b.ctypes.data, c.ctypes.data)
        entry = {}
        res = _abi.Result()
        wall, kms = [], []
        for i in range(args.reps + 1):
            t0 = time.perf_counter()
            assert L.enumgpu_solve(C.byref(p), C.byref(o), C.byref(res)) == _abi.OK, sm.last_error()
            if i >= 1:
                wall.append((time.perf_counter() - t0) * 1e3)
                kms.append(res.kernel_ms)
        entry["solve"] = {"wall_ms": summary(wall), "kernel_ms": summary(kms), "n_feasible": res.n_feasible,
                          "algo_used": res.algo_used}
        for k in [int(v) for v in args.ks.split(",")]:
            costs = np.ascontiguousarray(np.random.default_rng(k).standard_normal((k, n)))
            outs = (_abi.Result * k)()

            def call():
                rc = L.enumgpu_solve_objectives(C.byref(p), C.byref(o), k, costs.ctypes.data_as(C.POINTER(C.c_double)),
                                                n, 0, outs)
                assert rc == _abi.OK, sm.last_error()

            wall, kms = [], []
            for i in range(args.reps + 1):
                t0 = time.perf_counter()
                call()
                if i >= 1:
                    wall.append((time.perf_counter() - t0) * 1e3)
                    kms.append(outs[0].kernel_ms)
            e = {"wall_ms": summary(wall), "kernel_ms": summary(kms), "n_launches": outs[0].n_launches,
                 "pairs": int(outs[0].n_feasible) * k,
                 "vs_one_solve": statistics.median(wall) / entry["solve"]["wall_ms"]["median"]}
            kt = kernel_times(call)
            e["profile"] = kt if kt is not None else "not measured (torch.profiler unavailable)"
            entry[f"K{k}"] = e
        out[f"dense_{m}_{n}"] = entry
    out["device_after"] = device_facts()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
