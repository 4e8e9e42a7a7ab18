"""Times enumgpu_cost_ranges (cost ranging by enumeration) on one GPU and prints one JSON line.

For dense (12, 40) seed 1 (the headline LP, 5.59 G bases; the ray LP has C(40, 13) = 12.0 G) and dense (10, 30)
seed 1 (30.0 M bases; C(30, 11) = 54.6 M for the rays):
  wall_ms, kernel_ms     host clock around the call (it ends in a stream synchronisation), and its CUDA-event span
  n_vertex_bases, n_ray_bases
                         the feasible bases of each listing
  vertex_listing_ms      kernel_ms of enumgpu_list_feasible on the LP (the call's first listing on its own)
  ray_listing_ms         kernel_ms of enumgpu_list_feasible on the auxiliary LP [A; s*1'] d = (0, ..., 0, s)
  ranging_kernels_ms     device time of k_obj_values, k_ranging and k_ranging_finish in one call, from a separate
                         torch.profiler run with CUDA activities
and one enumgpu_solve of the LP for comparison.  Each entry is warmed up once and then timed `--reps` times; medians
and spreads are printed next to the device name, its power limit and its maximum SM clock, read in the same run.
Usage: python scripts/bench_ranging.py [--reps 5]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import simplexmethod_b200 as sm  # noqa: E402
from simplexmethod_b200 import _abi, lpgen  # noqa: E402
from scripts.bench_objectives import device_facts, summary  # noqa: E402


def ranging_kernel_ms(fn):
    """Device time (ms) of the ranging kernels in one call of fn, from torch.profiler; None if it is unavailable."""
    try:
        from torch.profiler import ProfilerActivity, profile
    except Exception:
        return None
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    out = {"k_obj_values_ms": 0.0, "k_ranging_ms": 0.0, "k_ranging_finish_ms": 0.0, "enumeration_ms": 0.0}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = getattr(e, "cuda_time_total", 0.0)
        name = e.key
        if "k_ranging_finish" in name:
            out["k_ranging_finish_ms"] += us * 1e-3
        elif "k_ranging" in name:
            out["k_ranging_ms"] += us * 1e-3
        elif "k_obj_values" in name:
            out["k_obj_values_ms"] += us * 1e-3
        elif "k_shared" in name or "k_independent" in name:
            out["enumeration_ms"] += us * 1e-3
    out["ranging_kernels_ms"] = out["k_obj_values_ms"] + out["k_ranging_ms"] + out["k_ranging_finish_ms"]
    return out


def problem(A, b, c, mx):
    A = np.asfortranarray(A, dtype=float)
    b = np.ascontiguousarray(b, dtype=float)
    c = np.ascontiguousarray(c, dtype=float)
    return _abi.Problem(A.shape[0], A.shape[1], A.shape[0], int(bool(mx)), A.ctypes.data, b.ctypes.data,
                        c.ctypes.data), (A, b, c)


def ray_lp(A):
    m, n = A.shape
    s = 2.0 ** (int(np.frexp(np.abs(A).max())[1]) - 1)       # the largest power of two <= max|A_ij|
    ba = np.zeros(m + 1)
    ba[m] = s
    return np.vstack([A, np.full(n, s)]), ba


def timed(fn, reps):
    wall, kms = [], []
    for i in range(reps + 1):
        t0 = time.perf_counter()
        k = fn()
        if i >= 1:
            wall.append((time.perf_counter() - t0) * 1e3)
            kms.append(k)
    return {"wall_ms": summary(wall), "kernel_ms": summary(kms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    L = sm.lib()
    if L.enumgpu_device_count() < 1:
        raise SystemExit("bench_ranging needs a CUDA device (libenumgpu has no CPU fallback)")
    out = device_facts()
    o = _abi.Options(-1.0, -1.0, 0, 0, 0, 0, None, None, 0, 0, 0, 0)
    for m, n in [(12, 40), (10, 30)]:
        A, b, c, mx = lpgen.dense_lp(m, n, 1)
        p, keep = problem(A, b, c, mx)
        res = _abi.Result()

        def solve():
            assert L.enumgpu_solve(C.byref(p), C.byref(o), C.byref(res)) == _abi.OK, sm.last_error()
            return res.kernel_ms

        entry = {"solve": timed(solve, args.reps)}
        rg = _abi.Ranging()

        def ranges():
            assert L.enumgpu_cost_ranges(C.byref(p), C.byref(o), C.byref(res), 1e-9, 0, C.byref(rg)) == _abi.OK, \
                sm.last_error()
            return rg.kernel_ms

        e = timed(ranges, args.reps)
        e.update(status=rg.status, n_vertex_bases=rg.n_vertex_bases, n_ray_bases=rg.n_ray_bases, n_launches=rg.n_launches,
                 finite_limits=sum(int(np.isfinite(rg.range[j].decrease)) + int(np.isfinite(rg.range[j].increase))
                                   for j in range(n)))
        pa, keep_a = problem(*ray_lp(A), np.zeros(n), False)
        for key, (P, count) in (("vertex_listing", (p, rg.n_vertex_bases)), ("ray_listing", (pa, rg.n_ray_bases))):
            ranks = np.zeros(max(1, count), dtype=np.uint64)
            n_listed = C.c_uint64()
            lr = _abi.Result()

            def listing():
                assert L.enumgpu_list_feasible(C.byref(P), C.byref(o), ranks.ctypes.data_as(C.POINTER(C.c_uint64)),
                                               len(ranks), C.byref(n_listed), C.byref(lr)) in (_abi.OK, _abi.NO_FEASIBLE), \
                    sm.last_error()
                assert lr.n_feasible == count
                return lr.kernel_ms

            e[key] = timed(listing, args.reps)
        kt = ranging_kernel_ms(ranges)
        e["profile"] = kt if kt is not None else "not measured (torch.profiler unavailable)"
        entry["cost_ranges"] = e
        out[f"dense_{m}_{n}"] = entry
    out["device_after"] = device_facts()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
