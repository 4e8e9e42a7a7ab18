"""Times the certificate entries of libenumgpu on one GPU and prints one JSON line.

  certify_headline   enumgpu_certify at the optimum of dense (12, 40) seed 1: one k_certify launch plus the copies
                     (host clock around the call, which ends in a stream synchronisation)
  find_ray_<m>_<n>   enumgpu_find_ray on dense (10, 30) and (12, 40): C(30, 11) = 54.6 M and C(40, 13) = 12.03 G
                     auxiliary bases; kernel_ms (CUDA events around the enumeration) and the wall time of the call
  window_<algo>      enumgpu_find_ray of (12, 40) over the first 2^30 auxiliary ranks with each kernel family

Each entry is warmed up first and then timed `--reps` times; the median and the spread are printed, next to the
device name, its power limit and its maximum SM clock.
Usage: python scripts/bench_certify.py [--reps 5]
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


def problem(A, b, c, mx):
    A = np.asfortranarray(A, dtype=float)
    b = np.ascontiguousarray(b, dtype=float)
    c = np.ascontiguousarray(c, dtype=float)
    return (A, b, c), _abi.Problem(A.shape[0], A.shape[1], A.shape[0], int(bool(mx)), A.ctypes.data, b.ctypes.data,
                                   c.ctypes.data)


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "n": len(xs)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    L = sm.lib()
    if L.enumgpu_device_count() < 1:
        raise SystemExit("bench_certify needs a CUDA device (libenumgpu has no CPU fallback)")
    out = device_facts()

    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    keep, p = problem(A, b, c, mx)
    o = _abi.Options(-1.0, -1.0, 0, 0, 0, 0, None, None, 0, 0, 0, 0)
    res = _abi.Result()
    assert L.enumgpu_solve(C.byref(p), C.byref(o), C.byref(res)) == _abi.OK
    basis = (C.c_int32 * 12)(*list(res.basis)[:12])
    cert = _abi.Certificate()
    wall = []
    for i in range(args.reps + 3):
        t0 = time.perf_counter()
        assert L.enumgpu_certify(C.byref(p), C.byref(o), basis, -1.0, C.byref(cert)) == _abi.OK
        if i >= 3:
            wall.append((time.perf_counter() - t0) * 1e3)
    out["certify_headline"] = {"status": cert.status, "wall_ms": summary(wall)}

    for m, n in [(10, 30), (12, 40)]:
        A, b, c, mx = lpgen.dense_lp(m, n, 1)
        keep, p = problem(A, b, c, mx)
        kms, wms = [], []
        for i in range(args.reps + 1):
            t0 = time.perf_counter()
            rc = L.enumgpu_find_ray(C.byref(p), C.byref(o), C.byref(res))
            w = (time.perf_counter() - t0) * 1e3
            assert rc in (_abi.OK, _abi.NO_FEASIBLE), sm.last_error()
            if i >= 1:
                kms.append(res.kernel_ms)
                wms.append(w)
        out[f"find_ray_{m}_{n}"] = {"aux_bases": res.n_bases, "rays": res.n_feasible, "algo_used": res.algo_used,
                                    "kernel_ms": summary(kms), "wall_ms": summary(wms)}

    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    keep, p = problem(A, b, c, mx)
    for name, algo in [("independent", _abi.ALGO_INDEPENDENT), ("shared", _abi.ALGO_SHARED)]:
        ow = _abi.Options(-1.0, -1.0, 0, 1 << 30, 0, algo, None, None, 0, 0, 0, 0)
        kms = []
        for i in range(args.reps + 1):
            rc = L.enumgpu_find_ray(C.byref(p), C.byref(ow), C.byref(res))
            assert rc in (_abi.OK, _abi.NO_FEASIBLE), sm.last_error()
            if i >= 1:
                kms.append(res.kernel_ms)
        out[f"window_{name}"] = {"aux_bases": res.n_bases, "algo_used": res.algo_used, "kernel_ms": summary(kms),
                                 "Gbases_per_s": res.n_bases / statistics.median(kms) * 1e-6}
    out["device_after"] = device_facts()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
