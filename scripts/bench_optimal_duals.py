"""Times the search for optimal duals (enumgpu_list_window, enumgpu_certify_optimum) on one GPU; prints one JSON line.

  list_window_headline  enumgpu_list_window on dense (12, 40) seed 1 with the bound key* + 1e-9 max(1, |key*|),
                        both kernel families: kernel_ms (CUDA events around the enumeration) and the call's wall time
  optimum_block_<m>     enumgpu_certify_optimum on the block LP of m rows and 2m columns (tests/test_optimal_duals.py:
                        block_lp; m = 16 is degenerate_block_16), whose winner is undecided: the window is every
                        feasible basis, 5^(m/2) of them, and the first OPTIMAL one sits near its end
  bounded_block_<m>     the same LP settled both ways: enumgpu_certify (BOUNDED through the C(2m, m+1) ray
                        enumeration) against enumgpu_certify_optimum (an OPTIMAL basis from the window)

Wall times are host clocks around calls that end in a stream synchronisation.  Each entry is warmed up once and then
timed `--reps` times; the median and the spread are printed next to the device name, its power limit and its
maximum SM clock.
Usage: python scripts/bench_optimal_duals.py [--reps 5]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402

import simplexmethod_b200 as sm  # noqa: E402
from simplexmethod_b200 import _abi, lpgen  # noqa: E402
from bench_certify import device_facts, problem, summary  # noqa: E402


def block_lp(m):
    n = 2 * m
    A = np.zeros((m, n), order="F")
    A[:, :m] = np.eye(m)
    c = np.zeros(n)
    for k in range(m // 2):
        A[2 * k, m + 2 * k], A[2 * k + 1, m + 2 * k] = 1.0, -1.0
        A[2 * k, m + 2 * k + 1], A[2 * k + 1, m + 2 * k + 1] = -1.0, 1.0
        c[m + 2 * k], c[m + 2 * k + 1] = -1.0, 2.0
    return A, np.zeros(m), c, False


def timed(fn, reps):
    fn()
    ws = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ws.append((time.perf_counter() - t0) * 1e3)
    return summary(ws)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    L = sm.lib()
    if L.enumgpu_device_count() < 1:
        raise SystemExit("bench_optimal_duals needs a CUDA device (libenumgpu has no CPU fallback)")
    out = device_facts()

    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    keep, p = problem(A, b, c, mx)
    res = _abi.Result()
    assert L.enumgpu_solve(C.byref(p), None, C.byref(res)) == _abi.OK
    bound = res.key + 1e-9 * max(1.0, abs(res.key))
    ranks = np.zeros(1 << 20, dtype=np.uint64)
    n_listed = C.c_uint64()
    for name, algo in [("independent", _abi.ALGO_INDEPENDENT), ("shared", _abi.ALGO_SHARED)]:
        o = _abi.Options(-1.0, -1.0, 0, 0, 0, algo, None, None, 0, 0, 0, 0)
        lr = _abi.Result()
        kms = []

        def run():
            assert L.enumgpu_list_window(C.byref(p), C.byref(o), bound, ranks.ctypes.data_as(C.POINTER(C.c_uint64)),
                                         ranks.size, C.byref(n_listed), C.byref(lr)) == _abi.OK, sm.last_error()
            kms.append(lr.kernel_ms)
        wall = timed(run, args.reps)
        out[f"list_window_headline_{name}"] = {"listed": n_listed.value, "algo_used": lr.algo_used,
                                               "kernel_ms": summary(kms[1:]), "wall_ms": wall}

    for m in (12, 14, 16):
        A, b, c, mx = block_lp(m)
        keep, p = problem(A, b, c, mx)
        assert L.enumgpu_solve(C.byref(p), None, C.byref(res)) == _abi.OK
        opt = _abi.Optimum()

        def run_opt():
            assert L.enumgpu_certify_optimum(C.byref(p), None, C.byref(res), -1.0, 0, C.byref(opt)) == _abi.OK, \
                sm.last_error()
        wall = timed(run_opt, args.reps)
        out[f"optimum_block_{m}"] = {"shape": [m, 2 * m], "status": opt.cert.status, "source": opt.source,
                                     "n_window": opt.n_window, "window_index": opt.window_index,
                                     "certificates": opt.window_index + 1, "n_launches": opt.n_launches,
                                     "wall_ms": wall}
        if m < 16:
            cert = _abi.Certificate()
            basis = (C.c_int32 * m)(*list(res.basis)[:m])

            def run_cert():
                assert L.enumgpu_certify(C.byref(p), None, basis, -1.0, C.byref(cert)) == _abi.OK, sm.last_error()
            wall_c = timed(run_cert, args.reps)
            out[f"bounded_block_{m}"] = {"certify_status": cert.status, "aux_bases": cert.n_aux_bases,
                                         "certify_wall_ms": wall_c, "optimum_status": opt.cert.status,
                                         "optimum_wall_ms": wall}
    out["device_after"] = device_facts()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
