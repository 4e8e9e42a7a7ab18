"""Times enumgpu_rhs_ranges (right-hand-side ranging by enumeration) on one GPU and prints one JSON line.

Cases (dense LPs of lpgen.dense_lp, seed 1 unless named):
  dense_12_40      the headline LP
  tied_12_40       the headline A with tied costs: c = A'y0 + s, s_j = 0 for the first 24 columns and random > 0
                   elsewhere, b = A x0 with x0 > 0 on those 24: every basis of them is optimal, so 24 columns are tight
                   and C(24, 12) = 2.70 M bases are ranged
  zero_10_30       c = 0 at 10 x 30: every column is tight, C(30, 10) = 30.0 M bases
  zero_12_40       c = 0 at 12 x 40: C(40, 12) = 5.59 G bases
For each: the enumgpu_solve and enumgpu_certify_optimum calls that produce the duals (kernel_ms), then the ranging
call: wall_ms (host clock around the call, which ends in a stream synchronisation) and kernel_ms (its CUDA-event span:
k_rhs_ranging plus k_rhs_ranging_finish), n_tight, n_bases, n_singular and the rate n_bases / kernel_ms.  The ranging
call is warmed up once and timed `--reps` times (once for zero_12_40); medians and spreads are printed next to the
device name, its power limit and its maximum SM clock, read in the same run.
Usage: python scripts/bench_rhs_ranging.py [--reps 3]
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
from scripts.bench_ranging import problem  # noqa: E402


def cases():
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    yield "dense_12_40", (A, b, c, mx), 3
    rng = np.random.default_rng(1)
    s = np.where(np.arange(40) < 24, 0.0, rng.uniform(0.5, 2.0, 40))
    x0 = np.where(np.arange(40) < 24, rng.uniform(0.5, 2.0, 40), 0.0)
    yield "tied_12_40", (A, A @ x0, A.T @ rng.uniform(-1.0, 1.0, 12) + s, False), 3
    A3, b3, _, mx3 = lpgen.dense_lp(10, 30, 1)
    yield "zero_10_30", (A3, b3, np.zeros(30), mx3), 3
    yield "zero_12_40", (A, b, np.zeros(40), mx), 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    L = sm.lib()
    if L.enumgpu_device_count() < 1:
        raise SystemExit("bench_rhs_ranging needs a CUDA device (libenumgpu has no CPU fallback)")
    out = device_facts()
    o = _abi.Options(-1.0, -1.0, 0, 0, 0, 0, None, None, 0, 0, 0, 0)
    for name, (A, b, c, mx), reps in cases():
        p, keep = problem(A, b, c, mx)
        res = _abi.Result()
        assert L.enumgpu_solve(C.byref(p), C.byref(o), C.byref(res)) == _abi.OK, sm.last_error()
        opt = _abi.Optimum()
        assert L.enumgpu_certify_optimum(C.byref(p), C.byref(o), C.byref(res), 1e-9, 0, C.byref(opt)) == _abi.OK
        entry = {"solve_kernel_ms": res.kernel_ms, "dual_status": opt.cert.status, "dual_source": opt.source}
        rr = _abi.RhsRanging()

        def ranges():
            assert L.enumgpu_rhs_ranges(C.byref(p), C.byref(o), C.byref(opt), 1e-9, C.byref(rr)) == _abi.OK, \
                sm.last_error()
            return rr.kernel_ms

        wall, kms = [], []
        for i in range(reps + (1 if reps > 1 else 0)):
            t0 = time.perf_counter()
            k = ranges()
            if reps == 1 or i >= 1:
                wall.append((time.perf_counter() - t0) * 1e3)
                kms.append(k)
        entry.update(wall_ms=summary(wall), kernel_ms=summary(kms), status=rr.status, n_tight=rr.n_tight,
                     n_bases=rr.n_bases, n_singular=rr.n_singular, n_launches=rr.n_launches,
                     bases_per_s=rr.n_bases / (summary(kms)["median"] * 1e-3),
                     finite_limits=sum(int(np.isfinite(rr.range[i].decrease)) + int(np.isfinite(rr.range[i].increase))
                                       for i in range(rr.m)))
        out[name] = entry
        print(name, json.dumps(entry), file=sys.stderr, flush=True)
    out["device_after"] = device_facts()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
