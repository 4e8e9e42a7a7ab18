"""Right-hand-side ranging by enumeration: enumgpu_rhs_ranges against a CPU twin, exact rationals, HiGHS and the textbook.

For every row i, the allowable decrease and increase of b_i over which the dual values y* stay optimal (DESIGN.md
§3.4): the maximum, over every nonsingular m-subset T of the tight columns J, of the ends of T's feasibility interval,
each one addition and one IEEE division of frozen per-basis bits.  The twin is tests/rhs_twin.c (the per-basis
arithmetic, compiled with the CPU oracle's flags); the reduction over bases is done here with numpy.  The GPU must
equal it bit for bit in every field.

Without a GPU: the twin against exact rational ranging on the tiny goldens; against HiGHS under moved right-hand sides
on the 200 general-form LPs of test_certificate.py, y* from the certificate twin's window search
(test_optimal_duals.py); against textbook ranging where J is the basis; against HiGHS's feasibility limits at c = 0;
self-checks that the generators reach every case; the struct layout; argument errors; the failure without a device.
"""
import ctypes as C
import json
import math
import os
import shutil
import subprocess
import tempfile
from fractions import Fraction
from itertools import combinations

import numpy as np
import pytest

import simplexmethod_b200 as sm
from simplexmethod_b200 import _abi, lpgen
from test_certificate import canonical_arrays, general_lp, symmetric_file
from test_cost_ranges import highs, options, problem
from test_optimal_duals import cpu_optimum, seed_optimum, twin_certify_many
from test_structured_parity import FAMILIES, bits, rank_of

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NCPU = os.cpu_count()
SEEDS = range(200)
U64 = _abi.UINT64_MAX
OPTIMAL, BOUNDED, UNBOUNDED, UNDECIDED = _abi.CERT_OPTIMAL, _abi.CERT_BOUNDED, _abi.CERT_UNBOUNDED, _abi.CERT_UNDECIDED
ABS, REL = _abi.PIVOT_ABSOLUTE, _abi.PIVOT_RELATIVE
with open(os.path.join(HERE, "golden", "tiny_lps.json")) as f:
    GOLD = json.load(f)


# --------------------------------------------------------------------------------------------- the CPU twin

_TWIN = None


def twin_lib():
    """tests/rhs_twin.c, built once per process into a temporary directory with the CPU oracle's flags."""
    global _TWIN
    if _TWIN is None:
        tmp = tempfile.mkdtemp(prefix="rhs_twin_")
        so = os.path.join(tmp, "librhs_twin.so")
        subprocess.check_call(["gcc", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra",
                               "-std=c11", "-shared", "-I", os.path.join(ROOT, "include"), "-o", so,
                               os.path.join(HERE, "rhs_twin.c"), "-lm"])
        L = C.CDLL(so)
        shutil.rmtree(tmp)
        L.rhs_twin_many.restype = None
        L.rhs_twin_many.argtypes = [C.POINTER(_abi.Problem), C.c_double, C.c_int, C.c_double, C.c_double, C.c_void_p,
                                    C.c_int, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p]
        _TWIN = L
    return _TWIN


class Dual:
    """What enumgpu_rhs_ranges reads of an enumgpu_optimum: the status, S*, its rank, y and the reduced costs."""

    def __init__(self, status, basis, rank, y, r):
        self.status, self.basis, self.rank = status, [int(j) for j in basis], int(rank)
        self.y, self.r = [float(v) for v in y], [float(v) for v in r]

    @staticmethod
    def of(opt, m, n):
        """From an _abi.Optimum or a test_optimal_duals.CpuOptimum."""
        return Dual(opt.cert.status, list(opt.basis)[:m], opt.rank, list(opt.cert.y)[:m], list(opt.cert.reduced_cost)[:n])


def tight_columns(dual, mx, n, eps_opt=1e-9):
    return [j for j in range(n) if j in dual.basis or ((-dual.r[j] if mx else dual.r[j]) <= eps_opt)]


def pivot_tol(A, m, eps_piv, pivot_rule):
    if pivot_rule == REL:
        return m * 2.0 ** -52 if eps_piv < 0 else eps_piv
    return (1e-9 if eps_piv < 0 else eps_piv) * float(np.abs(A).max())


def twin(A, b, c, mx, dual, eps_opt=1e-9, eps_feas=-1.0, eps_piv=-1.0, pivot_rule=ABS, chunk=1 << 16):
    """DESIGN.md §3.4 on the twin's per-basis bits.  Returns a dict with every field of enumgpu_rhs_ranging, plus
    'foreign' (S* singular or not containing 0: the entry refuses the dual) and diagnostics."""
    A = np.asfortranarray(A, dtype=np.float64)
    m, n = A.shape
    out = dict(status=dual.status, m=m, tight=[], n_bases=0, n_singular=0, foreign=False, star_rows=None,
               shadow_price=np.array(dual.y, dtype=np.float64) if dual.status == OPTIMAL else np.full(m, np.nan))
    if dual.status != OPTIMAL:
        out.update(decrease=np.full(m, np.nan), increase=np.full(m, np.nan), decrease_rank=np.full(m, U64, np.uint64),
                   increase_rank=np.full(m, U64, np.uint64))
        return out
    J = tight_columns(dual, mx, n, eps_opt)
    total = math.comb(len(J), m)
    out.update(tight=J, n_bases=total)
    p, keep = problem(A, b, c, mx)
    Jc = np.array(J, dtype=np.int32)
    ef = 1e-9 if eps_feas < 0 else eps_feas + 0.0
    tol = pivot_tol(A, m, eps_piv, pivot_rule)
    best = np.full((2, m), -1.0)
    brank = np.full((2, m), U64, dtype=np.uint64)
    for r0 in range(0, total, chunk):
        k = min(chunk, total - r0)
        rank = np.zeros(k, dtype=np.uint64)
        sing = np.zeros(k, dtype=np.int32)
        lo, hi = np.zeros((k, m)), np.zeros((k, m))
        ok = np.zeros((k, m), dtype=np.int32)
        twin_lib().rhs_twin_many(C.byref(p), ef, int(pivot_rule), tol, eps_opt, Jc.ctypes.data, len(J), r0, k,
                                 rank.ctypes.data, sing.ctypes.data, lo.ctypes.data, hi.ctypes.data, ok.ctypes.data)
        out["n_singular"] += int(sing.sum())
        valid = (sing == 0)[:, None] & (ok != 0)
        star = np.nonzero(rank == dual.rank)[0]
        if len(star):
            s = star[0]
            rows = valid[s] & (lo[s] <= 0) & (hi[s] >= 0)
            out["star_rows"] = (lo[s].copy(), hi[s].copy())
            out["foreign"] |= bool(sing[s]) or not rows.all()
        with np.errstate(invalid="ignore"):
            for t, vals in ((0, hi), (1, -lo)):
                for i in range(m):
                    sel = valid[:, i] & (vals[:, i] >= 0)
                    if not sel.any():
                        continue
                    v = vals[sel, i]
                    top = v.max()
                    rk = rank[sel][v == top].min()
                    if top > best[t, i] or (top == best[t, i] and rk < brank[t, i]):
                        best[t, i], brank[t, i] = top, rk
    brank[np.isinf(best)] = U64
    brank[best < 0] = U64
    best[best < 0] = np.nan
    out.update(increase=best[0], decrease=best[1], increase_rank=brank[0], decrease_rank=brank[1])
    if out["foreign"]:
        out["status"] = _abi.ERR_ARG
    return out


# --------------------------------------------------------------------------------------------- CPU duals

def cpu_dual(oracle, A, b, c, mx):
    """The certificate twin's window search (enumgpu_certify_optimum on the CPU) at the oracle's optimum, or None
    where the LP has no feasible basis.  The fallback is only taken on an unbounded or undecided LP: it reports
    the winner's certificate with status UNDECIDED, which is all twin() reads of it."""
    A = np.asfortranarray(A, dtype=np.float64)
    m, n = A.shape
    res, _ = oracle.solve(A, b, c, mx, n_threads=NCPU)
    if res.status != _abi.OK:
        return None
    winner = twin_certify_many(A, b, c, mx, [list(res.basis)[:m]])[1][0]

    def fallback():
        ct = _abi.Certificate.from_buffer_copy(bytes(winner))
        if ct.status == OPTIMAL:
            ct.status = UNDECIDED
        return ct
    return Dual.of(cpu_optimum(oracle, A, b, c, mx, res, winner, fallback), m, n), res


_SEED = {}


def seed_case(oracle, seed):
    """(A, b, c, mx, dual, twin) of general LP `seed`, y* from test_optimal_duals' CPU search."""
    if seed not in _SEED:
        A, b, c, mx = canonical_arrays(seed)
        m, n = A.shape
        d = Dual.of(seed_optimum(oracle, seed), m, n)
        _SEED[seed] = (A, b, c, mx, d, twin(A, b, c, mx, d))
    return _SEED[seed]


def objective_of(dual, b):
    return math.fsum(float(Fraction(bi) * Fraction(yi)) for bi, yi in zip(b, dual.y))


# --------------------------------------------------------------------------------------------- exact ranging

def exact_ranges(A, b, J, eps_opt=Fraction(1, 10**9), eps_feas=Fraction(1, 10**9)):
    """The definition over J in exact rationals (a basis is singular iff its exact determinant is 0):
    (decrease, increase) per row."""
    m = len(A)
    inc, dec = [Fraction(-1)] * m, [Fraction(-1)] * m
    for T in combinations(J, m):
        M = [[Fraction(A[r][j]) for j in T] + [Fraction(b[r])] + [Fraction(int(r == i)) for i in range(m)]
             for r in range(m)]
        singular = False
        for k in range(m):
            p = next((r for r in range(k, m) if M[r][k] != 0), None)
            if p is None:
                singular = True
                break
            M[k], M[p] = M[p], M[k]
            for r in range(m):
                if r != k and M[r][k] != 0:
                    f = M[r][k] / M[k][k]
                    M[r] = [a - f * bb for a, bb in zip(M[r], M[k])]
        if singular:
            continue
        x = [M[k][m] / M[k][k] for k in range(m)]
        for i in range(m):
            w = [M[k][m + 1 + i] / M[k][k] for k in range(m)]
            lo, hi, good = -math.inf, math.inf, True
            for k in range(m):
                s, v = x[k] + eps_feas, w[k]
                if v > eps_opt:
                    lo = max(lo, -s / v)
                elif v < -eps_opt:
                    hi = min(hi, s / -v)
                else:
                    good &= s >= 0
            if good and lo <= hi:
                if hi >= 0:
                    inc[i] = max(inc[i], hi)
                if -lo >= 0:
                    dec[i] = max(dec[i], -lo)
    return dec, inc


def gold_cases(oracle):
    for name in sorted(GOLD):
        g = GOLD[name]
        A = np.array(g["A"], dtype=float)
        for mx in (g["maximize"], not g["maximize"]):
            got = cpu_dual(oracle, A, g["b"], np.array(g["c"], dtype=float), mx)
            if got is not None and got[0].status == OPTIMAL:
                yield name, g, A, mx, got[0]


def test_twin_vs_exact_on_goldens(oracle):
    checked = 0
    for name, g, A, mx, d in gold_cases(oracle):
        t = twin(A, g["b"], g["c"], mx, d)
        assert t["status"] == OPTIMAL
        dec, inc = exact_ranges(g["A"], g["b"], t["tight"])
        for got, want in list(zip(t["decrease"], dec)) + list(zip(t["increase"], inc)):
            if want == math.inf:
                assert got == math.inf, name
            else:
                assert abs(Fraction(float(got)) - want) <= Fraction(1, 10**12) * max(1, abs(want)), (name, got, want)
        checked += 1
    assert checked >= 4


# --------------------------------------------------------------------------------------------- 200 general-form LPs

@pytest.mark.parametrize("seed", SEEDS)
def test_twin_vs_highs_moved_rhs(oracle, seed):
    """Inside each finite limit the optimum is y*.b'; 1 % past it the LP is infeasible or its optimum is no longer
    y*.b'; an infinite limit holds at a large move."""
    A, b, c, mx, d, t = seed_case(oracle, seed)
    m = A.shape[0]
    st, _ = highs(A, b, c, mx)
    assert (st == 3) == (d.status == UNBOUNDED)
    if d.status != OPTIMAL:
        return
    big = 1e3 * (1 + np.abs(b).max())
    for i in range(m):
        for side, lim in (("decrease", t["decrease"][i]), ("increase", t["increase"][i])):
            sgn = -1.0 if side == "decrease" else 1.0
            moves = [(0.999 * lim, True), (lim + max(1e-2, 1e-2 * lim), False)] if math.isfinite(lim) else [(big, True)]
            for mv, stays in moves:
                bp = b.copy()
                bp[i] += sgn * mv
                val = objective_of(d, bp)
                s2, v2 = highs(A, bp, c, mx)
                if stays:
                    # abs 1e-8: a limit can be as small as the feasibility tolerance eps_feas = 1e-9 allows
                    assert s2 == 0 and v2 == pytest.approx(val, rel=1e-9, abs=1e-8), (i, side, mv, s2, v2, val)
                else:
                    # y* stays dual feasible, so y*.b' bounds the optimum; past the limit the bound is not attained
                    if s2 != 2:
                        tol = 1e-9 * max(1, abs(val))
                        assert s2 == 0 and ((v2 < val - tol) if mx else (v2 > val + tol)), (i, side, mv, s2, v2, val)


def textbook(A, b, S, eps_feas=1e-9):
    """The range of basis S alone: x_B + delta * B^-1 e_i >= -eps_feas, the enumeration's feasibility test."""
    m = A.shape[0]
    B = A[:, S]
    x = np.linalg.solve(B, b) + eps_feas
    Binv = np.linalg.inv(B)
    dec, inc = np.full(m, np.inf), np.full(m, np.inf)
    for i in range(m):
        w = Binv[:, i]
        for k in range(m):
            if w[k] > 1e-9:
                dec[i] = min(dec[i], max(x[k], 0.0) / w[k])
            elif w[k] < -1e-9:
                inc[i] = min(inc[i], max(x[k], 0.0) / -w[k])
    return dec, inc


def test_twin_vs_textbook_where_J_is_the_basis(oracle):
    checked = 0
    for seed in SEEDS:
        A, b, c, mx, d, t = seed_case(oracle, seed)
        if d.status != OPTIMAL or len(t["tight"]) != A.shape[0]:
            continue
        checked += 1
        dec, inc = textbook(A, b, d.basis)
        for got, want in list(zip(t["decrease"], dec)) + list(zip(t["increase"], inc)):
            if math.isinf(want):
                assert math.isinf(got), seed
            else:
                assert got == pytest.approx(want, rel=1e-9, abs=1e-9), seed
    assert checked == 43


def zero_cost_lp(m, n, seed):
    A, b, c, mx = lpgen.dense_lp(m, n, seed)
    return A, b, np.zeros(n), mx


def highs_feasibility_limits(A, b, i):
    """max and min of delta subject to A x = b + delta e_i, x >= 0 (None: unbounded)."""
    from scipy.optimize import linprog
    m, n = A.shape
    Ae = np.hstack([A, -np.eye(m)[:, [i]]])
    out = []
    for sgn in (-1.0, 1.0):
        cc = np.zeros(n + 1)
        cc[n] = sgn
        r = linprog(cc, A_eq=Ae, b_eq=b, bounds=[(0, None)] * n + [(None, None)], method="highs")
        assert r.status in (0, 3)
        out.append(None if r.status == 3 else float(r.x[n]))
    return out            # [max delta, min delta]


@pytest.mark.parametrize("m,n,seed", [(3, 8, 1), (4, 9, 2), (5, 10, 3), (6, 12, 4)])
def test_twin_zero_cost_vs_highs(oracle, m, n, seed):
    """c = 0: y* = 0, J is every column, and the range is how far b_i can move with the LP still feasible."""
    A, b, c, mx = zero_cost_lp(m, n, seed)
    d, _ = cpu_dual(oracle, A, b, c, mx)
    t = twin(A, b, c, mx, d)
    assert t["status"] == OPTIMAL and t["tight"] == list(range(n)) and t["n_bases"] == math.comb(n, m)
    for i in range(m):
        hi, lo = highs_feasibility_limits(A, b, i)
        for got, want in ((t["increase"][i], hi), (t["decrease"][i], None if lo is None else -lo)):
            if want is None:
                assert got == math.inf
            else:
                assert got == pytest.approx(want, rel=1e-7, abs=1e-7), (i, got, want)


def test_selfcheck_generators_reach_every_case(oracle):
    """|J| > m with a range wider than the textbook one, an infinite limit, a singular T inside J, both senses, a
    non-OPTIMAL dual among the 200 LPs; m = 16 on a dense LP.  Also pins how many of the 200 have |J| > m."""
    seen = dict(wider=0, inf=0, singular=0, not_optimal=0, J_gt_m=0, optimal=0)
    for seed in SEEDS:
        A, b, c, mx, d, t = seed_case(oracle, seed)
        m = A.shape[0]
        if d.status != OPTIMAL:
            seen["not_optimal"] += 1
            continue
        seen["optimal"] += 1
        seen["inf"] += int(np.isinf(t["decrease"]).any() or np.isinf(t["increase"]).any())
        seen["singular"] += int(t["n_singular"] > 0)
        if len(t["tight"]) > m:
            seen["J_gt_m"] += 1
            dec, inc = textbook(A, b, d.basis)
            seen["wider"] += int(np.any(t["decrease"] > dec * (1 + 1e-9) + 1e-12) or
                                 np.any(t["increase"] > inc * (1 + 1e-9) + 1e-12))
    assert all(v > 0 for v in seen.values()), seen
    assert (seen["optimal"], seen["J_gt_m"]) == (132, 89), seen
    # the canonical forms of the 200 LPs share one sense: both senses, and m = 16, on dense LPs
    for m, n, mx in ((8, 14, False), (8, 14, True), (16, 18, False)):
        A, b, c, _ = lpgen.dense_lp(m, n, 2)
        d, _ = cpu_dual(oracle, A, b, c, mx)
        t = twin(A, b, c, mx, d)
        assert t["status"] == OPTIMAL and t["m"] == m and np.isfinite(t["decrease"]).any()


# --------------------------------------------------------------------------------------------- the C entry

def to_optimum(d, m):
    """An _abi.Optimum carrying a Dual (the fields enumgpu_rhs_ranges reads)."""
    o = _abi.Optimum()
    o.cert.status, o.cert.m, o.cert.n = d.status, m, len(d.r)
    for i, v in enumerate(d.y):
        o.cert.y[i] = v
    for j, v in enumerate(d.r):
        o.cert.reduced_cost[j] = v
    for i, j in enumerate(d.basis):
        o.basis[i] = j
    o.rank = d.rank
    return o


def call_rhs(L, A, b, c, mx, opt, eps_opt=1e-9, **o):
    ps, keep = problem(A, b, c, mx)
    out = _abi.RhsRanging()
    rc = L.enumgpu_rhs_ranges(C.byref(ps), C.byref(options(**o)), C.byref(opt), eps_opt, C.byref(out))
    return rc, out


def test_layout_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "enumgpu.h"\n'
                   'int (*f)(const enumgpu_problem*, const enumgpu_options*, const enumgpu_optimum*, double,'
                   ' enumgpu_rhs_ranging*) = enumgpu_rhs_ranges;\n'
                   'int main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n",sizeof(enumgpu_rhs_range),'
                   'sizeof(enumgpu_rhs_ranging),offsetof(enumgpu_rhs_ranging,n_bases),'
                   'offsetof(enumgpu_rhs_ranging,kernel_ms),offsetof(enumgpu_rhs_ranging,tight),'
                   'offsetof(enumgpu_rhs_ranging,range),offsetof(enumgpu_rhs_range,decrease_rank),'
                   'offsetof(enumgpu_rhs_range,increase));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", os.path.join(ROOT, "simplexmethod_b200"), "-lenumgpu"])
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "simplexmethod_b200"))
    got = [int(v) for v in subprocess.check_output([str(exe)], env=env).split()]
    T, R = _abi.RhsRanging, _abi.RhsRange
    assert got == [C.sizeof(R), C.sizeof(T), T.n_bases.offset, T.kernel_ms.offset, T.tight.offset, T.range.offset,
                   R.decrease_rank.offset, R.increase.offset]
    restype, argtypes = _abi.SYMBOLS["enumgpu_rhs_ranges"]
    assert restype is C.c_int
    assert argtypes == [C.POINTER(_abi.Problem), C.POINTER(_abi.Options), C.POINTER(_abi.Optimum), C.c_double,
                        C.POINTER(_abi.RhsRanging)]


def small_case(oracle):
    A, b, c, mx = lpgen.small_degenerate_lp()
    d, _ = cpu_dual(oracle, A, b, c, mx)
    assert d.status == OPTIMAL
    return A, b, c, mx, d


def test_argument_errors(oracle):
    """Each bad argument gives its code in the return value and out.status, with or without a GPU."""
    L = sm.lib()
    A, b, c, mx, d = small_case(oracle)
    m = A.shape[0]
    good = to_optimum(d, m)
    ps, keep = problem(A, b, c, mx)

    def call(o=None, op=good, p=ps, out=True):
        r = _abi.RhsRanging()
        rc = L.enumgpu_rhs_ranges(C.byref(p) if p is not None else None, C.byref(o) if o is not None else None,
                                  C.byref(op) if op is not None else None, 1e-9, C.byref(r) if out else None)
        return rc, r

    assert call(out=False)[0] == _abi.ERR_ARG
    for kw in (dict(p=None), dict(op=None), dict(o=options(rank_begin=0, rank_end=5)), dict(o=options(rank_begin=3)),
               dict(o=options(shard_index=0, shard_count=2)), dict(o=options(shard_index=1, shard_count=2)),
               dict(o=options(pivot_rule=5))):
        rc, r = call(**kw)
        assert rc == r.status == _abi.ERR_ARG, kw
    bad = []
    for field, value in (("rank", good.rank + 1), ("rank", U64)):
        o2 = _abi.Optimum.from_buffer_copy(bytes(good))
        setattr(o2, field, value)
        bad.append(o2)
    for field, value in (("m", m + 1), ("n", A.shape[1] - 1), ("status", _abi.ERR_CUDA)):
        o2 = _abi.Optimum.from_buffer_copy(bytes(good))
        setattr(o2.cert, field, value)
        bad.append(o2)
    o2 = _abi.Optimum.from_buffer_copy(bytes(good))
    o2.basis[0] = o2.basis[1]
    bad.append(o2)
    for o2 in bad:
        rc, r = call(op=o2)
        assert rc == r.status == _abi.ERR_ARG
        assert "dual" in sm.last_error()
    badA = A.copy()
    badA[0, 0] = np.nan
    pb, keep2 = problem(badA, b, c, mx)
    assert call(p=pb)[0] == _abi.ERR_NONFINITE


@pytest.mark.parametrize("status", [UNBOUNDED, BOUNDED, UNDECIDED])
def test_non_optimal_dual_launches_nothing(oracle, status):
    """No dual-feasible y*: no launch (so no device is needed), the status carried over, NaN ranges."""
    A, b, c, mx, d = small_case(oracle)
    m = A.shape[0]
    opt = to_optimum(d, m)
    opt.cert.status = status
    rc, out = call_rhs(sm.lib(), A, b, c, mx, opt)
    assert rc == _abi.OK and out.status == status and out.m == m and out.n_launches == 0 and out.n_bases == 0
    for i in range(m):
        r = out.range[i]
        assert all(math.isnan(v) for v in (r.shadow_price, r.decrease, r.increase))
        assert (r.decrease_rank, r.increase_rank) == (U64, U64)


@pytest.mark.skipif(sm.lib().enumgpu_device_count() > 0, reason="a GPU is present")
def test_no_gpu_means_loud_failure_not_fallback(oracle):
    A, b, c, mx, d = small_case(oracle)
    rc, out = call_rhs(sm.lib(), A, b, c, mx, to_optimum(d, A.shape[0]))
    assert rc == out.status == _abi.ERR_CUDA
    assert "no CPU fallback" in sm.last_error()
    with pytest.raises(sm.EnumGpuError, match="no CPU fallback"):
        sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(A.shape[0])), minimize=not mx)).rhsRanges()


# --------------------------------------------------------------------------------------------- GPU

def gpu_dual(L, A, b, c, mx, algo=_abi.ALGO_AUTO, **o):
    """enumgpu_solve then enumgpu_certify_optimum under the same options: (Optimum, Result)."""
    ps, keep = problem(A, b, c, mx)
    oo = options(algo=algo, **o)
    res = _abi.Result()
    assert L.enumgpu_solve(C.byref(ps), C.byref(oo), C.byref(res)) == _abi.OK, sm.last_error()
    opt = _abi.Optimum()
    assert L.enumgpu_certify_optimum(C.byref(ps), C.byref(oo), C.byref(res), -1.0, 0, C.byref(opt)) == _abi.OK
    return opt, res


def bits_of(values):
    return np.asarray(values, dtype=np.float64).view(np.uint64).tolist()


def assert_equal_to_twin(g, t):
    assert g.status == t["status"], (g.status, t["status"])
    m = t["m"]
    assert g.m == m
    assert list(g.tight)[:g.n_tight] == t["tight"]
    assert (g.n_bases, g.n_singular) == (t["n_bases"], t["n_singular"])
    for i in range(m):
        r = g.range[i]
        got = (bits(r.shadow_price), bits(r.decrease), bits(r.increase), r.decrease_rank, r.increase_rank)
        want = (bits(t["shadow_price"][i]), bits(t["decrease"][i]), bits(t["increase"][i]), int(t["decrease_rank"][i]),
                int(t["increase_rank"][i]))
        assert got == want, (i, got, want)


# (algo of the enumeration that gives the dual, pivot rule): the relative rule runs on the one-GE-per-basis family
VARIANTS = [(_abi.ALGO_INDEPENDENT, ABS), (_abi.ALGO_SHARED, ABS), (_abi.ALGO_INDEPENDENT, REL)]


def check(L, A, b, c, mx, variants=VARIANTS):
    """The entry against the twin for every variant's dual; returns the twins."""
    m, n = A.shape
    ts = []
    for algo, rule in variants:
        opt, res = gpu_dual(L, A, b, c, mx, algo=algo, pivot_rule=rule)
        d = Dual.of(opt, m, n)
        t = twin(A, b, c, mx, d, pivot_rule=rule)
        rc, g = call_rhs(L, A, b, c, mx, opt, pivot_rule=rule)
        assert rc == _abi.OK, sm.last_error()
        assert_equal_to_twin(g, t)
        if t["status"] == OPTIMAL:
            assert g.n_launches == 2 and g.kernel_ms > 0
        ts.append(t)
    return ts


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GOLD))
def test_gpu_tiny_goldens(gpu_lib, oracle, name):
    g = GOLD[name]
    A = np.array(g["A"], dtype=float)
    for mx in (g["maximize"], not g["maximize"]):
        if oracle.solve(A, g["b"], g["c"], mx)[0].status == _abi.OK:
            check(gpu_lib, A, np.array(g["b"], dtype=float), np.array(g["c"], dtype=float), mx)


@pytest.mark.gpu
@pytest.mark.parametrize("m", range(1, 17))
def test_gpu_dense_shapes(gpu_lib, oracle, m):
    A, b, c, _ = lpgen.dense_lp(m, m + 5, m)
    for mx in (False, True):
        check(gpu_lib, A, b, c, mx)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["small", "config5"])
def test_gpu_degenerate(gpu_lib, oracle, name):
    A, b, c, mx = {"small": lpgen.small_degenerate_lp, "config5": lpgen.degenerate_lp}[name]()
    for sense in (mx, not mx):
        if oracle.solve(A, b, c, sense)[0].status == _abi.OK:
            check(gpu_lib, A, b, c, sense)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(8, 20), (10, 22)])
@pytest.mark.parametrize("name", sorted(FAMILIES))
def test_gpu_structured_families(gpu_lib, oracle, name, m, n):
    A, b, c, _ = FAMILIES[name](m, n, 1)
    for mx in (False, True):
        if oracle.solve(A, b, c, mx)[0].status == _abi.OK:
            check(gpu_lib, A, b, c, mx, variants=VARIANTS[:2])


@pytest.mark.gpu
def test_gpu_general_lps(gpu_lib, oracle):
    """The 200 LPs: the GPU's own dual bit for bit against the CPU search's, then the ranges against the twin."""
    for seed in SEEDS:
        A, b, c, mx, d, t = seed_case(oracle, seed)
        m, n = A.shape
        for algo in (_abi.ALGO_INDEPENDENT, _abi.ALGO_SHARED):
            opt, _ = gpu_dual(gpu_lib, A, b, c, mx, algo=algo)
            g_d = Dual.of(opt, m, n)
            assert (g_d.status, g_d.basis, g_d.rank) == (d.status, d.basis, d.rank), seed
            assert bits_of(g_d.y) == bits_of(d.y) and bits_of(g_d.r) == bits_of(d.r), seed
            rc, g = call_rhs(gpu_lib, A, b, c, mx, opt)
            assert rc == _abi.OK, (seed, sm.last_error())
            assert_equal_to_twin(g, t)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(8, 24), (4, 64)])
def test_gpu_zero_cost_many_blocks(gpu_lib, oracle, m, n):
    """c = 0: every column is tight, C(24, 8) = 735 471 and C(64, 4) = 635 376 bases over many blocks."""
    A, b, c, mx = zero_cost_lp(m, n, 5)
    ts = check(gpu_lib, A, b, c, mx, variants=VARIANTS[:1])
    assert ts[0]["n_bases"] == math.comb(n, m) and ts[0]["n_singular"] >= 0


@pytest.mark.gpu
def test_gpu_wide_n64(gpu_lib, oracle):
    A, b, c, mx = lpgen.dense_lp(6, 64, 3)
    check(gpu_lib, A, b, c, mx, variants=VARIANTS[:2])


@pytest.mark.gpu
def test_gpu_zero_cost_10_30_vs_highs(gpu_lib):
    """C(30, 10) = 30 045 015 bases: against HiGHS's feasibility limits."""
    A, b, c, mx = zero_cost_lp(10, 30, 6)
    opt, _ = gpu_dual(gpu_lib, A, b, c, mx)
    rc, g = call_rhs(gpu_lib, A, b, c, mx, opt)
    assert rc == _abi.OK and g.status == OPTIMAL and g.n_bases == math.comb(30, 10)
    for i in range(10):
        hi, lo = highs_feasibility_limits(A, b, i)
        for got, want in ((g.range[i].increase, hi), (g.range[i].decrease, None if lo is None else -lo)):
            if want is None:
                assert got == math.inf
            else:
                assert got == pytest.approx(want, rel=1e-7, abs=1e-7), (i, got, want)


@pytest.mark.gpu
def test_gpu_foreign_dual_is_refused(gpu_lib, oracle):
    """A dual whose basis is infeasible at b (as from other options) is refused through the device flag."""
    A, b, c, mx = lpgen.dense_lp(6, 14, 2)
    m, n = A.shape
    opt, _ = gpu_dual(gpu_lib, A, b, c, mx)
    assert opt.cert.status == OPTIMAL
    ps, keep = problem(A, b, c, mx)
    x, z, cls = (C.c_double * m)(), C.c_double(), C.c_int32()
    for S in combinations(range(n), m):
        assert gpu_lib.enumgpu_eval_basis(C.byref(ps), None, (C.c_int32 * m)(*S), x, C.byref(z), C.byref(cls)) == 0
        if cls.value == _abi.BASIS_INFEASIBLE:
            break
    bad = _abi.Optimum.from_buffer_copy(bytes(opt))
    for i, j in enumerate(S):
        bad.basis[i] = j
    bad.rank = rank_of(n, m, list(S))
    rc, out = call_rhs(gpu_lib, A, b, c, mx, bad)
    assert rc == out.status == _abi.ERR_ARG
    assert "other options" in sm.last_error()


@pytest.mark.gpu
def test_gpu_python_adapter(gpu_lib, oracle):
    for A, b, c, mx in (lpgen.lab_symmetric_canonical(), lpgen.small_degenerate_lp(), zero_cost_lp(5, 12, 1)):
        m = A.shape[0]
        s = sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(m)), minimize=not mx))
        r = s.rhsRanges()
        opt, _ = gpu_dual(gpu_lib, A, b, c, mx)
        rc, g = call_rhs(gpu_lib, A, b, c, mx, opt)
        assert rc == _abi.OK and r.status == g.status
        for name in ("shadow_price", "decrease", "increase"):
            assert bits_of(getattr(r, name)) == bits_of([getattr(g.range[i], name) for i in range(m)])
        for name in ("decrease_rank", "increase_rank"):
            assert [int(v) for v in getattr(r, name)] == [getattr(g.range[i], name) for i in range(m)]
        assert (r.tight, r.n_bases, r.n_singular) == (list(g.tight)[:g.n_tight], g.n_bases, g.n_singular)
    hit = 0
    for seed in SEEDS:
        A, b, c, mx, d, t = seed_case(oracle, seed)
        if d.status == UNBOUNDED:
            hit += 1
            can = sm.Canonical(A, b, c, list(range(A.shape[0])), minimize=not mx)
            with pytest.raises(RuntimeError, match="objective is unbounded"):
                sm.EnumerationSolver(can).rhsRanges()
            if hit == 5:
                break
    assert hit == 5


@pytest.fixture(scope="module")
def certify_demo():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "simplexmethod_b200", "cpp"), "-s"])
    return os.path.join(ROOT, "simplexmethod_b200", "cpp", "build", "certify_demo")


@pytest.mark.gpu
def test_gpu_certify_demo_rhs_ranges(gpu_lib, oracle, certify_demo, tmp_path):
    """certify_demo --rhs-ranges prints the table of the Python adapter's ranges, on LPs with and without |J| > m."""
    chosen = {}
    for seed in SEEDS:
        A, b, c, mx, d, t = seed_case(oracle, seed)
        if d.status == OPTIMAL:
            chosen.setdefault(len(t["tight"]) > A.shape[0], seed)
    assert len(chosen) == 2
    for seed in chosen.values():
        f = tmp_path / f"lp{seed}.txt"
        symmetric_file(f, seed)
        out = subprocess.run([certify_demo, "--rhs-ranges", str(f)], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        r = sm.EnumerationSolver(general_lp(seed).ToSymmetrical().ToCanonical()).rhsRanges()
        lines = out.stdout.splitlines()
        head = lines[0].split()
        assert head[0] == "rhs_ranging" and [int(v) for v in head[1:]] == [r.status, len(r.tight), r.n_bases,
                                                                            r.n_singular]
        assert [int(v) for v in lines[1].split()[1:]] == r.tight
        rows = [ln.split() for ln in lines[2:] if ln.startswith("rhs ")]
        assert len(rows) == len(r.decrease)
        for row in rows:
            i = int(row[1])
            assert [float(v) for v in row[2:5]] == [float(r.shadow_price[i]), float(r.decrease[i]), float(r.increase[i])]
            assert [int(v) for v in row[5:7]] == [int(r.decrease_rank[i]), int(r.increase_rank[i])]
