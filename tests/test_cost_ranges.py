"""Cost ranging by enumeration: enumgpu_cost_ranges against a CPU twin, exact rationals, HiGHS and the textbook.

For every column j, the allowable decrease and increase of c_j over which the optimal vertex x* stays optimal
(DESIGN.md §3.3): the minimum over every feasible basis and every extreme ray of one subtraction and one division of
frozen per-basis bits.  The twin here builds the same answer from the CPU oracle's per-basis bits (enumcpu.list_class
and enumcpu.eval_basis; the rays from the oracle on the auxiliary LP, built here in Python) with numpy float64, whose
subtraction and division are IEEE correctly rounded.  The GPU must equal it bit for bit in every field.

Without a GPU: the twin against exact rational ranging on the tiny goldens, against HiGHS under perturbed costs on
the 200 general-form LPs of test_certificate.py, and against textbook basis-level ranging at nondegenerate optima;
self-checks that the generators reach every case; the struct layout; argument errors; the failure without a device.
"""
import ctypes as C
import json
import math
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

import simplexmethod_b200 as sm
from simplexmethod_b200 import _abi, lpgen
from oracle import exact
from test_certificate import canonical_arrays, certify_basis
from test_structured_parity import FAMILIES, bits, unrank

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NCPU = os.cpu_count()
ALGOS = [_abi.ALGO_INDEPENDENT, _abi.ALGO_SHARED]
SEEDS = range(200)
FEASIBLE = 0
U64 = _abi.UINT64_MAX
OPTIMAL, UNBOUNDED, UNDECIDED = _abi.CERT_OPTIMAL, _abi.CERT_UNBOUNDED, _abi.CERT_UNDECIDED
with open(os.path.join(HERE, "golden", "tiny_lps.json")) as f:
    GOLD = json.load(f)


# --------------------------------------------------------------------------------------------- the auxiliary LP

def ray_lp(A):
    """[A; s*1'] d = (0, ..., 0, s), cost 0: s the largest power of two <= max|A_ij|, found by search."""
    amax = float(np.abs(A).max())
    s = 1.0
    while s > amax:
        s /= 2
    while 2 * s <= amax:
        s *= 2
    m, n = A.shape
    ba = np.zeros(m + 1)
    ba[m] = s
    return np.asfortranarray(np.vstack([A, np.full(n, s)])), ba


# --------------------------------------------------------------------------------------------- the CPU twin

def oracle_bits(oracle, A, b, c, mx, eps_feas=-1.0, eps_piv=-1.0, pivot_rule=_abi.PIVOT_ABSOLUTE):
    """(ranks, S, X, z) of every feasible basis, from the oracle: list_class, then eval_basis per rank."""
    m, n = A.shape
    _, ranks, count = oracle.list_class(A, b, c, mx, FEASIBLE, capacity=1 << 22, n_threads=NCPU, eps_feas=eps_feas,
                                        eps_piv=eps_piv, pivot_rule=pivot_rule)
    assert len(ranks) == count
    hp = oracle.HostProblem(A, b, c, mx)
    if pivot_rule == _abi.PIVOT_RELATIVE:
        tol = m * 2.0 ** -52 if eps_piv < 0 else eps_piv
    else:
        tol = (1e-9 if eps_piv < 0 else eps_piv) * oracle.lib().enumcpu_scale(C.byref(hp.struct))
    ef = 1e-9 if eps_feas < 0 else eps_feas + 0.0
    S = np.array([unrank(n, m, int(r)) for r in ranks], dtype=np.int64).reshape(len(ranks), m)
    X = np.zeros((len(ranks), m))
    z = np.zeros(len(ranks))
    x, zz = (C.c_double * m)(), C.c_double()
    for i in range(len(ranks)):
        st = oracle.lib().enumcpu_eval_basis_rule(C.byref(hp.struct), ef, int(pivot_rule), tol,
                                                  (C.c_int32 * m)(*S[i]), x, C.byref(zz))
        assert st == FEASIBLE
        X[i] = list(x)
        z[i] = zz.value
    return ranks.astype(np.uint64), S, X, z


class Folder:
    """Running lexicographic minima of (ratio, rank) for n slots, fed in chunks."""

    def __init__(self, n):
        self.ratio = np.full(n, np.inf)
        self.rank = np.full(n, U64, dtype=np.uint64)

    def fold(self, ratio, ranks, mask):
        for j in range(ratio.shape[1]):
            sel = np.nonzero(mask[:, j])[0]
            if len(sel) == 0:
                continue
            r = ratio[sel, j]
            lo = r.min()
            rk = ranks[sel][r == lo].min()
            if lo < self.ratio[j] or (lo == self.ratio[j] and rk < self.rank[j]):
                self.ratio[j], self.rank[j] = lo, rk


def twin_ranges(n, m, mx, key_star, xs, eps_opt, vertex_chunks, ray_chunks):
    """The definition of DESIGN.md §3.3 on per-basis bits.  vertex_chunks: iterable of (ranks, S, X, z) with z under c;
    ray_chunks: None (no rays enumerated) or iterable of (ranks, S, D, ckd).  Returns a dict with status, the six
    range arrays, the listing counts and diagnostics (same_vertex: listed bases other than S* at x*)."""
    xs = np.asarray(xs, dtype=np.float64)
    tau = eps_opt * max(1.0, abs(key_star))
    tol = eps_opt * np.maximum(1.0, np.abs(xs))
    up, down, ray = Folder(n), Folder(n), Folder(n)
    out = dict(n_vertex=0, n_ray=0, same_vertex=0, below=False, unbounded=False)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        for ranks, S, X, z in vertex_chunks:
            N = len(ranks)
            out["n_vertex"] += N
            if N == 0:
                continue
            dk = (-z if mx else z) - key_star
            out["below"] |= bool(np.any(dk < 0))
            XB = np.zeros((N, n))
            XB[np.arange(N)[:, None], S] = X
            DX = XB - xs[None, :]
            ok = ~np.isnan(dk)[:, None] & ~np.isnan(DX) & (np.abs(DX) > tol[None, :])
            ratio = np.where(dk[:, None] <= tau, 0.0, dk[:, None] / np.abs(DX))
            ok &= ~np.isnan(ratio)
            out["same_vertex"] += int(np.sum(~ok.any(axis=1) & ~np.isnan(dk) & (dk <= tau)))
            up.fold(ratio, ranks, ok & (DX < 0))
            down.fold(ratio, ranks, ok & (DX > 0))
        if ray_chunks is not None:
            for ranks, S, D, ckd in ray_chunks:
                N = len(ranks)
                out["n_ray"] += N
                if N == 0:
                    continue
                out["unbounded"] |= bool(np.any(ckd < -eps_opt))
                DD = np.zeros((N, n))
                DD[np.arange(N)[:, None], S] = D
                ratio = np.where(ckd[:, None] <= eps_opt, 0.0, ckd[:, None] / DD)
                ok = ~np.isnan(ckd)[:, None] & ~(ckd < -eps_opt)[:, None] & (DD > eps_opt)
                ray.fold(ratio, ranks, ok)
    take = ray.ratio < down.ratio
    dn_r = np.where(take, ray.ratio, down.ratio)
    dn_k = np.where(take, ray.rank, down.rank)
    if mx:
        rng = (up.ratio, dn_r, up.rank, dn_k, np.zeros(n, bool), take)
    else:
        rng = (dn_r, up.ratio, dn_k, up.rank, take, np.zeros(n, bool))
    out.update(zip(("decrease", "increase", "decrease_rank", "increase_rank", "decrease_ray", "increase_ray"), rng))
    if out["below"]:
        out["status"] = _abi.ERR_ARG
    elif out["unbounded"]:
        out["status"] = UNBOUNDED
    else:
        out["status"] = UNDECIDED if (ray_chunks is None and n > m) else OPTIMAL
    return out


def twin(oracle, A, b, c, mx, opt=None, eps_opt=1e-9, **tol):
    """The twin on an LP from the oracle's bits.  opt: the winner (an oracle Result) unless given."""
    A = np.asfortranarray(A, dtype=np.float64)
    b, c = np.asarray(b, dtype=np.float64), np.asarray(c, dtype=np.float64)
    m, n = A.shape
    if opt is None:
        opt, _ = oracle.solve(A, b, c, mx, n_threads=NCPU, **tol)
    xs = np.zeros(n)
    xs[list(opt.basis)[:m]] = list(opt.x_B)[:m]
    vert = [oracle_bits(oracle, A, b, c, mx, **tol)]
    rays = None
    if m + 1 <= _abi.MAX_M and n > m:
        Aa, ba = ray_lp(A)
        ck = -c if mx else c
        rk, S, D, _ = oracle_bits(oracle, Aa, ba, np.zeros(n), False, **tol)
        ckd = np.array([oracle.eval_basis(Aa, ba, ck, False, list(s))[2] for s in S]) if len(rk) else np.zeros(0)
        rays = [(rk, S, D, ckd)]
    return twin_ranges(n, m, mx, opt.key, xs, eps_opt, vert, rays)


FIELDS = ("decrease", "increase", "decrease_rank", "increase_rank", "decrease_ray", "increase_ray")


def assert_equal_to_twin(g, t, n):
    """Every field of the GPU's enumgpu_ranging against the twin, doubles as bit patterns."""
    assert g.status == t["status"], (g.status, t["status"])
    assert (g.n, g.n_vertex_bases, g.n_ray_bases) == (n, t["n_vertex"], t["n_ray"])
    if g.status == UNBOUNDED:
        for j in range(n):
            r = g.range[j]
            assert math.isnan(r.decrease) and math.isnan(r.increase)
            assert (r.decrease_rank, r.increase_rank, r.decrease_ray, r.increase_ray) == (U64, U64, 0, 0)
        return
    for j in range(n):
        r = g.range[j]
        got = (bits(r.decrease), bits(r.increase), r.decrease_rank, r.increase_rank, r.decrease_ray, r.increase_ray)
        want = (bits(t["decrease"][j]), bits(t["increase"][j]), int(t["decrease_rank"][j]), int(t["increase_rank"][j]),
                int(t["decrease_ray"][j]), int(t["increase_ray"][j]))
        assert got == want, (j, got, want)


# --------------------------------------------------------------------------------------------- exact ranging

def exact_ranges(A, b, c, mx, eps=Fraction(1, 10**9)):
    """The definition in exact rationals: every vertex and every ray as Fractions."""
    m, n = len(A), len(A[0])
    ev = exact.enumerate_exact(A, b, c, mx)
    key_star = -ev["best_z"] if mx else ev["best_z"]
    xs = [Fraction(0)] * n
    for j, v in zip(ev["best_basis"], ev["best_x"]):
        xs[j] = v
    tau = eps * max(1, abs(key_star))
    inf = math.inf
    up, down, ray = [inf] * n, [inf] * n, [inf] * n
    from itertools import combinations
    for rank, S in enumerate(combinations(range(n), m)):
        if ev["status"][rank] != exact.FEASIBLE:
            continue
        z = ev["z"][rank]
        dk = (-z if mx else z) - key_star
        xb = [Fraction(0)] * n
        for j, v in zip(S, ev["x"][rank]):
            xb[j] = v
        for j in set(S) | set(ev["best_basis"]):
            dx = xb[j] - xs[j]
            if abs(dx) <= eps * max(1, abs(xs[j])):
                continue
            r = Fraction(0) if dk <= tau else dk / abs(dx)
            if dx < 0:
                up[j] = min(up[j], r)
            else:
                down[j] = min(down[j], r)
    if m + 1 <= _abi.MAX_M and n > m:
        Aa, ba = ray_lp(np.array(A, dtype=float))
        ck = [Fraction(-v if mx else v) for v in c]
        er = exact.enumerate_exact(Aa.tolist(), ba.tolist(), [0.0] * n, False)
        for rank, S in enumerate(combinations(range(n), m + 1)):
            if er["status"][rank] != exact.FEASIBLE:
                continue
            d = er["x"][rank]
            ckd = sum(ck[j] * v for j, v in zip(S, d))
            assert ckd >= -eps, "the goldens are bounded"
            for j, v in zip(S, d):
                if v > eps:
                    ray[j] = min(ray[j], Fraction(0) if ckd <= eps else ckd / v)
    dn = [min(a, r) for a, r in zip(down, ray)]
    return (up, dn) if mx else (dn, up)          # (decrease, increase)


@pytest.mark.parametrize("name", sorted(GOLD))
def test_twin_vs_exact_on_goldens(oracle, name):
    g = GOLD[name]
    A = np.array(g["A"], dtype=float)
    t = twin(oracle, A, g["b"], g["c"], g["maximize"])
    assert t["status"] == OPTIMAL
    dec, inc = exact_ranges(g["A"], g["b"], g["c"], g["maximize"])
    for got, want in list(zip(t["decrease"], dec)) + list(zip(t["increase"], inc)):
        if want == math.inf:
            assert got == math.inf
        else:
            assert abs(Fraction(float(got)) - want) <= Fraction(1, 10**12) * max(1, abs(want)), (got, want)


# --------------------------------------------------------------------------------------------- 200 general-form LPs

_TW = {}


def seed_twin(oracle, seed):
    if seed not in _TW:
        A, b, c, mx = canonical_arrays(seed)
        opt, _ = oracle.solve(A, b, c, mx, n_threads=NCPU)
        assert opt.status == _abi.OK
        _TW[seed] = (A, b, c, mx, opt, twin(oracle, A, b, c, mx, opt))
    return _TW[seed]


def highs(A, b, c, mx):
    from scipy.optimize import linprog
    r = linprog(-c if mx else c, A_eq=A, b_eq=b, bounds=[(0, None)] * A.shape[1], method="highs")
    return r.status, (None if r.status != 0 else (-r.fun if mx else r.fun))


@pytest.mark.parametrize("seed", SEEDS)
def test_twin_vs_highs_perturbed(oracle, seed):
    """Inside each finite limit x* stays optimal; past it the optimum improves (unbounded when a ray limits);
    an infinite limit holds at a large move."""
    A, b, c, mx, opt, t = seed_twin(oracle, seed)
    m, n = A.shape
    st, _ = highs(A, b, c, mx)
    assert (st == 3) == (t["status"] == UNBOUNDED)
    if t["status"] == UNBOUNDED:
        return
    xs = np.zeros(n)
    xs[list(opt.basis)[:m]] = list(opt.x_B)[:m]
    big = 1e3 * (1 + np.abs(c).max())
    better = (lambda v, w: v > w) if mx else (lambda v, w: v < w)
    for j in range(n):
        for side, lim, is_ray in (("decrease", t["decrease"][j], t["decrease_ray"][j]),
                                  ("increase", t["increase"][j], t["increase_ray"][j])):
            sgn = -1.0 if side == "decrease" else 1.0
            moves = [(0.999 * lim, True)] if math.isfinite(lim) else [(big, True)]
            if math.isfinite(lim):
                moves.append((lim + max(1e-2, 1e-2 * lim), False))
            for mv, stays in moves:
                cp = c.copy()
                cp[j] += sgn * mv
                val = float(cp @ xs)
                s2, v2 = highs(A, b, cp, mx)
                if stays:
                    assert s2 == 0 and v2 == pytest.approx(val, rel=1e-9, abs=1e-9), (j, side, mv, s2, v2, val)
                elif is_ray:
                    assert s2 == 3, (j, side, mv, s2, v2)
                else:
                    assert s2 == 3 or (s2 == 0 and better(v2, val + (1e-9 if mx else -1e-9) * max(1, abs(val)))), \
                        (j, side, mv, s2, v2, val)


def textbook(A, c, mx, S, r):
    """Basis-level ranging at basis S (key sense, then true sense): r the reduced costs (true sense), u_k = B^-1 a_k.
    Nonbasic j: rise without limit, fall r_j; basic S[i]: rise min rk_k / u_k[i] over u_k[i] > 0, fall over < 0."""
    m, n = A.shape
    u = np.linalg.solve(A[:, S], A)
    rk = -np.asarray(r) if mx else np.asarray(r)
    up, dn = np.full(n, np.inf), np.full(n, np.inf)
    nb = [k for k in range(n) if k not in S]
    for j in nb:
        dn[j] = rk[j]
    for i, j in enumerate(S):
        for k in nb:
            if u[i, k] > 1e-9:
                up[j] = min(up[j], rk[k] / u[i, k])
            elif u[i, k] < -1e-9:
                dn[j] = min(dn[j], rk[k] / -u[i, k])
    return (up, dn) if mx else (dn, up)


def nondegenerate(opt, m):
    return min(list(opt.x_B)[:m]) > 1e-9 * max(1.0, max(abs(v) for v in list(opt.x_B)[:m]))


def test_twin_vs_textbook_at_nondegenerate_optima(oracle):
    """Where the optimum is nondegenerate and the winner's certificate OPTIMAL, the exact ranges are the textbook ones
    from the winner's basis (this checks the ray side independently of the enumeration of rays)."""
    checked = 0
    for seed in SEEDS:
        A, b, c, mx, opt, t = seed_twin(oracle, seed)
        m, n = A.shape
        S = list(opt.basis)[:m]
        rc, cert = certify_basis(A, b, c, mx, S)
        if t["status"] != OPTIMAL or cert.status != OPTIMAL or not nondegenerate(opt, m):
            continue
        checked += 1
        dec, inc = textbook(A, c, mx, S, list(cert.reduced_cost)[:n])
        for got, want in list(zip(t["decrease"], dec)) + list(zip(t["increase"], inc)):
            if math.isinf(want):
                assert math.isinf(got), seed
            else:
                assert got == pytest.approx(want, rel=1e-9, abs=1e-12), seed
    assert checked >= 10


def test_selfcheck_generators_reach_every_case(oracle):
    """Degenerate optimum wider than the textbook, an alternative optimum, a ray-limited decrease, an infinite
    increase, an unbounded LP, a same-vertex basis dropped by the Delta x rule, and m = 16 UNDECIDED."""
    seen = dict(wider=0, zero=0, ray=0, inf_inc=0, unbounded=0, same_vertex=0, nondegenerate_textbook=0)
    for seed in SEEDS:
        A, b, c, mx, opt, t = seed_twin(oracle, seed)
        m, n = A.shape
        if t["status"] == UNBOUNDED:
            seen["unbounded"] += 1
            continue
        seen["zero"] += int(np.any(t["decrease"] == 0) or np.any(t["increase"] == 0))
        seen["ray"] += int(np.any(t["decrease_ray"]) or np.any(t["increase_ray"]))
        seen["inf_inc"] += int(np.any(np.isinf(t["increase"])))
        seen["same_vertex"] += int(t["same_vertex"] > 0)
        S = list(opt.basis)[:m]
        rc, cert = certify_basis(A, b, c, mx, S)
        if cert.status == OPTIMAL:
            dec, inc = textbook(A, c, mx, S, list(cert.reduced_cost)[:n])
            wide = np.any(t["decrease"] > dec * (1 + 1e-9) + 1e-12) or np.any(t["increase"] > inc * (1 + 1e-9) + 1e-12)
            if nondegenerate(opt, m):
                seen["nondegenerate_textbook"] += 1
            else:
                seen["wider"] += int(wide)
    assert all(v > 0 for v in seen.values()), seen
    A, b, c, mx = lpgen.dense_lp(16, 18, 2)
    t = twin(oracle, A, b, c, mx)
    assert t["status"] == UNDECIDED and t["n_ray"] == 0


# --------------------------------------------------------------------------------------------- the C entry

def options(algo=_abi.ALGO_AUTO, rank_begin=0, rank_end=0, eps_feas=-1.0, eps_piv=-1.0, pivot_rule=_abi.PIVOT_ABSOLUTE,
            shard_index=0, shard_count=0):
    return _abi.Options(eps_feas, eps_piv, rank_begin, rank_end, 0, algo, None, None, shard_index, shard_count,
                        pivot_rule, 0)


def problem(A, b, c, mx):
    A = np.asfortranarray(A, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    c = np.ascontiguousarray(c, dtype=np.float64)
    return _abi.Problem(A.shape[0], A.shape[1], A.shape[0], int(bool(mx)), A.ctypes.data, b.ctypes.data,
                        c.ctypes.data), (A, b, c)


def gpu_solve(L, A, b, c, mx, **opt):
    ps, keep = problem(A, b, c, mx)
    res = _abi.Result()
    L.enumgpu_solve(C.byref(ps), C.byref(options(**opt)), C.byref(res))
    return res


def gpu_ranges(L, A, b, c, mx, opt=None, eps_opt=1e-9, max_list=0, ropt=None, **o):
    """enumgpu_cost_ranges after enumgpu_solve under the same options; ropt: other options for the ranging call."""
    if opt is None:
        opt = gpu_solve(L, A, b, c, mx, **o)
        assert opt.status == _abi.OK, sm.last_error()
    ps, keep = problem(A, b, c, mx)
    out = _abi.Ranging()
    rc = L.enumgpu_cost_ranges(C.byref(ps), C.byref(options(**(o if ropt is None else ropt))), C.byref(opt), eps_opt,
                               max_list, C.byref(out))
    return rc, out, opt


def test_layout_matches_header(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "enumgpu.h"\n'
                   'int (*f)(const enumgpu_problem*, const enumgpu_options*, const enumgpu_result*, double, uint64_t,'
                   ' enumgpu_ranging*) = enumgpu_cost_ranges;\n'
                   'int main(){printf("%zu %zu %zu %zu %zu %zu\\n",sizeof(enumgpu_cost_range),sizeof(enumgpu_ranging),'
                   'offsetof(enumgpu_ranging,n_vertex_bases),offsetof(enumgpu_ranging,kernel_ms),'
                   'offsetof(enumgpu_ranging,range),offsetof(enumgpu_cost_range,decrease_ray));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", os.path.join(ROOT, "simplexmethod_b200"), "-lenumgpu"])
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "simplexmethod_b200"))
    got = [int(v) for v in subprocess.check_output([str(exe)], env=env).split()]
    assert got == [C.sizeof(_abi.CostRange), C.sizeof(_abi.Ranging), _abi.Ranging.n_vertex_bases.offset,
                   _abi.Ranging.kernel_ms.offset, _abi.Ranging.range.offset, _abi.CostRange.decrease_ray.offset]
    restype, argtypes = _abi.SYMBOLS["enumgpu_cost_ranges"]
    assert restype is C.c_int
    assert argtypes == [C.POINTER(_abi.Problem), C.POINTER(_abi.Options), C.POINTER(_abi.Result), C.c_double,
                        C.c_uint64, C.POINTER(_abi.Ranging)]


def oracle_opt(oracle, A, b, c, mx):
    opt, _ = oracle.solve(A, b, c, mx, n_threads=NCPU)
    return opt


def test_argument_errors(oracle):
    """Each bad argument gives its code in the return value and out.status, with or without a GPU."""
    L = sm.lib()
    A, b, c, mx = lpgen.small_degenerate_lp()
    opt = oracle_opt(oracle, A, b, c, mx)
    assert opt.status == _abi.OK
    ps, keep = problem(A, b, c, mx)

    def call(o=None, op=opt, p=ps, out=True):
        r = _abi.Ranging()
        rc = L.enumgpu_cost_ranges(C.byref(p) if p is not None else None, C.byref(o) if o is not None else None,
                                   C.byref(op) if op is not None else None, 1e-9, 0, C.byref(r) if out else None)
        return rc, r

    assert call(out=False)[0] == _abi.ERR_ARG
    for kw in (dict(p=None), dict(op=None), dict(o=options(rank_begin=0, rank_end=5)), dict(o=options(rank_begin=3)),
               dict(o=options(shard_index=0, shard_count=2)), dict(o=options(shard_index=1, shard_count=2)),
               dict(o=options(algo=7))):
        rc, r = call(**kw)
        assert rc == r.status == _abi.ERR_ARG, kw
    bad = []
    for field, value in (("status", _abi.NO_FEASIBLE), ("m", opt.m + 1), ("n_bases", opt.n_bases - 1),
                         ("best_rank", opt.best_rank + 1), ("best_rank", U64)):
        o2 = _abi.Result.from_buffer_copy(bytes(opt))
        setattr(o2, field, value)
        bad.append(o2)
    o2 = _abi.Result.from_buffer_copy(bytes(opt))
    o2.basis[0] = o2.basis[1]
    bad.append(o2)
    for o2 in bad:
        rc, r = call(op=o2)
        assert rc == r.status == _abi.ERR_ARG
        assert "opt" in sm.last_error()
    badA = A.copy()
    badA[0, 0] = np.nan
    pb, keep2 = problem(badA, b, c, mx)
    assert call(p=pb)[0] == _abi.ERR_NONFINITE
    # the Python adapter: a partial enumeration is not a whole-range optimum
    s = sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(A.shape[0])), minimize=not mx))
    s._res = opt
    opt2 = _abi.Result.from_buffer_copy(bytes(opt))
    opt2.n_bases = 3
    s._res = opt2
    with pytest.raises(ValueError):
        s.costRanges()


@pytest.mark.skipif(sm.lib().enumgpu_device_count() > 0, reason="a GPU is present")
def test_no_gpu_means_loud_failure_not_fallback(oracle):
    L = sm.lib()
    A, b, c, mx = lpgen.lab_symmetric_canonical()
    opt = oracle_opt(oracle, A, b, c, mx)
    rc, out, _ = gpu_ranges(L, A, b, c, mx, opt=opt)
    assert rc == out.status == _abi.ERR_CUDA
    assert "no CPU fallback" in sm.last_error()
    with pytest.raises(sm.EnumGpuError, match="no CPU fallback"):
        sm.EnumerationSolver(sm.Canonical(A, b, c, [3, 4], minimize=not mx)).costRanges()


# --------------------------------------------------------------------------------------------- GPU

def check(L, oracle, A, b, c, mx, algos=ALGOS, **o):
    """Both kernel families against the twin, bit for bit; returns the twin."""
    t = twin(oracle, A, b, c, mx, **{k: v for k, v in o.items() if k in ("eps_feas", "eps_piv", "pivot_rule")})
    n = A.shape[1]
    for algo in algos:
        rc, g, _ = gpu_ranges(L, A, b, c, mx, algo=algo, **o)
        assert rc == _abi.OK, sm.last_error()
        assert_equal_to_twin(g, t, n)
        assert g.n_launches >= 2 and g.kernel_ms > 0
    return t


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GOLD))
def test_gpu_tiny_goldens(gpu_lib, oracle, name):
    g = GOLD[name]
    A = np.array(g["A"], dtype=float)
    for mx in (g["maximize"], not g["maximize"]):
        if oracle_opt(oracle, A, g["b"], g["c"], mx).status == _abi.OK:
            check(gpu_lib, oracle, A, g["b"], np.array(g["c"], dtype=float), mx)


@pytest.mark.gpu
@pytest.mark.parametrize("m", range(1, 17))
def test_gpu_dense_shapes(gpu_lib, oracle, m):
    """Every m, both senses; m = 16 is UNDECIDED (no room for the ray LP's row)."""
    A, b, c, _ = lpgen.dense_lp(m, m + 5, m)
    for mx in (False, True):
        t = check(gpu_lib, oracle, A, b, c, mx)
        assert (t["status"] == UNDECIDED) == (m == 16)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["small", "config5"])
def test_gpu_degenerate(gpu_lib, oracle, name):
    A, b, c, mx = {"small": lpgen.small_degenerate_lp, "config5": lpgen.degenerate_lp}[name]()
    for sense in (mx, not mx):
        if oracle_opt(oracle, A, b, c, sense).status == _abi.OK:
            check(gpu_lib, oracle, A, b, c, sense)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(8, 20), (10, 22)])
@pytest.mark.parametrize("name", sorted(FAMILIES))
def test_gpu_structured_families(gpu_lib, oracle, name, m, n):
    """Dyadic ties, -0.0 components, +-inf and NaN keys; both kernel families, both senses."""
    A, b, c, _ = FAMILIES[name](m, n, 1)
    for mx in (False, True):
        if oracle_opt(oracle, A, b, c, mx).status == _abi.OK:
            check(gpu_lib, oracle, A, b, c, mx)


@pytest.mark.gpu
def test_gpu_general_lps(gpu_lib, oracle):
    for seed in SEEDS:
        A, b, c, mx, opt, t = seed_twin(oracle, seed)
        for algo in ALGOS:
            rc, g, _ = gpu_ranges(gpu_lib, A, b, c, mx, algo=algo)
            assert rc == _abi.OK, (seed, sm.last_error())
            assert_equal_to_twin(g, t, A.shape[1])


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ALGOS)
def test_gpu_max_list_splits_both_listings(gpu_lib, oracle, algo):
    """Lists too small for either listing: sub-ranges, some halved again; the same answer as one pass."""
    for A, b, c, mx in (lpgen.small_degenerate_lp(), FAMILIES["signed_duplicates"](8, 20, 1)):
        rc, whole, opt = gpu_ranges(gpu_lib, A, b, c, mx, algo=algo)
        assert rc == _abi.OK
        assert whole.n_vertex_bases > 40 and whole.n_ray_bases > 4
        for max_list in (3, whole.n_ray_bases - 1, whole.n_vertex_bases // 7, whole.n_vertex_bases - 1):
            rc, split, _ = gpu_ranges(gpu_lib, A, b, c, mx, opt=opt, max_list=max_list, algo=algo)
            assert rc == _abi.OK
            assert bytes(split.range) == bytes(whole.range)
            assert (split.status, split.n_vertex_bases, split.n_ray_bases) == \
                (whole.status, whole.n_vertex_bases, whole.n_ray_bases)
            assert split.n_launches > whole.n_launches


@pytest.mark.gpu
def test_gpu_opt_from_other_options_is_refused(gpu_lib, oracle):
    """An optimum under the default eps_feas, ranged under eps_feas = 0.5, where more bases are feasible and one beats
    its key."""
    A, b, c, mx = FAMILIES["sparse_dyadic"](8, 20, 2)
    loose = gpu_solve(gpu_lib, A, b, c, mx, eps_feas=0.5)
    tight = gpu_solve(gpu_lib, A, b, c, mx)
    assert loose.status == tight.status == _abi.OK and loose.key < tight.key
    rc, out, _ = gpu_ranges(gpu_lib, A, b, c, mx, opt=tight, ropt=dict(eps_feas=0.5))
    assert rc == out.status == _abi.ERR_ARG
    assert "other options" in sm.last_error()
    rc, out, _ = gpu_ranges(gpu_lib, A, b, c, mx, opt=loose, ropt=dict(eps_feas=0.5))
    assert rc == _abi.OK


@pytest.mark.gpu
def test_gpu_unbounded(gpu_lib, oracle):
    hit = 0
    for seed in SEEDS:
        A, b, c, mx, opt, t = seed_twin(oracle, seed)
        if t["status"] == UNBOUNDED:
            hit += 1
            can = sm.Canonical(A, b, c, list(range(A.shape[0])), minimize=not mx)
            with pytest.raises(RuntimeError, match="objective is unbounded"):
                sm.EnumerationSolver(can).costRanges()
    assert hit > 0


def gpu_bits(L, A, b, c, mx, ranks):
    """(ranks, S, x_B, z) of listed ranks from enumgpu_eval_ranks, a chunk at a time."""
    m, n = A.shape
    ps, keep = problem(A, b, c, mx)
    o = options()
    for lo in range(0, len(ranks), 1 << 20):
        r = np.ascontiguousarray(ranks[lo:lo + (1 << 20)], dtype=np.uint64)
        k = len(r)
        x = np.zeros(k * m)
        z = np.zeros(k)
        cls = np.zeros(k, dtype=np.int32)
        assert L.enumgpu_eval_ranks(C.byref(ps), C.byref(o), r.ctypes.data_as(C.POINTER(C.c_uint64)), k,
                                    x.ctypes.data_as(C.POINTER(C.c_double)), z.ctypes.data_as(C.POINTER(C.c_double)),
                                    cls.ctypes.data_as(C.POINTER(C.c_int32))) == _abi.OK
        assert np.all(cls == FEASIBLE)
        S = np.array([unrank(n, m, int(v)) for v in r], dtype=np.int64).reshape(k, m)
        yield r, S, x.reshape(k, m), z


def gpu_list(L, A, b, c, mx, cap):
    ps, keep = problem(A, b, c, mx)
    ranks = np.zeros(cap, dtype=np.uint64)
    n_listed = C.c_uint64()
    out = _abi.Result()
    assert L.enumgpu_list_feasible(C.byref(ps), C.byref(options()), ranks.ctypes.data_as(C.POINTER(C.c_uint64)), cap,
                                   C.byref(n_listed), C.byref(out)) == _abi.OK
    assert n_listed.value == out.n_feasible <= cap
    return np.sort(ranks[: n_listed.value])


@pytest.mark.gpu
def test_gpu_headline_12_40(gpu_lib):
    """One call on the headline LP; the twin from the GPU's own listing and enumgpu_eval_ranks bits."""
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    m, n = A.shape
    rc, g, opt = gpu_ranges(gpu_lib, A, b, c, mx)
    assert rc == _abi.OK, sm.last_error()
    xs = np.zeros(n)
    xs[list(opt.basis)[:m]] = list(opt.x_B)[:m]
    Aa, ba = ray_lp(A)
    ck = -c if mx else c
    ray_ranks = gpu_list(gpu_lib, Aa, ba, ck, False, max(1, g.n_ray_bases))
    t = twin_ranges(n, m, mx, opt.key, xs, 1e-9, gpu_bits(gpu_lib, A, b, c, mx, gpu_list(gpu_lib, A, b, c, mx,
                                                                                                 g.n_vertex_bases)),
                    gpu_bits(gpu_lib, Aa, ba, ck, False, ray_ranks))
    assert_equal_to_twin(g, t, n)
    for j in list(opt.basis)[:m]:
        assert math.isfinite(g.range[j].decrease) or math.isfinite(g.range[j].increase)


@pytest.mark.gpu
def test_gpu_python_adapter(gpu_lib, oracle):
    for A, b, c, mx in (lpgen.lab_symmetric_canonical(), lpgen.small_degenerate_lp()):
        m = A.shape[0]
        s = sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(m)), minimize=not mx))
        r = s.costRanges()
        rc, g, _ = gpu_ranges(gpu_lib, A, b, c, mx)
        assert rc == _abi.OK and r.status == g.status
        for name in FIELDS:
            assert [bits(v) if isinstance(v, float) else int(v) for v in getattr(r, name)] == \
                [bits(getattr(g.range[j], name)) if "rank" not in name and "ray" not in name else int(getattr(g.range[j], name))
                 for j in range(A.shape[1])]
        assert (r.n_vertex_bases, r.n_ray_bases) == (g.n_vertex_bases, g.n_ray_bases)


@pytest.fixture(scope="module")
def certify_demo():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "simplexmethod_b200", "cpp"), "-s"])
    return os.path.join(ROOT, "simplexmethod_b200", "cpp", "build", "certify_demo")


@pytest.mark.gpu
def test_gpu_certify_demo_ranges(gpu_lib, certify_demo, tmp_path):
    """certify_demo --ranges prints the table of the Python adapter's ranges."""
    sym_A = np.array([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0], [2.0, 1.0, 1.0]])
    sym_b = np.array([10.0, 20.0, 8.0])
    sym_c = np.array([7.0, 8.0, 3.0])
    f = tmp_path / "lp.txt"
    f.write_text("\n".join(["maximize", "objective:", " ".join(repr(float(v)) for v in sym_c), "constraints:"] +
                           [" ".join(repr(float(v)) for v in list(sym_A[i]) + [sym_b[i]]) for i in range(3)]) + "\n")
    out = subprocess.run([certify_demo, "--ranges", str(f)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    rows = {}
    for line in out.stdout.splitlines():
        if line.startswith("range "):
            _, j, dec, inc, dr, ir, dray, iray = line.split()
            rows[int(j)] = (float(dec), float(inc), int(dr), int(ir), int(dray), int(iray))
    can = sm.Symmetrical(sym_A, sym_b, sym_c, True).ToCanonical()
    r = sm.EnumerationSolver(can).costRanges()
    assert sorted(rows) == list(range(len(r.decrease)))
    for j, got in rows.items():
        assert got == (float(r.decrease[j]), float(r.increase[j]), int(r.decrease_rank[j]), int(r.increase_rank[j]),
                       int(r.decrease_ray[j]), int(r.increase_ray[j]))
