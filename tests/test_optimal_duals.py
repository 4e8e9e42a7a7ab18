"""Optimal duals at degenerate optima: the window of optimal bases and the search for a dual-feasible one.

enumgpu_list_window lists the feasible bases whose key is at most a bound; enumgpu_certify_bases certifies many
bases in one call; enumgpu_certify_optimum certifies the enumeration's winner and, when that is undecided, the
window key <= key* + eps_opt * max(1, |key*|) in ascending rank, and returns the lowest-rank OPTIMAL basis, else
enumgpu_certify's answer (DESIGN.md §3.1).

CPU: the same search built from the oracle (enumcpu.list_class, per-basis keys) and the certificate twin
(tests/certify_twin.c), against HiGHS and exact rationals on the 200 random general-form LPs of
test_certificate.py; self-checks that pin the window of two block LPs; the struct layout.
GPU: every entry against that CPU pipeline bit for bit, with both kernel families; the adapters.
"""
import ctypes as C
import math
import os
import shutil
import subprocess
import tempfile
from fractions import Fraction
from itertools import combinations, product

import numpy as np
import pytest

import simplexmethod_b200 as sm
from simplexmethod_b200 import _abi, lpgen
from test_certificate import (ALGOS, BOUNDED, GOLD, HERE, NCPU, OPTIMAL, ROOT, SEEDS, UNBOUNDED, UNDECIDED,
                              assert_cert_bits, bits, degenerate_block_16, general_lp, options, problem, seed_pipeline,
                              symmetric_file)
from test_certificate import certify_demo  # noqa: F401  (the C++ demo fixture)
from test_problem_types import highs_general
from test_structured_parity import FAMILIES, all_nan_keys, headline_windows

FEASIBLE = 0
WINNER, WINDOW, FALLBACK = _abi.OPT_WINNER, _abi.OPT_WINDOW, _abi.OPT_FALLBACK
INF = float("inf")
CHUNK = 4096          # bases per k_certify launch in the library


# --------------------------------------------------------------------------------------------- CPU twin, many bases

_TWIN = None


def twin_many():
    """tests/certify_twin.c + tests/certify_twin_many.c, built once per process with the CPU oracle's flags."""
    global _TWIN
    if _TWIN is None:
        tmp = tempfile.mkdtemp(prefix="certify_twin_many_")
        so = os.path.join(tmp, "libcertify_twin_many.so")
        subprocess.check_call(["gcc", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra",
                               "-std=c11", "-shared", "-I", os.path.join(ROOT, "include"), "-o", so,
                               os.path.join(HERE, "certify_twin.c"), os.path.join(HERE, "certify_twin_many.c"), "-lm"])
        L = C.CDLL(so)
        shutil.rmtree(tmp)
        L.certify_twin_many.restype = C.c_uint64
        L.certify_twin_many.argtypes = [C.POINTER(_abi.Problem), C.c_double, C.c_int, C.c_double, C.c_double,
                                        C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(_abi.Certificate)]
        _TWIN = L
    return _TWIN


def twin_certify_many(A, b, c, mx, bases, eps_opt=1e-9):
    """The twin's certificates (absolute pivot rule, default tolerances) at bases [k, m]: (rc [k], [Certificate])."""
    keep, p = problem(A, b, c, mx)
    bases = np.ascontiguousarray(bases, dtype=np.int32).reshape(-1, p.m)
    k = bases.shape[0]
    rc = np.zeros(k, dtype=np.int32)
    out = (_abi.Certificate * k)()
    twin_many().certify_twin_many(C.byref(p), 1e-9, _abi.PIVOT_ABSOLUTE, 1e-9 * float(np.abs(keep[0]).max()), eps_opt,
                                  bases.ctypes.data, k, rc.ctypes.data, out)
    return rc, list(out)


def unrank(oracle, n, m, r):
    S = (C.c_int32 * m)()
    assert oracle.lib().enumcpu_unrank(n, m, int(r), S) == 0
    return list(S)


def rank_of(oracle, n, m, S):
    return int(oracle.lib().enumcpu_rank(n, m, (C.c_int32 * m)(*S)))


def key_bound(key, eps_opt=1e-9):
    return key + eps_opt * max(1.0, abs(key))


def oracle_window(oracle, A, b, c, mx, key_max, **opt):
    """The oracle's feasible ranks (ascending) whose key is <= key_max; key_max = +inf: all of them."""
    _, ranks, count = oracle.list_class(A, b, c, mx, FEASIBLE, capacity=1 << 22, n_threads=NCPU, **opt)
    assert count == ranks.size
    if key_max == INF:
        return ranks
    m, n = A.shape
    keep = []
    for r in ranks:
        st, _, z = oracle.eval_basis(A, b, c, mx, unrank(oracle, n, m, r))
        assert st == FEASIBLE
        if (-z if mx else z) <= key_max:
            keep.append(r)
    return np.array(keep, dtype=np.uint64)


class CpuOptimum:
    """The search of enumgpu_certify_optimum built from the oracle and the twin."""

    def __init__(self, source, cert, basis, rank, window_index, n_window, bound):
        self.source, self.cert, self.basis, self.rank = source, cert, basis, rank
        self.window_index, self.n_window, self.key_bound = window_index, n_window, bound


def cpu_optimum(oracle, A, b, c, mx, res, winner_cert, fallback, window=None, max_window=1 << 24):
    """res: the oracle's enumeration; winner_cert: the twin's certificate at its winner; fallback() -> the
    certificate enumgpu_certify returns there (ray enumeration included); window: the ascending window, if known."""
    m, n = A.shape
    S, bound = list(res.basis)[:m], key_bound(res.key)
    if winner_cert.status in (OPTIMAL, UNBOUNDED):
        return CpuOptimum(WINNER, winner_cert, S, res.best_rank, _abi.UINT64_MAX, 0, bound)
    if window is None:
        window = oracle_window(oracle, A, b, c, mx, bound)
    if len(window) <= max_window:
        for i in range(0, len(window), CHUNK):
            bases = [unrank(oracle, n, m, r) for r in window[i:i + CHUNK]]
            rcs, certs = twin_certify_many(A, b, c, mx, bases)
            assert (rcs == _abi.OK).all()
            for j, ct in enumerate(certs):
                if ct.status == OPTIMAL:
                    return CpuOptimum(WINDOW, ct, bases[j], int(window[i + j]), i + j, len(window), bound)
    return CpuOptimum(FALLBACK, fallback(), S, res.best_rank, _abi.UINT64_MAX, len(window), bound)


_SEED_OPT = {}


def seed_optimum(oracle, seed):
    if seed not in _SEED_OPT:
        A, b, c, mx, res, cert, verdict, aux, ray = seed_pipeline(oracle, seed)

        def fallback():
            ct = _abi.Certificate()
            C.pointer(ct)[0] = cert
            ct.status = verdict
            if ray is not None:
                for j, v in enumerate(ray):
                    ct.ray[j] = v
            return ct
        _SEED_OPT[seed] = cpu_optimum(oracle, A, b, c, mx, res, cert, fallback)
    return _SEED_OPT[seed]


def block_lp(m):
    """degenerate_block_16's construction at any even m: the identity, then per pair of rows k the columns
    (1, -1) and (-1, 1) with costs -1 and +2; b = 0."""
    if m == 16:
        return degenerate_block_16()
    n = 2 * m
    A = np.zeros((m, n), order="F")
    A[:, :m] = np.eye(m)
    c = np.zeros(n)
    for k in range(m // 2):
        A[2 * k, m + 2 * k], A[2 * k + 1, m + 2 * k] = 1.0, -1.0
        A[2 * k, m + 2 * k + 1], A[2 * k + 1, m + 2 * k + 1] = -1.0, 1.0
        c[m + 2 * k], c[m + 2 * k + 1] = -1.0, 2.0
    return A, np.zeros(m), c, False


def block_window(oracle, m):
    """Every feasible basis of block_lp(m), by hand: b = 0 makes every nonsingular basis feasible with key 0, and a
    nonsingular basis takes two independent columns of each 2-row block: any pair of (e_2k, e_2k+1, p_k, q_k) but
    (p_k, q_k), 5 per block.  Ascending ranks."""
    pairs = []
    for k in range(m // 2):
        cols = [2 * k, 2 * k + 1, m + 2 * k, m + 2 * k + 1]
        pairs.append([pr for pr in combinations(cols, 2) if pr != (m + 2 * k, m + 2 * k + 1)])
    ranks = sorted(rank_of(oracle, 2 * m, m, sorted(sum(choice, ()))) for choice in product(*pairs))
    return np.array(ranks, dtype=np.uint64)


_BLOCK = {}


def block_optimum(oracle, m):
    """(LP, CpuOptimum, window, number of OPTIMAL bases in the window) of block_lp(m)."""
    if m not in _BLOCK:
        A, b, c, mx = block_lp(m)
        n = 2 * m
        window = block_window(oracle, m)
        res, _ = oracle.solve(A, b, c, mx, n_threads=NCPU, rank_begin=0, rank_end=int(window[0]) + 1)
        assert res.status == _abi.OK and res.best_rank == 0 and res.key == 0.0       # the winner: rank 0, key 0
        winner = twin_certify_many(A, b, c, mx, [list(range(m))])[1][0]
        opt = cpu_optimum(oracle, A, b, c, mx, res, winner, None, window=window)
        n_optimal = 0
        for i in range(0, len(window), 1 << 15):
            bases = [unrank(oracle, n, m, r) for r in window[i:i + (1 << 15)]]
            n_optimal += sum(ct.status == OPTIMAL for ct in twin_certify_many(A, b, c, mx, bases)[1])
        _BLOCK[m] = ((A, b, c, mx), opt, window, n_optimal)
    return _BLOCK[m]


def exact_dual_feasible(A, c, mx, S, y, eps=Fraction(1, 10**9)):
    """Every nonbasic reduced cost c_j - y.a_j (sense-adjusted), in exact rationals over the doubles, >= -eps."""
    m, n = A.shape
    Y = [Fraction(float(v)) for v in y[:m]]
    for j in range(n):
        if j in S:
            continue
        r = Fraction(float(c[j])) - sum(Y[i] * Fraction(float(A[i, j])) for i in range(m))
        if (-r if mx else r) < -eps:
            return False
    return True


# --------------------------------------------------------------------------------------------- CPU

@pytest.mark.parametrize("seed", SEEDS)
def test_cpu_pipeline_vs_highs(oracle, seed):
    A, b, c, mx, res, cert, verdict, aux, ray = seed_pipeline(oracle, seed)
    opt = seed_optimum(oracle, seed)
    st, z, _ = highs_general(general_lp(seed))
    assert st in (0, 3)
    assert opt.cert.status == (OPTIMAL if st == 0 else UNBOUNDED)
    m = A.shape[0]
    if opt.cert.status == OPTIMAL:
        assert exact_dual_feasible(A, c, mx, opt.basis, list(opt.cert.y))
        dual = math.fsum(float(Fraction(bi) * Fraction(yi)) for bi, yi in zip(b, list(opt.cert.y)[:m]))
        assert dual == pytest.approx(res.objective, rel=1e-9, abs=1e-9)
        assert opt.cert.objective == pytest.approx(res.objective, rel=1e-9, abs=1e-9)


def test_selfcheck_cpu_pipeline_counts(oracle):
    """132 OPTIMAL (68 at the winner, 64 from the window), 68 UNBOUNDED; every path of the search is reached."""
    by = {}
    for seed in SEEDS:
        opt = seed_optimum(oracle, seed)
        by.setdefault((opt.source, opt.cert.status), []).append(seed)
    counts = {k: len(v) for k, v in by.items()}
    assert counts.get((WINNER, OPTIMAL)) == 68 and counts.get((WINDOW, OPTIMAL)) == 64
    assert sum(v for (src, st), v in counts.items() if st == UNBOUNDED) == 68
    assert counts.get((FALLBACK, UNBOUNDED), 0) >= 1 and counts.get((WINNER, UNBOUNDED), 0) >= 1
    assert set(counts) <= {(WINNER, OPTIMAL), (WINDOW, OPTIMAL), (WINNER, UNBOUNDED), (FALLBACK, UNBOUNDED)}
    # the window seeds are exactly the ones test_certificate.py calls BOUNDED
    assert by[(WINDOW, OPTIMAL)] == [s for s in SEEDS if seed_pipeline(oracle, s)[6] == BOUNDED]


def test_selfcheck_block_12_24(oracle):
    (A, b, c, mx), opt, window, n_optimal = block_optimum(oracle, 12)
    assert len(window) == 15625
    assert oracle_window(oracle, A, b, c, mx, key_bound(0.0)).tolist() == window.tolist()     # the oracle agrees
    assert (opt.source, opt.cert.status, opt.window_index, opt.rank) == (WINDOW, OPTIMAL, 15561, 1829919)
    assert opt.basis == list(range(1, 12, 2)) + list(range(12, 24, 2))
    assert n_optimal == 64


def test_selfcheck_block_16_32(oracle):
    (A, b, c, mx), opt, window, n_optimal = block_optimum(oracle, 16)
    assert len(window) == 390625
    assert (opt.source, opt.cert.status, opt.window_index, opt.rank) == (WINDOW, OPTIMAL, 390369, 405183118)
    assert opt.basis == list(range(1, 16, 2)) + list(range(16, 32, 2))
    assert n_optimal == 256
    assert exact_dual_feasible(A, c, mx, opt.basis, list(opt.cert.y))
    # a max_window below the window's size takes the fallback
    small = cpu_optimum(oracle, A, b, c, mx, oracle.solve(A, b, c, mx, rank_begin=0, rank_end=1)[0],
                        twin_certify_many(A, b, c, mx, [list(range(16))])[1][0], lambda: "fallback", window=window,
                        max_window=len(window) - 1)
    assert small.source == FALLBACK and small.cert == "fallback"


def test_optimum_struct_layout_matches_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "enumgpu.h"\n'
                   'int main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",sizeof(enumgpu_optimum),'
                   'offsetof(enumgpu_optimum,basis),offsetof(enumgpu_optimum,source),'
                   'offsetof(enumgpu_optimum,n_launches),offsetof(enumgpu_optimum,rank),'
                   'offsetof(enumgpu_optimum,key_bound),offsetof(enumgpu_optimum,n_window),'
                   'offsetof(enumgpu_optimum,window_index),(size_t)ENUMGPU_OPT_FALLBACK);return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    T = _abi.Optimum
    assert got == [C.sizeof(T), T.basis.offset, T.source.offset, T.n_launches.offset, T.rank.offset,
                   T.key_bound.offset, T.n_window.offset, T.window_index.offset, _abi.OPT_FALLBACK]


# --------------------------------------------------------------------------------------------- GPU helpers

def gpu_list_window(L, A, b, c, mx, key_max, algo=_abi.ALGO_AUTO, rank_begin=0, rank_end=0, capacity=1 << 22):
    keep, p = problem(A, b, c, mx)
    ranks = np.zeros(capacity, dtype=np.uint64)
    n_listed = C.c_uint64()
    res = _abi.Result()
    rc = L.enumgpu_list_window(C.byref(p), C.byref(options(algo, rank_begin, rank_end)), key_max,
                               ranks.ctypes.data_as(C.POINTER(C.c_uint64)), capacity, C.byref(n_listed), C.byref(res))
    assert rc in (_abi.OK, _abi.NO_FEASIBLE), sm.last_error()
    return ranks[:n_listed.value].copy(), res


def gpu_certify_bases(L, A, b, c, mx, bases):
    keep, p = problem(A, b, c, mx)
    arr = np.ascontiguousarray(bases, dtype=np.int32).reshape(-1, p.m)
    out = (_abi.Certificate * arr.shape[0])()
    rc = L.enumgpu_certify_bases(C.byref(p), C.byref(options()), arr.ctypes.data_as(C.POINTER(C.c_int32)),
                                 arr.shape[0], -1.0, out)
    assert rc == _abi.OK, sm.last_error()
    return list(out)


def gpu_optimum(L, A, b, c, mx, algo=_abi.ALGO_AUTO, max_window=0):
    keep, p = problem(A, b, c, mx)
    o = options(algo)
    res = _abi.Result()
    assert L.enumgpu_solve(C.byref(p), C.byref(o), C.byref(res)) == _abi.OK
    opt = _abi.Optimum()
    rc = L.enumgpu_certify_optimum(C.byref(p), C.byref(o), C.byref(res), -1.0, max_window, C.byref(opt))
    assert rc == _abi.OK, sm.last_error()
    return opt, res


def assert_optimum_same(g, o, m):
    assert (g.source, g.rank, g.window_index, g.n_window) == (o.source, o.rank, o.window_index, o.n_window)
    assert list(g.basis)[:m] == list(o.basis)
    assert bits(g.key_bound) == bits(o.key_bound)
    assert_cert_bits(g.cert, o.cert)
    if o.cert.status == UNBOUNDED:
        assert bits(list(g.cert.ray)) == bits(list(o.cert.ray))


def window_lps():
    """(name, A, b, c, mx): the tiny goldens, small_degenerate_lp, config 5 and the structured families."""
    out = [(f"gold_{k}", np.array(g["A"], dtype=float), np.array(g["b"], dtype=float), np.array(g["c"], dtype=float),
            bool(g["maximize"])) for k, g in sorted(GOLD.items())]
    out.append(("small_degenerate",) + tuple(lpgen.small_degenerate_lp()))
    out.append(("config5",) + tuple(lpgen.degenerate_lp()))
    # the kernels compiled for n = 24 and n = 30, and the run-time-n one at (6, 18); tiny_rhs, whose bases are
    # nearly all feasible, only there
    shapes = {name: [(6, 18)] if name == "tiny_rhs" else [(8, 24)] for name in FAMILIES}
    shapes["sparse_dyadic"] = shapes["thirds"] = [(6, 18), (8, 24), (10, 30)]
    for name, fam in sorted(FAMILIES.items()):
        for m, n in shapes[name]:
            out.append((f"{name}_{m}_{n}",) + tuple(fam(m, n, 1)))
    out.append(("all_nan_keys_8_24",) + tuple(all_nan_keys(8, 24)))
    return out


WINDOW_LPS = window_lps()


def bounds_of(oracle, A, b, c, mx):
    """+inf, the optimum's window bound, and the median key of the feasible bases (a wider finite window)."""
    res, _ = oracle.solve(A, b, c, mx, n_threads=NCPU)
    out = [INF]
    if res.status == _abi.OK:
        out.append(key_bound(res.key))
    _, ranks, _ = oracle.list_class(A, b, c, mx, FEASIBLE, capacity=1 << 22, n_threads=NCPU)
    m, n = A.shape
    keys = sorted(k for k in ((lambda z: -z if mx else z)(oracle.eval_basis(A, b, c, mx, unrank(oracle, n, m, r))[2])
                              for r in ranks[:2000]) if not math.isnan(k))
    if keys:
        out.append(keys[len(keys) // 2])
    return out


# --------------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(WINDOW_LPS)), ids=[w[0] for w in WINDOW_LPS])
def test_list_window_vs_oracle(gpu_lib, oracle, case):
    name, A, b, c, mx = WINDOW_LPS[case]
    m, n = A.shape
    for key_max in bounds_of(oracle, A, b, c, mx):
        want = oracle_window(oracle, A, b, c, mx, key_max)
        for algo in ALGOS:
            got, res = gpu_list_window(gpu_lib, A, b, c, mx, key_max, algo)
            assert got.tolist() == want.tolist(), (name, key_max, algo)
            if key_max == INF:
                ranks = np.zeros(1 << 22, dtype=np.uint64)
                n_listed = C.c_uint64()
                keep, p = problem(A, b, c, mx)
                plain = _abi.Result()
                gpu_lib.enumgpu_list_feasible(C.byref(p), C.byref(options(algo)), ranks.ctypes.data_as(C.POINTER(C.c_uint64)),
                                              1 << 22, C.byref(n_listed), C.byref(plain))
                assert ranks[:n_listed.value].tolist() == got.tolist() and plain.n_feasible == res.n_feasible
    if name.startswith("all_nan"):
        assert len(oracle_window(oracle, A, b, c, mx, INF)) > 0
        assert gpu_list_window(gpu_lib, A, b, c, mx, 1e300)[0].size == 0        # a finite bound drops NaN keys


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_list_window_general_lps(gpu_lib, oracle, seed):
    A, b, c, mx, res, cert, verdict, aux, ray = seed_pipeline(oracle, seed)
    bound = key_bound(res.key)
    want = oracle_window(oracle, A, b, c, mx, bound)
    for algo in ALGOS:
        assert gpu_list_window(gpu_lib, A, b, c, mx, bound, algo)[0].tolist() == want.tolist()


@pytest.mark.gpu
def test_list_window_headline(gpu_lib, oracle):
    """dense (12, 40): k_shared<12,40> == k_independent == the oracle on rank windows, with a bound that lets a few
    hundred to a few thousand bases of each window in; and both kernels over the whole range."""
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    for lo, hi in headline_windows():
        _, ranks, _ = oracle.list_class(A, b, c, mx, FEASIBLE, n_threads=NCPU, rank_begin=lo, rank_end=hi)
        keys = sorted((lambda z: -z if mx else z)(oracle.eval_basis(A, b, c, mx, unrank(oracle, 40, 12, r))[2])
                      for r in ranks)
        bound = keys[min(1000, len(keys) - 1)]
        want = oracle_window(oracle, A, b, c, mx, bound, rank_begin=lo, rank_end=hi)
        assert 200 <= want.size <= 5000
        for algo in ALGOS:
            got, res = gpu_list_window(gpu_lib, A, b, c, mx, bound, algo, lo, hi)
            assert got.tolist() == want.tolist()
            assert res.algo_used == algo
    full = [gpu_list_window(gpu_lib, A, b, c, mx, 0.0, algo)[0] for algo in ALGOS]
    sh = gpu_list_window(gpu_lib, A, b, c, mx, 0.0, _abi.ALGO_SHARED)[1]
    assert full[0].tolist() == full[1].tolist() and sh.algo_used == _abi.ALGO_SHARED


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["small_degenerate", "config5", "block_12"])
def test_certify_bases_vs_twin(gpu_lib, oracle, case):
    """Every window basis (above one chunk of 4096 for the block LP), bit for bit; count = 1 == enumgpu_certify."""
    if case == "block_12":
        (A, b, c, mx), _, window, _ = block_optimum(oracle, 12)
    else:
        A, b, c, mx = lpgen.small_degenerate_lp() if case == "small_degenerate" else lpgen.degenerate_lp()
        window = oracle_window(oracle, A, b, c, mx, key_bound(oracle.solve(A, b, c, mx, n_threads=NCPU)[0].key))
    m, n = A.shape
    bases = [unrank(oracle, n, m, r) for r in window]
    got = gpu_certify_bases(gpu_lib, A, b, c, mx, bases)
    rcs, want = twin_certify_many(A, b, c, mx, bases)
    assert (rcs == _abi.OK).all()
    for g, w in zip(got, want):
        assert_cert_bits(g, w)
        assert bits(list(g.ray)) == bits(list(w.ray))
    # count = 1, in a permuted column order, against enumgpu_certify; and the error classes
    keep, p = problem(A, b, c, mx)
    for S in (bases[0][::-1], bases[-1], [0] * m, ):
        one = gpu_certify_bases(gpu_lib, A, b, c, mx, [S])[0]
        ref = _abi.Certificate()
        rc = gpu_lib.enumgpu_certify(C.byref(p), C.byref(options()), (C.c_int32 * m)(*S), -1.0, C.byref(ref))
        if rc == _abi.ERR_ARG:
            assert one.status == _abi.ERR_ARG and one.basis_class == ref.basis_class == _abi.BASIS_SINGULAR
        elif ref.status in (OPTIMAL, UNBOUNDED):
            assert_cert_bits(one, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_certify_optimum_general_lps(gpu_lib, oracle, seed):
    A, b, c, mx = seed_pipeline(oracle, seed)[:4]
    want = seed_optimum(oracle, seed)
    for algo in ALGOS:
        got, _ = gpu_optimum(gpu_lib, A, b, c, mx, algo)
        assert_optimum_same(got, want, A.shape[0])


@pytest.mark.gpu
@pytest.mark.parametrize("m", [12, 16])
def test_certify_optimum_block_lps(gpu_lib, oracle, m):
    (A, b, c, mx), want, window, _ = block_optimum(oracle, m)
    for algo in ALGOS:
        got, res = gpu_optimum(gpu_lib, A, b, c, mx, algo)
        assert_optimum_same(got, want, m)
        assert got.cert.status == OPTIMAL and got.n_launches > 2
    # enumgpu_certify on the same LP: undecided at m = 16 (bounded by the rays at m = 12)
    keep, p = problem(A, b, c, mx)
    ref = _abi.Certificate()
    assert gpu_lib.enumgpu_certify(C.byref(p), C.byref(options()), (C.c_int32 * m)(*range(m)), -1.0, C.byref(ref)) == 0
    assert ref.status == (UNDECIDED if m == 16 else BOUNDED)
    # a max_window below the window: enumgpu_certify's answer, window counted in full
    fb, _ = gpu_optimum(gpu_lib, A, b, c, mx, max_window=len(window) - 1)
    assert fb.source == FALLBACK and fb.n_window == len(window) and fb.window_index == _abi.UINT64_MAX
    assert list(fb.basis)[:m] == list(range(m)) and fb.rank == 0
    assert fb.cert.status == ref.status and fb.cert.n_aux_bases == ref.n_aux_bases
    assert_cert_bits(fb.cert, ref)


@pytest.mark.gpu
def test_certify_optimum_winner_is_certify(gpu_lib, oracle):
    """Where the winner decides, the certificate is enumgpu_certify's, bit for bit, and nothing is listed."""
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    got, res = gpu_optimum(gpu_lib, A, b, c, mx)
    keep, p = problem(A, b, c, mx)
    ref = _abi.Certificate()
    assert gpu_lib.enumgpu_certify(C.byref(p), C.byref(options()), res.basis, -1.0, C.byref(ref)) == 0
    assert got.source == WINNER and got.n_window == 0 and got.n_launches == 1 and got.rank == res.best_rank
    assert_cert_bits(got.cert, ref)
    # an opt that does not belong to the LP is an argument error
    bad = _abi.Result()
    C.pointer(bad)[0] = res
    bad.basis[0] += 1
    opt = _abi.Optimum()
    assert gpu_lib.enumgpu_certify_optimum(C.byref(p), None, C.byref(bad), -1.0, 0, C.byref(opt)) == _abi.ERR_ARG


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_solver_optimal_duals(gpu_lib, oracle, seed):
    A, b, c, mx, res, cert, verdict, aux, ray = seed_pipeline(oracle, seed)
    want = seed_optimum(oracle, seed)
    m, n = A.shape
    can = sm.Canonical(A, b, c, list(range(m)), minimize=not mx)
    plain = sm.EnumerationSolver(can)
    plain.solve()
    dflt = plain.certify()                                  # the default is enumgpu_certify at the winner
    assert dflt.status == verdict and plain.certificateBasis() == plain.optimalBasis()
    keep, p = problem(A, b, c, mx)
    ref = _abi.Certificate()
    gpu_lib.enumgpu_certify(C.byref(p), C.byref(options()), res.basis, -1.0, C.byref(ref))
    assert_cert_bits(dflt, ref)
    s = sm.EnumerationSolver(can, optimal_duals=True)
    s.solve()
    assert bits(s.dualValues()) == bits(list(want.cert.y)[:m])
    assert bits(s.reducedCosts()) == bits(list(want.cert.reduced_cost)[:n])
    assert s.certificateBasis() == list(want.basis)
    if verdict == BOUNDED:
        assert exact_dual_feasible(A, c, mx, s.certificateBasis(), s.dualValues())
    ranks = s.optimalBases()
    assert ranks.tolist() == oracle_window(oracle, A, b, c, mx, key_bound(res.key)).tolist()
    checked = sm.EnumerationSolver(can, check_unbounded=True, optimal_duals=True)
    if verdict == UNBOUNDED:
        with pytest.raises(RuntimeError, match="objective is unbounded"):
            checked.solve()
    else:
        checked.solve()
        assert checked.unboundedRay() is None


@pytest.mark.gpu
def test_cpp_adapter_optimal_duals(gpu_lib, oracle, certify_demo, tmp_path):
    """certify_demo --optimal-duals on LPs that take the window path; without the flag the output is unchanged."""
    seeds = [s for s in SEEDS if seed_optimum(oracle, s).source == WINDOW][:3]
    assert seeds
    for seed in seeds:
        A, b, c, mx = seed_pipeline(oracle, seed)[:4]
        want = seed_optimum(oracle, seed)
        f = tmp_path / f"lp{seed}.txt"
        symmetric_file(f, seed)
        plain = subprocess.run([certify_demo, str(f)], capture_output=True, text=True)
        out = subprocess.run([certify_demo, str(f), "--optimal-duals"], capture_output=True, text=True)
        assert out.returncode == 0 == plain.returncode, out.stderr
        facts = {ln.split()[0]: ln.split()[1:] for ln in out.stdout.splitlines()}
        assert int(facts["cert_status"][0]) == OPTIMAL and int(facts["source"][0]) == WINDOW
        assert [int(v) for v in facts["cert_basis"]] == list(want.basis)
        assert [float(v) for v in facts["y"]] == list(want.cert.y)[:A.shape[0]]
        assert facts["check_unbounded"] == ["0"]
        assert "cert_basis" not in plain.stdout and int(plain.stdout.split("cert_status")[1].split()[0]) == BOUNDED
