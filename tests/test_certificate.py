"""Certificate of the enumerated optimum: dual values, reduced costs and detection of unbounded LPs.

enumgpu_certify computes, at the enumeration's winning basis, u_j = B^-1 a_j, the reduced costs, the duals
y = B^-T c_B and a verdict: OPTIMAL (y dual feasible), UNBOUNDED (an edge ray), or undecided at a degenerate
vertex, where enumgpu_find_ray enumerates the extreme rays of {d >= 0, A d = 0, ck.d < 0} as the feasible
bases of an auxiliary LP with m+1 rows (DESIGN.md §3).

The CPU twin of the certificate kernel is tests/certify_twin.c, compiled here with the CPU oracle's flags.
CPU: the twin's certificate against exact rationals and HiGHS, the rays checked in exact
arithmetic, the reference's simplex, self-checks that the LP families reach every path, the struct layout.
GPU: enumgpu_certify == the twin bit for bit, enumgpu_find_ray == the oracle's enumeration of the auxiliary
LP built here in Python (a second statement of the construction), the adapters.
"""
import ctypes as C
import json
import math
import os
import shutil
import subprocess
import tempfile
from fractions import Fraction

import numpy as np
import pytest

import simplexmethod_b200 as sm
from simplexmethod_b200 import Common, ConstraintType as CT, VariableType as VT, _abi, lpgen
from oracle import exact, simplex_ref
from test_problem_types import highs_general
from test_structured_parity import network, signed_duplicates, sparse_dyadic

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
ALGOS = [_abi.ALGO_INDEPENDENT, _abi.ALGO_SHARED]
NCPU = os.cpu_count()
SEEDS = range(200)
OPTIMAL, BOUNDED, UNBOUNDED, UNDECIDED = _abi.CERT_OPTIMAL, _abi.CERT_BOUNDED, _abi.CERT_UNBOUNDED, _abi.CERT_UNDECIDED
with open(os.path.join(HERE, "golden", "tiny_lps.json")) as f:
    GOLD = json.load(f)


# --------------------------------------------------------------------------------------------- CPU twin

_TWIN = None


def twin():
    """tests/certify_twin.c, built once per process into a temporary directory with the CPU oracle's flags."""
    global _TWIN
    if _TWIN is None:
        tmp = tempfile.mkdtemp(prefix="certify_twin_")
        so = os.path.join(tmp, "libcertify_twin.so")
        subprocess.check_call(["gcc", "-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra",
                               "-std=c11", "-shared", "-I", os.path.join(ROOT, "include"), "-o", so,
                               os.path.join(HERE, "certify_twin.c"), "-lm"])
        L = C.CDLL(so)
        shutil.rmtree(tmp)                          # the loaded library stays mapped
        L.certify_twin.restype = C.c_int
        L.certify_twin.argtypes = [C.POINTER(_abi.Problem), C.c_double, C.c_int, C.c_double, C.c_double,
                                   C.POINTER(C.c_int32), C.POINTER(_abi.Certificate)]
        _TWIN = L
    return _TWIN


def certify_basis(A, b, c, maximize, S, eps_feas=1e-9, eps_piv=1e-9, eps_opt=1e-9):
    """The CPU twin's certificate at basis S (absolute pivot rule), without the ray fallback: (rc, Certificate)."""
    A = np.asfortranarray(A, dtype=float)
    b = np.ascontiguousarray(b, dtype=float)
    c = np.ascontiguousarray(c, dtype=float)
    m, n = A.shape
    p = _abi.Problem(m, n, m, int(bool(maximize)), A.ctypes.data, b.ctypes.data, c.ctypes.data)
    tol = eps_piv * float(np.abs(A).max())
    cert = _abi.Certificate()
    rc = twin().certify_twin(C.byref(p), eps_feas, _abi.PIVOT_ABSOLUTE, tol, eps_opt, (C.c_int32 * m)(*S), C.byref(cert))
    return rc, cert


# --------------------------------------------------------------------------------------------- LPs

def general_lp(seed):
    """The random general-form LP of test_problem_types.test_random_general_lps_vs_highs."""
    rng = np.random.default_rng(seed)
    m, n = int(rng.integers(2, 5)), int(rng.integers(2, 5))
    A = rng.integers(-4, 5, size=(m, n)).astype(float)
    x0 = rng.integers(-3, 4, size=n).astype(float)
    vts = [VT(int(k)) for k in rng.integers(0, 3, size=n)]
    x0 = np.array([abs(v) if t is VT.NonNegative else -abs(v) if t is VT.NonPositive else v for v, t in zip(x0, vts)])
    cts = [CT(int(k)) for k in rng.integers(0, 3, size=m)]
    slack = rng.integers(0, 3, size=m).astype(float)
    b = A @ x0 + np.array([s if t is CT.LessOrEqual else -s if t is CT.GreaterOrEqual else 0.0 for s, t in zip(slack, cts)])
    c = rng.integers(-5, 6, size=n).astype(float)
    return Common(A, b, c, cts, vts, bool(rng.integers(0, 2)))


def canonical_arrays(seed):
    can = general_lp(seed).ToCanonical()
    return (np.asfortranarray(can.GetConstraintsMatrix()), can.GetRightHandSide().copy(),
            can.GetObjectiveCoefficients().copy(), can.IsMaximization())


def aux_lp(A, c, maximize):
    """[A; s*ck'] d = (0, ..., 0, -1), cost 0, minimise; s the largest power of two with s*max|ck| <= max|A|.
    Found here by search, not by the library's frexp formula."""
    ck = -np.asarray(c, dtype=float) if maximize else np.asarray(c, dtype=float)
    amax, cmax = float(np.abs(A).max()), float(np.abs(ck).max())
    e = 0
    while math.ldexp(cmax, e) > amax:
        e -= 1
    while math.ldexp(cmax, e + 1) <= amax:
        e += 1
    m, n = A.shape
    row = np.array([math.ldexp(v, e) for v in ck])
    assert all(math.ldexp(v, -e) == w for v, w in zip(row, ck))
    ba = np.zeros(m + 1)
    ba[m] = -1.0
    return np.asfortranarray(np.vstack([A, row])), ba, np.zeros(n), False


def degenerate_block_16():
    """m = 16, n = 32, b = 0: columns 0..15 are the identity (the winner: every feasible basis is the vertex 0, the
    lowest rank wins the tie), and column 16 + 2k, 17 + 2k are (1, -1) and (-1, 1) on rows 2k, 2k+1, with costs -1 and
    +2.  At the winner column 16 + 2k improves (r = -1) but has a positive u, so the certificate is undecided; the
    cone {d >= 0, A d = 0} is d_{16+2k} = d_{17+2k}, along which the cost rises: bounded."""
    m, n = 16, 32
    A = np.zeros((m, n), order="F")
    A[:, :m] = np.eye(m)
    c = np.zeros(n)
    for k in range(m // 2):
        A[2 * k, 16 + 2 * k], A[2 * k + 1, 16 + 2 * k] = 1.0, -1.0
        A[2 * k, 17 + 2 * k], A[2 * k + 1, 17 + 2 * k] = -1.0, 1.0
        c[16 + 2 * k], c[17 + 2 * k] = -1.0, 2.0
    return A, np.zeros(m), c, False


# --------------------------------------------------------------------------------------------- oracle pipeline

def oracle_pipeline(oracle, A, b, c, mx):
    """Enumerate, certify the winner, and run the auxiliary LP through enumcpu_solve if undecided.
    Returns (winner Result, Certificate, verdict, aux Result | None, dense ray | None)."""
    res, _ = oracle.solve(A, b, c, mx, n_threads=4)
    assert res.status == _abi.OK
    m, n = A.shape
    rc, cert = certify_basis(A, b, c, mx, list(res.basis)[:m])
    assert rc == _abi.OK and cert.basis_class == _abi.BASIS_FEASIBLE
    verdict, aux, ray = cert.status, None, None
    if verdict == UNBOUNDED:
        ray = np.array(cert.ray[:n])
    elif verdict == UNDECIDED and m < _abi.MAX_M:
        aux, _ = oracle.solve(*aux_lp(A, c, mx), n_threads=4)
        if aux.status == _abi.OK:
            verdict = UNBOUNDED
            ray = np.zeros(n)
            ray[list(aux.basis)[:m + 1]] = list(aux.x_B)[:m + 1]
        elif aux.n_feasible == 0:
            verdict = BOUNDED
    return res, cert, verdict, aux, ray


def check_ray(A, c, mx, d):
    """d >= -eps, ck.d < 0, |A d|_inf <= 1e-9 max|A| |d|_1, in exact arithmetic on the doubles."""
    m, n = A.shape
    D = [Fraction(float(v)) for v in d]
    assert min(D) >= -Fraction(1, 10**9)
    ck = [Fraction(float(-v if mx else v)) for v in c]
    assert sum(x * y for x, y in zip(ck, D)) < 0
    amax = max(abs(Fraction(float(v))) for v in A.ravel())
    norm1 = sum(abs(x) for x in D)
    for i in range(m):
        assert abs(sum(Fraction(float(A[i, j])) * D[j] for j in range(n))) <= Fraction(1, 10**9) * amax * norm1


_PIPE = {}


def seed_pipeline(oracle, seed):
    if seed not in _PIPE:
        A, b, c, mx = canonical_arrays(seed)
        _PIPE[seed] = (A, b, c, mx) + oracle_pipeline(oracle, A, b, c, mx)
    return _PIPE[seed]


def path_of(cert, verdict):
    """Which of the four paths a seed takes: (verdict at the winner, verdict in the end)."""
    return cert.status, verdict


# --------------------------------------------------------------------------------------------- CPU

def exact_certificate(A, b, c, mx, S, eps_opt=Fraction(1, 10**9)):
    m, n = len(A), len(A[0])
    Af = [[Fraction(A[i][j]) for j in range(n)] for i in range(m)]
    cols = [[Af[i][j] for i in range(m)] for j in S]
    cf = [Fraction(v) for v in c]
    u = [exact.solve_exact(cols, [Af[i][j] for i in range(m)]) for j in range(n)]
    cB = [cf[j] for j in S]
    r = [cf[j] - sum(x * y for x, y in zip(cB, u[j])) for j in range(n)]
    y = exact.solve_exact([[Af[i][j] for j in S] for i in range(m)], cB)       # B^T y = c_B
    verdict, improving = OPTIMAL, False
    for j in range(n):
        if j in S:
            continue
        rk = -r[j] if mx else r[j]
        if rk < -eps_opt:
            improving = True
            if all(v <= eps_opt for v in u[j]):
                return UNBOUNDED, y, r
    return (UNDECIDED if improving else verdict), y, r


@pytest.mark.parametrize("name", sorted(GOLD))
def test_oracle_certificate_vs_exact_on_goldens(oracle, name):
    g = GOLD[name]
    A = np.array(g["A"], dtype=float)
    m, n = A.shape
    S = g["best_basis"]
    rc, cert = certify_basis(A, g["b"], g["c"], g["maximize"], S)
    assert rc == _abi.OK and cert.basis_class == _abi.BASIS_FEASIBLE
    verdict, y, r = exact_certificate(g["A"], g["b"], g["c"], g["maximize"], S)
    assert cert.status == verdict
    scale = max(abs(Fraction(v)) for v in g["c"]) or 1
    for got, want in zip(list(cert.y)[:m] + list(cert.reduced_cost)[:n], y + r):
        assert abs(Fraction(got) - want) <= Fraction(1, 10**12) * max(abs(want), scale)
    for got, want in zip(list(cert.x_B)[:m], g["best_x"]):
        assert abs(Fraction(got) - Fraction(want)) <= Fraction(1, 10**12) * max(1, abs(Fraction(want)))


@pytest.mark.parametrize("seed", SEEDS)
def test_oracle_verdict_vs_highs(oracle, seed):
    A, b, c, mx, res, cert, verdict, aux, ray = seed_pipeline(oracle, seed)
    st, z, _ = highs_general(general_lp(seed))
    assert st in (0, 3)
    assert verdict in ((OPTIMAL, BOUNDED) if st == 0 else (UNBOUNDED,))
    if verdict == UNBOUNDED:
        check_ray(A, c, mx, ray)
    if verdict == OPTIMAL:
        m = A.shape[0]
        dual = math.fsum(float(Fraction(bi) * Fraction(yi)) for bi, yi in zip(b, list(cert.y)[:m]))
        assert dual == pytest.approx(res.objective, rel=1e-9, abs=1e-9)


@pytest.mark.parametrize("seed", SEEDS)
def test_reference_simplex_from_the_winner(oracle, seed):
    """The reference's simplex (oracle/simplex_ref.py), started at the enumeration's winner, stops with
    "objective is unbounded" exactly on the seeds the certificate calls UNBOUNDED."""
    A, b, c, mx, res, cert, verdict, aux, ray = seed_pipeline(oracle, seed)
    m = A.shape[0]
    try:
        simplex_ref.solve_with_basis(A, b, c, list(res.basis)[:m], mx)
        unbounded = False
    except RuntimeError as e:
        unbounded = str(e) == "objective is unbounded"
    assert unbounded == (verdict == UNBOUNDED)


def test_selfcheck_every_path_is_reached(oracle):
    paths = {}
    for seed in SEEDS:
        _, _, _, _, _, cert, verdict, _, _ = seed_pipeline(oracle, seed)
        paths.setdefault(path_of(cert, verdict), []).append(seed)
    assert set(paths) == {(OPTIMAL, OPTIMAL), (UNDECIDED, BOUNDED), (UNBOUNDED, UNBOUNDED), (UNDECIDED, UNBOUNDED)}
    assert len(paths[(UNDECIDED, BOUNDED)]) >= 10 and len(paths[(UNBOUNDED, UNBOUNDED)]) >= 10


def test_selfcheck_degenerate_m16_is_undecided(oracle):
    A, b, c, mx = degenerate_block_16()
    rc, cert = certify_basis(A, b, c, mx, list(range(16)))
    assert rc == _abi.OK and cert.status == UNDECIDED and cert.entering == -1
    # the same construction at m = 4 (all bases enumerable here): the identity is the winner, undecided, bounded
    A4, c4 = np.asfortranarray(np.c_[A[:4, :4], A[:4, 16:20]]), np.r_[c[:4], c[16:20]]
    res, cert4, verdict, aux, _ = oracle_pipeline(oracle, A4, np.zeros(4), c4, False)
    assert list(res.basis)[:4] == [0, 1, 2, 3] and cert4.status == UNDECIDED and verdict == BOUNDED


def test_certificate_struct_layout_matches_header(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "enumgpu.h"\n'
                   'int main(){printf("%zu %zu %zu %zu %zu %zu %zu\\n",sizeof(enumgpu_certificate),'
                   'offsetof(enumgpu_certificate,objective),offsetof(enumgpu_certificate,y),'
                   'offsetof(enumgpu_certificate,reduced_cost),offsetof(enumgpu_certificate,x_B),'
                   'offsetof(enumgpu_certificate,ray),offsetof(enumgpu_certificate,n_rays));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    T = _abi.Certificate
    assert got == [C.sizeof(T), T.objective.offset, T.y.offset, T.reduced_cost.offset, T.x_B.offset, T.ray.offset,
                   T.n_rays.offset]


def test_check_unbounded_needs_the_whole_range():
    A, b, c, mx = lpgen.dense_lp(3, 6, 1)
    s = sm.EnumerationSolver(sm.Canonical(A, b, c, [0, 1, 2]), check_unbounded=True)
    with pytest.raises(ValueError, match="whole rank range"):
        s.solve(rank_begin=0, rank_end=5)


# --------------------------------------------------------------------------------------------- GPU

def problem(A, b, c, mx):
    A = np.asfortranarray(A, dtype=float)
    b = np.ascontiguousarray(b, dtype=float)
    c = np.ascontiguousarray(c, dtype=float)
    return (A, b, c), _abi.Problem(A.shape[0], A.shape[1], A.shape[0], int(bool(mx)), A.ctypes.data, b.ctypes.data,
                                   c.ctypes.data)


def options(algo=_abi.ALGO_AUTO, rank_begin=0, rank_end=0, devices=None, eps_feas=-1.0):
    o = _abi.Options(eps_feas, -1.0, rank_begin, rank_end, 0, algo, None, None, 0, 0, 0, 0)
    if devices:
        o.n_devices, o.devices = len(devices), (C.c_int32 * len(devices))(*devices)
    return o


def gpu_certify(L, A, b, c, mx, S, eps_opt=-1.0, algo=_abi.ALGO_AUTO):
    keep, p = problem(A, b, c, mx)
    cert = _abi.Certificate()
    rc = L.enumgpu_certify(C.byref(p), C.byref(options(algo)), (C.c_int32 * len(S))(*S), eps_opt, C.byref(cert))
    return rc, cert


def gpu_find_ray(L, A, c, mx, algo=_abi.ALGO_AUTO, **kw):
    keep, p = problem(A, np.zeros(A.shape[0]), c, mx)
    res = _abi.Result()
    rc = L.enumgpu_find_ray(C.byref(p), C.byref(options(algo, **kw)), C.byref(res))
    return rc, res


def bits(v):
    return np.asarray(v, dtype=np.float64).view(np.uint64).tolist()


def assert_cert_bits(g, o):
    assert (g.status, g.basis_class, g.entering, g.m, g.n) == (o.status, o.basis_class, o.entering, o.m, o.n)
    m, n = o.m, o.n
    assert bits(g.objective) == bits(o.objective)
    assert bits(list(g.x_B)[:m]) == bits(list(o.x_B)[:m])
    assert bits(list(g.y)[:m]) == bits(list(o.y)[:m])
    assert bits(list(g.reduced_cost)[:n]) == bits(list(o.reduced_cost)[:n])
    if o.status == UNBOUNDED:
        assert bits(list(g.ray)[:n]) == bits(list(o.ray)[:n])


def assert_record_same(g, o, m):
    assert g.status == o.status and g.m == o.m == m
    assert (g.n_bases, g.n_singular, g.n_infeasible, g.n_feasible, g.best_rank) == \
           (o.n_bases, o.n_singular, o.n_infeasible, o.n_feasible, o.best_rank)
    if o.status == _abi.OK:
        assert list(g.basis)[:m] == list(o.basis)[:m]
        assert bits(list(g.x_B)[:m]) == bits(list(o.x_B)[:m])


def certify_vs_oracle(L, oracle, A, b, c, mx):
    """Enumerate with the oracle, then certify its winner on the GPU and in the oracle; returns the GPU's."""
    o, _ = oracle.solve(A, b, c, mx, n_threads=NCPU)
    m = A.shape[0]
    S = list(o.basis)[:m]
    rc_o, want = certify_basis(A, b, c, mx, S)
    rc, got = gpu_certify(L, A, b, c, mx, S)
    assert rc == rc_o == _abi.OK
    if want.status == UNDECIDED:           # the GPU then decides with the auxiliary enumeration
        assert got.status in (BOUNDED, UNBOUNDED, UNDECIDED)
        got.status, got.entering = want.status, want.entering
    assert_cert_bits(got, want)
    assert bits(list(got.x_B)[:m]) == bits(list(o.x_B)[:m])          # the enumeration record's x_B
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GOLD))
def test_certify_tiny_goldens(gpu_lib, oracle, name):
    g = GOLD[name]
    certify_vs_oracle(gpu_lib, oracle, np.array(g["A"], dtype=float), np.array(g["b"], dtype=float),
                      np.array(g["c"], dtype=float), g["maximize"])


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,seed", [(1, 1, 1), (1, 7, 2), (2, 2, 3), (3, 9, 4), (4, 4, 5), (4, 11, 6), (5, 12, 7),
                                      (6, 13, 8), (7, 15, 9), (9, 14, 10), (11, 15, 11), (13, 15, 12), (16, 17, 13),
                                      (8, 24, 1), (10, 30, 1)])
def test_certify_dense_shapes(gpu_lib, oracle, m, n, seed):
    A, b, c, _ = lpgen.dense_lp(m, n, seed)
    for mx in (False, True):
        got = certify_vs_oracle(gpu_lib, oracle, A, b, c, mx)
        if n == m:
            assert got.status in (OPTIMAL, BOUNDED) and got.n_launches == 1 and got.n_aux_bases == 0


@pytest.mark.gpu
def test_certify_degenerate_config5(gpu_lib, oracle):
    A, b, c, mx = lpgen.degenerate_lp()
    certify_vs_oracle(gpu_lib, oracle, A, b, c, mx)


@pytest.mark.gpu
def test_certify_headline_golden_basis(gpu_lib, oracle):
    g = json.load(open(os.path.join(HERE, "golden", "dense_12_40_seed1.json")))
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    rc, got = gpu_certify(gpu_lib, A, b, c, mx, g["basis"])
    rc_o, want = certify_basis(A, b, c, mx, g["basis"])
    assert rc == rc_o == _abi.OK
    assert_cert_bits(got, want)
    assert [float(v).hex() for v in list(got.x_B)[:12]] == g["x_B"]
    assert float(got.objective).hex() == g["objective"]
    assert got.status == OPTIMAL and got.n_launches == 1
    nonbasic = [j for j in range(40) if j not in g["basis"]]
    assert min((-1 if mx else 1) * got.reduced_cost[j] for j in nonbasic) > 1e-3
    assert float(np.dot(b, list(got.y)[:12])) == pytest.approx(got.objective, rel=1e-12)


@pytest.mark.gpu
def test_certify_errors_and_m16_undecided(gpu_lib, oracle):
    A, b, c, mx = degenerate_block_16()
    total = gpu_lib.enumgpu_binomial(32, 16)
    s = sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(16))))
    s.solve()
    assert s.optimalBasis() == list(range(16)) and s.basesEvaluated() == total
    cert = s.certify()
    assert cert.status == UNDECIDED and cert.n_launches == 1 and cert.n_aux_bases == 0
    assert s.unboundedRay() is None
    # a singular and an infeasible basis are argument errors; the class says which
    rc, cert = gpu_certify(gpu_lib, A, b, c, mx, [0] * 15 + [1])
    assert rc == _abi.ERR_ARG and cert.basis_class == _abi.BASIS_SINGULAR
    A2, b2, c2, mx2 = lpgen.dense_lp(4, 8, 3)
    _, st = oracle.solve(A2, b2, c2, mx2, want_status=True)
    r_inf = int(np.flatnonzero(st == 1)[0])
    S = (C.c_int32 * 4)()
    gpu_lib.enumgpu_unrank(8, 4, r_inf, S)
    rc, cert = gpu_certify(gpu_lib, A2, b2, c2, mx2, list(S))
    assert rc == _abi.ERR_ARG and cert.basis_class == _abi.BASIS_INFEASIBLE
    # the auxiliary LP of m = 16 would need 17 rows
    rc, _ = gpu_find_ray(gpu_lib, A, c, mx)
    assert rc == _abi.ERR_ARG


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_certify_and_find_ray_on_general_lps(gpu_lib, oracle, seed):
    A, b, c, mx, res, cert, verdict, aux, ray = seed_pipeline(oracle, seed)
    m, n = A.shape
    rc, got = gpu_certify(gpu_lib, A, b, c, mx, list(res.basis)[:m])
    assert rc == _abi.OK and got.status == verdict
    if cert.status == UNDECIDED:
        got.status, got.entering = cert.status, cert.entering
    assert_cert_bits(got, cert)
    if verdict == UNBOUNDED:
        assert bits(list(got.ray)[:n]) == bits(list(ray))
    # the ray enumeration itself, against the oracle's enumeration of the auxiliary LP built here
    o, _ = oracle.solve(*aux_lp(A, c, mx), n_threads=4)
    for algo in ALGOS if m + 1 >= 6 else ALGOS[:1]:
        rc, g = gpu_find_ray(gpu_lib, A, c, mx, algo)
        assert rc == o.status
        assert_record_same(g, o, m + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("family", [sparse_dyadic, signed_duplicates, network], ids=lambda f: f.__name__)
@pytest.mark.parametrize("m,n", [(6, 18), (7, 21), (9, 22)])
def test_find_ray_structured(gpu_lib, oracle, family, m, n):
    """Dependent column pairs, exact ties and -0.0 components, in the auxiliary LP too."""
    A, b, c, _ = family(m, n, 1)
    for mx in (False, True):
        o, _ = oracle.solve(*aux_lp(A, c, mx), n_threads=NCPU)
        for algo in ALGOS:
            rc, g = gpu_find_ray(gpu_lib, A, c, mx, algo)
            assert rc == o.status
            assert_record_same(g, o, m + 1)


@pytest.mark.gpu
def test_find_ray_headline(gpu_lib, oracle):
    """dense (12, 40): lpgen builds c = A'y0 + s with s >= 0.1, so no ray exists among the C(40,13) aux bases."""
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    total = gpu_lib.enumgpu_binomial(40, 13)
    assert total == 12033222880
    rc, full = gpu_find_ray(gpu_lib, A, c, mx)
    assert rc == _abi.NO_FEASIBLE and full.n_feasible == 0 and full.n_bases == total
    assert full.n_singular + full.n_infeasible == total and full.algo_used == _abi.ALGO_SHARED
    Aa, ba, ca, _ = aux_lp(A, c, mx)
    S = [0, 2, 3, 5, 6, 7, 8, 9, 15, 21, 22, 23, 30]       # a window starting inside a child task
    inside_child = gpu_lib.enumgpu_rank(40, 13, (C.c_int32 * 13)(*S)) + 17
    for lo, hi in [(0, 1000000), (inside_child, inside_child + 300000)]:
        o, _ = oracle.solve(Aa, ba, ca, False, n_threads=NCPU, rank_begin=lo, rank_end=hi)
        for algo in ALGOS:
            rc, g = gpu_find_ray(gpu_lib, A, c, mx, algo, rank_begin=lo, rank_end=hi)
            assert_record_same(g, o, 13)
    if gpu_lib.enumgpu_device_count() >= 2:
        rc, two = gpu_find_ray(gpu_lib, A, c, mx, devices=[0, 1])
        assert_record_same(two, full, 13)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", SEEDS)
def test_solver_check_unbounded(gpu_lib, oracle, seed):
    A, b, c, mx, res, cert, verdict, aux, ray = seed_pipeline(oracle, seed)
    can = sm.Canonical(A, b, c, list(range(A.shape[0])), minimize=not mx)
    plain = sm.EnumerationSolver(can)
    x = plain.solve()                                   # the default is unchanged: a vertex, no exception
    assert plain.launches() == 1
    checked = sm.EnumerationSolver(can, check_unbounded=True)
    if verdict == UNBOUNDED:
        with pytest.raises(RuntimeError, match="objective is unbounded"):
            checked.solve()
        d = checked.unboundedRay()
        check_ray(A, c, mx, d)
    else:
        assert checked.solve().tolist() == x.tolist()
        assert checked.unboundedRay() is None
        if verdict == OPTIMAL:
            assert bits(checked.dualValues()) == bits(list(cert.y)[:A.shape[0]])
            assert bits(checked.reducedCosts()) == bits(list(cert.reduced_cost)[:A.shape[1]])
    assert (checked.findRay().status == _abi.OK) == (verdict == UNBOUNDED)        # the LP is feasible: ray <=> unbounded


@pytest.fixture(scope="module")
def certify_demo():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "simplexmethod_b200", "cpp"), "-s"])
    return os.path.join(ROOT, "simplexmethod_b200", "cpp", "build", "certify_demo")


def symmetric_file(path, seed):
    sym = general_lp(seed).ToSymmetrical()
    A, b, c = sym.GetConstraintsMatrix(), sym.GetRightHandSide(), sym.GetObjectiveCoefficients()
    lines = ["maximize" if sym.IsMaximization() else "minimize", "objective:", " ".join(repr(float(v)) for v in c),
             "constraints:"] + [" ".join(repr(float(v)) for v in list(A[i]) + [b[i]]) for i in range(A.shape[0])]
    path.write_text("\n".join(lines) + "\n")


@pytest.mark.gpu
def test_cpp_adapter_through_certify_demo(gpu_lib, oracle, certify_demo, tmp_path):
    """setCheckUnbounded / certify() of the C++ adapter on seeds of every path."""
    chosen = {}
    for seed in SEEDS:
        _, _, _, _, _, cert, verdict, _, _ = seed_pipeline(oracle, seed)
        chosen.setdefault(path_of(cert, verdict), [])
        if len(chosen[path_of(cert, verdict)]) < 3:
            chosen[path_of(cert, verdict)].append(seed)
    for seeds in chosen.values():
        for seed in seeds:
            A, b, c, mx, res, cert, verdict, aux, ray = seed_pipeline(oracle, seed)
            f = tmp_path / f"lp{seed}.txt"
            symmetric_file(f, seed)
            out = subprocess.run([certify_demo, str(f)], capture_output=True, text=True)
            assert out.returncode == 0, out.stderr
            facts = {l.split()[0]: l.split()[1:] for l in out.stdout.splitlines()}
            assert [int(v) for v in facts["basis"]] == list(res.basis)[:A.shape[0]]
            assert int(facts["cert_status"][0]) == verdict
            assert [float(v) for v in facts["y"]] == list(cert.y)[:A.shape[0]]
            assert [float(v) for v in facts["reduced_cost"]] == list(cert.reduced_cost)[:A.shape[1]]
            if verdict == UNBOUNDED:
                assert [float(v) for v in facts["ray"]] == list(ray)
            assert facts["check_unbounded"] == [str(int(verdict == UNBOUNDED))]
