"""Many objectives over one feasible set: enumgpu_solve_objectives against K separate enumgpu_solve calls and the oracle.

out[i] must be, bit for bit, the record enumgpu_solve gives for the problem with c = column i under the same options:
every field but kernel_ms and n_launches (which describe the whole call).  The GPU tests compare the raw bytes of the
two structs with those two fields cleared, and x_B, objective and key against the CPU oracle as bit patterns.

Without a GPU: the new prototype against the header, every argument error and its code (before any CUDA call), the
failure without a device, and self-checks that the cost sets reach what they are there for (equal keys everywhere,
+-c, unit vectors, z overflowing to +-inf and NaN, ties broken by rank).
"""
import ctypes as C
import json
import math
import os
import subprocess

import numpy as np
import pytest

import simplexmethod_b200 as sm
from simplexmethod_b200 import _abi, lpgen
from test_structured_parity import FAMILIES, all_nan_keys, assert_same, bits, headline_windows, network, unrank

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NCPU = os.cpu_count()
ALGOS = [_abi.ALGO_INDEPENDENT, _abi.ALGO_SHARED]
FEASIBLE = 0

with open(os.path.join(HERE, "golden", "tiny_lps.json")) as f:
    GOLD = json.load(f)


# --------------------------------------------------------------------------------------------- cost sets

def cost_set(A, c, n_random=6, seed=0):
    """(k, n) cost vectors: 0 (every key equal: the lowest-rank feasible basis wins), +c and -c, four unit vectors,
    three small-integer vectors (ties on data with integer vertices), n_random normal vectors, and one vector of
    +-2^1021 (z overflows to +-inf, or to NaN where terms of both signs overflow)."""
    n = A.shape[1]
    rng = np.random.default_rng(seed)
    cols = [np.zeros(n), np.asarray(c, dtype=np.float64), -np.asarray(c, dtype=np.float64)]
    cols += [np.eye(n)[j] for j in sorted(rng.choice(n, min(n, 4), replace=False))]
    cols += [rng.integers(-3, 4, n).astype(np.float64) for _ in range(3)]
    cols += [rng.standard_normal(n) for _ in range(n_random)]
    cols.append(rng.choice(np.array([-1.0, 1.0]), n) * 2.0 ** 1021)
    return np.ascontiguousarray(np.array(cols))


def options(algo=_abi.ALGO_AUTO, rank_begin=0, rank_end=0, eps_feas=-1.0, eps_piv=-1.0, pivot_rule=_abi.PIVOT_ABSOLUTE,
            shard_index=0, shard_count=0):
    return _abi.Options(eps_feas, eps_piv, rank_begin, rank_end, 0, algo, None, None, shard_index, shard_count,
                        pivot_rule, 0)


def problem(A, b, c, mx):
    A = np.asfortranarray(A, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    c = np.ascontiguousarray(c, dtype=np.float64)
    keep = (A, b, c)
    return _abi.Problem(A.shape[0], A.shape[1], A.shape[0], int(bool(mx)), A.ctypes.data, b.ctypes.data,
                        c.ctypes.data), keep


def call_objectives(L, A, b, costs, mx, max_list=0, ldc=None, k=None, **opt):
    """enumgpu_solve_objectives on the rows of costs; returns (rc, [Result] * k)."""
    costs = np.ascontiguousarray(costs, dtype=np.float64)
    ps, keep = problem(A, b, costs[0], mx)
    ps.c = None                                         # not read
    out = (_abi.Result * costs.shape[0])()              # an invalid k is refused before out is touched
    o = options(**opt)
    rc = L.enumgpu_solve_objectives(C.byref(ps), C.byref(o), costs.shape[0] if k is None else k,
                                    costs.ctypes.data_as(C.POINTER(C.c_double)), costs.shape[1] if ldc is None else ldc,
                                    max_list, out)
    return rc, [_abi.Result.from_buffer_copy(bytes(out[i])) for i in range(costs.shape[0])]


def gpu_solve(L, A, b, c, mx, **opt):
    ps, keep = problem(A, b, c, mx)
    res = _abi.Result()
    L.enumgpu_solve(C.byref(ps), C.byref(options(**opt)), C.byref(res))
    return res


def record_bytes(r):
    r = _abi.Result.from_buffer_copy(bytes(r))
    r.kernel_ms, r.n_launches = 0.0, 0
    return bytes(r)


def check_against_solves(L, A, b, costs, mx, results, **opt):
    """Every entry == enumgpu_solve with that column, byte for byte but kernel_ms / n_launches."""
    assert len(results) == costs.shape[0]
    for i, g in enumerate(results):
        want = gpu_solve(L, A, b, costs[i], mx, **opt)
        assert want.status in (_abi.OK, _abi.NO_FEASIBLE)
        assert record_bytes(g) == record_bytes(want), (i, g.status, want.status, g.best_rank, want.best_rank)
        assert g.kernel_ms == results[0].kernel_ms and g.n_launches == results[0].n_launches


def check_against_oracle(oracle, A, b, costs, mx, results, rank_begin=0, rank_end=0, **opt):
    m = A.shape[0]
    for i, g in enumerate(results):
        o, _ = oracle.solve(A, b, costs[i], mx, n_threads=NCPU, rank_begin=rank_begin, rank_end=rank_end, **opt)
        assert_same(g, o, m)


def run_and_check(L, oracle, A, b, costs, mx, with_oracle=True, **opt):
    rc, res = call_objectives(L, A, b, costs, mx, **opt)
    assert rc == _abi.OK, sm.last_error()
    check_against_solves(L, A, b, costs, mx, res, **opt)
    if with_oracle:
        o_opt = {k: v for k, v in opt.items() if k != "algo"}
        check_against_oracle(oracle, A, b, costs, mx, res, **o_opt)
    return res


# ------------------------------------------------------------------------------ without a GPU

def test_prototype_matches_header(tmp_path):
    """The declaration in enumgpu.h has the ctypes prototype's parameter types, and the structs it uses are unchanged."""
    src = tmp_path / "proto.c"
    src.write_text('#include <stdio.h>\n#include "enumgpu.h"\n'
                   'int (*f)(const enumgpu_problem*, const enumgpu_options*, int32_t, const double*, int32_t, uint64_t,'
                   ' enumgpu_result*) = enumgpu_solve_objectives;\n'
                   'int main(){printf("%zu %zu %zu\\n",sizeof(enumgpu_problem),sizeof(enumgpu_options),'
                   'sizeof(enumgpu_result));return 0;}\n')
    exe = tmp_path / "proto"
    subprocess.check_call(["gcc", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", os.path.join(ROOT, "simplexmethod_b200"), "-lenumgpu"])
    env = dict(os.environ, LD_LIBRARY_PATH=os.path.join(ROOT, "simplexmethod_b200"))
    got = [int(v) for v in subprocess.check_output([str(exe)], env=env).split()]
    assert got == [C.sizeof(_abi.Problem), C.sizeof(_abi.Options), C.sizeof(_abi.Result)]
    restype, argtypes = _abi.SYMBOLS["enumgpu_solve_objectives"]
    assert restype is C.c_int
    assert argtypes == [C.POINTER(_abi.Problem), C.POINTER(_abi.Options), C.c_int32, C.POINTER(C.c_double), C.c_int32,
                        C.c_uint64, C.POINTER(_abi.Result)]


def test_argument_errors_come_before_cuda():
    """Each bad argument gives its code, on every entry of out, whether or not a GPU is present."""
    L = sm.lib()
    A, b, c, mx = lpgen.dense_lp(3, 6, 1)
    costs = cost_set(A, c)[:5]
    cases = [
        (dict(k=0), _abi.ERR_ARG),
        (dict(k=_abi.MAX_OBJECTIVES + 1), _abi.ERR_ARG),
        (dict(ldc=5), _abi.ERR_ARG),
        (dict(shard_index=0, shard_count=2), _abi.ERR_ARG),
        (dict(shard_index=1, shard_count=2), _abi.ERR_ARG),
        (dict(rank_begin=10, rank_end=2), _abi.ERR_RANGE),
        (dict(algo=7), _abi.ERR_ARG),
    ]
    for kw, code in cases:
        rc, res = call_objectives(L, A, b, costs, mx, **kw)
        assert rc == code, (kw, rc)
        if kw.get("k", 1) >= 1 and kw.get("k", 1) <= _abi.MAX_OBJECTIVES:
            assert all(r.status == code for r in res), kw
    bad = costs.copy(); bad[3, 2] = np.nan
    rc, res = call_objectives(L, A, b, bad, mx)
    assert rc == _abi.ERR_NONFINITE and all(r.status == rc for r in res)
    assert "C(2,3)" in sm.last_error()
    bad[3, 2] = -np.inf
    assert call_objectives(L, A, b, bad, mx)[0] == _abi.ERR_NONFINITE
    badA = A.copy(); badA[1, 1] = np.inf
    assert call_objectives(L, badA, b, costs, mx)[0] == _abi.ERR_NONFINITE
    # NULL pointers
    ps, keep = problem(A, b, c, mx)
    out = (_abi.Result * 2)()
    assert L.enumgpu_solve_objectives(C.byref(ps), None, 2, None, 6, 0, out) == _abi.ERR_ARG
    assert out[0].status == out[1].status == _abi.ERR_ARG
    cc = np.ascontiguousarray(costs[:2])
    assert L.enumgpu_solve_objectives(None, None, 2, cc.ctypes.data_as(C.POINTER(C.c_double)), 6, 0, out) == _abi.ERR_ARG
    assert L.enumgpu_solve_objectives(C.byref(ps), None, 2, cc.ctypes.data_as(C.POINTER(C.c_double)), 6, 0, None) \
        == _abi.ERR_ARG
    # the Python adapter turns them into ValueError
    s = sm.EnumerationSolver(sm.Canonical(A, b, c, [0, 1, 2]))
    for bad_costs in (np.zeros((0, 6)), np.zeros((2, 5)), np.zeros(6), bad):
        with pytest.raises(ValueError):
            s.solveObjectives(bad_costs)
    with pytest.raises(ValueError):
        s.solveObjectives(costs, rank_begin=10, rank_end=2)


@pytest.mark.skipif(sm.lib().enumgpu_device_count() > 0, reason="a GPU is present")
def test_no_gpu_means_loud_failure_not_fallback():
    L = sm.lib()
    A, b, c, mx = lpgen.lab_symmetric_canonical()
    costs = cost_set(A, c)
    rc, res = call_objectives(L, A, b, costs, mx)
    assert rc == _abi.ERR_CUDA and all(r.status == _abi.ERR_CUDA for r in res)
    assert "no CPU fallback" in sm.last_error()
    can = sm.Canonical(A, b, c, [3, 4], minimize=False)
    with pytest.raises(sm.EnumGpuError, match="no CPU fallback"):
        sm.EnumerationSolver(can).solveObjectives(costs)


def test_selfcheck_equal_keys_pick_the_lowest_feasible_rank(oracle):
    """c = 0: every feasible key is +0.0 (or -0.0 when maximising), so the winner is the lowest feasible rank."""
    for A, b, c, mx in (lpgen.small_degenerate_lp(), lpgen.dense_lp(8, 24, 1), network(8, 20, 3)):
        _, ranks, count = oracle.list_class(A, b, c, mx, FEASIBLE, n_threads=NCPU)
        assert count > 1
        for sense in (False, True):
            o, _ = oracle.solve(A, b, cost_set(A, c)[0], sense, n_threads=NCPU)
            assert o.status == _abi.OK and o.best_rank == ranks[0] and o.objective == 0.0
            assert math.copysign(1.0, o.key) == (-1.0 if sense else 1.0)


def test_selfcheck_cost_set_contents():
    A, b, c, mx = lpgen.dense_lp(6, 18, 2)
    costs = cost_set(A, c)
    assert (costs[1] == c).all() and (costs[2] == -c).all()
    units = [i for i in range(costs.shape[0]) if (costs[i] != 0).sum() == 1 and costs[i].max() == 1.0]
    assert len(units) == 4
    assert np.isfinite(costs).all() and np.abs(costs[-1]).min() == 2.0 ** 1021


def test_selfcheck_overflow_reaches_inf_and_nan(oracle):
    """The +-2^1021 column overflows z: on the huge_rhs family (x_B infinite) and on plain data both infinite and
    NaN objectives of feasible bases occur, and the optimum's key is -inf for one sense or the other."""
    seen = {"z_inf": 0, "z_nan": 0}
    for A, b, c, mx in (FAMILIES["huge_rhs"](8, 24, 1), lpgen.dense_lp(8, 24, 1)):
        big = cost_set(A, c)[-1]
        _, ranks, _ = oracle.list_class(A, b, big, mx, FEASIBLE, n_threads=NCPU)
        for r in ranks[:: max(1, len(ranks) // 400)]:
            st, x, z = oracle.eval_basis(A, b, big, mx, unrank(24, 8, r))
            assert st == FEASIBLE
            seen["z_inf"] += math.isinf(z)
            seen["z_nan"] += math.isnan(z)
    assert seen["z_inf"] >= 5 and seen["z_nan"] >= 1, seen
    A, b, c, mx = FAMILIES["huge_rhs"](8, 24, 1)
    keys = [oracle.solve(A, b, cost_set(A, c)[-1], s, n_threads=NCPU)[0].key for s in (False, True)]
    assert -math.inf in keys


def test_selfcheck_ties_occur(oracle):
    """Small-integer costs on a network LP (integer vertices): several feasible bases share the optimal key."""
    A, b, c, mx = network(8, 20, 3)
    costs = cost_set(A, c)
    _, ranks, _ = oracle.list_class(A, b, c, mx, FEASIBLE, n_threads=NCPU)
    tied = 0
    for i in range(7, 10):
        zs = [oracle.eval_basis(A, b, costs[i], mx, unrank(20, 8, r))[2] for r in ranks]
        tied += sum(z == min(zs) for z in zs) > 1
    assert tied >= 2


# ------------------------------------------------------------------------------ on the GPU

@pytest.mark.gpu
@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("name", sorted(GOLD))
def test_tiny_goldens(gpu_lib, oracle, name, algo):
    g = GOLD[name]
    A = np.array(g["A"], dtype=np.float64)
    costs = cost_set(A, g["c"])
    res = run_and_check(gpu_lib, oracle, A, g["b"], costs, g["maximize"], algo=algo)
    assert res[1].best_rank == g["best_rank"]           # column 1 is the golden's own c


@pytest.mark.gpu
@pytest.mark.parametrize("m", range(1, 17))
def test_dense_shapes(gpu_lib, oracle, m):
    """Every m (register kernels for m <= 12, run-time m above), minimised and maximised."""
    A, b, c, _ = lpgen.dense_lp(m, m + 8, m)
    costs = cost_set(A, c, seed=m)
    for mx in (False, True):
        run_and_check(gpu_lib, oracle, A, b, costs, mx)


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("name", ["small", "config5"])
def test_degenerate_ties(gpu_lib, oracle, name, algo):
    """config 5 (C(30, 10) bases) against separate GPU solves only: its oracle parity is test_gpu_parity's."""
    A, b, c, mx = {"small": lpgen.small_degenerate_lp, "config5": lpgen.degenerate_lp}[name]()
    costs = cost_set(A, c)
    for sense in (mx, not mx):
        run_and_check(gpu_lib, oracle, A, b, costs, sense, with_oracle=name == "small", algo=algo)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(8, 20), (10, 22)])
@pytest.mark.parametrize("name", sorted(FAMILIES))
def test_structured_families(gpu_lib, oracle, name, m, n):
    """Dyadic ties, -0.0 components of network LPs, +-inf and NaN keys; both kernel families, both senses."""
    A, b, c, _ = FAMILIES[name](m, n, 1)
    costs = cost_set(A, c)
    for mx in (False, True):
        for algo in ALGOS:
            run_and_check(gpu_lib, oracle, A, b, costs, mx, with_oracle=algo == ALGOS[0], algo=algo)


@pytest.mark.gpu
def test_network_negative_zero_and_eps_feas_zero(gpu_lib, oracle):
    A, b, c, mx = network(8, 20, 3, b_vals=(0, 1, 2))
    costs = cost_set(A, c)
    for algo in ALGOS:
        run_and_check(gpu_lib, oracle, A, b, costs, mx, algo=algo, eps_feas=0.0)
        run_and_check(gpu_lib, oracle, A, b, costs, mx, algo=algo, eps_feas=-0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(6, 15), (8, 24), (12, 26)])
def test_all_nan_keys(gpu_lib, oracle, m, n):
    """Every feasible basis has a NaN objective under the LP's own c (column 1): NO_FEASIBLE with n_feasible > 0 there,
    while other columns have optima."""
    A, b, c, mx = all_nan_keys(m, n)
    costs = cost_set(A, c)
    res = run_and_check(gpu_lib, oracle, A, b, costs, mx)
    assert res[1].status == _abi.NO_FEASIBLE and res[1].n_feasible > 0
    assert any(r.status == _abi.OK for r in res)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["small", "dense_8_24", "sparse_dyadic"])
def test_relative_pivot_rule(gpu_lib, oracle, case):
    A, b, c, mx = {"small": lpgen.small_degenerate_lp, "dense_8_24": lambda: lpgen.dense_lp(8, 24, 3),
                   "sparse_dyadic": lambda: FAMILIES["sparse_dyadic"](8, 24, 1)}[case]()
    costs = cost_set(A, c)
    res = run_and_check(gpu_lib, oracle, A, b, costs, mx, pivot_rule=_abi.PIVOT_RELATIVE)
    assert all(r.algo_used == _abi.ALGO_INDEPENDENT for r in res)
    run_and_check(gpu_lib, oracle, A, b, costs, mx, pivot_rule=_abi.PIVOT_RELATIVE, eps_piv=1e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ALGOS)
def test_rank_subranges(gpu_lib, oracle, algo):
    for A, b, c, mx in (lpgen.small_degenerate_lp(), lpgen.dense_lp(10, 24, 1)):
        total = gpu_lib.enumgpu_binomial(A.shape[1], A.shape[0])
        costs = cost_set(A, c)
        for lo, hi in ((0, total // 3), (total // 3, total // 3 + 4097), (total - 1000, total), (5, 5)):
            run_and_check(gpu_lib, oracle, A, b, costs, mx, algo=algo, rank_begin=lo, rank_end=hi)


@pytest.mark.gpu
@pytest.mark.parametrize("algo", ALGOS)
def test_max_list_splits_the_range(gpu_lib, oracle, algo):
    """A list too small for the feasible bases: many sub-ranges, some halved again; the same records as one pass."""
    for A, b, c, mx in (lpgen.small_degenerate_lp(), FAMILIES["signed_duplicates"](8, 24, 1), all_nan_keys(8, 24)):
        costs = cost_set(A, c)
        rc, whole = call_objectives(gpu_lib, A, b, costs, mx, algo=algo)
        nf = int(whole[0].n_feasible)
        assert rc == _abi.OK and nf > 40
        check_against_solves(gpu_lib, A, b, costs, mx, whole, algo=algo)
        for max_list in (nf // 40, nf // 3, nf - 1):
            rc, split = call_objectives(gpu_lib, A, b, costs, mx, algo=algo, max_list=max_list)
            assert rc == _abi.OK
            assert [record_bytes(r) for r in split] == [record_bytes(r) for r in whole]
            assert split[0].n_launches > whole[0].n_launches
        rc, split = call_objectives(gpu_lib, A, b, costs, mx, algo=algo, max_list=5, rank_begin=100, rank_end=20000)
        check_against_solves(gpu_lib, A, b, costs, mx, split, algo=algo, rank_begin=100, rank_end=20000)


@pytest.mark.gpu
def test_many_objectives_small_lp(gpu_lib, oracle):
    """K = 3000 (several objective tiles, one slice) and K = 33 (a partial tile) against separate solves."""
    A, b, c, mx = lpgen.dense_lp(6, 18, 4)
    rng = np.random.default_rng(5)
    for k in (33, 3000):
        costs = rng.standard_normal((k, 18))
        costs[::7] = np.round(costs[::7])
        rc, res = call_objectives(gpu_lib, A, b, costs, mx)
        assert rc == _abi.OK
        pick = list(range(0, k, max(1, k // 60))) + [k - 1]
        for i in pick:
            assert record_bytes(res[i]) == record_bytes(gpu_solve(gpu_lib, A, b, costs[i], mx))


HEADLINE = os.path.join(HERE, "golden", "dense_12_40_seed1.json")


@pytest.mark.gpu
def test_headline_12_40(gpu_lib, oracle):
    """All C(40, 12) bases, K = 64: column 0 = the LP's own c reproduces the golden record, the others equal separate
    GPU solves; four windows of the rank range against the live oracle."""
    with open(HEADLINE) as f:
        g = json.load(f)
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    rng = np.random.default_rng(12)
    costs = np.vstack([c, -c, np.zeros(40), rng.standard_normal((61, 40))])
    rc, res = call_objectives(gpu_lib, A, b, costs, mx)
    assert rc == _abi.OK, sm.last_error()
    r0 = res[0]
    assert (r0.status, r0.n_bases, r0.n_singular, r0.n_infeasible, r0.n_feasible, r0.best_rank) == \
        (g["status"], g["n_bases"], g["n_singular"], g["n_infeasible"], g["n_feasible"], g["best_rank"])
    assert list(r0.basis)[:12] == g["basis"]
    assert [float(v).hex() for v in list(r0.x_B)[:12]] == g["x_B"]
    assert float(r0.objective).hex() == g["objective"]
    assert r0.algo_used == _abi.ALGO_SHARED
    check_against_solves(gpu_lib, A, b, costs, mx, res)
    small = costs[:6]
    for lo, hi in headline_windows()[:2] + [(0, 400000)]:
        rc, part = call_objectives(gpu_lib, A, b, small, mx, rank_begin=lo, rank_end=hi)
        assert rc == _abi.OK
        check_against_oracle(oracle, A, b, small, mx, part, rank_begin=lo, rank_end=hi)


@pytest.mark.gpu
def test_python_adapter_rows_equal_solve(gpu_lib, oracle):
    A, b, c, mx = lpgen.lab_symmetric_canonical()
    can = sm.Canonical(A, b, c, [3, 4], minimize=not mx)
    can.SetOriginalVariablesCount(3)
    costs = cost_set(A, c)[1:-1]
    s = sm.EnumerationSolver(can)
    X = s.solveObjectives(costs)
    assert X.shape == (costs.shape[0], 3)
    raw = s.enumerateObjectives(costs)
    for i in range(costs.shape[0]):
        can_i = sm.Canonical(A, b, costs[i], [3, 4], minimize=not mx)
        can_i.SetOriginalVariablesCount(3)
        one = sm.EnumerationSolver(can_i)
        x = one.solve()
        assert [bits(v) for v in X[i]] == [bits(v) for v in x]
        assert record_bytes(raw[i]) == record_bytes(one.enumerate())
    # rank ranges pass through; no feasible basis raises as solve() does
    total = gpu_lib.enumgpu_binomial(5, 2)
    assert s.solveObjectives(costs, 0, total).tolist() == X.tolist()
    A, b, c, mx = all_nan_keys(8, 24)
    s = sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(8))))
    with pytest.raises(RuntimeError, match="no feasible basic solution"):
        s.solveObjectives(cost_set(A, c))


@pytest.fixture(scope="module")
def objectives_demo():
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "simplexmethod_b200", "cpp"), "-s"])
    return os.path.join(ROOT, "simplexmethod_b200", "cpp", "build", "objectives_demo")


@pytest.mark.gpu
@pytest.mark.parametrize("sense", ["maximize", "minimize"])
def test_cpp_demo_equals_python_adapter(gpu_lib, objectives_demo, tmp_path, sense):
    """objectives_demo (Symmetrical file -> ToCanonical -> solveObjectives) against the Python adapter on the same
    canonical LP."""
    sym_A = np.array([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0], [2.0, 1.0, 1.0]])
    sym_b = np.array([10.0, 20.0, 8.0])
    sym_c = np.array([7.0, 8.0, 3.0])
    f = tmp_path / "lp.txt"
    f.write_text("\n".join([sense, "objective:", " ".join(repr(float(v)) for v in sym_c), "constraints:"] +
                           [" ".join(repr(float(v)) for v in list(sym_A[i]) + [sym_b[i]]) for i in range(3)]) + "\n")
    rng = np.random.default_rng(3)
    rows = np.vstack([sym_c, -sym_c, np.eye(3), np.round(rng.standard_normal((5, 3)), 3), np.zeros(3)])
    if sense == "minimize":
        rows = np.abs(rows)                          # bounded below: nonnegative costs over x >= 0
    cf = tmp_path / "costs.txt"
    cf.write_text("\n".join(" ".join(repr(float(v)) for v in r) for r in rows) + "\n")
    out = subprocess.run([objectives_demo, str(f), str(cf)], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    facts = {}
    for line in out.stdout.splitlines():
        key, i, *vals = line.split()
        facts[(key, int(i))] = vals
    sym = sm.Symmetrical(sym_A, sym_b, sym_c, sense == "maximize")
    can = sym.ToCanonical()
    n = can.GetConstraintsMatrix().shape[1]
    costs = np.zeros((rows.shape[0], n))
    costs[:, :3] = rows
    s = sm.EnumerationSolver(can)
    X = s.solveObjectives(costs)
    raw = s.enumerateObjectives(costs)
    for i in range(rows.shape[0]):
        assert int(facts[("status", i)][0]) == raw[i].status == _abi.OK
        assert [int(v) for v in facts[("basis", i)]] == list(raw[i].basis)[:raw[i].m]
        assert float(facts[("objective", i)][0]) == raw[i].objective
        assert [float(v) for v in facts[("x", i)]] == X[i].tolist()
