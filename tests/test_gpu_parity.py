"""GPU: libenumgpu (through the C ABI) against the CPU oracle, bit for bit."""
import ctypes as C
import json
import os
from fractions import Fraction

import numpy as np
import pytest

import simplexmethod_b200 as sm
from simplexmethod_b200 import _abi, lpgen

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ALGOS = [_abi.ALGO_INDEPENDENT, _abi.ALGO_SHARED]


def gpu_solve(A, b, c, mx, algo=_abi.ALGO_AUTO, devices=None, **rng):
    can = sm.Canonical(A, b, c, list(range(A.shape[0])), minimize=not mx)
    s = sm.EnumerationSolver(can, devices=devices, algo=algo)
    return s.enumerate(**rng)


def assert_same(g, o, m, bitexact=True):
    assert g.status == o.status
    assert (g.n_bases, g.n_singular, g.n_infeasible, g.n_feasible) == \
           (o.n_bases, o.n_singular, o.n_infeasible, o.n_feasible)
    assert g.best_rank == o.best_rank
    if o.status == 0:
        assert list(g.basis)[:m] == list(o.basis)[:m]
        if bitexact:
            assert g.objective == o.objective and g.key == o.key          # same bits (== also accepts +-0)
            assert list(g.x_B)[:m] == list(o.x_B)[:m]
        else:
            assert g.objective == pytest.approx(o.objective, rel=1e-9)


with open(os.path.join(HERE, "golden", "tiny_lps.json")) as f:
    GOLD = json.load(f)


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("name", sorted(GOLD))
def test_tiny_goldens(gpu_lib, oracle, name, algo):
    g = GOLD[name]
    A = np.array(g["A"]); m, n = A.shape
    res = gpu_solve(A, g["b"], g["c"], g["maximize"], algo)
    assert (res.n_singular, res.n_infeasible, res.n_feasible) == (g["n_singular"], g["n_infeasible"], g["n_feasible"])
    assert res.best_rank == g["best_rank"] and list(res.basis)[:m] == g["best_basis"]
    assert res.objective == pytest.approx(float(Fraction(g["best_z"])), rel=1e-12, abs=1e-12)
    o, _ = oracle.solve(A, g["b"], g["c"], g["maximize"])
    assert_same(res, o, m)


def test_reference_call_shape_config1(gpu_lib):
    """input_symmetric.txt -> ToCanonical -> EnumerationSolver(problem).solve() == (5,0,0), z = 35."""
    A, b, c, mx = lpgen.lab_symmetric_canonical()
    can = sm.Canonical(A, b, c, [3, 4], minimize=False)
    can.SetOriginalVariablesCount(3)
    s = sm.EnumerationSolver(can)
    x = s.solve()
    assert x.tolist() == [5.0, 0.0, 0.0] and s.objective() == 35.0 and s.optimalBasis() == [0, 3]
    assert (s.singularCount(), s.infeasibleCount(), s.feasibleCount(), s.basesEvaluated()) == (0, 3, 7, 10)
    assert can.Evaluate(np.r_[x, 0, 0]) == 35.0
    assert s.launches() == 1          # one kernel: the record is written by its last block (no finalize launch)


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("m,n,seed", [(1, 1, 1), (1, 7, 2), (2, 2, 3), (3, 9, 4), (4, 4, 5), (4, 11, 6), (5, 12, 7),
                                      (6, 13, 8), (7, 15, 9), (9, 14, 10), (11, 15, 11), (13, 15, 12), (16, 17, 13)])
def test_small_shapes_full_range(gpu_lib, oracle, m, n, seed, algo):
    A, b, c, mx = lpgen.dense_lp(m, n, seed)
    for maximize in (False, True):
        res = gpu_solve(A, b, c, maximize, algo)
        o, _ = oracle.solve(A, b, c, maximize, n_threads=4)
        assert_same(res, o, m)


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_config2_dense_8_24(gpu_lib, oracle, seed, algo):
    A, b, c, mx = lpgen.dense_lp(8, 24, seed)
    res = gpu_solve(A, b, c, mx, algo)
    o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count())
    assert res.n_bases == 735471
    assert_same(res, o, 8)


@pytest.mark.parametrize("algo", ALGOS)
def test_config3_dense_10_30(gpu_lib, oracle, algo):
    A, b, c, mx = lpgen.dense_lp(10, 30, 1)
    res = gpu_solve(A, b, c, mx, algo)
    o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count())
    assert res.n_bases == 30045015
    assert_same(res, o, 10)


@pytest.mark.parametrize("algo", ALGOS)
def test_config5_degenerate_tie_break(gpu_lib, oracle, algo):
    """Beale-style m=10, n=30: counters and best rank identical; lowest rank wins exact ties."""
    A, b, c, mx = lpgen.degenerate_lp()
    res = gpu_solve(A, b, c, mx, algo)
    o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count())
    assert o.n_singular > 10**6 and o.n_feasible > 1000
    assert_same(res, o, 10)


@pytest.mark.parametrize("algo", ALGOS)
def test_rank_ranges_and_merge(gpu_lib, oracle, algo):
    """Arbitrary half-open ranges, empty range, and merge of disjoint ranges == full run."""
    A, b, c, mx = lpgen.dense_lp(6, 16, 21)
    total = 8008
    full = gpu_solve(A, b, c, mx, algo)
    cuts = [0, 1, 17, 1000, 1001, 4097, 8007, total]
    acc = None
    for a, e in zip(cuts[:-1], cuts[1:]):
        part = gpu_solve(A, b, c, mx, algo, rank_begin=a, rank_end=e)
        o, _ = oracle.solve(A, b, c, mx, rank_begin=a, rank_end=e)
        assert_same(part, o, 6)
        acc = part if acc is None else acc
        if part is not acc:
            if (part.key, part.best_rank) < (acc.key, acc.best_rank) and part.status == 0:
                part.n_feasible += acc.n_feasible; part.n_infeasible += acc.n_infeasible
                acc = part
            else:
                acc.n_feasible += part.n_feasible; acc.n_infeasible += part.n_infeasible
    assert (acc.best_rank, acc.n_feasible, acc.n_infeasible) == (full.best_rank, full.n_feasible, full.n_infeasible)
    empty = gpu_solve(A, b, c, mx, algo, rank_begin=5, rank_end=5)
    assert empty.status == _abi.NO_FEASIBLE and empty.n_bases == 0


@pytest.mark.parametrize("algo", ALGOS)
def test_infeasible_lp_reports_no_feasible(gpu_lib, algo):
    A = np.asfortranarray(np.array([[1.0, 1.0, 1.0], [1.0, 2.0, 3.0]]))
    can = sm.Canonical(A, [-1.0, -1.0], [1.0, 1.0, 1.0], [0, 1])
    s = sm.EnumerationSolver(can, algo=algo)
    with pytest.raises(RuntimeError, match="no feasible"):
        s.solve()
    assert s.feasibleCount() == 0 and s.basesEvaluated() == 3


def test_lda_padding_and_device_entry(gpu_lib, oracle):
    """lda > m through the host entry; device-resident entry with torch-owned buffers and stream."""
    import torch
    A, b, c, mx = lpgen.dense_lp(7, 18, 33)
    o, _ = oracle.solve(A, b, c, mx, n_threads=4)
    pad = np.zeros((10, 18), order="F"); pad[:7] = A
    ps = _abi.Problem(7, 18, 10, 0, pad.ctypes.data, b.ctypes.data, c.ctypes.data)
    res = _abi.Result()
    assert gpu_lib.enumgpu_solve(C.byref(ps), None, C.byref(res)) == 0
    assert_same(res, o, 7)

    dA = torch.from_numpy(np.ascontiguousarray(A.T)).cuda()      # row-major (n, m) == column-major (m, n)
    db, dc = torch.from_numpy(b).cuda(), torch.from_numpy(c).cuda()
    pd = _abi.Problem(7, 18, 7, 0, dA.data_ptr(), db.data_ptr(), dc.data_ptr())
    for scale in (float(np.abs(A).max()), -1.0):
        opt = _abi.Options(-1, -1, 0, 0, 0, 0, None, torch.cuda.current_stream().cuda_stream)
        res2 = _abi.Result()
        assert gpu_lib.enumgpu_solve_device(C.byref(pd), scale, C.byref(opt), C.byref(res2)) == 0, sm.last_error()
        assert_same(res2, o, 7)
        assert res2.kernel_ms > 0


def test_enqueue_device_async_partial(gpu_lib, oracle):
    import torch
    A, b, c, mx = lpgen.dense_lp(8, 20, 5)
    o, _ = oracle.solve(A, b, c, mx, n_threads=4)
    dA = torch.from_numpy(np.ascontiguousarray(A.T)).cuda()
    db, dc = torch.from_numpy(b).cuda(), torch.from_numpy(c).cuda()
    pd = _abi.Problem(8, 20, 8, 0, dA.data_ptr(), db.data_ptr(), dc.data_ptr())
    half = 125970 // 2
    parts = []
    for a, e in ((0, half), (half, 125970)):
        buf = torch.zeros(256, dtype=torch.uint8, device="cuda")
        opt = _abi.Options(-1, -1, a, e, 0, 0, None, torch.cuda.current_stream().cuda_stream)
        nl = C.c_int32()
        assert gpu_lib.enumgpu_enqueue_device(C.byref(pd), float(np.abs(A).max()), C.byref(opt), buf.data_ptr(), C.byref(nl)) == 0
        assert nl.value >= 1
        parts.append(buf)
    torch.cuda.synchronize()
    recs = [_abi.Partial.from_buffer_copy(p.cpu().numpy().tobytes()) for p in parts]
    gpu_lib.enumgpu_merge_partial(C.byref(recs[0]), C.byref(recs[1]))
    res = _abi.Result()
    gpu_lib.enumgpu_partial_to_result(C.byref(recs[0]), C.byref(res))
    assert_same(res, o, 8)


def test_headline_12_40_prefix_and_windows(gpu_lib, oracle):
    """m=12, n=40: a 2e6-rank prefix and pseudo-random windows, GPU == oracle bit for bit."""
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    total = 5586853480
    rng = np.random.default_rng(12)
    starts = [0] + [int(v) for v in rng.integers(0, total - 400000, 4)] + [total - 300000]
    for s0 in starts:
        e0 = min(total, s0 + (2000000 if s0 == 0 else 300000))
        res = gpu_solve(A, b, c, mx, rank_begin=s0, rank_end=e0)
        o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count(), rank_begin=s0, rank_end=e0)
        assert_same(res, o, 12)


def test_headline_12_40_full_vs_golden(gpu_lib):
    """Full C(40,12) enumeration against the committed CPU-oracle golden (one-off 8-core run)."""
    path = os.path.join(HERE, "golden", "dense_12_40_seed1.json")
    if not os.path.exists(path):
        pytest.skip("golden for the full 12x40 run not generated")
    g = json.load(open(path))
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    res = gpu_solve(A, b, c, mx)
    assert res.status == g["status"] and res.n_bases == g["n_bases"] == 5586853480
    assert (res.n_singular, res.n_infeasible, res.n_feasible) == (g["n_singular"], g["n_infeasible"], g["n_feasible"])
    assert res.best_rank == g["best_rank"] and list(res.basis)[:12] == g["basis"]
    assert float(res.objective).hex() == g["objective"]
    assert [float(v).hex() for v in list(res.x_B)[:12]] == g["x_B"]
    # size-independent property: the optimum satisfies B x_B = b and is what HiGHS finds
    B = A[:, g["basis"]]
    assert np.allclose(B @ np.array(list(res.x_B)[:12]), b, rtol=0, atol=1e-9)
    from scipy.optimize import linprog
    h = linprog(c, A_eq=A, b_eq=b, bounds=(0, None), method="highs")
    assert res.objective == pytest.approx(h.fun, rel=1e-9)


def test_multi_device_in_process(gpu_lib, oracle):
    """n_devices > 1 inside one process: contiguous shards, host merge; same answer."""
    nd = gpu_lib.enumgpu_device_count()
    A, b, c, mx = lpgen.dense_lp(8, 24, 2)
    o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count())
    for devs in ([0], [0, 0, 0], list(range(nd))):
        res = gpu_solve(A, b, c, mx, devices=devs)
        assert_same(res, o, 8)


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("shards", [2, 3, 8])
def test_interleaved_shards_merge_to_full(gpu_lib, oracle, algo, shards):
    """enumgpu_options.shard_index/shard_count: the shards tile the range exactly and merge to the full result."""
    A, b, c, mx = lpgen.dense_lp(8, 24, 3)
    o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count())
    can = sm.Canonical(A, b, c, list(range(8)), minimize=not mx)
    for (lo, hi) in ((0, 0), (12345, 700001)):
        if (lo, hi) != (0, 0):
            o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count(), rank_begin=lo, rank_end=hi)
        parts = [sm.EnumerationSolver(can, algo=algo).enumerate(lo, hi, shard_index=i, shard_count=shards) for i in range(shards)]
        assert sum(p.n_bases for p in parts) == o.n_bases
        assert sum(p.n_feasible for p in parts) == o.n_feasible and sum(p.n_infeasible for p in parts) == o.n_infeasible
        best = min((p.key, p.best_rank) for p in parts if p.status == 0)
        assert best == (o.key, o.best_rank)
    with pytest.raises(ValueError):
        sm.EnumerationSolver(can).enumerate(shard_index=3, shard_count=3)


@pytest.mark.parametrize("name", ["test_canonical", "beale", "dense36"])
def test_strong_duality_by_enumeration(gpu_lib, oracle, name):
    """Lab step 5 / SURVEY N4: enumerate the primal and its dual (Canonical.GetDual, as the reference
    builds it) with the same kernel; optimal objectives coincide (strong duality)."""
    if name == "dense36":
        A, b, c, mx = lpgen.dense_lp(3, 6, 5)
    else:
        g = GOLD[name]
        A, b, c, mx = np.array(g["A"]), np.array(g["b"]), np.array(g["c"]), g["maximize"]
    assert not mx
    m, n = A.shape
    primal = sm.Canonical(A, b, c, list(range(m)), minimize=True)
    dual = primal.GetDual()
    assert dual.GetConstraintsMatrix().shape == (n, 2 * m + n) and dual.IsMaximization()
    sp_, sd_ = sm.EnumerationSolver(primal), sm.EnumerationSolver(dual)
    sp_.solve(); y2 = sd_.solve()
    assert sd_.objective() == pytest.approx(sp_.objective(), rel=1e-9, abs=1e-9)
    y = y2[:m] - y2[m:]                                   # y = y' - y''
    assert np.all(A.T @ y <= c + 1e-9)                    # dual feasibility
    od, _ = oracle.solve(dual.GetConstraintsMatrix(), dual.GetRightHandSide(), dual.GetObjectiveCoefficients(), True, n_threads=4)
    assert (sd_.bestRank(), sd_.feasibleCount(), sd_.singularCount()) == (od.best_rank, od.n_feasible, od.n_singular)


def test_shared_kernel_range_guard(gpu_lib, oracle):
    """eps_piv = 0 (or absurd scaling) takes the branch-free reciprocal of k_shared out of its proven range:
    the library must fall back to the independent kernel, and still match the oracle."""
    A, b, c, mx = lpgen.dense_lp(7, 16, 9)
    can = sm.Canonical(A, b, c, list(range(7)), minimize=not mx)
    res = sm.EnumerationSolver(can, algo=_abi.ALGO_SHARED, eps_piv=0.0).enumerate()
    o, _ = oracle.solve(A, b, c, mx, eps_piv=0.0)
    assert res.algo_used == _abi.ALGO_INDEPENDENT
    assert_same(res, o, 7)
    tiny = sm.Canonical(A * 1e-295, b * 1e-295, c, list(range(7)), minimize=not mx)
    res = sm.EnumerationSolver(tiny, algo=_abi.ALGO_SHARED).enumerate()
    o, _ = oracle.solve(A * 1e-295, b * 1e-295, c, mx)
    assert res.algo_used == _abi.ALGO_INDEPENDENT
    assert_same(res, o, 7)
    assert sm.EnumerationSolver(can, algo=_abi.ALGO_SHARED).enumerate().algo_used == _abi.ALGO_SHARED


@pytest.mark.parametrize("m,n,seed", [(6, 64, 3), (8, 40, 4), (16, 20, 5), (9, 33, 6)])
def test_wide_and_tall_shapes_shared_kernel(gpu_lib, oracle, m, n, seed):
    """Limits of the shared kernel: n = ENUMGPU_MAX_N (two columns per lane in the level code, fewer warps per
    CTA), m = ENUMGPU_MAX_M, and a shape where one child task has more than 32 candidate columns."""
    A, b, c, mx = lpgen.dense_lp(m, n, seed)
    res = gpu_solve(A, b, c, mx, _abi.ALGO_SHARED)
    assert res.algo_used == _abi.ALGO_SHARED
    o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count())
    assert_same(res, o, m)


@pytest.mark.parametrize("m,n,seed,eps", [(8, 24, 1, 1e300), (10, 30, 1, 1e300), (7, 40, 2, 1e300), (12, 20, 3, 1e300),
                                          (13, 19, 4, 1e300), (10, 30, 1, 5.0), (8, 24, 2, 3.0)])
def test_survivor_stacks_under_pressure(gpu_lib, oracle, m, n, seed, eps):
    """eps_feas so large that every basis (1e300) or a large share of them (5, 3) passes the five-component filter of
    the leaves: every lane of every d-loop trip pushes an entry, a batch fills its first-stage stack to the bound it
    was sized for (32 (n-4) on top of 31), and every basis goes through promote_fn and drain2_fn.  Counters, optimum
    and tie-break must still be the oracle's."""
    A, b, c, mx = lpgen.dense_lp(m, n, seed)
    can = sm.Canonical(A, b, c, list(range(m)), minimize=not mx)
    o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count(), eps_feas=eps)
    if eps > 1e10:
        assert o.n_infeasible == 0 and o.n_feasible + o.n_singular == o.n_bases
    else:
        assert o.n_feasible > o.n_bases // 10
    for algo in ALGOS:
        res = sm.EnumerationSolver(can, algo=algo, eps_feas=eps).enumerate()
        assert res.algo_used == algo
        assert_same(res, o, m)
    for shards in (3,):
        parts = [sm.EnumerationSolver(can, algo=_abi.ALGO_SHARED, eps_feas=eps).enumerate(shard_index=i, shard_count=shards)
                 for i in range(shards)]
        assert sum(p.n_feasible for p in parts) == o.n_feasible and sum(p.n_bases for p in parts) == o.n_bases
        assert min((p.key, p.best_rank) for p in parts if p.status == 0) == (o.key, o.best_rank)


def test_beyond_headline_size_properties(gpu_lib):
    """m=12, n=44 (21 090 682 613 bases, too many for the CPU oracle): size-independent properties —
    every rank falls in exactly one class, the optimum is HiGHS's, B x_B = b, and the result is the same for
    both kernel-independent shardings (1 shard vs 3 interleaved shards merged)."""
    from scipy.optimize import linprog
    m, n = 12, 44
    A, b, c, mx = lpgen.dense_lp(m, n, 7)
    can = sm.Canonical(A, b, c, list(range(m)), minimize=not mx)
    s = sm.EnumerationSolver(can)
    x = s.solve()
    total = gpu_lib.enumgpu_binomial(n, m)
    assert s.basesEvaluated() == total == 21090682613
    assert s.singularCount() + s.infeasibleCount() + s.feasibleCount() == total
    h = linprog(c, A_eq=A, b_eq=b, bounds=(0, None), method="highs")
    assert s.objective() == pytest.approx(h.fun, rel=1e-9)
    assert sorted(np.nonzero(h.x > 1e-9)[0].tolist()) == s.optimalBasis()
    assert np.allclose(A[:, s.optimalBasis()] @ np.array(s.basicValues()), b, rtol=0, atol=1e-9)
    parts = [sm.EnumerationSolver(can).enumerate(shard_index=i, shard_count=3) for i in range(3)]
    assert sum(p.n_bases for p in parts) == total
    assert sum(p.n_feasible for p in parts) == s.feasibleCount()
    assert sum(p.n_singular for p in parts) == s.singularCount()
    assert min((p.key, p.best_rank) for p in parts if p.status == 0) == (s._res.key, s.bestRank())


@pytest.mark.parametrize("algo", ALGOS)
def test_list_feasible_bases_and_vertices(gpu_lib, oracle, algo):
    """enumgpu_list_feasible / enumgpu_eval_ranks: the extreme points themselves.  Ranks == the oracle's
    per-rank classification; x_B of every listed basis == the oracle's; vertices of the lab LP == SURVEY A.1."""
    A, b, c, mx = lpgen.dense_lp(8, 20, 5)
    o, status = oracle.solve(A, b, c, mx, want_status=True)
    want = np.nonzero(status == 0)[0]
    s = sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(8)), minimize=not mx), algo=algo)
    ranks = s.listFeasibleBases()
    assert ranks.tolist() == want.tolist() and s.feasibleCount() == want.size and s.bestRank() == o.best_rank
    few = s.listFeasibleBases(capacity=10)                       # too small: some 10 of them, ascending
    assert few.size == 10 and set(few.tolist()) <= set(want.tolist()) and (np.diff(few.astype(np.int64)) > 0).all()
    assert s.feasibleCount() == want.size
    bases, xB, z, cls = s.evaluateBases(ranks[:50])
    assert (cls == 0).all()
    for i in range(50):
        st, xo, zo = oracle.eval_basis(A, b, c, mx, bases[i].tolist())
        assert st == 0 and xB[i].tolist() == xo and z[i] == zo
    _, _, _, cls_mixed = s.evaluateBases([0, 1, 2, int(want[0])])
    assert cls_mixed.tolist() == [int(status[0]), int(status[1]), int(status[2]), 0]
    # the reference's lab LP: 7 feasible bases, 4 distinct vertices (SURVEY A.1)
    A, b, c, mx = lpgen.lab_symmetric_canonical()
    s = sm.EnumerationSolver(sm.Canonical(A, b, c, [3, 4], minimize=False), algo=algo)
    assert s.listFeasibleBases().tolist() == [1, 2, 4, 5, 7, 8, 9]
    X, zz = s.feasibleVertices()
    assert X.shape == (4, 5) and sorted(np.round(zz, 9).tolist()) == [0.0, 10.0, 32.0, 35.0]


def test_reentrant_from_two_host_threads(gpu_lib, oracle):
    """The ABI promises re-entrancy (no global mutable state but a thread-local error string): two host
    threads enumerate different LPs at the same time, repeatedly, and both get the oracle's answers."""
    import threading
    lps = [lpgen.dense_lp(8, 22, 11), lpgen.dense_lp(9, 21, 12)]
    want = [oracle.solve(*lp, n_threads=4)[0] for lp in lps]
    errors = []

    def work(i):
        try:
            A, b, c, mx = lps[i]
            for _ in range(5):
                res = gpu_solve(A, b, c, mx)
                assert_same(res, want[i], A.shape[0])
        except BaseException as e:       # noqa: BLE001 - reported to the main thread
            errors.append(e)

    ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors


# ---------------------------------------------------------------------------------------------
# round 2: the parity gaps VERDICT r1 named — ties and singular subtrees through the SHARDED path,
# the singular bases of the headline LP, the Eigen-like relative rule, handles, the reciprocal.

_DEGENERATE = {"small": lpgen.small_degenerate_lp, "config5": lpgen.degenerate_lp}
_ORACLE_CACHE = {}


def _oracle_cached(oracle, name, **opt):
    key = (name, tuple(sorted(opt.items())))
    if key not in _ORACLE_CACHE:
        A, b, c, mx = _DEGENERATE[name]()
        _ORACLE_CACHE[key] = oracle.solve(A, b, c, mx, n_threads=os.cpu_count(), **opt)[0]
    return _ORACLE_CACHE[key]


def _merge_results(parts):
    """What enumgpu_merge_partial does, on result structs: counters add, lexicographic min on (key, rank)."""
    tot = [sum(getattr(p, f) for p in parts) for f in ("n_bases", "n_singular", "n_infeasible", "n_feasible")]
    ok = [p for p in parts if p.status == 0]
    win = min(ok, key=lambda p: (p.key, p.best_rank)) if ok else None
    return tot, win


def _assert_merged_equals(parts, o, m):
    tot, win = _merge_results(parts)
    assert tot == [o.n_bases, o.n_singular, o.n_infeasible, o.n_feasible]
    if o.status == 0:
        assert win is not None and win.best_rank == o.best_rank and win.key == o.key
        assert list(win.basis)[:m] == list(o.basis)[:m] and list(win.x_B)[:m] == list(o.x_B)[:m]
        assert win.objective == o.objective
    else:
        assert win is None


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("shards", [2, 3, 8])
@pytest.mark.parametrize("name", ["small", "config5"])
def test_degenerate_lps_through_interleaved_shards(gpu_lib, oracle, name, shards, algo):
    """Config 5 (29 M singular bases, exact ties at the optimum) and a small degenerate LP through
    shard_index/shard_count: ties that straddle shard windows and singular children split across windows
    (k_shared's ns_bulk share) must merge to the oracle's best rank and all four counters."""
    A, b, c, mx = _DEGENERATE[name]()
    m = A.shape[0]
    o = _oracle_cached(oracle, name)
    assert o.n_singular > 1000 and o.n_feasible > 100
    can = sm.Canonical(A, b, c, list(range(m)), minimize=not mx)
    s = sm.EnumerationSolver(can, algo=algo)
    parts = []
    for i in range(shards):
        r = s.enumerate(shard_index=i, shard_count=shards)
        parts.append(_abi.Result.from_buffer_copy(bytes(r)))
    _assert_merged_equals(parts, o, m)


@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("shards", [1, 3])
def test_subrange_cut_inside_a_singular_child(gpu_lib, oracle, algo, shards):
    """Columns 0 and 1 of the small degenerate LP are identical: every child task (0, 1, s) is singular as a
    whole.  Rank ranges cut INSIDE such a child (ragged head/tail on the independent kernel, the core on the
    shared one) and inside later children, optionally sharded, must reproduce the oracle range by range."""
    A, b, c, mx = lpgen.small_degenerate_lp()
    total = 31824
    child0 = 1365                                   # C(15,4) bases with prefix (0,1,2): ranks [0, 1365), all singular
    st = oracle.solve(A, b, c, mx, want_status=True)[1]
    assert (st[:child0] == 2).all()
    can = sm.Canonical(A, b, c, list(range(7)), minimize=not mx)
    s = sm.EnumerationSolver(can, algo=algo)
    cuts = [0, 700, child0 + 333, 9000, 9001, 20000, total]
    for a, e in zip(cuts[:-1], cuts[1:]):
        o, _ = oracle.solve(A, b, c, mx, rank_begin=a, rank_end=e)
        parts = [_abi.Result.from_buffer_copy(bytes(s.enumerate(a, e, shard_index=i, shard_count=shards if shards > 1 else 0)))
                 for i in range(shards)]
        _assert_merged_equals(parts, o, 7)


def test_headline_singular_bases_under_both_rules(gpu_lib, oracle):
    """The 9 bases of dense(12,40,1) that the default ABSOLUTE rule (|pivot| <= 1e-9 max|A|) calls singular —
    the only place where that rule and the reference's FullPivLU::isInvertible (SimplexSolover.h:124-126,
    relative threshold eps*m) can differ on the headline LP.  Evaluated one by one on the GPU and by the oracle
    under both rules: absolute -> singular (as counted in the golden); relative (Eigen-like) -> NOT singular,
    infeasible (the pivots are ~1e-10, far above 12*2^-52 relative), i.e. n_singular moves to n_infeasible and
    n_feasible is unaffected.  tests/test_reference_code.py asks the reference's own code about the same ranks."""
    g = json.load(open(os.path.join(HERE, "golden", "dense_12_40_seed1.json")))
    ranks = g.get("singular_ranks")
    if not ranks:
        pytest.skip("golden without singular_ranks")
    assert len(ranks) == g["n_singular"] == 9
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    can = sm.Canonical(A, b, c, list(range(12)), minimize=not mx)
    for rule, want_cls in ((_abi.PIVOT_ABSOLUTE, 2), (_abi.PIVOT_RELATIVE, 1)):
        s = sm.EnumerationSolver(can, pivot_rule=rule)
        bases, xB, z, cls = s.evaluateBases(ranks)
        assert cls.tolist() == [want_cls] * 9
        for i, r in enumerate(ranks):
            st, xo, zo = oracle.eval_basis(A, b, c, mx, bases[i].tolist(), pivot_rule=rule)
            assert st == want_cls
            if st != 2:
                assert xB[i].tolist() == xo and z[i] == zo
        # the same through the enumeration kernels on 1-rank windows (both kernel families for the absolute rule)
        for r in ranks[:3]:
            for algo in ALGOS:
                res = sm.EnumerationSolver(can, pivot_rule=rule, algo=algo).enumerate(r, r + 1)
                assert (res.n_singular, res.n_infeasible, res.n_feasible) == ((1, 0, 0) if want_cls == 2 else (0, 1, 0))


@pytest.mark.parametrize("name", ["small", "config5", "dense_8_24", "beale", "tiny_shapes"])
def test_relative_pivot_rule_parity(gpu_lib, oracle, name):
    """ENUMGPU_PIVOT_RELATIVE (Eigen-like: min|pivot| > eps * max|pivot|, eps = m * 2^-52 by default) against its
    oracle twin, bit for bit: counters, best rank, x_B, objective; explicit eps too.  Runs on the independent kernel."""
    if name == "tiny_shapes":
        lps = [lpgen.dense_lp(m, n, 40 + m) for (m, n) in [(1, 3), (2, 5), (5, 11), (7, 14), (13, 15), (16, 17)]]
    elif name == "dense_8_24":
        lps = [lpgen.dense_lp(8, 24, 2)]
    elif name == "beale":
        lps = [lpgen.beale_lp(), lpgen.main_cpp_canonical()]
    else:
        lps = [_DEGENERATE[name]()]
    for A, b, c, mx in lps:
        m = A.shape[0]
        can = sm.Canonical(A, b, c, list(range(m)), minimize=not mx)
        for eps in (-1.0, 1e-6):
            o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count(), pivot_rule=_abi.PIVOT_RELATIVE, eps_piv=eps)
            res = sm.EnumerationSolver(can, pivot_rule=_abi.PIVOT_RELATIVE, eps_piv=eps, algo=_abi.ALGO_SHARED).enumerate()
            assert res.algo_used == _abi.ALGO_INDEPENDENT
            assert_same(res, o, m)
    with pytest.raises(ValueError):
        sm.EnumerationSolver(can, pivot_rule=7).enumerate()


def test_rcp_nobranch_equals_drcp_rn_on_1e9_operands(gpu_lib):
    """The shared kernel's branch-free reciprocal against __drcp_rn, bitwise, on the device: every power of two
    in 2^-1000..2^1000 with both neighbours and both signs, then > 1e9 random operands with uniformly distributed
    exponents (enumgpu_selftest_rcp).  Bit-identity of every basis k_shared evaluates rests on this."""
    bad, first = C.c_uint64(123), C.c_double()
    for seed, count in ((1, 1 << 30), (2026, 1 << 24)):
        assert gpu_lib.enumgpu_selftest_rcp(count, seed, C.byref(bad), C.byref(first)) == 0, sm.last_error()
        assert bad.value == 0, f"{bad.value} mismatches, first at {first.value!r}"


def test_handles_reuse_and_recover(gpu_lib, oracle):
    """enumgpu_create / enumgpu_solve_h / enumgpu_destroy: one handle, many solves of different shapes (the
    control block must come back zeroed every time), a failing call in between, and two handles side by side."""
    h1, h2 = C.c_void_p(), C.c_void_p()
    assert gpu_lib.enumgpu_create(-1, C.byref(h1)) == 0 and gpu_lib.enumgpu_create(0, C.byref(h2)) == 0
    try:
        for rep in range(3):
            for (m, n, seed) in [(8, 20, 5), (3, 9, 4), (6, 30, 2), (12, 18, 3)]:
                A, b, c, mx = lpgen.dense_lp(m, n, seed)
                o, _ = oracle.solve(A, b, c, mx, n_threads=4)
                ps = _abi.Problem(m, n, m, int(mx), A.ctypes.data, b.ctypes.data, c.ctypes.data)
                for h in (h1, h2):
                    res = _abi.Result()
                    assert gpu_lib.enumgpu_solve_h(h, C.byref(ps), None, C.byref(res)) == 0, sm.last_error()
                    assert_same(res, o, m)
                    assert res.n_launches == 1 and res.kernel_ms > 0
            bad = _abi.Options(-1, -1, 10, 2, 0, 0, None, None)          # bad range: an error, then business as usual
            res = _abi.Result()
            assert gpu_lib.enumgpu_solve_h(h1, C.byref(ps), C.byref(bad), C.byref(res)) == _abi.ERR_RANGE
        # ragged range: shared kernel + independent head and tail in one enqueue, one record
        A, b, c, mx = lpgen.dense_lp(8, 24, 1)
        ps = _abi.Problem(8, 24, 8, int(mx), A.ctypes.data, b.ctypes.data, c.ctypes.data)
        opt = _abi.Options(-1, -1, 12345, 700001, 0, 0, None, None)
        o, _ = oracle.solve(A, b, c, mx, n_threads=4, rank_begin=12345, rank_end=700001)
        res = _abi.Result()
        assert gpu_lib.enumgpu_solve_h(h1, C.byref(ps), C.byref(opt), C.byref(res)) == 0
        assert_same(res, o, 8)
        assert res.n_launches == 3
    finally:
        gpu_lib.enumgpu_destroy(h1); gpu_lib.enumgpu_destroy(h2)
    assert gpu_lib.enumgpu_solve_h(None, C.byref(ps), None, C.byref(res)) == _abi.ERR_ARG


def test_enqueue_h_back_to_back_on_one_stream(gpu_lib, oracle):
    """enumgpu_enqueue_h: the handle's scratch is reused by consecutive enqueues on one stream without any
    host synchronisation in between; every record must be right."""
    import torch
    h = C.c_void_p()
    assert gpu_lib.enumgpu_create(-1, C.byref(h)) == 0
    try:
        A, b, c, mx = lpgen.dense_lp(8, 20, 5)
        o, _ = oracle.solve(A, b, c, mx, n_threads=4)
        dA = torch.from_numpy(np.ascontiguousarray(A.T)).cuda()
        db, dc = torch.from_numpy(b).cuda(), torch.from_numpy(c).cuda()
        pd = _abi.Problem(8, 20, 8, 0, dA.data_ptr(), db.data_ptr(), dc.data_ptr())
        bufs = [torch.zeros(256, dtype=torch.uint8, device="cuda") for _ in range(6)]
        torch.cuda.synchronize()
        nl = C.c_int32()
        side = torch.cuda.Stream()                        # a caller-owned stream: every enqueue of this handle goes there
        opt = _abi.Options(-1, -1, 0, 0, 0, 0, None, side.cuda_stream)
        for buf in bufs[:3]:
            assert gpu_lib.enumgpu_enqueue_h(h, C.byref(pd), float(np.abs(A).max()), C.byref(opt), buf.data_ptr(), C.byref(nl)) == 0
            assert nl.value == 1
        side.synchronize()
        opt.stream = None                                 # NULL: the handle's own stream
        for buf in bufs[3:]:
            assert gpu_lib.enumgpu_enqueue_h(h, C.byref(pd), float(np.abs(A).max()), C.byref(opt), buf.data_ptr(), C.byref(nl)) == 0
        torch.cuda.ExternalStream(gpu_lib.enumgpu_handle_stream(h)).synchronize()
        for buf in bufs:
            rec = _abi.Partial.from_buffer_copy(buf.cpu().numpy().tobytes())
            res = _abi.Result()
            gpu_lib.enumgpu_partial_to_result(C.byref(rec), C.byref(res))
            assert_same(res, o, 8)
    finally:
        gpu_lib.enumgpu_destroy(h)


@pytest.mark.skipif(sm.lib().enumgpu_device_count() < 2, reason="needs two CUDA devices in one process")
def test_multi_device_distinct_devices_in_process(gpu_lib, oracle):
    """devices=[0, 1] (and all of them) inside ONE process: one handle per device, interleaved windows, host merge."""
    nd = gpu_lib.enumgpu_device_count()
    for lp, m in ((lpgen.dense_lp(8, 24, 2), 8), (lpgen.degenerate_lp(), 10)):
        A, b, c, mx = lp
        o, _ = oracle.solve(A, b, c, mx, n_threads=os.cpu_count())
        for devs in ([0, 1], [1, 0], list(range(nd))):
            res = gpu_solve(A, b, c, mx, devices=devs)
            assert_same(res, o, m)


def test_eval_basis_any_size(gpu_lib, oracle):
    """Canonical.GetBasicSolution / IsFeasibleBasis stand on enumgpu_eval_basis, which — like the reference's
    methods (Canonical.cpp:165-197) — takes a Canonical of ANY size and any index list: the dual of the headline
    LP (40 x 64), an LP beyond the enumeration limits (m = 40, n = 100), repeated indices (singular, no error)."""
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    dual = sm.Canonical(A, b, c, list(range(12)), minimize=True).GetDual()
    assert dual.GetConstraintsMatrix().shape == (40, 64)
    assert dual.IsFeasibleBasis() == bool(np.all(dual.GetRightHandSide() >= -1e-9))     # slack basis: x = c
    x = dual.GetBasicSolution()
    assert np.array_equal(x[24:], dual.GetRightHandSide()) and not x[:24].any()
    rng = np.random.default_rng(5)
    m, n = 40, 100
    Ab = rng.uniform(-1, 1, (m, n)); xb = rng.uniform(0.5, 1.5, m)
    basis = sorted(rng.choice(n, m, replace=False).tolist())
    bb = Ab[:, basis] @ xb
    big = sm.Canonical(Ab, bb, rng.uniform(-1, 1, n), basis)
    assert big.IsFeasibleBasis()
    assert np.allclose(big.GetBasicSolution()[basis], xb, rtol=0, atol=1e-9)
    # the same arithmetic as the enumeration: bit-identical to the oracle where both apply
    A8, b8, c8, _ = lpgen.dense_lp(8, 24, 1)
    for S in ([0, 1, 2, 3, 4, 5, 6, 7], [3, 5, 8, 9, 13, 17, 20, 23]):
        st, xo, zo = oracle.eval_basis(A8, b8, c8, False, S)
        can = sm.Canonical(A8, b8, c8, S)
        assert can.IsFeasibleBasis() == (st == 0)
        assert can.GetBasicSolution()[S].tolist() == xo
    rep = sm.Canonical(A8, b8, c8, [0, 1, 2, 3, 4, 5, 6, 6])
    assert rep.IsFeasibleBasis() is False
    with pytest.raises(RuntimeError, match="Singular"):
        rep.GetBasicSolution()
    # eps_feas = eps_piv = -0.0 mean 0 (enumgpu.h): the oracle's answer with both tolerances 0
    zero = _abi.Options(-0.0, -0.0, 0, 0, 0, 0, None, None, 0, 0, _abi.PIVOT_ABSOLUTE, 0)
    ps = _abi.Problem(8, 24, 8, 0, A8.ctypes.data, b8.ctypes.data, c8.ctypes.data)
    for S in ([0, 1, 2, 3, 4, 5, 6, 7], [3, 5, 8, 9, 13, 17, 20, 23], [0, 1, 2, 3, 4, 5, 6, 6]):
        x, z, cls = (C.c_double * 8)(), C.c_double(), C.c_int32()
        assert gpu_lib.enumgpu_eval_basis(C.byref(ps), C.byref(zero), (C.c_int32 * 8)(*S), x, C.byref(z), C.byref(cls)) == 0
        st, xo, zo = oracle.eval_basis(A8, b8, c8, False, S, eps_feas=0.0, eps_piv=0.0)
        assert cls.value == st
        if st != _abi.BASIS_SINGULAR:
            assert list(x) == xo and z.value == zo


def test_sharded_enumeration_host_path_single_rank(gpu_lib, oracle):
    """dist.ShardedEnumeration.solve (enumgpu_enqueue_host_h + gather + enumgpu_merge_records) with WORLD = 1:
    the host-buffer path a one-process-per-GPU job runs on every rank (bench.py's e2e at N > 1), without NCCL."""
    from simplexmethod_b200 import dist as edist
    se = edist.ShardedEnumeration(0, 0, 1)
    try:
        for lp, m in ((lpgen.dense_lp(8, 24, 2), 8), (lpgen.small_degenerate_lp(), 7), (lpgen.dense_lp(6, 16, 21), 6)):
            A, b, c, mx = lp
            o, _ = oracle.solve(A, b, c, mx, n_threads=4)
            for _ in range(2):
                assert_same(se.solve(A, b, c, mx), o, m)
        A, b, c, mx = lpgen.dense_lp(8, 24, 2)
        o, _ = oracle.solve(A, b, c, mx, n_threads=4, rank_begin=1000, rank_end=500000)
        assert_same(se.solve(A, b, c, mx, rank_begin=1000, rank_end=500000), o, 8)
    finally:
        se.close()
