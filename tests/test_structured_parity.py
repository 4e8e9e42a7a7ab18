"""Structured and boundary LPs: both kernel families against the CPU oracle, bit for bit.

lpgen.dense_lp has uniform random entries: no exact zeros, no ties in |pivot|, all magnitudes O(1), no
degeneracy.  The families here are built to reach what such data never does:

  sparse_dyadic      entries from {+-1/2, +-1, +-3/2, +-2, +-3}, many zeros: singular subtrees at every level and
                     frequent exact ties for the pivot (the frozen arithmetic takes the FIRST maximum)
  thirds             entries k/3: ties between non-dyadic values, where the wrong row also changes the rounding
  signed_duplicates  dense_lp with dependent column pairs (c, -c), (c, 2c) placed so that prefixes of every depth
                     are singular as a whole, a duplicated late column, and +-1, -+1 in rows 0 and 1 of every
                     second column (ties of |pivot| with opposite signs)
  network            [I | e_i - e_k, +-e_i]: totally unimodular, every x_B an integer, so components sit exactly
                     on the feasibility boundary (-1, -2, -0.0)
  column_scaled      dense_lp with columns scaled by 2^k, k in [-36, 12]: whole columns below the pivot threshold
  huge_rhs, huge_cost, tiny_rhs, all_nan_keys
                     overflow of x_B or z to +-inf / NaN, subnormal x_B, and an LP whose feasible bases all have a
                     NaN objective (NO_FEASIBLE with n_feasible > 0)

The tests without the gpu marker check that each family still reaches what it is there for, so that an edit to a
generator cannot quietly take a case away.  All generators are deterministic: small finite value sets drawn with
numpy's PCG64, and right-hand sides formed exactly.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest

from simplexmethod_b200 import _abi, lpgen

ALGOS = [_abi.ALGO_INDEPENDENT, _abi.ALGO_SHARED]
NCPU = os.cpu_count()
FEASIBLE, INFEASIBLE, SINGULAR = 0, 1, 2


# --------------------------------------------------------------------------------------------- generators

def sparse_dyadic(m, n, seed, density=0.5):
    rng = np.random.default_rng(seed)
    mag = rng.choice(np.array([0.5, 1.0, 1.5, 2.0, 3.0]), (m, n))
    sign = rng.choice(np.array([-1.0, 1.0]), (m, n))
    keep = rng.random((m, n)) < density
    A = np.asfortranarray(np.where(keep, mag * sign, 0.0))
    x0 = rng.integers(1, 4, m).astype(np.float64)
    b = A[:, :m] @ x0                       # halves times small integers: exact in any summation order
    c = rng.integers(-3, 4, n).astype(np.float64)
    return A, b, c, False


def thirds(m, n, seed, density=0.7):
    rng = np.random.default_rng(seed)
    K = rng.integers(-6, 7, (m, n)) * (rng.random((m, n)) < density)
    x0 = rng.integers(1, 4, m)
    A = np.asfortranarray(K / 3.0)
    b = (K[:, :m] @ x0) / 3.0               # integer product, one rounding
    c = rng.integers(-6, 7, n) / 3.0
    return A, b, c, False


def dup_pairs(m):
    """Column pairs (j, j+1) of signed_duplicates: column j+1 = -column j, and 2 x column j' at j' = j + 3."""
    j1 = max(m - 6, 0)
    return j1, j1 + 3


def signed_duplicates(m, n, seed):
    """dense_lp(m, n, seed) with dependent columns.  The pair (j1, j1+1), j1 = m - 6, fits at prefix positions
    (i, i+1) for every i <= j1, so whole subtrees are singular at every elimination step up to the child pivot:
    the rebuild of depth q-1 from A, the node and parent level steps and the child's pivot."""
    A, b, c, mx = lpgen.dense_lp(m, n, seed)
    A = A.copy(order="F")
    c = c.copy()
    j1, j2 = dup_pairs(m)
    A[:, j1 + 1] = -A[:, j1]
    A[:, j2 + 1] = 2.0 * A[:, j2]
    A[:, n - 2] = A[:, n - 5]
    for j in range(0, n, 2):                 # the largest entries of these columns: +-1 in row 0, the opposite in row 1
        if j not in (j1, j1 + 1, j2, j2 + 1, n - 5, n - 2):
            A[0, j] = 1.0 if A[0, j] >= 0 else -1.0
            A[1, j] = -A[0, j]
    return A, b, c, mx


def network(m, n, seed, b_vals=range(-3, 6)):
    """[I | e_i - e_k or +-e_i]: totally unimodular, so every pivot is +-1, every x_B an integer."""
    rng = np.random.default_rng(seed)
    A = np.zeros((m, n), order="F")
    A[:, :m] = np.eye(m)
    for j in range(m, n):
        i, k = rng.choice(m, 2, replace=False)
        A[i, j] = 1.0
        if rng.random() < 0.75:
            A[k, j] = -1.0
        elif rng.random() < 0.5:
            A[i, j] = -1.0
    b = rng.choice(np.array(list(b_vals), dtype=np.float64), m)
    c = rng.integers(-4, 5, n).astype(np.float64)
    return A, b, c, False


def column_scaled(m, n, seed):
    A, b, c, mx = lpgen.dense_lp(m, n, seed)
    k = np.random.default_rng(seed).integers(-36, 13, n)
    return np.asfortranarray(A * np.ldexp(1.0, k)), b, c, mx


def huge_rhs(m, n, seed):
    A, b, c, mx = lpgen.dense_lp(m, n, seed)
    return A, b * 2.0 ** 1020, c, mx


def huge_cost(m, n, seed):
    A, b, c, mx = lpgen.dense_lp(m, n, seed)
    return A, b, c * 2.0 ** 1021, mx


def tiny_rhs(m, n, seed):
    A, b, c, mx = sparse_dyadic(m, n, seed)
    return A, b * 2.0 ** -1070, c, mx


def all_nan_keys(m, n, seed=0):
    """Column 0 = e_0 / 2 is the only column with an entry in row 0, so it is S[0] of every nonsingular basis,
    and b[0] = 2^1023 makes x[0] = +inf (feasible).  x[0] is the last component the back substitution computes,
    so nothing else turns NaN; every other component is 4.  c[0] = 0 then gives the objective 0 * inf = NaN
    for every feasible basis."""
    A = np.zeros((m, n), order="F")
    A[0, 0] = 0.5
    for j in range(1, n):
        A[1 + (j - 1) % (m - 1), j] = 1.0
    b = np.full(m, 4.0)
    b[0] = 2.0 ** 1023
    c = np.ones(n)
    c[0] = 0.0
    return A, b, c, False


FAMILIES = {"sparse_dyadic": sparse_dyadic, "thirds": thirds, "signed_duplicates": signed_duplicates,
            "network": network, "column_scaled": column_scaled, "huge_rhs": huge_rhs, "huge_cost": huge_cost,
            "tiny_rhs": tiny_rhs}
# the run-time-n instantiation across m (m >= 12 also runs the odd-column copy of the d loop), n = 64, and the
# three shapes with kernels compiled for their n
SHAPES = [(6, 18), (7, 21), (9, 22), (11, 23), (12, 26), (13, 24), (16, 24), (6, 64), (8, 24), (10, 30)]


# --------------------------------------------------------------------------------------------- helpers

def bits(v):
    return np.float64(v).view(np.uint64).item()


def rank_of(n, m, S):
    from oracle import enumcpu
    return int(enumcpu.lib().enumcpu_rank(n, m, (C.c_int32 * m)(*S)))


def unrank(n, m, r):
    from oracle import enumcpu
    S = (C.c_int32 * m)()
    enumcpu.lib().enumcpu_unrank(n, m, int(r), S)
    return list(S)


def scale_of(A):
    return float(np.abs(A).max())


def exact_eps_piv(A, thr):
    """eps_piv with eps_piv * max|A| == thr exactly (the threshold is that one product)."""
    e = thr / scale_of(A)
    assert e * scale_of(A) == thr
    return e


def assert_same(g, o, m):
    """Bit-for-bit: counters, status, best rank and basis, and the bits of x_B, objective and key."""
    assert (g.n_bases, g.n_singular, g.n_infeasible, g.n_feasible) == \
           (o.n_bases, o.n_singular, o.n_infeasible, o.n_feasible)
    assert g.status == o.status and g.best_rank == o.best_rank
    if o.status == _abi.OK:
        assert list(g.basis)[:m] == list(o.basis)[:m]
        assert [bits(v) for v in list(g.x_B)[:m]] == [bits(v) for v in list(o.x_B)[:m]]
        assert bits(g.objective) == bits(o.objective) and bits(g.key) == bits(o.key)


def merged(parts):
    """What enumgpu_merge_partial does: counters add, lexicographic minimum of (key, rank) over the OK parts."""
    out = _abi.Result()
    for f in ("n_bases", "n_singular", "n_infeasible", "n_feasible"):
        setattr(out, f, sum(getattr(p, f) for p in parts))
    ok = [p for p in parts if p.status == _abi.OK]
    if not ok:
        out.status, out.best_rank = _abi.NO_FEASIBLE, (1 << 64) - 1
        return out
    w = min(ok, key=lambda p: (p.key, p.best_rank))
    out.status, out.best_rank, out.m = _abi.OK, w.best_rank, w.m
    out.objective, out.key = w.objective, w.key
    for i in range(w.m):
        out.basis[i], out.x_B[i] = w.basis[i], w.x_B[i]
    return out


def ge_ties(A, S):
    """Pivot steps of the partial-pivot GE of basis S at which the maximum |M[r][k]| (nonzero) is attained by
    more than one row.  Plain numpy, no FMA: only has to show that ties occur."""
    M = np.array(A[:, S], dtype=np.float64)
    m = M.shape[0]
    ties = 0
    for k in range(m):
        col = np.abs(M[k:, k])
        best = col.max()
        if not best > 0:
            return ties
        ties += int((col == best).sum() > 1)
        p = k + int(np.argmax(col))
        M[[k, p]] = M[[p, k]]
        M[k + 1:] -= np.outer(M[k + 1:, k] / M[k, k], M[k])
    return ties


def sample_ranks(n, m, count, seed):
    from oracle import enumcpu
    total = int(enumcpu.lib().enumcpu_binomial(n, m))
    return np.random.default_rng(seed).integers(0, total, min(count, total))


# ---------------------------------------------------------------------------- self-checks (no GPU)

THRESHOLD_CASES = [("sparse_dyadic", 8, 24, 1, 0.5), ("sparse_dyadic", 9, 22, 2, 0.25), ("thirds", 8, 24, 3, 1.0)]


@pytest.mark.parametrize("name,m,n,seed,thr", THRESHOLD_CASES)
def test_selfcheck_pivots_exactly_at_threshold(oracle, name, m, n, seed, thr):
    """Some pivots equal thr exactly: n_singular moves when eps_piv moves one ulp down."""
    A, b, c, mx = FAMILIES[name](m, n, seed)
    e = exact_eps_piv(A, thr)
    at, _ = oracle.solve(A, b, c, mx, n_threads=NCPU, eps_piv=e)
    below, _ = oracle.solve(A, b, c, mx, n_threads=NCPU, eps_piv=np.nextafter(e, 0.0))
    assert at.n_singular > below.n_singular > 0


NETWORK_FEAS = [(8, 20, 3), (9, 22, 3)]


@pytest.mark.parametrize("m,n,seed", NETWORK_FEAS)
def test_selfcheck_network_on_the_feasibility_boundary(oracle, m, n, seed):
    """x_B components equal -1 and -2 exactly: n_feasible moves when eps_feas moves one ulp below 1 or 2."""
    A, b, c, mx = network(m, n, seed)
    for eps in (1.0, 2.0):
        at, _ = oracle.solve(A, b, c, mx, n_threads=NCPU, eps_feas=eps)
        below, _ = oracle.solve(A, b, c, mx, n_threads=NCPU, eps_feas=np.nextafter(eps, 0.0))
        assert at.n_feasible > below.n_feasible


def test_selfcheck_network_negative_zero_components(oracle):
    """With b >= 0, feasible bases at eps_feas = 0 have x_B components equal to -0.0."""
    A, b, c, mx = network(8, 20, 3, b_vals=(0, 1, 2))
    _, ranks, count = oracle.list_class(A, b, c, mx, FEASIBLE, n_threads=NCPU, eps_feas=0.0)
    assert count > 100
    neg_zero = 0
    for r in ranks:
        st, x, _ = oracle.eval_basis(A, b, c, mx, unrank(20, 8, r), eps_feas=0.0)
        assert st == FEASIBLE
        neg_zero += any(v == 0.0 and math.copysign(1.0, v) < 0 for v in x)
    assert neg_zero > 20


@pytest.mark.parametrize("name,floor", [("sparse_dyadic", 400), ("thirds", 400), ("signed_duplicates", 200)])
def test_selfcheck_pivot_ties(name, floor):
    """Exact ties for the maximum |pivot| are frequent (dense_lp has none)."""
    for m, n in ((8, 24), (12, 40)):
        A = FAMILIES[name](m, n, 1)[0]
        ties = sum(ge_ties(A, unrank(n, m, r)) for r in sample_ranks(n, m, 2000, 7))
        assert ties >= floor, (m, n, ties)
    A = lpgen.dense_lp(8, 24, 1)[0]
    assert sum(ge_ties(A, unrank(24, 8, r)) for r in sample_ranks(24, 8, 2000, 7)) == 0


def test_selfcheck_magnitudes(oracle):
    """Non-finite x_B (huge_rhs), infinite objectives of feasible bases (huge_cost: the optimum is a tie of -inf
    keys), subnormal x_B (tiny_rhs), and NaN objectives of all feasible bases (all_nan_keys)."""
    m, n = 8, 24
    seen = {"x_inf": 0, "x_nan": 0, "z_inf": 0, "x_sub": 0}
    for name in ("huge_rhs", "huge_cost", "tiny_rhs"):
        A, b, c, mx = FAMILIES[name](m, n, 1)
        for r in sample_ranks(n, m, 3000, 3):
            st, x, z = oracle.eval_basis(A, b, c, mx, unrank(n, m, r))
            if st == SINGULAR:
                continue
            x = np.array(x)
            if name == "huge_rhs":
                seen["x_inf"] += bool(np.isinf(x).any())
                seen["x_nan"] += bool(np.isnan(x).any())
            elif name == "huge_cost":
                seen["z_inf"] += st == FEASIBLE and math.isinf(z)
            else:
                seen["x_sub"] += bool(((x != 0) & (np.abs(x) < np.finfo(np.float64).tiny)).any())
    assert min(seen.values()) >= 10, seen
    o, _ = oracle.solve(*huge_cost(m, n, 1), n_threads=NCPU)
    assert o.status == _abi.OK and o.key == -math.inf
    for m, n in ((6, 15), (8, 24)):
        o, _ = oracle.solve(*all_nan_keys(m, n), n_threads=NCPU)
        assert o.status == _abi.NO_FEASIBLE and o.n_feasible > 0


def test_selfcheck_bulk_singular_prefixes(oracle):
    """signed_duplicates: the subtree of prefix (0, .., L-3, j1, j1+1) is singular as a whole for every prefix
    length L up to the child's (m - 4) — detected in the rebuild from A (L <= m - 7), at the node and parent
    steps (L = m - 6, m - 5) and at the child's pivot (L = m - 4)."""
    m, n = 10, 30
    A, b, c, mx = signed_duplicates(m, n, 1)
    j1, _ = dup_pairs(m)
    for L in range(2, m - 3):
        S = list(range(L - 2)) + [j1, j1 + 1]
        S += list(range(j1 + 2, j1 + 2 + m - L))
        lo = rank_of(n, m, S)
        size = math.comb(n - 1 - (j1 + 1), m - L)
        o, st = oracle.solve(A, b, c, mx, n_threads=NCPU, want_status=True, rank_begin=lo, rank_end=lo + size)
        assert size > 0 and (st == SINGULAR).all() and o.n_singular == size


# ---------------------------------------------------------------------------- GPU parity

def gpu_solve(A, b, c, mx, algo, rank_begin=0, rank_end=0, shard_index=0, shard_count=0, **opt):
    import simplexmethod_b200 as sm
    can = sm.Canonical(A, b, c, list(range(A.shape[0])), minimize=not mx)
    res = sm.EnumerationSolver(can, algo=algo, **opt).enumerate(rank_begin, rank_end, shard_index, shard_count)
    return _abi.Result.from_buffer_copy(bytes(res))


def both_algos_vs_oracle(oracle, A, b, c, mx, rank_begin=0, rank_end=0, shared_expected=True, **opt):
    m = A.shape[0]
    o, _ = oracle.solve(A, b, c, mx, n_threads=NCPU, rank_begin=rank_begin, rank_end=rank_end, **opt)
    out = []
    for algo in ALGOS:
        g = gpu_solve(A, b, c, mx, algo, rank_begin, rank_end, **opt)
        assert g.algo_used == (algo if shared_expected else _abi.ALGO_INDEPENDENT)
        assert_same(g, o, m)
        out.append(g)
    return o, out


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", SHAPES)
@pytest.mark.parametrize("name", sorted(FAMILIES))
def test_family_full_range(gpu_lib, oracle, name, m, n):
    """Every family at every shape, minimise and maximise, both kernel families against the oracle."""
    A, b, c, _ = FAMILIES[name](m, n, 1)
    for mx in (False, True):
        both_algos_vs_oracle(oracle, A, b, c, mx)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(6, 15), (8, 24), (12, 26)])
def test_all_nan_keys(gpu_lib, oracle, m, n):
    """Every feasible basis has a NaN objective: no optimum, yet n_feasible > 0 — on both sides."""
    A, b, c, mx = all_nan_keys(m, n)
    o, _ = both_algos_vs_oracle(oracle, A, b, c, mx)
    assert o.status == _abi.NO_FEASIBLE and o.n_feasible > 0


HEADLINE_TOTAL = 5586853480


def headline_windows():
    """Four 300 000-rank windows of C(40, 12): starting inside a large child task, starting inside a tail group
    (children whose column is among the last 11, pooled by k_shared), running from a child into a tail group, and
    the end of the range."""
    n, m = 40, 12
    inside_child = rank_of(n, m, [0, 2, 3, 5, 6, 7, 8, 9, 15, 21, 22, 23]) + 17
    tail_first = rank_of(n, m, [1, 2, 3, 4, 5, 6, 7, 29, 30, 31, 32, 33])
    inside_tail = rank_of(n, m, [0, 1, 3, 4, 6, 8, 9, 31, 32, 34, 36, 38]) + 3
    w = 300000
    return [(inside_child, inside_child + w), (inside_tail, inside_tail + w), (tail_first - w // 2, tail_first + w // 2),
            (HEADLINE_TOTAL - w, HEADLINE_TOTAL)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sparse_dyadic", "signed_duplicates"])
def test_headline_12_40_structured(gpu_lib, oracle, name):
    """m = 12, n = 40 (the kernel compiled for n = 40): k_shared == k_independent over all C(40,12) bases, every
    field of the record; the oracle on a 2e6-rank prefix and four windows; three interleaved shards merged."""
    A, b, c, mx = FAMILIES[name](12, 40, 1)
    ind = gpu_solve(A, b, c, mx, _abi.ALGO_INDEPENDENT)
    sh = gpu_solve(A, b, c, mx, _abi.ALGO_SHARED)
    assert ind.n_bases == HEADLINE_TOTAL and sh.algo_used == _abi.ALGO_SHARED
    assert ind.n_singular > 0 and ind.n_feasible > 0
    assert_same(sh, ind, 12)
    for lo, hi in [(0, 2000000)] + headline_windows():
        both_algos_vs_oracle(oracle, A, b, c, mx, lo, hi)
    parts = [gpu_solve(A, b, c, mx, _abi.ALGO_SHARED, shard_index=i, shard_count=3) for i in range(3)]
    assert_same(merged(parts), ind, 12)


@pytest.mark.gpu
@pytest.mark.parametrize("name,m,n", [("signed_duplicates", 8, 24), ("sparse_dyadic", 10, 30), ("thirds", 10, 30)])
def test_interleaved_shards_structured(gpu_lib, oracle, name, m, n):
    """Three interleaved shards of a structured LP (singular subtrees and ties cut by shard windows), merged."""
    A, b, c, mx = FAMILIES[name](m, n, 2)
    o, _ = oracle.solve(A, b, c, mx, n_threads=NCPU)
    assert o.n_singular > 0 and o.n_feasible > 0
    for algo in ALGOS:
        parts = [gpu_solve(A, b, c, mx, algo, shard_index=i, shard_count=3) for i in range(3)]
        assert_same(merged(parts), o, m)


@pytest.mark.gpu
def test_list_feasible_bases_structured(gpu_lib, oracle):
    """listFeasibleBases through k_shared (listing in drain2_fn) on data with ties == the oracle's feasible ranks."""
    import simplexmethod_b200 as sm
    A, b, c, mx = sparse_dyadic(8, 24, 1)
    o, want, count = oracle.list_class(A, b, c, mx, FEASIBLE, n_threads=NCPU)
    assert 0 < count == want.size
    s = sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(8)), minimize=not mx), algo=_abi.ALGO_SHARED)
    got = s.listFeasibleBases()
    assert s._res.algo_used == _abi.ALGO_SHARED
    assert got.tolist() == want.tolist() and s.feasibleCount() == o.n_feasible and s.bestRank() == o.best_rank


@pytest.mark.gpu
@pytest.mark.parametrize("name,m,n,seed,thr", THRESHOLD_CASES)
def test_pivot_threshold_boundary(gpu_lib, oracle, name, m, n, seed, thr):
    """eps_piv such that thr = eps_piv max|A| is hit exactly by some pivots, and its two neighbours."""
    A, b, c, mx = FAMILIES[name](m, n, seed)
    e = exact_eps_piv(A, thr)
    for eps in (e, np.nextafter(e, 0.0), np.nextafter(e, 1.0)):
        both_algos_vs_oracle(oracle, A, b, c, mx, eps_piv=float(eps))


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,seed", NETWORK_FEAS + [(12, 26, 3)])
def test_feasibility_boundary(gpu_lib, oracle, m, n, seed):
    """network LPs: x_B components exactly -1, -2 and -0.0 against eps_feas in {0, 1, 2} and their neighbours."""
    A, b, c, mx = network(m, n, seed)
    for eps in (1.0, 2.0):
        for e in (eps, np.nextafter(eps, 0.0), np.nextafter(eps, 4.0)):
            both_algos_vs_oracle(oracle, A, b, c, mx, eps_feas=float(e))
    A, b, c, mx = network(m, n, seed, b_vals=(0, 1, 2))
    for e in (0.0, -0.0, 5e-324):
        both_algos_vs_oracle(oracle, A, b, c, mx, eps_feas=e)


NEG_ZERO_CASES = [(8, 24, 0, 0), (10, 30, 0, 0), (9, 22, 0, 0),
                  (12, 40, 0, 2000000), (12, 40, 3000000000, 3000300000)]


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,lo,hi", NEG_ZERO_CASES)
def test_eps_feas_negative_zero(gpu_lib, oracle, m, n, lo, hi):
    """eps_feas = -0.0 is not < 0, so it asks for 0, not for the default: both kernel families must give the
    oracle's result, and the same as for +0.0.  (k_shared once took -(-0.0) = +0.0 as the bound of its leaf
    filter and dropped every basis with a positive leaf component.)"""
    A, b, c, mx = lpgen.dense_lp(m, n, 1)
    o, _ = oracle.solve(A, b, c, mx, n_threads=NCPU, rank_begin=lo, rank_end=hi, eps_feas=0.0)
    assert o.n_feasible > 0
    for algo in ALGOS:
        neg = gpu_solve(A, b, c, mx, algo, lo, hi, eps_feas=-0.0)
        pos = gpu_solve(A, b, c, mx, algo, lo, hi, eps_feas=0.0)
        assert neg.algo_used == algo
        assert_same(neg, o, m)
        assert_same(pos, o, m)


@pytest.mark.gpu
def test_eps_piv_negative_zero(gpu_lib, oracle):
    """eps_piv = -0.0 means a zero threshold, outside k_shared's range: the independent kernel runs, == oracle."""
    A, b, c, mx = sparse_dyadic(8, 24, 1)
    o, _ = both_algos_vs_oracle(oracle, A, b, c, mx, shared_expected=False, eps_piv=-0.0)
    assert o.n_singular > 0
