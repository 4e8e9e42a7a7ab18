"""The wide shapes: n = 41 to 64 and m = 6 to 16, on rank windows, bit for bit against the CPU oracle.

The header accepts n up to ENUMGPU_MAX_N = 64, and several paths are reached only there: the run-time-n
instantiations k_shared<M> for every M at n > 40, the survivor stacks at their largest (queue1_cap(n) = 32 (n - 3)
entries per warp, regrown by a handle made for n = 40), k_objectives' largest shared-memory configuration, k_certify's
widest slab and the largest binomials of unrank.  All of C(64, m) cannot be enumerated for most m, so the enumeration
tests run on rank windows that start where the shared kernel's work splits: the start of the space, inside a large
child task (all bases with the same first m - 4 columns), inside a tail group (the children of a parent whose column is
among the last kTailR = 11, which k_shared pools), across a child into a tail group, and the end of the space.

Without a GPU: self-checks that every window starts where its name says, has a child-aligned core that k_shared runs
on, that the pressure cases really fill the stacks, that the objectives case reaches its shared-memory size, and that
the LP families have singular and (at eps_feas = 3) many feasible bases in every window.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest

import simplexmethod_b200 as sm
from simplexmethod_b200 import _abi, lpgen
from test_certificate import assert_cert_bits, certify_basis, problem
from test_objectives import call_objectives, check_against_oracle, check_against_solves, cost_set, record_bytes
from test_optimal_duals import gpu_certify_bases, gpu_list_window, oracle_window, twin_certify_many
from test_structured_parity import (assert_same, bits, dup_pairs, gpu_solve, merged, rank_of, signed_duplicates,
                                    sparse_dyadic, unrank)

ALGOS = [_abi.ALGO_INDEPENDENT, _abi.ALGO_SHARED]
NCPU = os.cpu_count()
FEASIBLE, INFEASIBLE, SINGULAR = 0, 1, 2
KT = 4                 # k_shared's per-lane levels: a child task fixes the first m - 4 columns
KTAIL_R = 11           # k_shared's kTailR: children whose column is among the last 11 form their parent's tail group
PRESSURE = 1e300       # eps_feas under which every nonsingular basis is feasible: every leaf survives to the stacks

# one or two shapes for every m, n = 64 for m in {6, 7, 12, 14, 16}, odd n among them
SHAPES = [(6, 64), (7, 64), (8, 57), (9, 48), (10, 61), (11, 63), (12, 64), (13, 41), (14, 64), (15, 55), (16, 64)]


def sparse_dyadic_wide(m, n, seed):
    """sparse_dyadic with 30 % nonzeros.  The bases of a window share most of their first m - 4 columns, and at the
    family's default density of 50 % they are then almost never singular for m >= 12."""
    return sparse_dyadic(m, n, seed, density=0.3)


FAMILIES = {"dense_lp": lpgen.dense_lp, "sparse_dyadic": sparse_dyadic_wide, "signed_duplicates": signed_duplicates}
EPS_FEAS = [-1.0, 3.0, 10.0]        # -1: the default (1e-9)
W_MIN, W_MAX = 300_000, 2_000_000


# --------------------------------------------------------------------------------------------- windows

def piece_of(n, m, r):
    """The atomic piece of k_shared's work that holds rank r, as enqueue_range cuts the range: (first rank, size,
    tail).  A child task is every basis with the first P = m - 4 columns of r's basis; its first basis continues
    with the 4 columns after S[P-1].  If S[P-1] >= t0 = max(S[P-2] + 1, n - kTailR), the child belongs to the tail
    group of its parent: the children t0 .. n-5 together, starting with the basis (S[0..P-2], t0, .., t0 + 4)."""
    S = unrank(n, m, r)
    P = m - KT
    t0 = max(S[P - 2] + 1, n - KTAIL_R)
    if S[P - 1] >= t0:
        return rank_of(n, m, S[:P - 1] + list(range(t0, t0 + KT + 1))), math.comb(n - t0, KT + 1), True
    s = S[P - 1]
    return rank_of(n, m, S[:P] + list(range(s + 1, s + 1 + KT))), math.comb(n - 1 - s, KT), False


def core_pieces(n, m, lo, hi):
    """The pieces of the child-aligned core of [lo, hi): what k_shared runs; the rest goes to the independent
    kernel as ragged head and tail."""
    total = math.comb(n, m)
    f, c, _ = piece_of(n, m, lo)
    a = lo if f == lo else f + c
    b = hi if hi == total else piece_of(n, m, hi)[0]
    out = []
    while a < b:
        f, c, tail = piece_of(n, m, a)
        assert f == a
        out.append((f, c, tail))
        a += c
    return out


def spread(k):
    return [i + (i + 1) // 2 for i in range(k)]


def width_from(n, m, lo):
    """At least W_MIN ranks, and enough that the window's core holds two whole pieces."""
    f, c, _ = piece_of(n, m, lo)
    a = lo if f == lo else f + c
    for _ in range(2):
        a += piece_of(n, m, a)[1]
    return max(W_MIN, a - lo + 1)


def windows(m, n):
    """{name: (lo, hi)}: the start of the space, a window starting inside a large child task (17 ranks in), one
    starting inside a tail group (3 ranks in), one running from the children before a tail group into it, and the end
    of the space.  Widths between W_MIN and W_MAX, grown where the pieces are large."""
    total = math.comb(n, m)
    P = m - KT
    pre = spread(P)
    s = pre[-1]
    inside_child = rank_of(n, m, pre + [s + 3, s + 8, s + 9, s + 12]) + 17
    inside_tail = rank_of(n, m, spread(P - 1) + [n - 9, n - 8, n - 6, n - 4, n - 2]) + 3
    t0 = n - KTAIL_R
    tail_first = rank_of(n, m, list(range(1, P)) + list(range(t0, t0 + KT + 1)))
    out = {}
    for name, lo in (("start", 0), ("inside_child", inside_child), ("inside_tail", inside_tail)):
        out[name] = (lo, lo + width_from(n, m, lo))
    w = W_MIN
    out["child_into_tail"] = (tail_first - w // 2, tail_first + w // 2)
    out["end"] = (total - w, total)
    return out


# --------------------------------------------------------------------------------------------- oracle, cached

_ORACLE = {}


def lp_of(family, m, n):
    return FAMILIES[family](m, n, 1)


def oracle_result(oracle, family, m, n, lo, hi, eps_feas=-1.0, mx=None):
    """The oracle's record of [lo, hi) (hi = 0: the whole space); mx None: the family's own sense."""
    A, b, c, mx0 = lp_of(family, m, n)
    mx = mx0 if mx is None else mx
    key = (family, m, n, lo, hi, eps_feas, mx)
    if key not in _ORACLE:
        _ORACLE[key] = oracle.solve(A, b, c, mx, n_threads=NCPU, rank_begin=lo, rank_end=hi, eps_feas=eps_feas)[0]
    return _ORACLE[key]


# ---------------------------------------------------------------------------- self-checks (no GPU)

def test_selfcheck_shapes_cover_every_m():
    assert sorted({m for m, _ in SHAPES}) == list(range(6, 17))
    assert all(41 <= n <= 64 for _, n in SHAPES)
    assert {m for m, n in SHAPES if n == 64} >= {6, 7, 12, 14, 16}
    assert {(8, 57), (11, 63), (13, 41), (15, 55)} <= set(SHAPES)


def test_selfcheck_piece_of_matches_the_child_definition():
    """piece_of against a direct reading of the definition on sampled ranks: every basis of the piece shares the
    first P - 1 columns, the child's column S[P-1] (or, in a tail group, a column >= t0), and the piece is contiguous
    in rank order."""
    rng = np.random.default_rng(3)
    for m, n in SHAPES:
        P = m - KT
        total = math.comb(n, m)
        for r in [0, total - 1] + rng.integers(0, total, 20).tolist():
            f, c, tail = piece_of(n, m, r)
            assert f <= r < f + c
            S, F, L = unrank(n, m, r), unrank(n, m, f), unrank(n, m, f + c - 1)
            assert F[:P - 1] == L[:P - 1] == S[:P - 1]
            t0 = max(S[P - 2] + 1, n - KTAIL_R)
            if tail:
                assert F[P - 1] == t0 and L[P - 1] == n - KT - 1 and S[P - 1] >= t0
            else:
                assert F[P - 1] == L[P - 1] == S[P - 1] < t0
                assert L[P:] == list(range(n - KT, n))
            if f > 0:                                  # the piece before ends where this one starts
                assert piece_of(n, m, f - 1)[0] + piece_of(n, m, f - 1)[1] == f


@pytest.mark.parametrize("m,n", SHAPES)
def test_selfcheck_windows_start_where_named(m, n):
    total = math.comb(n, m)
    W = windows(m, n)
    assert set(W) == {"start", "inside_child", "inside_tail", "child_into_tail", "end"}
    for name, (lo, hi) in W.items():
        assert 0 <= lo < hi <= total and W_MIN <= hi - lo <= W_MAX, (name, lo, hi)
    assert W["start"][0] == 0 and W["end"][1] == total
    f, c, tail = piece_of(n, m, W["inside_child"][0])
    assert not tail and f < W["inside_child"][0] and c >= 1000          # strictly inside a child of 1000+ bases
    f, c, tail = piece_of(n, m, W["inside_tail"][0])
    assert tail and f < W["inside_tail"][0] < f + c
    lo, hi = W["child_into_tail"]
    pieces = core_pieces(n, m, lo, hi)
    first_tail = next(i for i, p in enumerate(pieces) if p[2])
    assert first_tail >= 1 and not pieces[first_tail - 1][2]            # whole children, then a tail group


@pytest.mark.parametrize("m,n", SHAPES)
def test_selfcheck_windows_have_a_core(m, n):
    """Every window's core holds at least two whole pieces (k_shared runs, the window is not all head and tail),
    and the shape has windows whose core holds a tail group."""
    with_tail = 0
    for name, (lo, hi) in windows(m, n).items():
        pieces = core_pieces(n, m, lo, hi)
        assert len(pieces) >= 2, name
        with_tail += any(t for _, _, t in pieces)
    assert with_tail >= 1


def largest_batch_push(n, m, s):
    """Stage-1 stack entries that one batch of 32 leaf items can push in child s (its column S[P-1] = s) when every
    leaf survives: items are the colex triples (a, b, c) of the child's columns s+1 .. n-1, and a triple has
    trips = n - 1 - c bases (the last column d runs over c+1 .. n-1)."""
    cols = range(s + 1, n)
    trips = [n - 1 - c for c in cols for b in range(s + 1, c) for a in range(s + 1, b)]     # colex: c, then b, then a
    return max(sum(trips[i:i + 32]) for i in range(0, len(trips), 32))


def queue1_cap(n):
    return 32 * (n - 3)


def test_selfcheck_pressure_fills_the_stacks():
    """Under eps_feas = 1e300 the first batch of child (0, 1) at (6, 64) pushes >= 90 % of queue1_cap(64) entries
    (the sizing leaves room for 31 more).  The pressure tests check n_infeasible == 0 on the oracle side."""
    push = largest_batch_push(64, 6, 1)
    assert 0.9 * queue1_cap(64) <= push <= queue1_cap(64) - 31
    assert push == 59 + 3 * 58 + 6 * 57 + 10 * 56 + 12 * 55


def objectives_smem(M, n, k):
    W = 1
    while W < k and W < 256:
        W *= 2
    return M * 256 * 9 + 256 * 8 + n * W * 8


def test_selfcheck_objectives_smem():
    assert objectives_smem(16, 64, OBJ_K) == 169984 >= 160 * 1024
    assert OBJ_K > 256 and OBJ_K % 256 != 0                             # two tiles, the second ragged


@pytest.mark.parametrize("m,n", SHAPES)
def test_selfcheck_families_in_every_window(oracle, m, n):
    """sparse_dyadic and signed_duplicates have singular bases in every window, dense_lp at most a handful.  At
    eps_feas = 3 every dense_lp window has feasible bases in the thousands, and so do at least three windows of each
    other family.  A signed_duplicates window is singular as a whole exactly where its bases start with the
    dependent pair (j1, j1 + 1) (the bulk-singular path)."""
    j1, _ = dup_pairs(m)
    for family in FAMILIES:
        many = 0
        for name, (lo, hi) in windows(m, n).items():
            o = oracle_result(oracle, family, m, n, lo, hi, eps_feas=3.0)
            assert o.n_bases == hi - lo
            many += o.n_feasible >= 1000
            if family == "dense_lp":
                assert o.n_singular <= 10 and o.n_feasible >= 1000, (name, o.n_singular, o.n_feasible)
            else:
                assert o.n_singular > 0, (family, name)
            if family == "signed_duplicates":
                pair = all({j1, j1 + 1} <= set(unrank(n, m, r)) for r in (lo, hi - 1))
                assert (o.n_singular == o.n_bases) == pair, name
        assert many >= 3, family


# ---------------------------------------------------------------------------- GPU: enumeration windows

def both_vs_oracle(o, A, b, c, mx, lo, hi, **opt):
    m = A.shape[0]
    for algo in ALGOS:
        g = gpu_solve(A, b, c, mx, algo, lo, hi, **opt)
        assert g.algo_used == algo
        assert_same(g, o, m)


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", SHAPES)
@pytest.mark.parametrize("family", sorted(FAMILIES))
def test_enumeration_windows(gpu_lib, oracle, family, m, n):
    """Every window, eps_feas in {default, 3, 10}, both senses for dense_lp: both kernel families == the oracle."""
    A, b, c, mx0 = lp_of(family, m, n)
    senses = (False, True) if family == "dense_lp" else (mx0,)
    for name, (lo, hi) in windows(m, n).items():
        for eps in EPS_FEAS:
            for mx in senses:
                o = oracle_result(oracle, family, m, n, lo, hi, eps_feas=eps, mx=mx)
                both_vs_oracle(o, A, b, c, mx, lo, hi, eps_feas=eps)


# ---------------------------------------------------------------------------- GPU: the stacks under pressure

@pytest.mark.gpu
def test_pressure_full_range_6_64(gpu_lib, oracle):
    """All C(64, 6) bases of dense (6, 64) with every nonsingular basis feasible."""
    A, b, c, mx = lp_of("dense_lp", 6, 64)
    o = oracle_result(oracle, "dense_lp", 6, 64, 0, 0, eps_feas=PRESSURE)
    assert o.n_bases == math.comb(64, 6) == 74974368 and o.n_infeasible == 0 and o.status == _abi.OK
    both_vs_oracle(o, A, b, c, mx, 0, 0, eps_feas=PRESSURE)


@pytest.mark.gpu
@pytest.mark.parametrize("m", range(7, 17))
def test_pressure_windows_n64(gpu_lib, oracle, m):
    """The windows of the smallest children (the largest pushes) and the end of the space, under pressure."""
    A, b, c, mx = lp_of("dense_lp", m, 64)
    W = windows(m, 64)
    for name in ("start", "inside_child", "end"):
        lo, hi = W[name]
        o = oracle_result(oracle, "dense_lp", m, 64, lo, hi, eps_feas=PRESSURE)
        assert o.n_infeasible == 0 and o.n_feasible > 0
        both_vs_oracle(o, A, b, c, mx, lo, hi, eps_feas=PRESSURE)


@pytest.mark.gpu
@pytest.mark.parametrize("shards", [3, 8])
def test_pressure_interleaved_shards(gpu_lib, oracle, shards):
    A, b, c, mx = lp_of("dense_lp", 12, 64)
    lo, hi = windows(12, 64)["start"]
    o = oracle_result(oracle, "dense_lp", 12, 64, lo, hi, eps_feas=PRESSURE)
    assert o.n_infeasible == 0
    for algo in ALGOS:
        parts = [gpu_solve(A, b, c, mx, algo, lo, hi, shard_index=i, shard_count=shards, eps_feas=PRESSURE)
                 for i in range(shards)]
        assert_same(merged(parts), o, 12)


# ---------------------------------------------------------------------------- GPU: listing

@pytest.mark.gpu
@pytest.mark.parametrize("m", [6, 16])
@pytest.mark.parametrize("case", ["pressure", "default"])
def test_list_window_wide(gpu_lib, oracle, case, m):
    """enumgpu_list_window with key bound +inf == the oracle's feasible ranks; a capacity below the count gives a
    subset, ascending, and the full count."""
    n = 64
    family, eps = ("dense_lp", PRESSURE) if case == "pressure" else ("sparse_dyadic", -1.0)
    A, b, c, mx = lp_of(family, m, n)
    lo, hi = windows(m, n)["inside_child"]
    want = oracle_window(oracle, A, b, c, mx, math.inf, rank_begin=lo, rank_end=hi, eps_feas=eps)
    assert want.size >= 50
    for algo in ALGOS:
        got, res = gpu_list_window(gpu_lib, A, b, c, mx, math.inf, algo, lo, hi, capacity=want.size + 7,
                                   eps_feas=eps)
        assert res.algo_used == algo and res.n_feasible == want.size
        assert got.tolist() == want.tolist()
        few, res = gpu_list_window(gpu_lib, A, b, c, mx, math.inf, algo, lo, hi, capacity=want.size // 3,
                                   eps_feas=eps)
        assert few.size == want.size // 3 and res.n_feasible == want.size
        assert set(few.tolist()) <= set(want.tolist()) and (np.diff(few.astype(np.int64)) > 0).all()


# ---------------------------------------------------------------------------- GPU: per-basis kernels

@pytest.mark.gpu
@pytest.mark.parametrize("family", ["dense_lp", "sparse_dyadic"])
def test_eval_ranks_16_64(gpu_lib, oracle, family):
    """enumgpu_eval_ranks at the largest binomials: sampled ranks of C(64, 16) ~ 4.9e14 and its last 64 ranks, the
    class of every basis, x_B and objective bits of every nonsingular one; enumgpu_eval_basis on some of them."""
    m, n = 16, 64
    A, b, c, mx = lp_of(family, m, n)
    total = math.comb(n, m)
    ranks = np.r_[np.random.default_rng(11).integers(0, total, 400, dtype=np.uint64),
                  np.arange(total - 64, total, dtype=np.uint64)]
    s = sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(m)), minimize=not mx))
    bases, xB, z, cls = s.evaluateBases(ranks)
    seen = {FEASIBLE: 0, INFEASIBLE: 0, SINGULAR: 0}
    keep, p = problem(A, b, c, mx)
    for i, r in enumerate(ranks):
        S = unrank(n, m, int(r))
        assert bases[i].tolist() == S
        st, xo, zo = oracle.eval_basis(A, b, c, mx, S)
        assert cls[i] == st, (i, int(r))
        seen[st] += 1
        if st != SINGULAR:
            assert [bits(v) for v in xB[i]] == [bits(v) for v in xo]
            assert bits(z[i]) == bits(zo)
        if i % 29 == 0 or i >= len(ranks) - 3:
            x, zz, cl = (C.c_double * m)(), C.c_double(), C.c_int32()
            assert gpu_lib.enumgpu_eval_basis(C.byref(p), None, (C.c_int32 * m)(*S), x, C.byref(zz), C.byref(cl)) == 0
            assert cl.value == st
            if st != SINGULAR:
                assert [bits(v) for v in x] == [bits(v) for v in xo] and bits(zz.value) == bits(zo)
    assert seen[INFEASIBLE] > 0
    if family == "sparse_dyadic":
        assert seen[SINGULAR] > 0


CERT_SHAPES = [(16, 64), (12, 64), (6, 64)]


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", CERT_SHAPES)
def test_certify_bases_wide(gpu_lib, oracle, m, n):
    """enumgpu_certify_bases on every feasible basis of a window at eps_feas = 3 == the certificate twin, bit for
    bit, ray included: dense_lp minimised (undecided verdicts) and maximised, and signed_duplicates maximised (edge
    rays); at (16, 64) the signed_duplicates call takes three launches of at most 4096 bases."""
    lo, hi = cert_window(m, n)
    seen = set()
    for family, mx in (("dense_lp", False), ("dense_lp", True), ("signed_duplicates", True)):
        A, b, c, _ = lp_of(family, m, n)
        ranks = oracle_window(oracle, A, b, c, mx, math.inf, rank_begin=lo, rank_end=hi, eps_feas=3.0)
        assert ranks.size > 1000
        bases = [unrank(n, m, int(r)) for r in ranks]
        got = gpu_certify_bases(gpu_lib, A, b, c, mx, bases, eps_feas=3.0)
        rcs, want = twin_certify_many(A, b, c, mx, bases, eps_feas=3.0)
        assert (rcs == _abi.OK).all()
        for g, w in zip(got, want):
            assert w.basis_class == _abi.BASIS_FEASIBLE
            assert_cert_bits(g, w)
            assert [bits(v) for v in g.ray] == [bits(v) for v in w.ray]
            seen.add(w.status)
        rc, one = certify_basis(A, b, c, mx, bases[-1], eps_feas=3.0)       # the single-basis twin agrees
        assert rc == _abi.OK
        assert_cert_bits(got[-1], one)
        if (m, n) == (16, 64) and family == "signed_duplicates":
            assert len(bases) > 2 * 4096
    assert seen == {_abi.CERT_UNDECIDED, _abi.CERT_UNBOUNDED}


def cert_window(m, n):
    lo = windows(m, n)["inside_child"][0]
    return lo, lo + (40_000 if m >= 12 else 20_000)


# ---------------------------------------------------------------------------- GPU: objectives

OBJ_K = 300


@pytest.mark.gpu
@pytest.mark.parametrize("m", [16, 6])
def test_objectives_largest_smem(gpu_lib, oracle, m):
    """k = 300 cost vectors (tiles of 256: the second one ragged) at n = 64: every checked out[i] == enumgpu_solve
    with c = column i, raw bytes; four columns == the oracle; a max_list below the feasible count splits the range
    and gives the same records."""
    n = 64
    A, b, c, mx = lp_of("dense_lp", m, n)
    lo, hi = cert_window(m, n)
    costs = cost_set(A, c, n_random=OBJ_K - 11, seed=m)
    assert costs.shape == (OBJ_K, n)
    opt = dict(rank_begin=lo, rank_end=hi, eps_feas=3.0)
    rc, res = call_objectives(gpu_lib, A, b, costs, mx, **opt)
    assert rc == _abi.OK, sm.last_error()
    nf = int(res[0].n_feasible)
    assert nf > 500
    pick = list(range(0, 11)) + [20, 100, 255, 256, 257, 280, 297, 298, OBJ_K - 1]      # OBJ_K - 1: the +-2^1021 column
    pick += list(range(30, 256, 37))
    assert len(pick) >= 24
    check_against_solves(gpu_lib, A, b, costs[pick], mx, [res[i] for i in pick], **opt)
    four = [1, 5, 256, OBJ_K - 1]
    check_against_oracle(oracle, A, b, costs[four], mx, [res[i] for i in four], **opt)
    rc, split = call_objectives(gpu_lib, A, b, costs, mx, max_list=nf // 3, **opt)
    assert rc == _abi.OK
    assert [record_bytes(r) for r in split] == [record_bytes(r) for r in res]
    assert split[0].n_launches > res[0].n_launches


# ---------------------------------------------------------------------------- GPU: one raw handle across widths

def handle_cases(oracle):
    """(LP, options, oracle record): n = 24, then (12, 64) under pressure (the stacks regrow past the handle's n = 40
    reservation), then n = 41, then n = 64 again at the default tolerance."""
    cases = []
    for family, m, n, window, eps in (("dense_lp", 8, 24, None, -1.0), ("dense_lp", 12, 64, "start", PRESSURE),
                                      ("sparse_dyadic", 13, 41, "child_into_tail", -1.0),
                                      ("signed_duplicates", 16, 64, "inside_child", -1.0)):
        lo, hi = (0, 0) if window is None else windows(m, n)[window]
        A, b, c, mx = lp_of(family, m, n)
        o = oracle_result(oracle, family, m, n, lo, hi, eps_feas=eps)
        cases.append(((A, b, c, mx), _abi.Options(eps, -1.0, lo, hi, 0, _abi.ALGO_SHARED, None, None, 0, 0, 0, 0), o))
    return cases


@pytest.mark.gpu
def test_one_handle_across_widths(gpu_lib, oracle):
    h = C.c_void_p()
    assert gpu_lib.enumgpu_create(-1, C.byref(h)) == 0, sm.last_error()
    try:
        for (A, b, c, mx), opt, o in handle_cases(oracle):
            keep, p = problem(A, b, c, mx)
            res = _abi.Result()
            assert gpu_lib.enumgpu_solve_h(h, C.byref(p), C.byref(opt), C.byref(res)) == o.status, sm.last_error()
            assert res.algo_used == _abi.ALGO_SHARED
            assert_same(res, o, A.shape[0])
    finally:
        gpu_lib.enumgpu_destroy(h)


@pytest.mark.gpu
def test_one_handle_across_widths_enqueue_host(gpu_lib, oracle):
    """The same sequence through enumgpu_enqueue_host_h on a caller-owned torch stream."""
    import torch
    h = C.c_void_p()
    assert gpu_lib.enumgpu_create(-1, C.byref(h)) == 0, sm.last_error()
    try:
        side = torch.cuda.Stream()
        for (A, b, c, mx), opt, o in handle_cases(oracle):
            keep, p = problem(A, b, c, mx)
            opt.stream = side.cuda_stream
            buf = torch.zeros(C.sizeof(_abi.Partial), dtype=torch.uint8, device="cuda")
            torch.cuda.synchronize()
            nl = C.c_int32()
            assert gpu_lib.enumgpu_enqueue_host_h(h, C.byref(p), C.byref(opt), buf.data_ptr(), C.byref(nl)) == 0, \
                sm.last_error()
            side.synchronize()
            rec = _abi.Partial.from_buffer_copy(buf.cpu().numpy().tobytes())
            res = _abi.Result()
            gpu_lib.enumgpu_partial_to_result(C.byref(rec), C.byref(res))
            assert res.algo_used == _abi.ALGO_SHARED
            assert_same(res, o, A.shape[0])
    finally:
        gpu_lib.enumgpu_destroy(h)
