"""Parity against the REFERENCE'S OWN CODE: the original SimplexMethod project's sources —
src/ProblemTypes/{Canonical,Symmetrical,Common}.cpp, src/SymmetricalParser.cpp, src/SimplexSolover.h.

Every test compares this project's code with tests/golden/reference_outputs.json: the original's outputs for
these inputs, for every quantity compared exactly (see tests/golden/make_reference_goldens.py for where they come
from).  Where the original is available — oracle/_ref/libsimplexref.so, built by ``make -C oracle ref`` from the
sources SIMPLEX_REFERENCE points at, with oracle/eigen_shim standing in for Eigen (NOT Eigen: the control flow,
tolerances and conversions are the reference's, the LU/QR underneath are the shim's) — the tests also compare
with it live, which checks the stored outputs too.

  * conversions and parser: the host types of this repo must reproduce the reference's outputs exactly;
  * per basis: Canonical::GetBasicSolution / IsFeasibleBasis / Evaluate (Householder QR) against the
    oracle's frozen partial-pivot GE — x and z within 1e-9 relative, same class (live only);
  * the enumeration path composed from those primitives (ref_enumerate: what EnumerationSolver would be,
    SURVEY 3.3) against the oracle and, on the GPU, against libenumgpu: identical class of every basis,
    optimal basis and counts; objective and x within 1e-9 relative (live) — the north star's parity statement;
  * the reference's simplex Solver against the enumeration optimum (README.md:42; live only).
"""
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import simplexmethod_b200 as sm
from simplexmethod_b200 import Common, ConstraintType as CT, Symmetrical, SymmetricalParser, VariableType as VT, lpgen
from oracle import simplexref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP = os.path.join(ROOT, "simplexmethod_b200", "cpp")
GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_outputs.json")
with open(GOLDEN) as f:
    GOLD = json.load(f)
LIVE = R.available()
live_only = pytest.mark.skipif(not LIVE, reason="compares with the original SimplexMethod code at run time: build "
                                                "oracle/_ref from its sources (SIMPLEX_REFERENCE=<checkout>)")
REL = 1e-9          # north star: objective and x within 1e-9 relative

TINY = {"lab_symmetric": lpgen.lab_symmetric_canonical, "main_cpp": lpgen.main_cpp_canonical,
        "test_canonical": lpgen.test_canonical_fixture, "beale": lpgen.beale_lp, "readme_shaped": lpgen.readme_shaped_lp}
DENSE = [(4, 12, 1), (6, 16, 1), (6, 16, 2), (6, 16, 3), (8, 24, 1)]
HEADLINE_WINDOWS = [(826_255_000, 826_267_000), (5_586_850_000, 5_586_853_480)]


def close(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return np.all(np.abs(a - b) <= REL * np.maximum(1.0, np.maximum(np.abs(a), np.abs(b))))


def problem_dict(mine) -> dict:
    """This project's problem object in the form oracle/simplexref.py returns the reference's."""
    d = {"A": np.asarray(mine.GetConstraintsMatrix()).tolist(), "b": np.asarray(mine.GetRightHandSide()).tolist(),
         "c": np.asarray(mine.GetObjectiveCoefficients()).tolist(), "maximize": bool(mine.IsMaximization())}
    if isinstance(mine, Common):
        d.update(kind=R.COMMON, row_types=[t.value for t in mine.GetConstraintTypes()],
                 var_types=[t.value for t in mine.GetVariableTypes()])
    elif isinstance(mine, Symmetrical):
        d.update(kind=R.SYMMETRICAL)
    else:
        d.update(kind=R.CANONICAL, basis=list(mine.GetBasisIndices()), n_orig=mine.GetOriginalVariablesCount())
    return d


def same_problem(ref: dict, mine):
    assert np.array_equal(ref["A"], np.asarray(mine.GetConstraintsMatrix()))
    assert np.array_equal(ref["b"], mine.GetRightHandSide()) and np.array_equal(ref["c"], mine.GetObjectiveCoefficients())
    assert ref["maximize"] == mine.IsMaximization()
    if ref["kind"] == R.COMMON:
        assert ref["row_types"] == [t.value for t in mine.GetConstraintTypes()]
        assert ref["var_types"] == [t.value for t in mine.GetVariableTypes()]
    if ref["kind"] == R.CANONICAL:
        assert ref["basis"] == list(mine.GetBasisIndices()) and ref["n_orig"] == mine.GetOriginalVariablesCount()


def status_sha256(status) -> str:
    return hashlib.sha256(np.ascontiguousarray(status, dtype=np.uint8).tobytes()).hexdigest()


def enumeration_record(res, status, m, winner=True) -> dict:
    """What the composed enumeration's record says, in the form stored in the golden file."""
    rec = {"status": res.status, "n_bases": res.n_bases, "counts": [res.n_singular, res.n_infeasible, res.n_feasible],
           "class_sha256": status_sha256(status)}
    if winner:
        rec.update(best_rank=res.best_rank, basis=list(res.basis)[:m])
    return rec


# ---- host types and parser reproduce the reference's conversions exactly -----------------------

def conversion_cases(seed):
    """(label, kind, op, A, b, c, maximize, reference keywords, this project's converted problem) for one seed."""
    rng = np.random.default_rng(100 + seed)
    m, n = int(rng.integers(1, 6)), int(rng.integers(1, 6))
    A = rng.integers(-9, 10, size=(m, n)).astype(float)
    b, c = rng.integers(-9, 10, size=m).astype(float), rng.integers(-9, 10, size=n).astype(float)
    rt, vt = rng.integers(0, 3, size=m).tolist(), rng.integers(0, 3, size=n).tolist()
    for mx in (True, False):
        com = Common(A, b, c, [CT(t) for t in rt], [VT(t) for t in vt], mx)
        kw = dict(row_types=rt, var_types=vt)
        yield f"{mx}/common/to_symmetrical", R.COMMON, R.TO_SYMMETRICAL, A, b, c, mx, kw, com.ToSymmetrical()
        yield f"{mx}/common/to_canonical", R.COMMON, R.TO_CANONICAL, A, b, c, mx, kw, com.ToCanonical()
        yield f"{mx}/common/dual", R.COMMON, R.GET_DUAL, A, b, c, mx, kw, com.GetDual()
        sym = Symmetrical(A, b, c, mx)
        yield f"{mx}/symmetrical/to_canonical", R.SYMMETRICAL, R.TO_CANONICAL, A, b, c, mx, {}, sym.ToCanonical()
        yield f"{mx}/symmetrical/to_common", R.SYMMETRICAL, R.TO_COMMON, A, b, c, mx, {}, sym.ToCommon()
        yield f"{mx}/symmetrical/dual", R.SYMMETRICAL, R.GET_DUAL, A, b, c, mx, {}, sym.GetDual()
        if m <= n:
            basis = sorted(rng.choice(n, size=m, replace=False).tolist())
            n_orig = int(rng.integers(1, n + 1))
            can = sm.Canonical(A, b, c, basis, minimize=not mx)
            can.SetOriginalVariablesCount(n_orig)
            kw = dict(basis=basis, n_orig=n_orig)
            yield f"{mx}/canonical/dual", R.CANONICAL, R.GET_DUAL, A, b, c, mx, kw, can.GetDual()
            yield f"{mx}/canonical/to_common", R.CANONICAL, R.TO_COMMON, A, b, c, mx, kw, can.ToCommon()
            yield f"{mx}/canonical/to_symmetrical", R.CANONICAL, R.TO_SYMMETRICAL, A, b, c, mx, kw, can.ToSymmetrical()


@pytest.mark.parametrize("seed", range(10))
def test_conversions_equal_the_reference(seed):
    want = GOLD["conversions"][str(seed)]
    labels = []
    for label, kind, op, A, b, c, mx, kw, mine in conversion_cases(seed):
        labels.append(label)
        same_problem(want[label], mine)
        if LIVE:
            same_problem(R.convert(kind, op, A, b, c, mx, **kw), mine)
    assert sorted(labels) == sorted(want)


def test_constructor_errors_like_the_reference():
    A = np.ones((2, 3))
    with pytest.raises(ValueError):
        sm.Canonical(A, [1, 2], [1, 2, 3], [0, 1]).SetOriginalVariablesCount(4)
    with pytest.raises(ValueError):
        sm.Canonical(A, [1, 2], [1, 2, 3], [0, 7])
    assert GOLD["constructor_errors"] == {"n_orig_out_of_range": "rejected", "basis_index_out_of_range": "rejected"}
    if LIVE:
        with pytest.raises(RuntimeError):       # n_orig out of range (Canonical.cpp:156-163)
            R.convert(R.CANONICAL, R.GET_DUAL, A, [1, 2], [1, 2, 3], False, basis=[0, 1], n_orig=4)
        with pytest.raises(RuntimeError):       # basis index out of range (Canonical.cpp:40-46)
            R.convert(R.CANONICAL, R.GET_DUAL, A, [1, 2], [1, 2, 3], False, basis=[0, 7], n_orig=3)


PARSER_TEXTS = [
    "\n  maximize\n\n objective:\n 3 5\n\n constraints:\n 1 2 10\n 3 4 20\n",
    "minimize\nobjective:\n7 8\nsubject to:\n1 1 5\n2 3 12\n",
    "# c\nmax\nobjective:\n1 2 3  # more\nconstraints:\n1 0 0 5 # a\r\n0 1 0 6\r\n0 0 1 7\r\n",
    "min\nobjective\n1.5 -2e1\n.5 4\nconstraints\n1 2 3 4 5\n",          # objective over two lines
    "maximize\n# nothing else\n",
    "1 2 3\n",
    "max\nobjective:\n1 2\nconstraints:\n1 2 3 4\n",
    "max\nobjective:\n1 2\nconstraints:\n7\n",
    "max\nobjective:\n1 x 2\nconstraints:\n1 2 3\n",
    open(os.path.join(ROOT, "tests", "golden", "lab_lp_symmetric.txt")).read(),
]


@pytest.mark.parametrize("k", range(len(PARSER_TEXTS)))
def test_parser_equals_the_reference(k):
    text = PARSER_TEXTS[k]
    mine = SymmetricalParser().ParseFromString(text)
    for ref in [GOLD["parser"][k]] + ([R.parse(text)] if LIVE else []):
        assert (ref is None) == (mine is None)
        if ref is not None:
            same_problem(ref, mine)


def print_fixture():
    """The three forms of test_print_layouts_equal_the_reference: (reference kind, A, b, c, maximize, keywords, ours)."""
    A = np.array([[1, -2, 0.5], [0, 4, -6], [7, 8.25, 9]])
    b, c = np.array([10, -11, 1e-7]), np.array([1.0, -2.0, 0.0])
    rt, vt = [0, 1, 2], [0, 1, 2]
    Ac, bc, cc = np.array([[1, -2, 1, 0], [3, 4.5, 0, 1]]), np.array([5.0, 6.0]), np.array([7.0, -8.0, 0.0, 0.0])
    can = sm.Canonical(Ac, bc, cc, [2, 3], minimize=False)
    can.SetOriginalVariablesCount(2)
    return [(R.COMMON, A, b, c, False, dict(row_types=rt, var_types=vt),
             Common(A, b, c, [CT(t) for t in rt], [VT(t) for t in vt], False)),
            (R.SYMMETRICAL, A, b, c, True, {}, Symmetrical(A, b, c, True)),
            (R.SYMMETRICAL, A, b, c, False, {}, Symmetrical(A, b, c, False)),
            (R.CANONICAL, Ac, bc, cc, True, dict(basis=[2, 3], n_orig=2), can)]


def test_print_layouts_equal_the_reference():
    """IProblem::Print() of the three forms: the Python mirror and the C++ host types (cpp/tests/host_tests --print)
    write the reference's text character for character (Common.cpp:86-137, Symmetrical.cpp:70-97, Canonical.cpp:88-123)."""
    fixture = print_fixture()
    want = GOLD["print"]
    if LIVE:
        assert [R.print_problem(kind, A, b, c, mx, **kw) for kind, A, b, c, mx, kw, _ in fixture] == want
    assert [mine.PrintText() for *_, mine in fixture] == want
    assert "1*x1-2*x2 + 0*x3" in want[0] and "0x1 + 4x2-6x3>=-11" in want[0] and "x1: ∈R" in want[0]      # what the layout looks like
    subprocess.check_call(["make", "-C", CPP, "-s"])
    out = subprocess.run([os.path.join(CPP, "build", "host_tests"), "--print"], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.split("---\n") == want


FUZZ_WORDS = ["maximize", "max", "minimize", "min", "objective:", "objective", "constraints:", "constraints", "subject to:",
              "subject to", "", "# note", "1 2 3", "4 5 6 7", "1.5 -2 3e1", "0 0", "7", "1 2 # tail", "  3   4  ", "x 1 2",
              "1 x 2", "-1 -2 -3", ".5 .25 8", "1e-3 2 3 4", "maximise", "Objective:", "2 3"]


def fuzz_texts():
    """150 seeded line soups from the format's vocabulary, a good share of them well-formed."""
    rng = np.random.default_rng(3)
    texts = []
    for k in range(150):
        lines = [FUZZ_WORDS[i] for i in rng.integers(0, len(FUZZ_WORDS), size=int(rng.integers(0, 10)))]
        if k % 3 == 0:                                      # make a good share of them well-formed
            rows4 = ["4 5 6 7", "1e-3 2 3 4", "1 2 3 4 # c", "-1 -2 -3 9", "  0 0 1 .5"]
            lines = ["max" if k % 2 else "minimize", "objective:", "1 2 3", "constraints:"] + \
                    [rows4[i] for i in rng.integers(0, len(rows4), size=int(rng.integers(1, 5)))] + (lines[:1] if k % 9 == 0 else [])
        texts.append("\n".join(lines) + "\n")
    return texts


def parse_line(line):
    """One line of cpp/tests/host_tests --parse: "null" or "maximize m n A(row-major) b c" -> dict like R.parse's."""
    if line == "null":
        return None
    v = [float(t) for t in line.split()]
    m, n = int(v[1]), int(v[2])
    return {"kind": R.SYMMETRICAL, "maximize": bool(v[0]), "A": np.reshape(v[3:3 + m * n], (m, n)).tolist(),
            "b": v[3 + m * n:3 + m * n + m], "c": v[3 + m * n + m:]}


def test_parser_fuzz_equals_the_reference():
    """Seeded line soups from the format's vocabulary: the Python parser accepts, rejects and reads exactly what the
    reference's parser does; live, also random soups drawn by hypothesis (the C++ parser shares its structure and is
    checked on the same soups below)."""
    texts, want = fuzz_texts(), GOLD["parser_fuzz"]
    assert len(want) == len(texts) and sum(w is not None for w in want) >= 20
    for text, ref in zip(texts, want):
        mine = SymmetricalParser().ParseFromString(text)
        assert (ref is None) == (mine is None), text
        if ref is not None:
            same_problem(ref, mine)
    if not LIVE:
        return
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=400, deadline=None)
    @given(st.lists(st.sampled_from(FUZZ_WORDS), min_size=0, max_size=9), st.sampled_from(["\n", "\r\n"]))
    def check(lines, eol):
        text = eol.join(lines) + eol
        ref, mine = R.parse(text), SymmetricalParser().ParseFromString(text)
        assert (ref is None) == (mine is None), text
        if ref is not None:
            same_problem(ref, mine)

    check()


def test_cpp_parser_fuzz_equals_the_reference(tmp_path):
    """The same soups through the C++ parser (cpp/tests/host_tests --parse): 150 files in one process."""
    texts, files = fuzz_texts(), []
    for k, text in enumerate(texts):
        files.append(tmp_path / f"lp{k}.txt")
        files[-1].write_text(text)
    subprocess.check_call(["make", "-C", CPP, "-s"])
    out = subprocess.run([os.path.join(CPP, "build", "host_tests"), "--parse"] + [str(f) for f in files], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    got = out.stdout.splitlines()
    assert len(got) == len(texts)
    n_ok = 0
    for text, line, ref in zip(texts, got, GOLD["parser_fuzz"]):
        assert parse_line(line) == ref, text
        if LIVE:
            live, mine = R.parse(text), parse_line(line)
            assert (live is None) == (mine is None), text
            if live is not None:
                assert live["maximize"] == mine["maximize"] and np.array_equal(live["A"], mine["A"])
                assert np.array_equal(live["b"], mine["b"]) and np.array_equal(live["c"], mine["c"])
        n_ok += ref is not None
    assert n_ok >= 20


# ---- per basis: the reference's QR-based primitives vs the oracle's frozen GE --------------------

@live_only
@pytest.mark.parametrize("name", sorted(TINY))
def test_per_basis_primitives_vs_oracle_tiny(oracle, name):
    from itertools import combinations
    A, b, c, mx = TINY[name]()
    m, n = A.shape
    for S in combinations(range(n), m):
        st, xo, zo = oracle.eval_basis(A, b, c, mx, list(S))
        if st == oracle.SINGULAR:
            continue                       # GetBasicSolution has no singularity test (Canonical.cpp:179-197); ref_enumerate covers it
        x, feas, z = R.basic_solution(A, b, c, list(S), minimize=not mx)
        assert close(x[list(S)], xo) and close(z, zo)
        assert feas == (st == oracle.FEASIBLE)
        assert np.count_nonzero(np.delete(x, list(S))) == 0


@live_only
def test_per_basis_primitives_vs_oracle_dense_sample(oracle):
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    rng = np.random.default_rng(7)
    for _ in range(300):
        S = sorted(rng.choice(40, size=12, replace=False).tolist())
        st, xo, zo = oracle.eval_basis(A, b, c, mx, S)
        x, feas, z = R.basic_solution(A, b, c, S, minimize=not mx)
        assert st != oracle.SINGULAR and close(x[S], xo) and close(z, zo)
        if min(xo) < -1e-8 or min(xo) > -1e-10:          # away from the -1e-9 boundary the classes must agree
            assert feas == (st == oracle.FEASIBLE)


# ---- the composed enumeration path vs the oracle ------------------------------------------------

def _compare(res_ref, res, m, exact_counts=True):
    assert res_ref.status == res.status
    assert list(res_ref.basis)[:m] == list(res.basis)[:m] and res_ref.best_rank == res.best_rank
    if res.status == 0:
        assert close(res_ref.objective, res.objective) and close(list(res_ref.x_B)[:m], list(res.x_B)[:m])
    assert res_ref.n_bases == res.n_bases
    if exact_counts:
        assert (res_ref.n_singular, res_ref.n_infeasible, res_ref.n_feasible) == (res.n_singular, res.n_infeasible, res.n_feasible)


@pytest.mark.parametrize("name", sorted(TINY))
def test_reference_enumeration_vs_oracle_tiny(oracle, name):
    A, b, c, mx = TINY[name]()
    res, st = oracle.solve(A, b, c, mx, want_status=True)
    assert enumeration_record(res, st, A.shape[0]) == GOLD["enumeration"][f"tiny/{name}"]    # class of every basis too
    if LIVE:
        ref, st_ref = R.enumerate_bases(A, b, c, mx, want_status=True)
        assert np.array_equal(st_ref, st)                     # class of every basis, singular ones included
        _compare(ref, res, A.shape[0])


@pytest.mark.parametrize("m,n,seed", DENSE)
def test_reference_enumeration_vs_oracle_dense(oracle, m, n, seed):
    A, b, c, mx = lpgen.dense_lp(m, n, seed)
    res, st = oracle.solve(A, b, c, mx, n_threads=4, want_status=True)
    assert enumeration_record(res, st, m) == GOLD["enumeration"][f"dense/{m}_{n}_{seed}"]
    if LIVE:
        ref, st_ref = R.enumerate_bases(A, b, c, mx, want_status=True)
        assert np.array_equal(st_ref, st)
        _compare(ref, res, m)


def small_degenerate_lp(seed, m=5, n=13):
    """Small-integer LP with duplicated, scaled and summed columns (exactly singular bases), a right-hand side built
    from a vertex with only m-2 positive components (degenerate vertices) and tied costs (exact ties at the optimum)."""
    rng = np.random.default_rng(seed)
    A = rng.integers(-3, 4, size=(m, n)).astype(float)
    A[:, n - 1] = A[:, 0]; A[:, n - 2] = 2 * A[:, 1]; A[:, n - 3] = A[:, 2] + A[:, 3]
    x0 = np.zeros(n)
    x0[rng.choice(n - 3, size=m - 2, replace=False)] = rng.integers(1, 4, size=m - 2)
    c = rng.integers(-4, 5, size=n).astype(float)
    c[n - 1] = c[0]; c[n - 2] = 2 * c[1]
    return np.asfortranarray(A), A @ x0, c, bool(seed % 2)


@pytest.mark.parametrize("seed", range(24))
def test_degenerate_lps_classes_agree_ties_may_not(oracle, seed):
    """Degenerate LPs: the class of every basis (hundreds of exactly singular ones) and all counters agree with the
    reference's code.  The winner need not: tied vertices have objectives that differ in the last bits, differently
    under Householder QR (reference) and partial-pivot GE (frozen arithmetic), so 'first strict improvement' lands on
    different members of the tie — the north star asks for the identical basis on non-degenerate problems only.
    Both winners are optimal to 1e-9 (checked live); GPU and oracle share one arithmetic and agree exactly
    (test_gpu_parity)."""
    A, b, c, mx = small_degenerate_lp(seed)
    res, st = oracle.solve(A, b, c, mx, want_status=True)
    assert res.n_singular > 100
    assert enumeration_record(res, st, A.shape[0], winner=False) == GOLD["enumeration"][f"degenerate/{seed}"]
    if not LIVE:
        return
    ref, st_ref = R.enumerate_bases(A, b, c, mx, want_status=True)
    assert np.array_equal(st_ref, st)
    assert (ref.n_singular, ref.n_infeasible, ref.n_feasible) == (res.n_singular, res.n_infeasible, res.n_feasible)
    assert ref.status == res.status
    if res.status == 0:
        assert close(ref.objective, res.objective)
        # each side's winner, evaluated by the other side, is a tie
        st_o, x_o, z_o = oracle.eval_basis(A, b, c, mx, list(ref.basis)[:A.shape[0]])
        assert st_o == oracle.FEASIBLE and close(z_o, res.objective)


def test_reference_enumeration_vs_oracle_headline_window(oracle):
    """m=12, n=40: 12 000 ranks around the optimum (rank 826 261 626) and a window of the densest region."""
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    for lo, hi in HEADLINE_WINDOWS:
        res, st = oracle.solve(A, b, c, mx, want_status=True, rank_begin=lo, rank_end=hi)
        assert enumeration_record(res, st, 12) == GOLD["enumeration"][f"headline/{lo}_{hi}"]
        if LIVE:
            ref, st_ref = R.enumerate_bases(A, b, c, mx, want_status=True, rank_begin=lo, rank_end=hi)
            assert np.array_equal(st_ref, st)
            _compare(ref, res, 12)


def test_headline_singular_bases_reference_vs_both_rules(oracle):
    """The 9 bases of dense(12,40,1) that the default ABSOLUTE pivot rule rejects (|pivot| <= 1e-9 max|A|; their
    condition numbers are 3e10..3e11): the ONLY ranks of the headline LP where the rule can disagree with the
    reference's Solver::computeBFS test, FullPivLU::isInvertible (SimplexSolover.h:124-126, relative threshold
    eps*m).  Asked one by one: the reference's own code says NOT singular -> infeasible (x_B ~ -1e9); so does
    ENUMGPU_PIVOT_RELATIVE; the absolute rule says singular.  n_feasible and the optimum are the same under
    both; only 9 bases move between n_singular and n_infeasible (DESIGN.md section 2)."""
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "dense_12_40_seed1.json")))
    ranks = g["singular_ranks"]
    assert len(ranks) == g["n_singular"] == 9
    assert GOLD["headline_singular_ranks"] == {"ranks": ranks, "class": "infeasible", "counts": [0, 1]}
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    import ctypes as C
    S = (C.c_int32 * 12)()
    for r in ranks:
        assert sm.lib().enumgpu_unrank(40, 12, r, S) == 0
        basis = list(S)
        assert 1e10 < np.linalg.cond(A[:, basis]) < 1e12
        assert oracle.eval_basis(A, b, c, mx, basis)[0] == oracle.SINGULAR                       # absolute rule
        st_rel, x_rel, _ = oracle.eval_basis(A, b, c, mx, basis, pivot_rule=1)                   # Eigen-like rule
        assert st_rel == oracle.INFEASIBLE and min(x_rel) < -1e8
        if LIVE:
            ref, st_ref = R.enumerate_bases(A, b, c, mx, want_status=True, rank_begin=r, rank_end=r + 1)
            assert st_ref.tolist() == [oracle.INFEASIBLE] and (ref.n_singular, ref.n_infeasible) == (0, 1)
        # a 1-rank window of the oracle enumeration under each rule says the same as eval_basis; under the
        # relative rule it gives the reference's counts
        for rule, want in ((0, [1, 0]), (1, GOLD["headline_singular_ranks"]["counts"])):
            o, _ = oracle.solve(A, b, c, mx, rank_begin=r, rank_end=r + 1, pivot_rule=rule)
            assert [o.n_singular, o.n_infeasible] == want


# ---- the reference's simplex Solver vs the enumeration optimum (README.md:42) -------------------

@live_only
@pytest.mark.parametrize("case", ["lab_symmetric", "main_cpp", "dense1", "dense2", "dense3", "dense_12_40"])
def test_reference_simplex_vs_enumeration(oracle, case):
    if case in TINY:
        A, b, c, mx = TINY[case]()
        basis, n_orig = [3, 4], 3
        res, _ = oracle.solve(A, b, c, mx)
    elif case == "dense_12_40":
        A, b, c, mx = lpgen.dense_lp(12, 40, 1)
        basis, n_orig = list(range(12)), 40
        g = json.load(open(os.path.join(ROOT, "tests", "golden", "dense_12_40_seed1.json")))
        x_enum = np.zeros(40)
        st, xo, zo = oracle.eval_basis(A, b, c, mx, g["basis"])
        x_enum[g["basis"]] = xo
        assert close(R.simplex_solve(A, b, c, basis, minimize=not mx, n_orig=n_orig), x_enum)
        return
    else:
        A, b, c, mx = lpgen.dense_lp(8, 24, int(case[-1]))
        basis, n_orig = list(range(8)), 24
        res, _ = oracle.solve(A, b, c, mx, n_threads=4)
    m = A.shape[0]
    x_enum = np.zeros(A.shape[1])
    x_enum[list(res.basis)[:m]] = list(res.x_B)[:m]
    x = R.simplex_solve(A, b, c, basis, minimize=not mx, n_orig=n_orig)
    assert close(x, x_enum[:n_orig])


# ---- GPU: libenumgpu vs the reference's code ----------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(TINY) + ["dense_4_12", "dense_6_16", "dense_8_24"])
def test_gpu_enumeration_vs_reference_code(gpu_lib, case):
    """north star: 'identical optimal basis index set, identical feasible-vertex counts, objective and x within
    1e-9 relative' — libenumgpu against the enumeration composed from the reference's own primitives."""
    if case in TINY:
        A, b, c, mx = TINY[case]()
        want = GOLD["enumeration"][f"tiny/{case}"]
    else:
        m, n = (int(v) for v in case.split("_")[1:])
        A, b, c, mx = lpgen.dense_lp(m, n, 1)
        want = GOLD["enumeration"][f"dense/{m}_{n}_1"]
    m = A.shape[0]
    ref = R.enumerate_bases(A, b, c, mx)[0] if LIVE else None
    for algo in ((sm._abi.ALGO_INDEPENDENT, sm._abi.ALGO_SHARED) if m >= 6 else (sm._abi.ALGO_INDEPENDENT,)):
        s = sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(m)), minimize=not mx), algo=algo)
        s.solve()
        assert s.optimalBasis() == want["basis"] and s.bestRank() == want["best_rank"]
        assert [s.basesEvaluated(), s.singularCount(), s.infeasibleCount(), s.feasibleCount()] == [want["n_bases"]] + want["counts"]
        if ref is not None:
            assert s.optimalBasis() == list(ref.basis)[:m] and s.bestRank() == ref.best_rank
            assert (s.basesEvaluated(), s.singularCount(), s.infeasibleCount(), s.feasibleCount()) == \
                   (ref.n_bases, ref.n_singular, ref.n_infeasible, ref.n_feasible)
            assert close(s.objective(), ref.objective) and close(s.basicValues(), list(ref.x_B)[:m])


@live_only
@pytest.mark.gpu
def test_gpu_vs_reference_simplex_headline(gpu_lib):
    """m=12, n=40: the GPU enumeration optimum is the vertex the reference's simplex Solver walks to."""
    A, b, c, mx = lpgen.dense_lp(12, 40, 1)
    s = sm.EnumerationSolver(sm.Canonical(A, b, c, list(range(12)), minimize=not mx))
    x_gpu = s.solve()
    assert close(R.simplex_solve(A, b, c, list(range(12)), minimize=not mx), x_gpu)


@live_only
@pytest.mark.gpu
def test_dropin_with_the_reference_types(gpu_lib, tmp_path):
    """INTEGRATION.md §1 for real (oracle/dropin_demo.cpp): our EnumerationSolver.h in place of the reference's
    stub, compiled with the reference's own Canonical / Symmetrical / parser / Solver; the reference user's flow
    ParseFromFile -> ToCanonical -> Solver.solve() and EnumerationSolver.solve() gives the same vertex."""
    assert os.path.exists(R.DROPIN), "oracle/_ref/dropin_demo was not built (make -C oracle dropin)"
    rng = np.random.default_rng(5)
    A = rng.integers(1, 10, size=(6, 10))
    text = "maximize\nobjective:\n" + " ".join(str(v) for v in rng.integers(1, 10, size=10)) + "\nconstraints:\n" + \
           "\n".join(" ".join(str(v) for v in row) + f" {int(rng.integers(20, 60))}" for row in A) + "\n"
    big = tmp_path / "sym_6_10.txt"
    big.write_text(text)
    for path, want in ((os.path.join(ROOT, "tests", "golden", "lab_lp_symmetric.txt"), [5.0, 0.0, 0.0]), (str(big), None)):
        out = subprocess.run([R.DROPIN, path], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        facts = {l.split()[0]: [float(v) for v in l.split()[1:]] for l in out.stdout.splitlines()}
        assert close(facts["simplex_x"], facts["enumeration_x"])
        if want:
            assert facts["enumeration_x"] == want and facts["objective"] == [35.0]
        else:
            sym = SymmetricalParser().ParseFromString(text)
            assert close(sym.Evaluate(facts["enumeration_x"]), facts["objective"][0]) and facts["counts"][0] == 8008
