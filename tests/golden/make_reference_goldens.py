"""Writes tests/golden/reference_outputs.json: what the original SimplexMethod code returns for the inputs of
tests/test_reference_code.py, for every quantity that module compares EXACTLY — the results of the conversions,
the parser's results on the fixed texts and on 150 seeded soups, the Print() text, and for each composed
enumeration the class of every basis (as a SHA-256 of the status bytes), the counters, the status and, where the
winner is unique, the best rank and optimal basis.

    python tests/golden/make_reference_goldens.py

Where the values come from.  The original's sources are not part of this repository, so they are recorded from
this project's own code — the Python problem types and parser, the C++ parser of cpp/tests/host_tests, the CPU
oracle — which is unchanged since commit 22d0033.  At that commit tests/test_reference_code.py ran in full against
the original's code (oracle/_ref, built from its sources) and passed, and it asserted each of these quantities
EQUAL to the original's: so they are the original's values for these inputs.  Quantities that module compared
only within 1e-9 (x, z, simplex solutions) and the winners of tied degenerate LPs differ in the last bits between
the two codes and are not recorded; the tests that need them compare live only.  Wherever the original is
available (SIMPLEX_REFERENCE), tests/test_reference_code.py compares with it live as well, which checks this file.
"""
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
OUT = os.path.join(HERE, "reference_outputs.json")
if not os.path.exists(OUT):                  # the test module reads the file when imported
    with open(OUT, "w") as f:
        f.write("{}\n")

import test_reference_code as T  # noqa: E402
from oracle import enumcpu  # noqa: E402
from simplexmethod_b200 import SymmetricalParser, lpgen  # noqa: E402


def main():
    out = {"conversions": {}, "enumeration": {}}
    for seed in range(10):
        out["conversions"][str(seed)] = {label: T.problem_dict(mine) for label, *_, mine in T.conversion_cases(seed)}
    out["constructor_errors"] = {"n_orig_out_of_range": "rejected", "basis_index_out_of_range": "rejected"}
    parsed = [SymmetricalParser().ParseFromString(t) for t in T.PARSER_TEXTS]
    out["parser"] = [None if p is None else T.problem_dict(p) for p in parsed]
    out["print"] = [mine.PrintText() for *_, mine in T.print_fixture()]

    subprocess.check_call(["make", "-C", T.CPP, "-s"])
    with tempfile.TemporaryDirectory() as tmp:
        files = []
        for k, text in enumerate(T.fuzz_texts()):
            files.append(os.path.join(tmp, f"lp{k}.txt"))
            with open(files[-1], "w") as f:
                f.write(text)
        lines = subprocess.check_output([os.path.join(T.CPP, "build", "host_tests"), "--parse"] + files, text=True)
    out["parser_fuzz"] = [T.parse_line(line) for line in lines.splitlines()]

    def record(key, A, b, c, mx, winner=True, **opt):
        res, st = enumcpu.solve(A, b, c, mx, n_threads=os.cpu_count(), want_status=True, **opt)
        out["enumeration"][key] = T.enumeration_record(res, st, A.shape[0], winner)

    for name, fn in T.TINY.items():
        record(f"tiny/{name}", *fn())
    for m, n, seed in T.DENSE:
        record(f"dense/{m}_{n}_{seed}", *lpgen.dense_lp(m, n, seed))
    for seed in range(24):
        record(f"degenerate/{seed}", *T.small_degenerate_lp(seed), winner=False)
    for lo, hi in T.HEADLINE_WINDOWS:
        record(f"headline/{lo}_{hi}", *lpgen.dense_lp(12, 40, 1), rank_begin=lo, rank_end=hi)
    with open(os.path.join(HERE, "dense_12_40_seed1.json")) as f:
        ranks = json.load(f)["singular_ranks"]
    out["headline_singular_ranks"] = {"ranks": ranks, "class": "infeasible", "counts": [0, 1]}

    with open(OUT, "w") as f:
        json.dump(out, f, indent=0)
        f.write("\n")
    print("wrote", OUT)


if __name__ == "__main__":
    main()
