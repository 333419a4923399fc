"""Freeze the reference's known-answer LPs into fixtures.

Sources (files of coin-or/Clp):
  * test/test_racing_lp.cpp generators (glibc srand/rand, restated in clp_b200/generators.py) +
    test/test_racing_reference.txt expected LP bounds -> <name>.npz with known_objective
  * src/unitTest.cpp:1415-1431 3x5 LP -> unitTest-3x5.npz
  * examples/modified_afiro.mps, examples/hello.mps (copied verbatim next to this script) parsed
    with THIS repo's MPS reader ->
    .npz (no reference value is printed for them; the expected objective stored is the
    independent HiGHS dual simplex optimum, see SURVEY.md 8c item 3)
Every fixture without a reference-published objective gets `known_objective` from HiGHS
(scipy.optimize.linprog method='highs-ds') and is cross-checked against the CPU oracle.
Usage:  python tests/golden/make_golden.py
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from clp_b200 import generators as G  # noqa: E402


def highs_objective(lp):
    import scipy.sparse as sp
    from scipy.optimize import linprog

    A = lp.to_scipy().tocsr()
    inf = 1e29
    rl, ru = lp.row_lower, lp.row_upper
    eq = rl == ru
    up = (~eq) & (ru < inf)
    lo = (~eq) & (rl > -inf)
    Aub = sp.vstack([A[up], -A[lo]]) if (up.any() or lo.any()) else None
    bub = np.concatenate([ru[up], -rl[lo]])
    Aeq = A[eq] if eq.any() else None
    bounds = [(l if l > -inf else None, u if u < inf else None)
              for l, u in zip(lp.col_lower, lp.col_upper)]
    r = linprog(lp.objective, A_ub=Aub, b_ub=bub if Aub is not None else None, A_eq=Aeq,
                b_eq=rl[eq] if Aeq is not None else None, bounds=bounds, method="highs-ds")
    return r.status, (float(r.fun) if r.status == 0 else None)


def main():
    from oracle.oracle import OracleSimplex

    cases = [G.unit_test_3x5()] + G.racing_suite()
    # reduced shapes of BASELINE.json configs[3] (staircase) and configs[4] (degenerate transportation);
    # no reference value exists for them: pinned by HiGHS dual simplex, cross-checked by the oracle
    cases += [G.staircase_lp(8, 60, 3), G.staircase_lp(10, 100, 4), G.transportation_lp(10, 200, 5),
              G.transportation_lp(20, 500, 6)]
    # the reference's example MPS files (kept here verbatim) through our own reader (host-only code
    # path, no GPU needed)
    import clp_b200

    for fn in ("modified_afiro.mps", "hello.mps"):
        s = clp_b200.ClpSimplex()
        assert s.readMps(os.path.join(HERE, fn)) == 0
        lp = s.getProblem()
        lp.name = fn.replace(".mps", "")
        cases.append(lp)
    manifest = {}
    for lp in cases:
        src = "reference"
        if lp.known_objective is None and lp.expect_status == 0:
            st, obj = highs_objective(lp)
            assert st == 0, (lp.name, st)
            lp.known_objective = obj
            src = "highs-ds"
        o = OracleSimplex(lp)
        st = o.dual()
        assert st == lp.expect_status, (lp.name, st)
        if st == 0:
            tol = 1e-4 if src == "reference" else 1e-7
            assert abs(o.objective_value - lp.known_objective) <= tol * (1 + abs(lp.known_objective)), \
                (lp.name, o.objective_value, lp.known_objective)
        lp.save(os.path.join(HERE, lp.name + ".npz"))
        manifest[lp.name] = {"m": lp.m, "n": lp.n, "nnz": lp.nnz, "expect_status": lp.expect_status,
                             "known_objective": lp.known_objective, "objective_source": src,
                             "oracle_objective": o.objective_value if st == 0 else None,
                             "oracle_iterations": o.iterations}
        print(lp.name, manifest[lp.name])
    with open(os.path.join(HERE, "manifest.json"), "w") as f:
        json.dump(manifest, f, indent=1, sort_keys=True)


if __name__ == "__main__":
    main()
