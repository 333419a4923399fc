"""Primal simplex measurement (not a pytest test): one JSON line per case; with --out FILE the lines
are also written there as one JSON list.
  c5     C5 transportation 5 050 x 250 000: primal vs dual from the all-slack basis
  c4     C4 staircase 20 000 x 20 000: primal vs dual from the all-slack basis
  c5hot  C5 after a 1 % cost change: hot primal (hotStart=1, from the previous optimum) vs cold dual
Wall time to the end of the solve, iterations and iterations per second of the solve loop, at default
settings (no scaling, no perturbation).  Every line carries the GPU name and its power limit.
  python tests/primal_probe.py [c5] [c4] [c5hot] [maximumSeconds=...] [--out FILE]"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, ".")
import numpy as np

import clp_b200
from clp_b200 import generators as G

args = sys.argv[1:]
out_file = None
if "--out" in args:
    i = args.index("--out")
    out_file = args[i + 1]
    del args[i:i + 2]
extra = {a.split("=")[0]: float(a.split("=")[1]) for a in args if "=" in a}
which = [a for a in args if "=" not in a] or ["c5", "c5hot", "c4"]
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()[0]


def solve(lp, algorithm, model=None, **params):
    s = model or clp_b200.ClpSimplex()
    if model is None:
        s.loadLP(lp)
    params = dict({"maximumSeconds": 240}, **params, **extra)
    for k, v in params.items():
        s.setParameter(k, v)
    t = time.time()
    st = getattr(s, algorithm)()
    el = time.time() - t
    return s, {"algorithm": algorithm, "params": params, "status": st, "objective": s.objectiveValue(),
               "iterations": s.numberIterations(), "refactorizations": s.numberRefactorizations(),
               "seconds": round(el, 3), "seconds_in_loop": round(s.secondsInLoop(), 3),
               "iterations_per_sec": round(s.numberIterations() / max(1e-9, s.secondsInLoop()), 1),
               "hot": s.lastSolveWasHot()}


def emit(case, lp, r, out):
    r = dict({"case": case, "gpu": gpu, "m": lp.m, "n": lp.n, "nnz": lp.nnz}, **r)
    print(json.dumps(r), flush=True)
    out.append(r)


out = []
for w in which:
    if w in ("c5", "c4"):
        case, lp = (("C5 transport-50x5000", G.transportation_lp(50, 5000, 20260926)) if w == "c5" else
                    ("C4 staircase-20000", G.staircase_lp(40, 500, 20260925)))
        for algorithm in ("primal", "dual"):
            emit(case, lp, solve(lp, algorithm)[1], out)
    elif w == "c5hot":
        case, lp = "C5 transport-50x5000, 1% cost change", G.transportation_lp(50, 5000, 20260926)
        s, r0 = solve(lp, "dual")
        assert r0["status"] == 0, r0
        c = lp.objective * (1.0 + 0.01 * np.random.default_rng(1).choice([-1.0, 1.0], lp.n))
        s.chgObjCoefficients(c)
        _, r = solve(lp, "primal", model=s, hotStart=1)
        emit(case, lp, r, out)
        changed = G.LP("changed", lp.m, lp.n, lp.col_start, lp.row_index, lp.element, lp.col_lower, lp.col_upper,
                       c, lp.row_lower, lp.row_upper)
        _, rc = solve(changed, "dual")
        rc["rel_diff_to_hot"] = abs(rc["objective"] - r["objective"]) / (1 + abs(rc["objective"]))
        emit(case, lp, rc, out)
if out_file:
    os.makedirs(os.path.dirname(os.path.abspath(out_file)), exist_ok=True)
    json.dump(out, open(out_file, "w"), indent=1)
