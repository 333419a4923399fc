import os, sys, time, json
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE))); sys.path.insert(0, HERE)
import numpy as np
from clp_b200 import generators as G
from make_golden import highs_objective
res = {}
for name, lp in (("C5 transport-50x5000", G.transportation_lp(50, 5000, 20260926)), ("C4 staircase-20000", G.staircase_lp(40, 500, 20260925))):
    t = time.time()
    st, obj = highs_objective(lp)
    res[name] = {"status": st, "objective": obj, "seconds": time.time() - t, "m": lp.m, "n": lp.n, "nnz": lp.nnz}
    print(name, res[name], flush=True)
json.dump(res, open(os.path.join(HERE, 'fullsize_highs.json'), 'w'))
