"""Primal simplex on the device (-m gpu): ClpSimplex::primal with Devex / Dantzig pricing, the
re-solve after a cost change, and its two hot kernels against numpy restatements written here."""
import json
import os

import numpy as np
import pytest

from conftest import ROOT, load_golden

import clp_b200
from clp_b200 import generators as G
from oracle import oracle as O

pytestmark = pytest.mark.gpu

MANIFEST = json.load(open(os.path.join(ROOT, "tests", "golden", "manifest.json")))
ALL = sorted(MANIFEST)
INF = 1e30


def engine(lp, **params):
    s = clp_b200.ClpSimplex()
    s.loadLP(lp)
    params.setdefault("maximumSeconds", 300)  # a stalled solve fails the test instead of hanging the suite
    for k, v in params.items():
        s.setParameter(k, v)
    return s


def kkt(lp, s):
    return O.kkt_violations(lp, s.primalColumnSolution(), s.primalRowSolution(), s.dualColumnSolution())


def close(a, b, tol=1e-8):
    return abs(a - b) <= tol * (1 + abs(b))


# ------------------------------------------------------------------ whole solves
@pytest.mark.parametrize("name", ALL)
def test_golden_fixture_primal(name):
    lp = load_golden(name)
    s = engine(lp)
    st = s.primal()
    assert st == lp.expect_status, (name, st, s.numberIterations())
    if st == 0:
        tol = 1e-4 if MANIFEST[name]["objective_source"] == "reference" else 1e-8
        assert close(s.objectiveValue(), lp.known_objective, tol)
        assert close(s.objectiveValue(), MANIFEST[name]["oracle_objective"])
        assert kkt(lp, s) == 0
        assert int((s.statusArray() == 1).sum()) == lp.m


@pytest.mark.parametrize("pivot", [0, 1])
@pytest.mark.parametrize("shape", [(300, 3000, 0.02, 7), (1000, 10000, 0.01, 20260923)])
def test_planted_random_lp_primal(shape, pivot):
    m, n, dens, seed = shape
    lp = G.random_sparse_lp(m, n, dens, seed)
    s = engine(lp, primalColumnPivot=pivot)
    assert s.primal() == 0
    assert close(s.objectiveValue(), lp.known_objective)
    assert kkt(lp, s) == 0
    d = engine(lp)
    assert d.dual() == 0
    assert close(s.objectiveValue(), d.objectiveValue())


@pytest.mark.parametrize("mode", [1, 2, 3])
@pytest.mark.parametrize("name", ["TSP-MTZ-40", "UFL-30x100", "modified_afiro", "staircase-480", "SetCover-50x200",
                                  "NQueens-20", "hello"])
def test_scaled_primal_matches_unscaled(name, mode):
    lp = load_golden(name)
    s = engine(lp)
    s.scaling(mode)
    assert s.primal() == 0
    assert close(s.objectiveValue(), lp.known_objective, 1e-7)
    assert close(s.objectiveValue(), MANIFEST[name]["oracle_objective"], 1e-7)
    assert kkt(lp, s) == 0
    assert int((s.statusArray() == 1).sum()) == lp.m


@pytest.mark.parametrize("name", ["TSP-MTZ-40", "staircase-480"])
def test_primal_is_deterministic_across_batch_and_graph(name):
    lp = load_golden(name)
    runs = []
    for params in ({"batch": 1}, {"batch": 7}, {"batch": 32}, {"useGraph": 0}):
        s = engine(lp, **params)
        assert s.primal() == 0
        runs.append((s.numberIterations(), s.objectiveValue()))
    assert all(r == runs[0] for r in runs), runs


def test_reoptimize_after_cost_change_is_hot():
    lp = G.random_sparse_lp(300, 3000, 0.02, 7)
    s = engine(lp)
    assert s.dual() == 0
    rng = np.random.default_rng(11)
    c = lp.objective * (1.0 + rng.uniform(0.01, 0.05, lp.n) * rng.choice([-1.0, 1.0], lp.n))
    s.chgObjCoefficients(c)
    s.setParameter("hotStart", 1)
    assert s.primal() == 0
    assert s.lastSolveWasHot()
    hot_iterations = s.numberIterations()
    changed = G.LP("changed", lp.m, lp.n, lp.col_start, lp.row_index, lp.element, lp.col_lower, lp.col_upper,
                   c, lp.row_lower, lp.row_upper)
    assert kkt(changed, s) == 0
    cold_dual = engine(changed)
    assert cold_dual.dual() == 0
    assert close(s.objectiveValue(), cold_dual.objectiveValue())
    cold_primal = engine(changed)
    assert cold_primal.primal() == 0
    assert hot_iterations < cold_primal.numberIterations(), (hot_iterations, cold_primal.numberIterations())


def test_warm_start_from_optimal_basis():
    lp = load_golden("TSP-MTZ-40")
    d = engine(lp)
    assert d.dual() == 0
    s = engine(lp)
    s.copyinStatus(d.statusArray())
    assert s.primal() == 0
    assert s.numberIterations() <= 2
    assert close(s.objectiveValue(), d.objectiveValue())


@pytest.mark.parametrize("name,objective", [("afiro", -4.6475314286e+02), ("modified_afiro", None)])
def test_initial_primal_solve(name, objective):
    lp = load_golden(name)
    s = engine(lp)
    assert s.initialPrimalSolve() == 0
    target = objective if objective is not None else lp.known_objective
    assert close(s.objectiveValue(), target)


def test_stops_on_iteration_limit_with_consistent_rows():
    lp = load_golden("TSP-MTZ-40")
    s = engine(lp, maximumIterations=5)
    assert s.primal() == 3
    x, y = s.primalColumnSolution(), s.primalRowSolution()
    ax = lp.to_scipy() @ x
    assert np.abs(ax - y).max() <= 1e-7 * (1 + np.abs(ax).max())


def test_transportation_c5_shape_primal():
    """C5's shape (5 050 x 250 000, fully degenerate) from the slack basis, certified by the duality gap."""
    from test_fullsize import duality_gap

    lp = G.transportation_lp(50, 5000, 0)
    s = engine(lp, maximumSeconds=400)
    assert s.primal() == 0, (s.status(), s.numberIterations())
    print(f"C5 shape: {s.numberIterations()} iterations, {s.secondsInLoop():.2f} s")
    primal, dual, bad = duality_gap(lp, s.primalColumnSolution(), s.dualRowSolution(), s.dualColumnSolution())
    assert bad <= 1e-7
    assert abs(primal - dual) <= 1e-8 * (1 + abs(primal))
    assert close(s.objectiveValue(), primal)


# ------------------------------------------------------------------ hot kernels on explicit vectors
def _key_bits(v):
    return np.asarray(v, dtype=np.float64).view(np.uint64) & np.uint64(~0xFFFFF & 0xFFFFFFFFFFFFFFFF)


def np_primal_column_pivot(dj, status, weights, mode, tol=1e-7):
    """ClpPrimalColumnPivot::pivotColumn restated: the largest packed (score, 0xFFFFF - j) key."""
    dj = np.asarray(dj, dtype=np.float64)
    cand = (((status == 3) & (dj < -tol)) | ((status == 2) & (dj > tol)) |
            (((status == 0) | (status == 4)) & (np.abs(dj) > tol)))
    score = dj * dj if mode == 1 else dj * dj / weights
    cand &= score > 0
    if not cand.any():
        return -1
    keys = _key_bits(np.where(cand, score, 0.0)) | (np.uint64(0xFFFFF) - np.arange(len(dj), dtype=np.uint64))
    keys[~cand] = 0
    return int(0xFFFFF - (int(keys.max()) & 0xFFFFF))


def np_primal_row(alpha, x, lo, up, direction, rng_, phase, tol=1e-7, acceptable=1e-7):
    """ClpSimplexPrimal::primalRow restated (Harris two passes): (row | -1 | -2, theta)."""
    def block(a, xv, l, u, relax):
        if a > 0:
            if phase == 1 and xv < l - tol:
                return None
            to_upper = phase == 1 and xv > u + tol and l <= -INF
            b = u if to_upper else l
            if b <= -INF:
                return None
            r = (xv - b + relax) / a
        else:
            if phase == 1 and xv > u + tol:
                return None
            to_upper = not (phase == 1 and xv < l - tol and u >= INF)
            b = u if to_upper else l
            if b >= INF:
                return None
            r = (b - xv + relax) / -a
        return r if r > 0 else 0.0

    m = len(alpha)
    theta_max = np.inf
    for p in range(m):
        a = direction * alpha[p]
        if abs(a) >= acceptable:
            r = block(a, x[p], lo[p], up[p], tol)
            if r is not None:
                theta_max = min(theta_max, r)
    best = 0
    for p in range(m):
        a = direction * alpha[p]
        if abs(a) >= acceptable:
            r = block(a, x[p], lo[p], up[p], 0.0)
            if r is not None and r <= theta_max:
                key = int(_key_bits([abs(alpha[p])])[0]) | (0xFFFFF - p)
                best = max(best, key)
    if rng_ < 1e29 and rng_ <= theta_max:
        return -2, rng_
    if best == 0:
        return -1, None
    r = 0xFFFFF - (best & 0xFFFFF)
    return r, block(direction * alpha[r], x[r], lo[r], up[r], 0.0)


@pytest.fixture(scope="module")
def plugin_model():
    lp = G.random_sparse_lp(64, 200, 0.05, 3)
    return engine(lp), lp


def test_primal_column_pivot_matches_restatement(plugin_model):
    s, lp = plugin_model
    nm = lp.n + lp.m
    rng = np.random.default_rng(5)
    for trial in range(20):
        dj = rng.standard_normal(nm) * (10.0 ** rng.uniform(-9, 1, nm))
        status = rng.choice(np.array([0, 1, 2, 3, 4, 5], np.uint8), nm, p=[0.05, 0.2, 0.25, 0.4, 0.05, 0.05])
        weights = 10.0 ** rng.uniform(-1, 2, nm)
        if trial % 4 == 0:  # ties: equal scores at several sequences -> the smallest sequence
            idx = rng.choice(nm, 6, replace=False)
            dj[idx] = -3.0
            status[idx] = 3
            weights[idx] = 2.0
        for mode in (0, 1):
            assert s.primalColumnPivot(dj, status, weights, mode) == np_primal_column_pivot(dj, status, weights, mode), \
                (trial, mode)
    # nothing attractive
    assert s.primalColumnPivot(np.zeros(nm), np.full(nm, 3, np.uint8), np.ones(nm), 0) == -1


def _check_row(s, m, alpha, x, lo, up, direction, rng_, phase):
    got, theta = s.primalRow(alpha, x, lo, up, direction, rng_, phase)
    want, wtheta = np_primal_row(alpha, x, lo, up, direction, rng_, phase)
    assert got == want, (got, want)
    if wtheta is not None:
        assert abs(theta - wtheta) <= 1e-15 * (1 + abs(wtheta)), (theta, wtheta)
    return got


def test_primal_row_matches_restatement(plugin_model):
    s, lp = plugin_model
    m = lp.m
    rng = np.random.default_rng(9)
    for trial in range(30):
        alpha = rng.standard_normal(m) * (rng.random(m) < 0.5)
        lo = np.where(rng.random(m) < 0.8, rng.uniform(-5, 0, m), -INF)
        up = np.where(rng.random(m) < 0.8, rng.uniform(0, 5, m), INF)
        x = np.clip(rng.uniform(-6, 6, m), np.maximum(lo, -6), np.minimum(up, 6))
        phase = 2
        if trial % 3 == 0:  # phase 1: some basics outside their bounds
            phase = 1
            out = rng.random(m) < 0.3
            x = np.where(out, rng.uniform(-8, 8, m), x)
        direction = 1 if trial % 2 else -1
        rng_ = [INF, 0.5, 1e-3][trial % 3]
        _check_row(s, m, alpha, x, lo, up, direction, rng_, phase)


def test_primal_row_adversarial(plugin_model):
    s, lp = plugin_model
    m = lp.m
    lo, up, x = np.zeros(m), np.full(m, INF), np.ones(m)
    # ties: equal |alpha| and equal ratios -> the smaller row
    alpha = np.zeros(m)
    alpha[[7, 3, 40]] = 2.0
    assert _check_row(s, m, alpha, x, lo, up, 1, INF, 2) == 3
    # |alpha| just below acceptablePivot is ignored although its ratio would be the smallest
    alpha2 = alpha.copy()
    alpha2[1] = 0.999e-7
    x2 = 10.0 * x
    x2[1] = 0.0
    assert _check_row(s, m, alpha2, x2, lo, up, 1, INF, 2) == 3
    # the entering range is the smallest step: bound flip
    assert _check_row(s, m, alpha, x, lo, up, 1, 0.25, 2) == -2
    # nothing blocks and no range: unbounded ray
    assert _check_row(s, m, -alpha, x, lo, up, 1, INF, 2) == -1
    # phase 1: a basic below its lower bound passes it and blocks at its upper bound only
    lo1, up1 = np.zeros(m), np.full(m, 10.0)
    x1 = np.full(m, 5.0)
    x1[3] = -4.0
    a1 = np.zeros(m)
    a1[3] = -1.0   # x_3 increases with the entering variable: reaches 10 after a step of 14
    a1[9] = 0.25   # x_9 decreases: reaches 0 after a step of 20
    assert _check_row(s, m, a1, x1, lo1, up1, 1, INF, 1) == 3
    # a basic infeasible within the tolerance that moves further out: its negative step clamps to 0
    x1[9] = -1e-8
    got, theta = s.primalRow(a1, x1, lo1, up1, 1, INF, 2)
    assert got == 9 and theta == 0.0
